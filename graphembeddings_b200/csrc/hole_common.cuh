// Shared declarations for libhole_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>

#include "../../include/hole_b200.h"

// ---------------------------------------------------------------------------------------
// error handling + launch accounting
// ---------------------------------------------------------------------------------------
extern thread_local std::string g_hole_err;
extern thread_local int64_t g_hole_launches;

int hole_set_error(int code, const char* fmt, ...);

#define HOLE_CUDA_TRY(expr)                                                              \
  do {                                                                                   \
    cudaError_t _e = (expr);                                                             \
    if (_e != cudaSuccess)                                                               \
      return hole_set_error(HOLE_ERR_CUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #expr,  \
                            cudaGetErrorString(_e));                                     \
  } while (0)

#define HOLE_CHECK_ARG(cond)                                                             \
  do {                                                                                   \
    if (!(cond)) return hole_set_error(HOLE_ERR_ARG, "%s: bad argument: %s", __func__, #cond); \
  } while (0)

// Count a kernel launch and surface launch-configuration errors immediately.
#define HOLE_LAUNCHED()                                                                  \
  do {                                                                                   \
    ++g_hole_launches;                                                                   \
    HOLE_CUDA_TRY(cudaGetLastError());                                                   \
  } while (0)

// ---------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------
struct hole_rank_ws;       // hole_rank.cu
struct hole_shard_state;   // hole_shard.cuh

// Update plan of a chunk of S steps (integer-only; built ahead of the steps that use it).
struct hole_plan {
  uint32_t* keysA = nullptr;     // [S][4B] the step's row keys by position (kept: --log_loss reads them)
  uint32_t* keysB = nullptr;     // [S][4B] keys of the duplicated uses, compacted: sort ping
  uint32_t* keysC = nullptr;     // [S][4B] sort pong
  uint32_t* seen = nullptr;      // [S][n_rows/32] bitmap: row used by the step
  uint32_t* dup = nullptr;       // [S][n_rows/32] bitmap: row used more than once (second half of `seen`'s allocation)
  size_t bitmap_words = 0;
  unsigned* done = nullptr;      // [S] "last tile block of the step" tickets of the sort (zero between uses)
  int* blkcnt = nullptr;         // [S][tiles+1] duplicated uses per tile -> offsets; total last
  int* mdup = nullptr;           // [S] duplicated uses of the step
  uint32_t* valsA = nullptr;
  uint32_t* valsB = nullptr;
  uint32_t* ghist = nullptr;     // [S][256][tiles] radix histograms
  uint32_t* skey = nullptr;      // sorted keys of the duplicated uses (points into keysB or keysC)
  uint32_t* spos = nullptr;      // sorted original positions (points into valsA or valsB)
  uint32_t* gslot = nullptr;     // [S][4B] per ORIGINAL position: G row of that use, or UNIQUE
  uint4* heads = nullptr;        // [S][heads_cap] leaves of the combine trees {j, seg start, n, row}
  int* nheads = nullptr;         // [S]
  int32_t* neg = nullptr;        // [S*B] corrupt entity per triple
  int32_t* perm = nullptr;       // [S*B] triples grouped by relation (K1's processing order)
  int heads_cap = 0;
  int T = 1;                     // triples per K1 lane group
  cudaEvent_t ready = nullptr;     // recorded by the builder when the plan is complete
  cudaEvent_t released = nullptr;  // recorded by the consumer when it no longer needs the plan
  bool used = false;
  // hole_train_step_plan: plan built ahead for exactly these buffers
  const int32_t* prepared_pos = nullptr;
  const int32_t* prepared_neg = nullptr;
  int64_t prepared_B = -1;
};

struct hole_ctx {
  int device = 0;
  int64_t n_rows = 0;
  int dim = 0;         // embedding_dim (even)
  int H = 0;           // dim / 2
  int nvec = 0;        // float4s per (padded) half = round_up(H, 4) / 4
  int row_stride = 0;  // floats per device row = 8 * nvec
  int gs = 0, v = 0;   // lanes per row and float4s per lane per half (kernel variant)
  int sm_count = 0;
  int key_bits = 0;    // bits needed for a row id
  bool k1_ready = false;   // kernel attributes set (lazily, on the first training call)
  int k1v2_smem = 0;   // dynamic shared memory of hole_k1_kernel
  int k1_groups = 0;   // lane groups resident on the whole GPU (sizes T, the triples per group)
  int ramp_first = 0;  // hole_train_steps: steps in the first planned chunk, then x ramp_factor; 0 = no ramp
  int host_first = 0;  // hole_train_steps_host: steps in a short first chunk; 0 = off (measured slower: r02_e2e_ab.jsonl)
  int ramp_factor = 4; //   (HOLE_PLAN_RAMP=first,factor; measured slower than no ramp, profiles/r02_train_ab.txt:
                       //   a plan's latency is ~120 us of dependent launches whatever its size)
  int score_mode = 0;  // HOLE_SCORE_COMPLEX (live holE.py) or HOLE_SCORE_CCORR_TANH (archived variant, hole_ccorr.cuh)
  bool cc_ready = false;   // shared-memory attributes of the ccorr kernels set
  int optimizer = 0;   // HOLE_OPT_SGD or HOLE_OPT_ADAGRAD (hole_ctx_set_optimizer)
  float* accum = nullptr;  // AdaGrad accumulator [n_rows, row_stride] (caller-owned, kept by reference)
  int sort_small = 1;          // plan: one-launch sort + segments while the steps seen so far were small enough
                               //   (HOLE_SORT_SMALL: 0 never, 1 adaptive, 2 always -- tests of its large-step path)
  int64_t dup_seen_B = -1;     //   batch size the observation below belongs to
  int dup_seen_max = -1;       //   largest duplicated-use count of a step in the last plan of either slot (-1: none yet)
  int* dup_max_host = nullptr;     //   mapped pinned int[2] the plans report into, one word per plan slot (host view)
  int* dup_max_host_dev = nullptr; //   ... its device address
  int row_passes = 1;  // 8-bit radix passes for row keys
  int rel_passes = 1;  // ... for relation ids (hole_ctx_set_relations)
  int64_t n_rel_hint = int64_t(1) << 40;   // relation ids are < this (hole_ctx_set_relations); default: no promise

  // ---- training workspace (grown on demand; owned by the context)
  int64_t cap_B = 0, cap_S = 0;
  float* G = nullptr;            // [4B, row_stride] staged gradient rows of ONE step
  int* counters = nullptr;       // [LEVELS][4B] tree-combine tickets (self-resetting)
  float* loss = nullptr;         // [S*B] scratch when the caller passes no loss_out
  float* loss_sum = nullptr;     // [S]
  hole_plan plan[2];             // double-buffered: chunk c+1 is planned while chunk c trains
  cudaStream_t plan_stream = nullptr;
  cudaEvent_t ev_entry = nullptr;
  int32_t* triples_stage[2] = {nullptr, nullptr};  // device staging for the host-buffer path
  int64_t cap_stage = 0;
  float* loss_sum_pinned = nullptr;   // pinned host mirror of loss sums (e2e path)
  int64_t cap_pinned = 0;
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_copy[2] = {nullptr, nullptr};

  int plan_toggle = 0;                 // slot the next hole_train_step_plan call uses
  hole_rank_ws* rank = nullptr;
  hole_shard_state* shard_state = nullptr;   // row-sharded step (hole_shard_init)
  // multi-GPU step routing (hole_shard_route): sort scratch for 3B entity keys
  uint32_t* route_buf = nullptr;
  unsigned* route_done = nullptr;
  int64_t route_cap = 0;

  // ---- measurement hooks
  bool profile = false;
  std::vector<cudaEvent_t> prof_ev;   // 3 per measured step
  size_t prof_used = 0;
};

// run_step / K3 `flags`: bits 0-1 = loss mode (0 hinge, 1 / 2 log-loss pass with / without the
// positive term: K1 runs in DM 3, which always adds to the delta table), bit 2 = K3 adds to the
// delta table instead of overwriting it
constexpr int HOLE_K1_ACCUMULATE = 4;
constexpr int HOLE_TREE_C = 32;      // fan-in of the deterministic gradient combine tree
constexpr int HOLE_TREE_LEVELS = 6;  // 32^6 > any 4B

// device addresses of one buffer on every rank (peer memory mapped with CUDA IPC)
struct hole_peer_ptrs { void* p[HOLE_MAX_RANKS]; };

int hole_ws_reserve(hole_ctx* ctx, int64_t B, int64_t S);
void hole_rank_ws_free(hole_ctx* ctx);
void hole_rank_cache_invalidate(hole_ctx* ctx);   // a training call changes the table: drop the packed operand

// ---------------------------------------------------------------------------------------
// Philox4x32-10 (must match oracle/philox.py bit for bit)
// ---------------------------------------------------------------------------------------
#define HOLE_STREAM_SIDE   0x5EED0001u
#define HOLE_STREAM_ENTITY 0x5EED0002u

__host__ __device__ inline void hole_philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint64_t p0 = (uint64_t)M0 * c[0];
    uint64_t p1 = (uint64_t)M1 * c[2];
    uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0;
    uint32_t hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
    uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
    c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
    k0 += W0; k1 += W1;
  }
}

__host__ __device__ inline int hole_side_coin(uint64_t seed, uint64_t step) {
  uint32_t c[4] = {(uint32_t)step, (uint32_t)(step >> 32), 0u, HOLE_STREAM_SIDE};
  hole_philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
  return (int)(c[0] & 1u);
}

// floor(r64 * cnt / 2^64), cnt < 2^32
__host__ __device__ inline uint32_t hole_mulhi64_u32(uint32_t r_lo, uint32_t r_hi, uint32_t cnt) {
  uint64_t lo = (uint64_t)r_lo * cnt;
  uint64_t hi = (uint64_t)r_hi * cnt;
  return (uint32_t)((hi + (lo >> 32)) >> 32);
}

__host__ __device__ inline uint32_t hole_entity_draw(uint64_t seed, uint64_t step, uint32_t index,
                                                     uint32_t cnt) {
  uint32_t c[4] = {index, (uint32_t)step, (uint32_t)(step >> 32), HOLE_STREAM_ENTITY};
  hole_philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
  return hole_mulhi64_u32(c[0], c[1], cnt);
}
