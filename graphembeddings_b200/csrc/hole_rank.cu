// All-candidate link-prediction ranking for sm_100a: a dense bf16 contraction
// S = Q . C^T on tcgen05 tensor cores (TMEM accumulators, TMA-fed shared-memory operands)
// whose epilogue counts, per query row, the candidates that rank before the true one.
// The Q x N score matrix is never written.
//
// Reference seams: the scoring loop of infer_triples (holE.py:564-573) and the heap of
// eval_link_prediction (holE.py:427-469); GEMM form: SURVEY.md App. A.4, rank rule App. A.5.
//
// Kernel anatomy (one CTA per SM, persistent over work items = (query tile, candidate chunk)):
//   warp 0      TMA producer: query tile once per item, candidate k-blocks through a ring
//   warp 1      MMA issuer (one elected lane): tcgen05.mma cta_group::1, M=128 N=256 K=16,
//               accumulators double-buffered in TMEM (2 x 256 columns)
//   warps 2..9  epilogue: tcgen05.ld 32 columns at a time, compare against the row's
//               threshold, count, and merge-join the row's filter slice with the counted columns;
//               two warps per TMEM lane quarter split the columns
#include <cuda.h>
#include <cuda_bf16.h>

#include <algorithm>
#include <climits>

#include "hole_common.cuh"
#include "hole_ccorr_core.cuh"

namespace {

constexpr int BM = 128;            // query rows per tile (UMMA M)
constexpr int BN = 256;            // candidates per tile (UMMA N)
constexpr int BK = 64;             // bf16 elements per k-block = one 128-byte swizzle row
constexpr int UMMA_K = 16;
constexpr int A_KB_BYTES = BM * BK * 2;   // 16 KB
constexpr int B_KB_BYTES = BN * BK * 2;   // 32 KB
constexpr int EPI_WARPS = 8;       // two warps per TMEM lane quarter, 128 columns each (16 warps x 64
                                   // columns measured 3 % slower on the FB15k shape)
constexpr int RANK_THREADS = 64 + 32 * EPI_WARPS;
// The SM's warp arbiter favours higher warp ids (B300_MICROARCH.md): the two single-lane roles
// that feed the tensor pipe must not be starved by the epilogue warps, so they come last.
constexpr int WARP_TMA = EPI_WARPS, WARP_MMA = EPI_WARPS + 1, WARP_EPI0 = 0;
constexpr int EPI_COLS = 256 / (EPI_WARPS / 4);    // columns of the 256-wide tile one warp owns
constexpr int MAX_STAGES = 4;     // candidate k-block ring slots and their barriers; a fifth 32 KB stage measured no gain
constexpr int SMEM_LIMIT = 227 * 1024;

enum { MODE_COUNT = 0, MODE_DIAG = 1 };
// epilogue of hole_rank_kernel, chosen at compile time: EPI_RANK runs MODE_COUNT / MODE_DIAG, EPI_TOPK keeps
// each thread's k best candidates (hole_topk)
enum { EPI_RANK = 0, EPI_TOPK = 1 };

struct RankParams {
  int mode;
  int num_kb;        // k-blocks of ONE operand part: round_up(D, 64) / 64
  int parts;         // 1 = bf16 operands; 2 = split-bf16: operand columns are [hi | lo] and the
                     //     contraction is hi.hi + lo.hi + hi.lo (HOLE_RANK_BF16X3)
  int last_kb_mmas;  // K=16 slices of the last k-block that hold real columns (the rest is zero padding)
  int stages;        // ring depth for candidate k-blocks
  int m_tiles;       // query tiles
  int n_tiles;       // candidate tiles (COUNT mode)
  int chunk_tiles;   // candidate tiles per work item
  int n_chunks;
  int Q;             // valid queries
  int Nc;            // valid candidates in this shard
  const float* true_score;     // [Q]   COUNT: thresholds
  const int32_t* true_idx;     // [Qpad] shard-local index of the true candidate (may be out of range)
  int32_t* raw_cnt;            // [Q]   COUNT: += count
  int32_t* filt_cnt;           // [Q]   COUNT: += count minus the filtered candidates among it
  float* true_out;             // [Q]   DIAG: score of the true candidate if it lives in this shard
  // top-k epilogue (EPI_TOPK)
  int topk;                    // k
  uint64_t* tk_keys;           // [Qpad][n_chunks][2][k] per-thread candidate lists (binary max-heaps)
  // COUNT and EPI_TOPK
  const int64_t* f_off;        // [Q+1] filter CSR, or null
  const int32_t* f_ids;        //       ids ascending within a query's slice
  int64_t ent_begin;
  const int32_t* tk_self;      // [Qpad] hole_neighbors: shard-local index each query never returns (itself); else null
};

// ------------------------------------------------------------------------------------ PTX
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra WAIT_DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t"
      "}" ::"r"(smem_u32(bar)), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar,
                                            int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)map) : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)),
               "r"(cols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, bf16 in, fp32 accumulate
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on an mbarrier when all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]),
        "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]),
        "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]),
        "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// The same load without the wait: the registers are valid only after tmem_ld_wait(v).
__device__ __forceinline__ void tmem_ld32_async(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]),
        "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]),
        "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]),
        "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
// Waits for every tcgen05.ld of this thread; the registers pass through the statement so that no
// use of them can be scheduled ahead of the wait.
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.wait::ld.sync.aligned;"
      : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]),
        "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]),
        "+r"(v[15]), "+r"(v[16]), "+r"(v[17]), "+r"(v[18]), "+r"(v[19]), "+r"(v[20]), "+r"(v[21]),
        "+r"(v[22]), "+r"(v[23]), "+r"(v[24]), "+r"(v[25]), "+r"(v[26]), "+r"(v[27]), "+r"(v[28]),
        "+r"(v[29]), "+r"(v[30]), "+r"(v[31])
      :
      : "memory");
}

// K-major, 128-byte-swizzled operand tile whose rows are 128 bytes (64 bf16): 8-row groups
// are 1024 bytes apart (SBO); LBO is unused for swizzled K-major layouts (canonical value 1).
// Bits: [0,14) addr>>4, [16,30) LBO>>4, [32,46) SBO>>4, [46,48) version=1, [61,64) layout=2.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  return (uint64_t)((smem_addr >> 4) & 0x3FFFu) | (1ull << 16) | (64ull << 32) | (1ull << 46) |
         (2ull << 61);
}
// kind::f16 instruction descriptor: D=f32 (bit 4), A=B=bf16 (bits 7, 10), both K-major,
// N>>3 at [17,23), M>>4 at [24,29)
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// A thread's place in its query row's filter slice (known-true candidates, holE.py:454-461), whose ids are
// ascending: the thread meets its columns in ascending order, so the slice is merge-joined with them.
struct FilterCursor {
  int64_t fp, f1;            // f_ids[fp .. f1): ids not yet passed
  int next, after;           // shard-local indices of f_ids[fp] and f_ids[fp + 1], INT_MAX past the end; `after`
                             // is loaded one step ahead, so that a step of the cursor does not wait for memory
};

__device__ __forceinline__ int filter_id_at(const int32_t* __restrict__ ids, int64_t i, int64_t f1, int64_t ent_begin) {
  return i < f1 ? (int)((int64_t)ids[i] - ent_begin) : INT_MAX;
}

// First id of f_ids[lo, hi) that is >= id (hi if none).
__device__ __forceinline__ int64_t lower_bound_id(const int32_t* __restrict__ ids, int64_t lo, int64_t hi, int64_t id) {
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if ((int64_t)ids[mid] < id) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// Moves the cursor past every copy of the id it stands on (a repeated id is one candidate).
__device__ __forceinline__ void filter_advance(FilterCursor& f, const int32_t* __restrict__ ids, int64_t ent_begin) {
  const int cur = f.next;
  do {
    ++f.fp;
    f.next = f.after;
    f.after = filter_id_at(ids, f.fp + 1, f.f1, ent_begin);
  } while (f.next <= cur);
}

// Rank-count epilogue of 32 accumulator columns held by one thread (one query row): how many of the
// candidates j0 .. j0+31 rank before the true one (c0), and how many of those are filtered (fc).
// thr_hi = nextafter(thr): s <= thr <=> s < thr_hi; candidates with index < tie win ties (holE.py:427-469
// walks the heap in index order).  A filtered column is subtracted exactly when this very compare counted
// it, so filt_before is exact with respect to raw_before; the true column itself never counts (s == thr,
// j == tie), whether or not it is filtered.
__device__ __forceinline__ void epi_count32(const uint32_t (&v)[32], int j0, float thr, float thr_hi, int tie,
                                            int Nc, int& c0, FilterCursor& f, const int32_t* __restrict__ f_ids,
                                            int64_t ent_begin, int& fc) {
  const bool slow = (j0 < tie && tie < j0 + 32) || (j0 + 32 > Nc) || (f.next < j0 + 32);
  if (!__any_sync(0xffffffffu, slow)) {
    const float tt = (j0 + 32 <= tie) ? thr_hi : thr;
    // (A two-instruction FSETP + predicated-add form on four independent counters measured 2-5 %
    // slower end to end than this select chain: the call is power-bound, see DESIGN.md section 9.)
#pragma unroll
    for (int k = 0; k < 32; ++k) c0 += (__uint_as_float(v[k]) < tt) ? 1 : 0;
  } else {
#pragma unroll
    for (int k = 0; k < 32; ++k) {
      const int j = j0 + k;
      const float tt = (j < tie) ? thr_hi : thr;
      c0 += (j < Nc && __uint_as_float(v[k]) < tt) ? 1 : 0;
    }
    // ids below j0 (the other column group's half of a tile, or before this thread's first column) are passed
    // without a compare
    while (f.next < j0 + 32) {
      const int j = f.next, c = j - j0;
      if (c >= 0) {
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < 32; ++i) s = (i == c) ? __uint_as_float(v[i]) : s;     // no dynamic register index
        const float tt = (j < tie) ? thr_hi : thr;
        fc += (j < Nc && s < tt) ? 1 : 0;
      }
      filter_advance(f, f_ids, ent_begin);
    }
    __syncwarp();          // reconverge before the next .sync.aligned tcgen05 instruction
  }
}
// 128 columns (four chunks) of one accumulator row; the TMEM load of a chunk is in flight while
// the previous one is counted.
__device__ __forceinline__ void epi_count128(uint32_t taddr0, int j0, float thr, float thr_hi, int tie, int Nc,
                                             int& c0, FilterCursor& f, const int32_t* __restrict__ f_ids,
                                             int64_t ent_begin, int& fc) {
  uint32_t va[32], vb[32];
  tmem_ld32_async(taddr0, va);
  tmem_ld_wait(va);
  tmem_ld32_async(taddr0 + 32, vb);
  epi_count32(va, j0, thr, thr_hi, tie, Nc, c0, f, f_ids, ent_begin, fc);
  tmem_ld_wait(vb);
  tmem_ld32_async(taddr0 + 64, va);
  epi_count32(vb, j0 + 32, thr, thr_hi, tie, Nc, c0, f, f_ids, ent_begin, fc);
  tmem_ld_wait(va);
  tmem_ld32_async(taddr0 + 96, vb);
  epi_count32(va, j0 + 64, thr, thr_hi, tie, Nc, c0, f, f_ids, ent_begin, fc);
  tmem_ld_wait(vb);
  epi_count32(vb, j0 + 96, thr, thr_hi, tie, Nc, c0, f, f_ids, ent_begin, fc);
}

// ---- top-k epilogue.  A candidate is the 64-bit key (order-preserving bits of s, local index j): ascending
// keys are ascending (s, id), the reference heap's pop order (holE.py:434, 446-453).  -0 is folded into +0 so
// that the float compare and the key order agree.
constexpr uint64_t TOPK_EMPTY = ~0ull;      // larger than every real key
__device__ __forceinline__ uint32_t f32_order_bits(float s) {
  const uint32_t u = __float_as_uint(s + 0.0f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float f32_from_order_bits(uint32_t b) {
  return __uint_as_float((b & 0x80000000u) ? (b & 0x7fffffffu) : ~b);
}
__device__ __forceinline__ uint64_t topk_key(float s, uint32_t j) {
  return ((uint64_t)f32_order_bits(s) << 32) | j;
}

// One thread's list: a binary max-heap of at most k keys in global memory; thr = the float of its root once
// it is full (+inf before).  Candidates arrive in increasing index order, so a later candidate with the
// root's score loses the tie and `s < thr` is the whole admission test.
struct TopkList {
  uint64_t* heap;
  int n, k;
  float thr;
  int64_t f0, f1;            // the query's filter slice [f0, f1) of f_ids
  int self;                  // local index never admitted (hole_neighbors: the query's own row), -1 for none
};

__device__ __forceinline__ bool in_filter(const int32_t* __restrict__ ids, int64_t lo, int64_t hi, int32_t id) {
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    const int32_t v = ids[mid];
    if (v == id) return true;
    if (v < id) lo = mid + 1; else hi = mid;
  }
  return false;
}

__device__ __forceinline__ void topk_insert(TopkList& L, uint64_t key) {
  uint64_t* h = L.heap;
  if (L.n < L.k) {                                // sift up from the new leaf
    int i = L.n++;
    while (i > 0) {
      const int par = (i - 1) >> 1;
      const uint64_t pk = h[par];
      if (pk >= key) break;
      h[i] = pk;
      i = par;
    }
    h[i] = key;
  } else {                                        // replace the root (key < root), sift down
    int i = 0;
    for (;;) {
      int c = 2 * i + 1;
      if (c >= L.k) break;
      uint64_t ck = h[c];
      if (c + 1 < L.k) {
        const uint64_t rk = h[c + 1];
        if (rk > ck) { ck = rk; ++c; }
      }
      if (ck <= key) break;
      h[i] = ck;
      i = c;
    }
    h[i] = key;
  }
  if (L.n == L.k) L.thr = f32_from_order_bits((uint32_t)(h[0] >> 32));
}

// Hot path: one compare per score of 32 accumulator columns, and a warp vote.
__device__ __forceinline__ bool epi_topk_vote(const uint32_t (&v)[32], float thr) {
  bool hit = false;
#pragma unroll
  for (int c = 0; c < 32; ++c) hit |= __uint_as_float(v[c]) < thr;
  return __any_sync(0xffffffffu, hit);
}
// Slow path, only for a warp in which some lane admits a candidate of columns j0 .. j0+31: bounds, filter,
// heap insert.  Runs while no tcgen05.ld is in flight (the loaded registers are final).
__device__ __forceinline__ void epi_topk_admit(const uint32_t (&v)[32], int j0, TopkList& L, int Nc,
                                               const int32_t* __restrict__ f_ids, int64_t ent_begin) {
  uint32_t m = 0;
#pragma unroll
  for (int c = 0; c < 32; ++c) m |= (__uint_as_float(v[c]) < L.thr ? 1u : 0u) << c;
  while (m != 0) {
    const int c = __ffs(m) - 1;
    m &= m - 1;
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 32; ++i) s = (i == c) ? __uint_as_float(v[i]) : s;     // no dynamic register index
    const int j = j0 + c;
    if (!(s < L.thr) || j >= Nc || j == L.self) continue;                      // thr may have dropped
    if (L.f0 < L.f1 && in_filter(f_ids, L.f0, L.f1, (int32_t)(ent_begin + j))) continue;
    topk_insert(L, topk_key(s, (uint32_t)j));
  }
  __syncwarp();          // reconverge before the next .sync.aligned tcgen05 instruction
}
// 128 columns of one accumulator row.  The next chunk's TMEM load is in flight during the vote on the current
// one; the slow path of a chunk runs after that load has landed.
__device__ __forceinline__ void epi_topk128(uint32_t taddr0, int j0, TopkList& L, int Nc,
                                            const int32_t* __restrict__ f_ids, int64_t ent_begin) {
  uint32_t va[32], vb[32];
  tmem_ld32_async(taddr0, va);
  tmem_ld_wait(va);
  tmem_ld32_async(taddr0 + 32, vb);
  bool h = epi_topk_vote(va, L.thr);
  tmem_ld_wait(vb);
  if (h) epi_topk_admit(va, j0, L, Nc, f_ids, ent_begin);
  tmem_ld32_async(taddr0 + 64, va);
  h = epi_topk_vote(vb, L.thr);
  tmem_ld_wait(va);
  if (h) epi_topk_admit(vb, j0 + 32, L, Nc, f_ids, ent_begin);
  tmem_ld32_async(taddr0 + 96, vb);
  h = epi_topk_vote(va, L.thr);
  tmem_ld_wait(vb);
  if (h) epi_topk_admit(va, j0 + 64, L, Nc, f_ids, ent_begin);
  if (epi_topk_vote(vb, L.thr)) epi_topk_admit(vb, j0 + 96, L, Nc, f_ids, ent_begin);
}

struct SmemLayout {
  uint64_t full[MAX_STAGES];
  uint64_t empty[MAX_STAGES];
  uint64_t a_full;
  uint64_t a_empty;
  uint64_t tmem_full[2];
  uint64_t tmem_empty[2];
  uint32_t tmem_base;
};

// ------------------------------------------------------------------------------------ kernel
// PARTS = 1 plain bf16, 2 split-bf16 (compile-time, so that the bf16 instantiation's single-thread
// producer / issue loops carry none of the split mode's bookkeeping); EPI = EPI_RANK / EPI_TOPK (compile-time,
// so that the counting epilogue carries none of the top-k code).
// p is __grid_constant__ so that its fields are read in place from parameter space where they are used.  Passed
// by value, the struct (136 bytes) is loaded into registers at entry, and each top-k instantiation compiles to
// 112 more instructions.
template <int PARTS, int EPI>
__global__ void __launch_bounds__(RANK_THREADS, 1)
hole_rank_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const __grid_constant__ RankParams p) {
  extern __shared__ uint8_t smem_raw[];
  // 128-byte swizzle atoms repeat every 1024 bytes: align the operand area explicitly
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int nkb_all = p.num_kb * PARTS;                     // k-blocks of a whole operand row
  uint8_t* sA = smem;                                       // nkb_all x 16 KB
  uint8_t* sB = smem + (size_t)nkb_all * A_KB_BYTES;        // stages x 32 KB
  SmemLayout* sl = reinterpret_cast<SmemLayout*>(sB + (size_t)p.stages * B_KB_BYTES);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_items = p.m_tiles * p.n_chunks;

  if (warp == WARP_TMA && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < p.stages; ++s) { mbar_init(&sl->full[s], 1); mbar_init(&sl->empty[s], 1); }
    mbar_init(&sl->a_full, 1);
    mbar_init(&sl->a_empty, 1);
    for (int s = 0; s < 2; ++s) { mbar_init(&sl->tmem_full[s], 1); mbar_init(&sl->tmem_empty[s], EPI_WARPS); }
    fence_barrier_init();
  }
  if (warp == WARP_MMA) tmem_alloc(&sl->tmem_base, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = sl->tmem_base;

  if (warp == WARP_TMA) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0, a_phase = 0;
      // DIAG: only the tile's own 128 true rows are needed (the map's box is 128 rows there)
      const uint32_t b_bytes = (p.mode == MODE_DIAG) ? B_KB_BYTES / 2 : B_KB_BYTES;
      for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        const int m_tile = item / p.n_chunks, chunk = item % p.n_chunks;
        mbar_wait(&sl->a_empty, a_phase ^ 1);
        mbar_expect_tx(&sl->a_full, (uint32_t)nkb_all * A_KB_BYTES);
        for (int kb = 0; kb < nkb_all; ++kb)
          tma_load_2d(sA + (size_t)kb * A_KB_BYTES, &tmA, &sl->a_full, kb * BK, m_tile * BM);
        a_phase ^= 1;
        const int t0 = chunk * p.chunk_tiles;
        const int t1 = (p.mode == MODE_DIAG) ? t0 + 1 : min(p.n_tiles, t0 + p.chunk_tiles);
        for (int t = t0; t < t1; ++t) {
          const int row0 = (p.mode == MODE_DIAG) ? m_tile * BM : t * BN;
          for (int kb = 0; kb < nkb_all; ++kb) {
            mbar_wait(&sl->empty[stage], phase ^ 1);
            mbar_expect_tx(&sl->full[stage], b_bytes);
            tma_load_2d(sB + (size_t)stage * B_KB_BYTES, &tmB, &sl->full[stage], kb * BK, row0);
            if (++stage == p.stages) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == WARP_MMA) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t idesc = (p.mode == MODE_DIAG) ? umma_idesc_bf16(BM, BM) : umma_idesc_bf16(BM, BN);
      const int a_lo_off = p.num_kb * A_KB_BYTES;   // query lo part sits after the hi part
      int stage = 0; uint32_t phase = 0, a_phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        const int chunk = item % p.n_chunks;
        mbar_wait(&sl->a_full, a_phase);
        a_phase ^= 1;
        tc_fence_after();
        const int t0 = chunk * p.chunk_tiles;
        const int t1 = (p.mode == MODE_DIAG) ? t0 + 1 : min(p.n_tiles, t0 + p.chunk_tiles);
        for (int t = t0; t < t1; ++t) {
          mbar_wait(&sl->tmem_empty[acc], acc_phase ^ 1);
          tc_fence_after();
          const uint32_t d_addr = tmem_base + (uint32_t)acc * BN;
          int kk = 0;                                // kb modulo num_kb: k-block inside its operand part
          for (int kb = 0; kb < nkb_all; ++kb) {
            mbar_wait(&sl->full[stage], phase);
            tc_fence_after();
            const uint32_t b_addr = smem_u32(sB + (size_t)stage * B_KB_BYTES);
            // The issuing thread is on the critical path (the k-block's MMAs must be queued before
            // the previous block's retire), so both loops below are kept free of divisions and
            // nested runtime loops: measured 59 -> 52 ms on 100 k x 1.2 M against a generic loop.
            const uint32_t a_addr = smem_u32(sA + (size_t)kk * A_KB_BYTES);
            const int nk = (kk == p.num_kb - 1) ? p.last_kb_mmas : BK / UMMA_K;   // skip all-zero slices
#pragma unroll
            for (int k = 0; k < BK / UMMA_K; ++k) {
              if (k < nk) {
                const uint64_t da = umma_desc_sw128(a_addr + k * UMMA_K * 2);
                const uint64_t db = umma_desc_sw128(b_addr + k * UMMA_K * 2);
                umma_bf16(d_addr, da, db, idesc, (kb | k) != 0 ? 1u : 0u);
              }
            }
            if (PARTS == 2 && kb < p.num_kb) {
              // split-bf16: a candidate hi block also meets the query lo block (hi.hi + lo.hi + hi.lo;
              // the candidate lo blocks, kb >= num_kb, meet the query hi block only)
              const uint32_t a_lo = a_addr + (uint32_t)a_lo_off;
#pragma unroll
              for (int k = 0; k < BK / UMMA_K; ++k) {
                if (k < nk) {
                  const uint64_t da = umma_desc_sw128(a_lo + k * UMMA_K * 2);
                  const uint64_t db = umma_desc_sw128(b_addr + k * UMMA_K * 2);
                  umma_bf16(d_addr, da, db, idesc, 1u);
                }
              }
            }
            if (PARTS == 2) { if (++kk == p.num_kb) kk = 0; } else { kk = kb + 1; }
            umma_commit(&sl->empty[stage]);          // frees the smem slot when the MMAs retire
            if (++stage == p.stages) { stage = 0; phase ^= 1; }
          }
          umma_commit(&sl->tmem_full[acc]);          // accumulator ready for the epilogue
          if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
        umma_commit(&sl->a_empty);                   // query tile may be overwritten
      }
    }
  } else if constexpr (EPI == EPI_TOPK) {
    // ===================== top-k epilogue =====================
    // Each thread keeps the k best of its 128 columns of every tile of the work item: list
    // [q][chunk][cgrp] of p.tk_keys, unused slots TOPK_EMPTY.  hole_topk_merge_kernel combines the lists.
    const int ew = warp - WARP_EPI0;
    const int quarter = warp & 3;
    const int cgrp = ew >> 2;
    const int row_in_tile = quarter * 32 + lane;
    int acc = 0; uint32_t acc_phase = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
      const int m_tile = item / p.n_chunks, chunk = item % p.n_chunks;
      const int q = m_tile * BM + row_in_tile;
      const bool qok = q < p.Q;
      TopkList L;
      L.heap = p.tk_keys + (((size_t)q * p.n_chunks + chunk) * 2 + cgrp) * p.topk;
      L.n = 0; L.k = p.topk;
      L.thr = qok ? INFINITY : -INFINITY;            // rows past Q admit nothing
      L.f0 = L.f1 = 0;
      if (qok && p.f_off != nullptr) { L.f0 = p.f_off[q]; L.f1 = p.f_off[q + 1]; }
      L.self = (qok && p.tk_self != nullptr) ? p.tk_self[q] : -1;
      const int t0 = chunk * p.chunk_tiles;
      const int t1 = min(p.n_tiles, t0 + p.chunk_tiles);
      for (int t = t0; t < t1; ++t) {
        mbar_wait(&sl->tmem_full[acc], acc_phase);
        tc_fence_after();
        const uint32_t taddr0 = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * BN + cgrp * EPI_COLS);
        epi_topk128(taddr0, t * BN + cgrp * EPI_COLS, L, p.Nc, p.f_ids, p.ent_begin);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&sl->tmem_empty[acc]);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
      if (qok)
        for (int i = L.n; i < L.k; ++i) L.heap[i] = TOPK_EMPTY;
    }
  } else {
    // ===================== epilogue =====================
    const int ew = warp - WARP_EPI0;         // 0..EPI_WARPS-1
    const int quarter = warp & 3;            // TMEM lane quarter this warp may access
    const int cgrp = ew >> 2;                // which EPI_COLS columns of the tile
    const int row_in_tile = quarter * 32 + lane;
    int acc = 0; uint32_t acc_phase = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
      const int m_tile = item / p.n_chunks, chunk = item % p.n_chunks;
      const int q = m_tile * BM + row_in_tile;
      const bool qok = q < p.Q;
      const int t0 = chunk * p.chunk_tiles;
      const int t1 = (p.mode == MODE_DIAG) ? t0 + 1 : min(p.n_tiles, t0 + p.chunk_tiles);
      float thr = -INFINITY, thr_hi = -INFINITY;
      int tie = 0;
      FilterCursor fcur{0, 0, INT_MAX, INT_MAX};
      if (p.mode == MODE_COUNT && qok) {
        int64_t f0 = 0;
        if (p.f_off != nullptr) { f0 = p.f_off[q]; fcur.f1 = p.f_off[q + 1]; }
        thr = p.true_score[q];
        const int ti = p.true_idx[q];
        if (p.f_off != nullptr) {
          // A long slice is entered by binary search at this thread's first column; a short one from its start
          // (the merge-join passes ids below the thread's columns).
          if (fcur.f1 - f0 > 16)
            f0 = lower_bound_id(p.f_ids, f0, fcur.f1, p.ent_begin + (int64_t)t0 * BN + cgrp * EPI_COLS);
          fcur.fp = f0;
          fcur.next = filter_id_at(p.f_ids, f0, fcur.f1, p.ent_begin);
          fcur.after = filter_id_at(p.f_ids, f0 + 1, fcur.f1, p.ent_begin);
        }
        thr_hi = nextafterf(thr, INFINITY);          // s <= thr  <=>  s < thr_hi
        tie = ti < 0 ? 0 : (ti > p.Nc ? p.Nc : ti);  // candidates with local index < tie win ties
      }
      int cnt = 0, fcnt = 0;
      for (int t = t0; t < t1; ++t) {
        mbar_wait(&sl->tmem_full[acc], acc_phase);
        tc_fence_after();
        const uint32_t taddr0 = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * BN + cgrp * EPI_COLS);
        if (p.mode == MODE_COUNT) {
          static_assert(EPI_COLS == 128, "epi_count128 covers 128 columns per warp");
          epi_count128(taddr0, t * BN + cgrp * EPI_COLS, thr, thr_hi, tie, p.Nc, cnt, fcur, p.f_ids, p.ent_begin,
                       fcnt);
        } else if (cgrp == (quarter * 32) / EPI_COLS) {
          // DIAG: row i of the tile wants column i, which lives in chunk `quarter`, register `lane`
          uint32_t v[32];
          tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * BN + quarter * 32), v);
          float s = 0.f;
#pragma unroll
          for (int k = 0; k < 32; ++k) s = (k == lane) ? __uint_as_float(v[k]) : s;
          if (qok) {
            const int ti = p.true_idx[q];
            if (ti >= 0 && ti < p.Nc) p.true_out[q] = s;
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&sl->tmem_empty[acc]);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
      if (p.mode == MODE_COUNT && qok && cnt != 0) {
        atomicAdd(&p.raw_cnt[q], cnt);
        atomicAdd(&p.filt_cnt[q], cnt - fcnt);
      }
    }
  }
  __syncwarp();          // the single-lane roles rejoin their warps
  tc_fence_before();
  __syncthreads();
  if (warp == WARP_MMA) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------ operand packing
// One warp per row.  Candidate operand: clip(E_j) rounded to bf16, [Re | Im | 0-pad] of K columns; with
// `normalize` (hole_neighbors) E_j / |E_j| instead, and zero for a zero row.
__global__ void __launch_bounds__(256)
hole_rank_pack_cand_kernel(const float* __restrict__ table, int stride, int H, int64_t ent_begin,
                           int Nc, int Npad, int K, int parts, int normalize, __nv_bfloat16* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (r >= Npad) return;
  __nv_bfloat16* o = out + (size_t)r * K * parts;       // row = [hi part (K) | lo part (K)]
  if (r >= Nc) {
    for (int k = lane; k < K * parts; k += 32) o[k] = __float2bfloat16(0.f);
    return;
  }
  const float* x = table + (size_t)(ent_begin + r) * stride;
  const int Hp = stride / 2;
  float ss = 0.f;
  for (int k = lane; k < H; k += 32) { float a = x[k], b = x[Hp + k]; ss = fmaf(a, a, fmaf(b, b, ss)); }
#pragma unroll
  for (int o2 = 16; o2 > 0; o2 >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o2);
  const float sc = normalize ? (ss > 0.f ? __frsqrt_rn(ss) : 0.f) : fminf(__frsqrt_rn(ss), 1.0f);
  for (int k = lane; k < K; k += 32) {
    float v = 0.f;
    if (k < H) v = x[k] * sc;
    else if (k < 2 * H) v = x[Hp + (k - H)] * sc;
    const __nv_bfloat16 hi = __float2bfloat16(v);
    o[k] = hi;
    if (parts == 2) o[K + k] = __float2bfloat16(v - __bfloat162float(hi));
  }
}

// Query operand (App. A.4): tail side q = h * r; head side q = r * conj(t) with the imaginary
// half negated; relation side q = h * conj(t) with the imaginary half negated (the head side's product
// with h as the first factor: s is linear in the relation row, App. A.3's ds/dy_r).  Also records the
// shard-local index of the true candidate (t, h or r).
// One warp per query; a lane holds groups of four complex components of both factor rows
// (float4 loads of the [Re | pad | Im | pad] row layout) in registers between the norm pass and
// the product pass.  PQ_ITERS = ceil(Hp / 128), at most 3 for the dimensions the ranking kernel's smem admits.
template <int PQ_ITERS>
__global__ void __launch_bounds__(256)
hole_rank_pack_query_kernel(const float* __restrict__ table, int stride, int H,
                            const int32_t* __restrict__ queries, int Q, int Qpad, int side,
                            int64_t ent_begin, int K, int parts, __nv_bfloat16* __restrict__ out,
                            int32_t* __restrict__ true_idx, float* __restrict__ qf) {
  extern __shared__ uint4 pq_smem[];                    // one operand row per warp, written out as 16-byte vectors
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int64_t qi = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (qi >= Qpad) return;
  const int row_vecs = K * parts / 8;                   // K is a multiple of 64
  uint4* o4 = reinterpret_cast<uint4*>(out + (size_t)qi * K * parts);      // row = [hi part (K) | lo part (K)]
  if (qi >= Q) {
    for (int k = lane; k < row_vecs; k += 32) o4[k] = make_uint4(0, 0, 0, 0);
    if (lane == 0) true_idx[qi] = -1;
    return;
  }
  uint4* row4 = pq_smem + (size_t)wib * row_vecs;
  __nv_bfloat16* row = reinterpret_cast<__nv_bfloat16*>(row4);
#pragma unroll 1
  for (int k = lane; k < row_vecs; k += 32) row4[k] = make_uint4(0, 0, 0, 0);      // the padding stays zero
  // HOLE_SIDE_BOTH: Q = 2 * Qsrc rows, the first half ranks tails, the second half heads
  int64_t src = qi;
  if (side == HOLE_SIDE_BOTH) {
    const int64_t half = Q / 2;
    side = (qi < half) ? HOLE_SIDE_TAIL : HOLE_SIDE_HEAD;
    src = (qi < half) ? qi : qi - half;
  }
  const int h = queries[3 * src], t = queries[3 * src + 1], r = queries[3 * src + 2];
  const int Hp = stride / 2, G4 = Hp / 4;
  const float4* x1 = reinterpret_cast<const float4*>(table + (size_t)(side == HOLE_SIDE_HEAD ? r : h) * stride);
  const float4* x2 = reinterpret_cast<const float4*>(table + (size_t)(side == HOLE_SIDE_TAIL ? r : t) * stride);
  float4 A[PQ_ITERS], Bv[PQ_ITERS], C[PQ_ITERS], Dv[PQ_ITERS];   // (A,Bv) = first factor re/im, (C,Dv) = second
  float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int it = 0; it < PQ_ITERS; ++it) {
    const int g = lane + 32 * it;
    A[it] = Bv[it] = C[it] = Dv[it] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (g < G4) {          // components H..Hp-1 of a half row are zero padding
      A[it] = x1[g]; Bv[it] = x1[G4 + g]; C[it] = x2[g]; Dv[it] = x2[G4 + g];
      s1 += A[it].x * A[it].x + A[it].y * A[it].y + A[it].z * A[it].z + A[it].w * A[it].w +
            Bv[it].x * Bv[it].x + Bv[it].y * Bv[it].y + Bv[it].z * Bv[it].z + Bv[it].w * Bv[it].w;
      s2 += C[it].x * C[it].x + C[it].y * C[it].y + C[it].z * C[it].z + C[it].w * C[it].w +
            Dv[it].x * Dv[it].x + Dv[it].y * Dv[it].y + Dv[it].z * Dv[it].z + Dv[it].w * Dv[it].w;
    }
  }
#pragma unroll
  for (int o2 = 16; o2 > 0; o2 >>= 1) {
    s1 += __shfl_xor_sync(0xffffffffu, s1, o2);
    s2 += __shfl_xor_sync(0xffffffffu, s2, o2);
  }
  const float c1 = fminf(__frsqrt_rn(s1), 1.0f), c2 = fminf(__frsqrt_rn(s2), 1.0f);
  const float c1s = (side == HOLE_SIDE_TAIL) ? c1 : -c1;
  __syncwarp();
#pragma unroll
  for (int it = 0; it < PQ_ITERS; ++it) {
    const int g = lane + 32 * it;
    if (g < G4) {
      const float a[4] = {A[it].x * c1, A[it].y * c1, A[it].z * c1, A[it].w * c1};        // clipped factors
      const float b[4] = {Bv[it].x * c1s, Bv[it].y * c1s, Bv[it].z * c1s, Bv[it].w * c1s};   // head side: -Im
      const float c[4] = {C[it].x * c2, C[it].y * c2, C[it].z * c2, C[it].w * c2};
      const float d[4] = {Dv[it].x * c2, Dv[it].y * c2, Dv[it].z * c2, Dv[it].w * c2};
      float re[4], im[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        // tail: (a,b)=h (c,d)=r, q = h*r;  head: (a,b)=r (c,d)=t with b negated: q = (ac+bd, ad-bc);
        // relation: (a,b)=h (c,d)=t with b negated, the same product
        re[i] = a[i] * c[i] - b[i] * d[i];
        im[i] = a[i] * d[i] + b[i] * c[i];
      }
      const int k0 = 4 * g;
      if (qf != nullptr) {     // hole_topk: the fp32 query vector before rounding, [Re | Im] of K floats
        float* qrow = qf + (size_t)qi * K;
#pragma unroll
        for (int i = 0; i < 4; ++i)
          if (k0 + i < H) { qrow[k0 + i] = re[i]; qrow[H + k0 + i] = im[i]; }
      }
      if (k0 + 4 <= H) {       // whole group: the real part is 8-byte aligned in the row
        __nv_bfloat162 p0 = __floats2bfloat162_rn(re[0], re[1]), p1 = __floats2bfloat162_rn(re[2], re[3]);
        uint2 u;
        u.x = *reinterpret_cast<uint32_t*>(&p0);
        u.y = *reinterpret_cast<uint32_t*>(&p1);
        *reinterpret_cast<uint2*>(row + k0) = u;
#pragma unroll
        for (int i = 0; i < 4; ++i) row[H + k0 + i] = __float2bfloat16(im[i]);
      } else {
#pragma unroll
        for (int i = 0; i < 4; ++i)
          if (k0 + i < H) { row[k0 + i] = __float2bfloat16(re[i]); row[H + k0 + i] = __float2bfloat16(im[i]); }
      }
      if (parts == 2) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
          if (k0 + i < H) {
            row[K + k0 + i] = __float2bfloat16(re[i] - __bfloat162float(__float2bfloat16(re[i])));
            row[K + H + k0 + i] = __float2bfloat16(im[i] - __bfloat162float(__float2bfloat16(im[i])));
          }
      }
    }
  }
  __syncwarp();
#pragma unroll 1
  for (int k = lane; k < row_vecs; k += 32) o4[k] = row4[k];
  if (lane == 0)
    true_idx[qi] = (int32_t)((int64_t)(side == HOLE_SIDE_TAIL ? t : (side == HOLE_SIDE_HEAD ? h : r)) - ent_begin);
}

// Query operand of the ARCHIVED score variant (hole_ccorr.cuh): s = Re sum_k rho_k c_k with rho = (1 - i) r is
// linear in the candidate entity, so the all-candidate form is the same dense contraction with another
// query vector:   tail side  s(h, r, .) = [Re t ; Im t] . [Re w ; -Im w],  w_m = sum_k rho_k conj(h_{m-k})
//                 head side  s(., r, t) = [Re h ; Im h] . [Re u ;  Im u],  u_j = sum_k rho_k t_{j+k}
//                 relation   s(h, ., t) = [Re r ; Im r] . [Re c + Im c ; Re c - Im c],  c_k = sum_j conj(h_j) t_{j+k}
// One warp per query, one direct O(H^2) correlation out of shared memory.  tanh is monotone: ranking on s.
template <int NV>
__global__ void __launch_bounds__(256)
hole_rank_pack_query_ccorr_kernel(const float* __restrict__ table, int stride, int H,
                                  const int32_t* __restrict__ queries, int Q, int Qpad, int side,
                                  int64_t ent_begin, int K, int parts, __nv_bfloat16* __restrict__ out,
                                  int32_t* __restrict__ true_idx, float* __restrict__ qf) {
  extern __shared__ float pqc_smem[];                   // per warp: entity row doubled (4H), rho or h (2H)
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int64_t qi = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (qi >= Qpad) return;
  __nv_bfloat16* o = out + (size_t)qi * K * parts;
  if (qi >= Q) {
    for (int k = lane * 8; k < K * parts; k += 256) *reinterpret_cast<uint4*>(o + k) = make_uint4(0, 0, 0, 0);
    if (lane == 0) true_idx[qi] = -1;
    return;
  }
  int64_t src = qi;
  if (side == HOLE_SIDE_BOTH) {
    const int64_t half = Q / 2;
    side = (qi < half) ? HOLE_SIDE_TAIL : HOLE_SIDE_HEAD;
    src = (qi < half) ? qi : qi - half;
  }
  const int h = queries[3 * src], t = queries[3 * src + 1], r = queries[3 * src + 2];
  const int Hp = stride / 2;
  float* sm = pqc_smem + (size_t)wib * (6 * H);
  float *e_re = sm, *e_im = sm + 2 * H, *rho_re = sm + 4 * H, *rho_im = sm + 5 * H;
  const bool rel = side == HOLE_SIDE_RELATION;
  CVec<NV> yr;
  // The fixed operand's row lands in the entity buffers first (overwritten below) and is kept in registers:
  // cc_load_row writes a doubled row, which does not fit the 2H floats of the rho slot.
  // rho = (1 - i) r, or for the relation side h itself.
  cc_load_row<NV>(table + (size_t)(rel ? h : r) * stride, H, Hp, lane, e_re, e_im, &yr);
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const int k = lane + 32 * v;
    if (k < H) {
      rho_re[k] = rel ? yr.re[v] : yr.re[v] + yr.im[v];
      rho_im[k] = rel ? yr.im[v] : yr.im[v] - yr.re[v];
    }
  }
  __syncwarp();
  cc_load_row<NV>(table + (size_t)(side == HOLE_SIDE_TAIL ? h : t) * stride, H, Hp, lane, e_re, e_im, nullptr);
  __syncwarp();
  CVec<NV> qv;
  if (side == HOLE_SIDE_TAIL) {
    cc_corr<NV, false, true, false>(qv, rho_re, rho_im, e_re, e_im, H, lane);       // w; q = [Re w ; -Im w]
#pragma unroll
    for (int v = 0; v < NV; ++v) qv.im[v] = -qv.im[v];
  } else if (rel) {
    cc_corr<NV, true, false, true>(qv, rho_re, rho_im, e_re, e_im, H, lane);        // c; q = [Re c + Im c ; Re c - Im c]
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      const float cr = qv.re[v], ci = qv.im[v];
      qv.re[v] = cr + ci;
      qv.im[v] = cr - ci;
    }
  } else {
    cc_corr<NV, false, false, true>(qv, rho_re, rho_im, e_re, e_im, H, lane);       // u; q = [Re u ; Im u]
  }
  for (int k = 2 * H + lane; k < K; k += 32) {
    o[k] = __float2bfloat16(0.f);
    if (parts == 2) o[K + k] = __float2bfloat16(0.f);
  }
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const int k = lane + 32 * v;
    if (k < H) {
      if (qf != nullptr) { qf[(size_t)qi * K + k] = qv.re[v]; qf[(size_t)qi * K + H + k] = qv.im[v]; }
      const __nv_bfloat16 rh = __float2bfloat16(qv.re[v]), ih = __float2bfloat16(qv.im[v]);
      o[k] = rh;
      o[H + k] = ih;
      if (parts == 2) {
        o[K + k] = __float2bfloat16(qv.re[v] - __bfloat162float(rh));
        o[K + H + k] = __float2bfloat16(qv.im[v] - __bfloat162float(ih));
      }
    }
  }
  if (lane == 0) true_idx[qi] = (int32_t)((int64_t)(side == HOLE_SIDE_TAIL ? t : (rel ? r : h)) - ent_begin);
}

// Query operand of hole_neighbors: -E_q / |E_q| (zero for a zero row) of the row ids[q], negated so that the
// ascending top-k epilogue selects the most similar candidates.  The norm is reduced in the candidate packer's
// order, so a row and its own candidate row are exact negatives of each other.  Also writes the fp32 vector
// before rounding (qf, [Re | Im] of K floats) and the shard-local index of the row itself, which the epilogue
// never admits.  One warp per query.
__global__ void __launch_bounds__(256)
hole_neighbors_pack_query_kernel(const float* __restrict__ table, int stride, int H, const int32_t* __restrict__ ids,
                                 int Q, int Qpad, int64_t ent_begin, int K, int parts,
                                 __nv_bfloat16* __restrict__ out, int32_t* __restrict__ true_idx,
                                 float* __restrict__ qf) {
  const int lane = threadIdx.x & 31;
  const int64_t qi = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (qi >= Qpad) return;
  __nv_bfloat16* o = out + (size_t)qi * K * parts;       // row = [hi part (K) | lo part (K)]
  if (qi >= Q) {
    for (int k = lane; k < K * parts; k += 32) o[k] = __float2bfloat16(0.f);
    if (lane == 0) true_idx[qi] = -1;
    return;
  }
  const int id = ids[qi];
  const float* x = table + (size_t)id * stride;
  const int Hp = stride / 2;
  float ss = 0.f;
  for (int k = lane; k < H; k += 32) { float a = x[k], b = x[Hp + k]; ss = fmaf(a, a, fmaf(b, b, ss)); }
#pragma unroll
  for (int o2 = 16; o2 > 0; o2 >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o2);
  const float sc = ss > 0.f ? -__frsqrt_rn(ss) : 0.f;
  float* qrow = qf + (size_t)qi * K;
  for (int k = lane; k < K; k += 32) {
    float v = 0.f;
    if (k < H) v = x[k] * sc;
    else if (k < 2 * H) v = x[Hp + (k - H)] * sc;
    if (k < 2 * H) qrow[k] = v;
    const __nv_bfloat16 hi = __float2bfloat16(v);
    o[k] = hi;
    if (parts == 2) o[K + k] = __float2bfloat16(v - __bfloat162float(hi));
  }
  if (lane == 0) true_idx[qi] = (int32_t)((int64_t)id - ent_begin);
}

// T[q] = packed candidate row of q's true candidate (zeros when it is not in this shard).
// Eight lanes per row, four rows per warp: the kernel is two dependent loads deep, so rows in
// flight per SM are what sets its speed.
__global__ void __launch_bounds__(256)
hole_rank_gather_true_kernel(const __nv_bfloat16* __restrict__ cand, const int32_t* __restrict__ true_idx,
                             int Nc, int rows, int K, __nv_bfloat16* __restrict__ out) {
  const int sub = threadIdx.x & 7;
  const int64_t qi = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 3;
  if (qi >= rows) return;
  const int ti = true_idx[qi];
  const bool ok = ti >= 0 && ti < Nc;
  const uint4* src = reinterpret_cast<const uint4*>(cand + (size_t)(ok ? ti : 0) * K);
  uint4* dst = reinterpret_cast<uint4*>(out + (size_t)qi * K);
  const int nv = K / 8;                                  // a multiple of 8 (K is a multiple of 64)
#pragma unroll 4
  for (int k = sub; k < nv; k += 8) dst[k] = ok ? src[k] : make_uint4(0, 0, 0, 0);
}

// hole_topk, after the contraction: one block per output row.
//  1. the k smallest keys of the row's n_lists partial lists (k keys each, TOPK_EMPTY-padded): an 8-pass
//     MSB-first radix select finds the k-th smallest key K*, then every key < K* and K* itself are taken
//     (real keys are unique -- each candidate lives in one list -- so only TOPK_EMPTY repeats);
//  2. each selected candidate is rescored in fp32: the clipped fp32 table row times the fp32 query vector qf;
//  3. the row is sorted by (fp32 score, id); slots without a candidate get id -1 and score +inf.
// neighbors (hole_neighbors): the candidate row is unit-normalised instead of clipped, the score written is the
// similarity -s, and empty slots get -inf.
constexpr int TOPK_MAX = 128;
constexpr int MERGE_THREADS = 256;
__global__ void __launch_bounds__(MERGE_THREADS)
hole_topk_merge_kernel(const uint64_t* __restrict__ keys, int n_lists, int k, const float* __restrict__ table,
                       int stride, int H, int64_t ent_begin, const float* __restrict__ qf, int K, int neighbors,
                       int32_t* __restrict__ ids_out, float* __restrict__ scores_out) {
  __shared__ uint32_t hist[256];
  __shared__ uint64_t sel[TOPK_MAX];
  __shared__ float sc[TOPK_MAX];
  __shared__ uint64_t prefix_s;
  __shared__ int kk_s, cnt_s;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t q = blockIdx.x;
  int32_t* ido = ids_out + q * k;
  float* sco = scores_out + q * k;
  const float pad = neighbors ? -INFINITY : INFINITY;
  if (n_lists == 0) {                                  // empty candidate range
    for (int i = tid; i < k; i += MERGE_THREADS) { ido[i] = -1; sco[i] = pad; }
    return;
  }
  const int64_t L = (int64_t)n_lists * k;              // >= 2k: the k-th smallest key exists
  const uint64_t* kr = keys + q * L;
  uint64_t prefix = 0, mask = 0;
  int kk = k;                                          // rank of K* among the keys matching prefix
  for (int shift = 56; shift >= 0; shift -= 8) {
    for (int i = tid; i < 256; i += MERGE_THREADS) hist[i] = 0;
    __syncthreads();
    for (int64_t i = tid; i < L; i += MERGE_THREADS) {
      const uint64_t x = kr[i];
      if ((x & mask) == prefix) atomicAdd(&hist[(x >> shift) & 255], 1u);
    }
    __syncthreads();
    if (warp == 0) {                                   // digit of K*: lane l scans bins 8l .. 8l+7
      uint32_t c[8], tot = 0;
#pragma unroll
      for (int i = 0; i < 8; ++i) { c[i] = hist[lane * 8 + i]; tot += c[i]; }
      uint32_t inc = tot;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += y;
      }
      uint32_t cum = inc - tot;
      if (cum < (uint32_t)kk && (uint32_t)kk <= inc) {
        int d = -1;
#pragma unroll
        for (int i = 0; i < 8; ++i)
          if (d < 0) {
            if (cum + c[i] >= (uint32_t)kk) d = lane * 8 + i; else cum += c[i];
          }
        kk_s = kk - (int)cum;
        prefix_s = prefix | ((uint64_t)d << shift);
      }
    }
    __syncthreads();
    kk = kk_s;
    prefix = prefix_s;
    mask |= 0xffull << shift;
  }
  if (tid == 0) cnt_s = 0;
  __syncthreads();
  for (int64_t i = tid; i < L; i += MERGE_THREADS) {
    const uint64_t x = kr[i];
    if (x < prefix) sel[atomicAdd(&cnt_s, 1)] = x;     // k - kk keys
  }
  __syncthreads();
  for (int i = k - kk + tid; i < k; i += MERGE_THREADS) sel[i] = prefix;
  __syncthreads();
  const float* qrow = qf + q * K;
  const int Hp = stride / 2;
  for (int i = warp; i < k; i += MERGE_THREADS / 32) {
    const uint64_t x = sel[i];
    if (x == TOPK_EMPTY) continue;
    const float* row = table + (size_t)(ent_begin + (uint32_t)x) * stride;
    float ss = 0.f;
    for (int c = lane; c < H; c += 32) { const float a = row[c], b = row[Hp + c]; ss = fmaf(a, a, fmaf(b, b, ss)); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    const float scl = neighbors ? (ss > 0.f ? __frsqrt_rn(ss) : 0.f) : fminf(__frsqrt_rn(ss), 1.0f);
    float d = 0.f;
    for (int c = lane; c < H; c += 32) d = fmaf(row[c] * scl, qrow[c], fmaf(row[Hp + c] * scl, qrow[H + c], d));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
    if (lane == 0) sc[i] = d;
  }
  __syncthreads();
  uint64_t mine = TOPK_EMPTY;
  if (tid < k && sel[tid] != TOPK_EMPTY) mine = topk_key(sc[tid], (uint32_t)sel[tid]);
  __syncthreads();
  if (tid < k) sel[tid] = mine;
  __syncthreads();
  if (tid < k) {
    int r = 0;
    for (int i = 0; i < k; ++i) { const uint64_t o = sel[i]; r += (o < mine || (o == mine && i < tid)) ? 1 : 0; }
    if (mine == TOPK_EMPTY) { ido[r] = -1; sco[r] = pad; }
    else {
      const float s = f32_from_order_bits((uint32_t)(mine >> 32));
      ido[r] = (int32_t)(ent_begin + (uint32_t)mine);
      sco[r] = neighbors ? 0.f - s : s;                // 0 - s: a zero similarity is +0
    }
  }
}

// ------------------------------------------------------------------------------------ host
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn == nullptr) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(ptr);
  }
  return fn;
}

// bf16 [rows, K] row-major, box = 64 columns x box_rows rows, 128-byte swizzle
int make_map(CUtensorMap* map, const void* base, int64_t rows, int K, int box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  if (fn == nullptr) return hole_set_error(HOLE_ERR_CUDA, "cuTensorMapEncodeTiled entry point not found");
  cuuint64_t gdim[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t gstr[1] = {(cuuint64_t)K * 2};
  cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstr, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return hole_set_error(HOLE_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  return HOLE_OK;
}

}  // namespace

struct hole_rank_ws {
  __nv_bfloat16* cand = nullptr;   // [Npad, K]
  __nv_bfloat16* qp = nullptr;     // [Qpad, K]
  __nv_bfloat16* tq = nullptr;     // [Qpad + BN, K] gathered true rows
  int32_t* true_idx = nullptr;     // [Qpad]
  size_t cand_cap = 0, q_cap = 0, tq_cap = 0;  // elements
  float* qf = nullptr;             // hole_topk: [Qpad, K] fp32 query vectors
  uint64_t* tk_keys = nullptr;     // hole_topk: [Qpad][n_chunks][2][k] partial lists
  size_t qf_cap = 0, tk_cap = 0;   // elements
  bool attr_set = false;
  int64_t last_npad = 0, last_qpad = 0;
  int last_K = 0;
  // packed candidate operand kept across calls (hole_rank_prepare): valid for exactly this table / range
  const float* cache_table = nullptr;
  int64_t cache_begin = -1, cache_end = -1;
  int cache_parts = 0;
  bool cache_valid = false;
};

void hole_rank_cache_invalidate(hole_ctx* c) {
  if (c->rank != nullptr) c->rank->cache_valid = false;
}

void hole_rank_ws_free(hole_ctx* c) {
  if (c->rank == nullptr) return;
  cudaFree(c->rank->cand); cudaFree(c->rank->qp); cudaFree(c->rank->tq); cudaFree(c->rank->true_idx);
  cudaFree(c->rank->qf); cudaFree(c->rank->tk_keys);
  delete c->rank;
  c->rank = nullptr;
}

// Work items of hole_rank_kernel: enough to balance the persistent CTAs, chunks of at least 8 candidate tiles.
static void split_chunks(RankParams& p, int sm_count) {
  const int want_items = 8 * sm_count;
  const int chunks = std::max(1, std::min(p.n_tiles / 8, (want_items + p.m_tiles - 1) / p.m_tiles));
  p.chunk_tiles = (p.n_tiles + chunks - 1) / chunks;
  p.n_chunks = (p.n_tiles + p.chunk_tiles - 1) / p.chunk_tiles;
}

struct TopkArgs {
  int k;
  int32_t* ids_out;
  float* scores_out;
  bool neighbors;      // hole_neighbors: `queries` is an id list [Q], cosine over unit-normalised operands
};

// prepare_only: pack (and keep) the candidate operand, nothing else
// tk != null: hole_topk (the k best candidates per row instead of counts / true scores), or hole_neighbors.
// hole_neighbors packs its own normalised candidate operand over the cache's buffer: it never reads the
// cache and always drops it, so a clipped operand never meets a cosine query and a normalised one never
// serves a ranking call.
static int rank_impl(hole_ctx* c, const float* table, int64_t ent_begin, int64_t ent_end,
                     const float* query_table, const int32_t* queries, int64_t Q, int side, int precision,
                     const int64_t* filter_off, const int32_t* filter_ids, float* true_score_io,
                     int compute_true, int32_t* raw_before, int32_t* filt_before, void* stream,
                     bool prepare_only, const TopkArgs* tk = nullptr) {
  HOLE_CHECK_ARG(c && Q >= 0 && ent_begin >= 0 && ent_end >= ent_begin && ent_end <= c->n_rows);
  HOLE_CHECK_ARG(side == HOLE_SIDE_TAIL || side == HOLE_SIDE_HEAD || side == HOLE_SIDE_BOTH ||
                 side == HOLE_SIDE_RELATION);
  const bool topk = tk != nullptr;
  const bool nb = topk && tk->neighbors;
  if (topk && Q > 0 && ent_end == ent_begin) {       // no candidates: every output row is padding
    HOLE_CHECK_ARG(queries != nullptr);
    HOLE_CUDA_TRY(cudaSetDevice(c->device));
    const int64_t rows = (side == HOLE_SIDE_BOTH) ? 2 * Q : Q;
    HOLE_CHECK_ARG(rows < (int64_t(1) << 30));
    hole_topk_merge_kernel<<<(unsigned)rows, MERGE_THREADS, 0, (cudaStream_t)stream>>>(
        nullptr, 0, tk->k, nullptr, 0, 0, 0, nullptr, 0, nb ? 1 : 0, tk->ids_out, tk->scores_out);
    HOLE_LAUNCHED();
    return HOLE_OK;
  }
  if ((Q == 0 && !prepare_only) || ent_end == ent_begin) return HOLE_OK;
  if (side == HOLE_SIDE_BOTH) Q *= 2;    // output rows: [tail ranks of all queries | head ranks]
  const bool count = raw_before != nullptr;          // without count buffers: true scores only
  HOLE_CHECK_ARG(table != nullptr && (prepare_only || (queries && (topk || true_score_io))));
  HOLE_CHECK_ARG((raw_before == nullptr) == (filt_before == nullptr));
  HOLE_CHECK_ARG(prepare_only || topk || count || compute_true);
  if (query_table == nullptr) query_table = table;
  HOLE_CHECK_ARG((filter_off == nullptr) == (filter_ids == nullptr));
  HOLE_CHECK_ARG(precision == HOLE_RANK_BF16 || precision == HOLE_RANK_BF16X3);
  const int parts = (precision == HOLE_RANK_BF16X3) ? 2 : 1;
  HOLE_CHECK_ARG(Q < (int64_t(1) << 30) && ent_end - ent_begin < (int64_t(1) << 30));
  HOLE_CUDA_TRY(cudaSetDevice(c->device));
  cudaStream_t st = (cudaStream_t)stream;

  const int Nc = (int)(ent_end - ent_begin);
  const int K = (c->dim + BK - 1) / BK * BK;
  const int num_kb = K / BK;
  const int Npad = (Nc + BN - 1) / BN * BN;
  const int Qpad = (int)((Q + BM - 1) / BM * BM);
  const int Kall = K * parts;                                  // operand columns in memory
  const int a_bytes = num_kb * parts * A_KB_BYTES;
  const int stages = std::min((SMEM_LIMIT - a_bytes - 2048) / B_KB_BYTES, MAX_STAGES);
  if (stages < 2)
    return hole_set_error(HOLE_ERR_UNSUPPORTED, "embedding_dim %d too large for the ranking kernel's smem budget at precision %d",
                          c->dim, precision);
  const int smem_bytes = a_bytes + stages * B_KB_BYTES + 2048;   // + alignment slack + barriers

  if (c->rank == nullptr) c->rank = new hole_rank_ws();
  hole_rank_ws* w = c->rank;
  if ((size_t)Npad * Kall > w->cand_cap) {
    HOLE_CUDA_TRY(cudaStreamSynchronize(st));
    cudaFree(w->cand); w->cand = nullptr; w->cand_cap = 0;
    w->cache_valid = false;
    if (cudaMalloc((void**)&w->cand, (size_t)Npad * Kall * 2) != cudaSuccess) {
      cudaGetLastError();
      return hole_set_error(HOLE_ERR_ALLOC, "ranking candidate operand allocation failed");
    }
    w->cand_cap = (size_t)Npad * Kall;
  }
  if ((size_t)Qpad * Kall > w->q_cap) {
    HOLE_CUDA_TRY(cudaStreamSynchronize(st));
    cudaFree(w->qp); cudaFree(w->true_idx);
    w->qp = nullptr; w->true_idx = nullptr; w->q_cap = 0;
    if (cudaMalloc((void**)&w->qp, (size_t)Qpad * Kall * 2) != cudaSuccess ||
        cudaMalloc((void**)&w->true_idx, (size_t)Qpad * 4) != cudaSuccess) {
      cudaGetLastError();
      return hole_set_error(HOLE_ERR_ALLOC, "ranking query operand allocation failed");
    }
    w->q_cap = (size_t)Qpad * Kall;
  }
  // the gathered true rows serve only the diagonal pass: top-k and neighbour calls do not allocate them
  if (compute_true && (size_t)(Qpad + BN) * Kall > w->tq_cap) {
    HOLE_CUDA_TRY(cudaStreamSynchronize(st));
    cudaFree(w->tq); w->tq = nullptr; w->tq_cap = 0;
    if (cudaMalloc((void**)&w->tq, (size_t)(Qpad + BN) * Kall * 2) != cudaSuccess) {
      cudaGetLastError();
      return hole_set_error(HOLE_ERR_ALLOC, "ranking true-row allocation failed");
    }
    w->tq_cap = (size_t)(Qpad + BN) * Kall;
  }
  RankParams p{};
  p.m_tiles = Qpad / BM;
  if (topk) {
    p.n_tiles = Npad / BN;
    split_chunks(p, c->sm_count);
    const size_t n_keys = (size_t)Qpad * p.n_chunks * 2 * tk->k;
    if ((size_t)Qpad * K > w->qf_cap || n_keys > w->tk_cap) {
      const size_t qf_n = std::max((size_t)Qpad * K, w->qf_cap), tk_n = std::max(n_keys, w->tk_cap);
      HOLE_CUDA_TRY(cudaStreamSynchronize(st));
      cudaFree(w->qf); cudaFree(w->tk_keys);
      w->qf = nullptr; w->tk_keys = nullptr; w->qf_cap = w->tk_cap = 0;
      if (cudaMalloc((void**)&w->qf, qf_n * sizeof(float)) != cudaSuccess ||
          cudaMalloc((void**)&w->tk_keys, tk_n * sizeof(uint64_t)) != cudaSuccess) {
        cudaGetLastError();
        cudaFree(w->qf); w->qf = nullptr;
        return hole_set_error(HOLE_ERR_ALLOC, "top-k workspace allocation failed (%zu candidate keys)", tk_n);
      }
      w->qf_cap = qf_n; w->tk_cap = tk_n;
    }
  }
  if (!w->attr_set) {
    HOLE_CUDA_TRY(cudaFuncSetAttribute(hole_rank_kernel<1, EPI_RANK>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    HOLE_CUDA_TRY(cudaFuncSetAttribute(hole_rank_kernel<2, EPI_RANK>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    HOLE_CUDA_TRY(cudaFuncSetAttribute(hole_rank_kernel<1, EPI_TOPK>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    HOLE_CUDA_TRY(cudaFuncSetAttribute(hole_rank_kernel<2, EPI_TOPK>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    w->attr_set = true;
  }

  w->last_npad = Npad; w->last_K = Kall;
  // operands: the candidate operand is reused when hole_rank_prepare packed exactly this table / range
  const bool cached = !nb && w->cache_valid && w->cache_table == table && w->cache_begin == ent_begin &&
                      w->cache_end == ent_end && w->cache_parts == parts;
  if (!cached) {
    w->cache_valid = false;
    hole_rank_pack_cand_kernel<<<(unsigned)((Npad + 7) / 8), 256, 0, st>>>(table, c->row_stride, c->H, ent_begin, Nc, Npad, K, parts,
                                                                           nb ? 1 : 0, w->cand);
    HOLE_LAUNCHED();
  }
  if (prepare_only) {
    w->cache_table = table; w->cache_begin = ent_begin; w->cache_end = ent_end; w->cache_parts = parts;
    w->cache_valid = true;
    return HOLE_OK;
  }
  w->last_qpad = Qpad;
  if (nb) {
    // cosine does not depend on the score mode: one query packer for both
    hole_neighbors_pack_query_kernel<<<(unsigned)((Qpad + 7) / 8), 256, 0, st>>>(table, c->row_stride, c->H, queries,
                                                                                 (int)Q, Qpad, ent_begin, K, parts,
                                                                                 w->qp, w->true_idx, w->qf);
    HOLE_LAUNCHED();
  } else if (c->score_mode == HOLE_SCORE_CCORR_TANH) {
    // archived score variant: another query vector, the same contraction (see the kernel's comment)
    const int nv = (c->row_stride / 2 + 31) / 32;
    const int warps = std::max(1, std::min(8, (200 * 1024) / (6 * c->H * (int)sizeof(float))));
    const unsigned grid = (unsigned)((Qpad + warps - 1) / warps);
    const size_t smem = (size_t)warps * 6 * c->H * sizeof(float);
#define HOLE_PQC_LAUNCH(N)                                                                                           \
    do {                                                                                                             \
      HOLE_CUDA_TRY(cudaFuncSetAttribute(hole_rank_pack_query_ccorr_kernel<N>,                                       \
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));                 \
      hole_rank_pack_query_ccorr_kernel<N><<<grid, 32 * warps, smem, st>>>(query_table, c->row_stride, c->H, queries, \
                                                                           (int)Q, Qpad, side, ent_begin, K, parts,  \
                                                                           w->qp, w->true_idx, topk ? w->qf : nullptr); \
    } while (0)
    if (nv <= 1) HOLE_PQC_LAUNCH(1);
    else if (nv <= 2) HOLE_PQC_LAUNCH(2);
    else if (nv <= 3) HOLE_PQC_LAUNCH(3);
    else if (nv <= 4) HOLE_PQC_LAUNCH(4);
    else if (nv <= 6) HOLE_PQC_LAUNCH(6);
    else if (nv <= 8) HOLE_PQC_LAUNCH(8);
    else HOLE_PQC_LAUNCH(12);
#undef HOLE_PQC_LAUNCH
    HOLE_LAUNCHED();
  } else {
    const unsigned pq_grid = (unsigned)((Qpad + 7) / 8);
    const size_t pq_smem = (size_t)8 * Kall * 2;
    const int pq_iters = (c->row_stride / 2 + 127) / 128;
#define HOLE_PQ_LAUNCH(N)                                                                                          \
    hole_rank_pack_query_kernel<N><<<pq_grid, 256, pq_smem, st>>>(query_table, c->row_stride, c->H, queries, (int)Q, \
                                                                  Qpad, side, ent_begin, K, parts, w->qp, w->true_idx, \
                                                                  topk ? w->qf : nullptr)
    if (pq_iters == 1) HOLE_PQ_LAUNCH(1);
    else if (pq_iters == 2) HOLE_PQ_LAUNCH(2);
    else if (pq_iters == 3) HOLE_PQ_LAUNCH(3);
    else return hole_set_error(HOLE_ERR_UNSUPPORTED, "embedding_dim %d too large for the ranking query packer", c->dim);
#undef HOLE_PQ_LAUNCH
    HOLE_LAUNCHED();
  }

  CUtensorMap mapA, mapB;
  int rc = make_map(&mapA, w->qp, Qpad, Kall, BM);
  if (rc) return rc;

  p.num_kb = num_kb;
  p.parts = parts;
  p.last_kb_mmas = (c->dim - (num_kb - 1) * BK + UMMA_K - 1) / UMMA_K;
  p.stages = stages;
  p.Q = (int)Q;
  p.Nc = Nc;
  p.true_idx = w->true_idx;

  if (topk) {
    rc = make_map(&mapB, w->cand, Npad, Kall, BN);
    if (rc) return rc;
    p.mode = MODE_COUNT;
    p.topk = tk->k;
    p.tk_keys = w->tk_keys;
    p.f_off = filter_off;
    p.f_ids = filter_ids;
    p.ent_begin = ent_begin;
    p.tk_self = nb ? w->true_idx : nullptr;
    const int grid = std::min(p.m_tiles * p.n_chunks, c->sm_count);
    if (parts == 2) hole_rank_kernel<2, EPI_TOPK><<<grid, RANK_THREADS, smem_bytes, st>>>(mapA, mapB, p);
    else hole_rank_kernel<1, EPI_TOPK><<<grid, RANK_THREADS, smem_bytes, st>>>(mapA, mapB, p);
    HOLE_LAUNCHED();
    hole_topk_merge_kernel<<<(unsigned)Q, MERGE_THREADS, 0, st>>>(w->tk_keys, p.n_chunks * 2, tk->k, table,
                                                                  c->row_stride, c->H, ent_begin, w->qf, K,
                                                                  nb ? 1 : 0, tk->ids_out, tk->scores_out);
    HOLE_LAUNCHED();
    return HOLE_OK;
  }

  if (compute_true) {
    const int rows = Qpad + BN;
    hole_rank_gather_true_kernel<<<(unsigned)((Qpad + 31) / 32), 256, 0, st>>>(w->cand, w->true_idx, Nc, Qpad, Kall, w->tq);
    HOLE_LAUNCHED();
    HOLE_CUDA_TRY(cudaMemsetAsync(w->tq + (size_t)Qpad * Kall, 0, (size_t)BN * Kall * 2, st));
    rc = make_map(&mapB, w->tq, rows, Kall, BN / 2);      // DIAG tiles: the query tile's own 128 true rows
    if (rc) return rc;
    p.mode = MODE_DIAG;
    p.n_tiles = 1; p.chunk_tiles = 1; p.n_chunks = 1;
    p.true_out = true_score_io;
    const int grid = std::min(p.m_tiles, c->sm_count);
    if (parts == 2) hole_rank_kernel<2, EPI_RANK><<<grid, RANK_THREADS, smem_bytes, st>>>(mapA, mapB, p);
    else hole_rank_kernel<1, EPI_RANK><<<grid, RANK_THREADS, smem_bytes, st>>>(mapA, mapB, p);
    HOLE_LAUNCHED();
  }

  if (!count) return HOLE_OK;                      // true scores only (first phase of the sharded ranking)
  rc = make_map(&mapB, w->cand, Npad, Kall, BN);
  if (rc) return rc;
  p.mode = MODE_COUNT;
  p.n_tiles = Npad / BN;
  split_chunks(p, c->sm_count);
  p.true_score = true_score_io;
  p.raw_cnt = raw_before;
  p.filt_cnt = filt_before;
  p.f_off = filter_off;
  p.f_ids = filter_ids;
  p.ent_begin = ent_begin;
  const int grid = std::min(p.m_tiles * p.n_chunks, c->sm_count);
  if (parts == 2) hole_rank_kernel<2, EPI_RANK><<<grid, RANK_THREADS, smem_bytes, st>>>(mapA, mapB, p);
  else hole_rank_kernel<1, EPI_RANK><<<grid, RANK_THREADS, smem_bytes, st>>>(mapA, mapB, p);
  HOLE_LAUNCHED();
  return HOLE_OK;
}

extern "C" int hole_rank(hole_ctx* c, const float* table, int64_t ent_begin, int64_t ent_end,
                         const int32_t* queries, int64_t Q, int side, int precision,
                         const int64_t* filter_off, const int32_t* filter_ids, float* true_score_io,
                         int compute_true, int32_t* raw_before, int32_t* filt_before, void* stream) {
  return rank_impl(c, table, ent_begin, ent_end, nullptr, queries, Q, side, precision, filter_off, filter_ids,
                   true_score_io, compute_true, raw_before, filt_before, stream, false);
}

extern "C" int hole_rank_ex(hole_ctx* c, const float* table, int64_t ent_begin, int64_t ent_end,
                            const float* query_table, const int32_t* queries, int64_t Q, int side, int precision,
                            const int64_t* filter_off, const int32_t* filter_ids, float* true_score_io,
                            int compute_true, int32_t* raw_before, int32_t* filt_before, void* stream) {
  return rank_impl(c, table, ent_begin, ent_end, query_table, queries, Q, side, precision, filter_off, filter_ids,
                   true_score_io, compute_true, raw_before, filt_before, stream, false);
}

extern "C" int hole_topk(hole_ctx* c, const float* table, int64_t ent_begin, int64_t ent_end,
                         const int32_t* queries, int64_t Q, int side, int precision, int k,
                         const int64_t* filter_off, const int32_t* filter_ids,
                         int32_t* ids_out, float* scores_out, void* stream) {
  HOLE_CHECK_ARG(c && k >= 1 && k <= TOPK_MAX && ids_out != nullptr && scores_out != nullptr);
  const TopkArgs tk{k, ids_out, scores_out, false};
  return rank_impl(c, table, ent_begin, ent_end, nullptr, queries, Q, side, precision, filter_off, filter_ids,
                   nullptr, 0, nullptr, nullptr, stream, false, &tk);
}

extern "C" int hole_neighbors(hole_ctx* c, const float* table, int64_t ent_begin, int64_t ent_end,
                              const int32_t* ids, int64_t Q, int precision, int k,
                              const int64_t* filter_off, const int32_t* filter_ids,
                              int32_t* ids_out, float* sim_out, void* stream) {
  HOLE_CHECK_ARG(c && k >= 1 && k <= TOPK_MAX && ids_out != nullptr && sim_out != nullptr);
  const TopkArgs tk{k, ids_out, sim_out, true};
  return rank_impl(c, table, ent_begin, ent_end, nullptr, ids, Q, HOLE_SIDE_TAIL, precision, filter_off, filter_ids,
                   nullptr, 0, nullptr, nullptr, stream, false, &tk);
}

extern "C" int hole_rank_prepare(hole_ctx* c, const float* table, int64_t ent_begin, int64_t ent_end,
                                 int precision, void* stream) {
  return rank_impl(c, table, ent_begin, ent_end, nullptr, nullptr, 0, HOLE_SIDE_TAIL, precision, nullptr, nullptr,
                   nullptr, 0, nullptr, nullptr, stream, true);
}

extern "C" int hole_rank_invalidate(hole_ctx* c) {
  HOLE_CHECK_ARG(c != nullptr);
  hole_rank_cache_invalidate(c);
  return HOLE_OK;
}

extern "C" int hole_rank_debug_operands(hole_ctx* c, void* cand_out, void* query_out, int64_t* n_pad,
                                        int64_t* q_pad, int* K, void* stream) {
  HOLE_CHECK_ARG(c && n_pad && q_pad && K);
  if (c->rank == nullptr || c->rank->last_K == 0)
    return hole_set_error(HOLE_ERR_ARG, "hole_rank has not been called on this context");
  hole_rank_ws* w = c->rank;
  *n_pad = w->last_npad; *q_pad = w->last_qpad; *K = w->last_K;
  HOLE_CUDA_TRY(cudaSetDevice(c->device));
  if (cand_out)
    HOLE_CUDA_TRY(cudaMemcpyAsync(cand_out, w->cand, (size_t)w->last_npad * w->last_K * 2,
                                  cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  if (query_out)
    HOLE_CUDA_TRY(cudaMemcpyAsync(query_out, w->qp, (size_t)w->last_qpad * w->last_K * 2,
                                  cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return HOLE_OK;
}
