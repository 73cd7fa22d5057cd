// HolE training hot path for sm_100a: Philox type-safe corruption (K2), update-plan sort,
// fused gather + norm-clip + Hermitian score + sigmoid + hinge + backward (K1) and the
// deterministic tree-combined sparse SGD update (K3).
//
// Reference seams: corrupt_batch holE.py:97-158 (+ host subsample 343-347),
// get_embedding 161-168, evaluate_triples 179-202, evaluate_batch 222-234,
// GradientDescentOptimizer.minimize 296.  Arithmetic: SURVEY.md App. A/B.
//
// All kernels are HBM/L2-bandwidth bound integer/fp32 work: no tensor cores here.  A row
// is handled by a group of GS lanes, each owning V float4s of the real half and the
// matching V float4s of the imaginary half, so every complex product is lane-local and
// every global access is a coalesced 16-byte vector.
#include <stdarg.h>
#include <string.h>

#include <algorithm>

#include "hole_common.cuh"

thread_local std::string g_hole_err;
thread_local int64_t g_hole_launches = 0;

int hole_set_error(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_hole_err = buf;
  return code;
}

// ---------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------
// Programmatic dependent launch: K1 and K3 of consecutive steps form a dependent chain; each
// is launched with programmatic stream serialization so that its prologue (plan / triple
// loads that do not depend on the table) overlaps the tail of its predecessor, and waits
// here before touching anything the predecessor writes.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <int V>
struct Row {
  float re[4 * V];
  float im[4 * V];
};

__device__ __forceinline__ float4 ld_nc(const float4* p) { return __ldg(p); }
__device__ __forceinline__ float4 ld_cg(const float4* p) { return __ldcg(p); }

template <int GS, int V, bool NC>
__device__ __forceinline__ void row_load(Row<V>& x, const float* base, int lane, int nvec) {
  const float4* p = reinterpret_cast<const float4*>(base);
#pragma unroll
  for (int v = 0; v < V; ++v) {
    int idx = lane + v * GS;
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
    if (idx < nvec) {
      a = NC ? ld_nc(p + idx) : ld_cg(p + idx);
      b = NC ? ld_nc(p + nvec + idx) : ld_cg(p + nvec + idx);
    }
    x.re[4 * v + 0] = a.x; x.re[4 * v + 1] = a.y; x.re[4 * v + 2] = a.z; x.re[4 * v + 3] = a.w;
    x.im[4 * v + 0] = b.x; x.im[4 * v + 1] = b.y; x.im[4 * v + 2] = b.z; x.im[4 * v + 3] = b.w;
  }
}

template <int GS, int V, bool FULL = false>
__device__ __forceinline__ void row_store(const Row<V>& x, float* base, int lane, int nvec) {
  float4* p = reinterpret_cast<float4*>(base);
#pragma unroll
  for (int v = 0; v < V; ++v) {
    int idx = lane + v * GS;
    if (FULL || idx < nvec) {
      p[idx] = make_float4(x.re[4 * v], x.re[4 * v + 1], x.re[4 * v + 2], x.re[4 * v + 3]);
      p[nvec + idx] = make_float4(x.im[4 * v], x.im[4 * v + 1], x.im[4 * v + 2], x.im[4 * v + 3]);
    }
  }
}

template <int GS>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int o = GS / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <int V>
__device__ __forceinline__ float row_sumsq(const Row<V>& x) {
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < 4 * V; ++k) s = fmaf(x.re[k], x.re[k], s);
#pragma unroll
  for (int k = 0; k < 4 * V; ++k) s = fmaf(x.im[k], x.im[k], s);
  return s;
}

template <int V>
__device__ __forceinline__ float row_dot(const Row<V>& x, const Row<V>& y) {
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < 4 * V; ++k) s = fmaf(x.re[k], y.re[k], s);
#pragma unroll
  for (int k = 0; k < 4 * V; ++k) s = fmaf(x.im[k], y.im[k], s);
  return s;
}

// clip_by_norm(row, 1): y = x * min(rsqrt(sum x^2), 1)  (App. B; holE.py:162 max_norm=1).
// Returns inv = rsqrt(sum x^2); the row is "clipped" (gradient takes the rsqrt branch)
// when inv <= 1.
template <int V>
__device__ __forceinline__ void row_clip(Row<V>& x, float inv) {
  float sc = fminf(inv, 1.0f);
#pragma unroll
  for (int k = 0; k < 4 * V; ++k) { x.re[k] *= sc; x.im[k] *= sc; }
}

template <int V>
__device__ __forceinline__ void row_zero(Row<V>& x) {
#pragma unroll
  for (int k = 0; k < 4 * V; ++k) { x.re[k] = 0.f; x.im[k] = 0.f; }
}
template <int V>
__device__ __forceinline__ void row_add(Row<V>& acc, const Row<V>& x) {
#pragma unroll
  for (int k = 0; k < 4 * V; ++k) { acc.re[k] += x.re[k]; acc.im[k] += x.im[k]; }
}

#ifdef HOLE_FAST_SIGMOID   // A/B only: ex2.approx + approximate division (|d sigma| ~ 1e-7)
__device__ __forceinline__ float sigmoidf_precise(float s) { return __fdividef(1.0f, 1.0f + __expf(-s)); }
#else
__device__ __forceinline__ float sigmoidf_precise(float s) { return 1.0f / (1.0f + expf(-s)); }
#endif

// dx = clipped ? (dy - y (y.dy)) * inv : dy      (App. A.3)
template <int V>
__device__ __forceinline__ void clip_backward(Row<V>& dy, const Row<V>& y, float proj, float inv) {
  if (inv <= 1.0f) {
#pragma unroll
    for (int k = 0; k < 4 * V; ++k) {
      dy.re[k] = (dy.re[k] - y.re[k] * proj) * inv;
      dy.im[k] = (dy.im[k] - y.im[k] * proj) * inv;
    }
  }
}

// ---------------------------------------------------------------------------------------
// layout conversion
// ---------------------------------------------------------------------------------------
__global__ void hole_pack_rows_kernel(const float* __restrict__ src, float* __restrict__ dst,
                                      int64_t n, int dim, int H, int Hp) {
  int64_t total = n * 2 * Hp;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total;
       t += (int64_t)gridDim.x * blockDim.x) {
    int64_t row = t / (2 * Hp);
    int c = (int)(t % (2 * Hp));
    int half = c / Hp, k = c % Hp;
    dst[t] = (k < H) ? src[row * dim + half * H + k] : 0.0f;
  }
}

__global__ void hole_unpack_rows_kernel(const float* __restrict__ src, float* __restrict__ dst,
                                        int64_t n, int dim, int H, int Hp) {
  int64_t total = n * dim;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total;
       t += (int64_t)gridDim.x * blockDim.x) {
    int64_t row = t / dim;
    int c = (int)(t % dim);
    int half = c / H, k = c % H;
    dst[t] = src[row * 2 * Hp + half * Hp + k];
  }
}

// ---------------------------------------------------------------------------------------
// K2: corruption sampler + update-plan keys
// ---------------------------------------------------------------------------------------
constexpr uint32_t HOLE_KEY_ABSENT = 0xFFFFFFFFu;   // sorts after every real row id
constexpr uint32_t HOLE_SLOT_UNIQUE = 0xFFFFFFFFu;  // gslot value: row used once in the step

// Stand-alone sampler (hole_corrupt): for step s (grid.y) and triple i,
// neg = csr_ids[off[ty] + draw] with ty the type of the replaced entity.
__global__ void hole_corrupt_kernel(const int32_t* __restrict__ triples, int64_t B, int n_steps,
                                    const int32_t* __restrict__ type_of,
                                    const int64_t* __restrict__ csr_off,
                                    const int32_t* __restrict__ csr_ids, uint64_t seed,
                                    uint64_t first_step, uint64_t index_base,
                                    int32_t* __restrict__ neg_out,
                                    int32_t* __restrict__ side_out) {
  int s = blockIdx.y;
  uint64_t step = first_step + (uint64_t)s;
  int side = hole_side_coin(seed, step);
  if (side_out != nullptr && blockIdx.x == 0 && threadIdx.x == 0) side_out[s] = side;
  const int32_t* tr = triples + (size_t)s * B * 3;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < B;
       i += (int64_t)gridDim.x * blockDim.x) {
    int ent = side ? tr[3 * i] : tr[3 * i + 1];
    int ty = type_of[ent];
    int64_t lo = csr_off[ty];
    uint32_t cnt = (uint32_t)(csr_off[ty + 1] - lo);
    neg_out[(size_t)s * B + i] = csr_ids[lo + hole_entity_draw(seed, step, (uint32_t)(index_base + (uint64_t)i), cnt)];
  }
}

// relation id of every triple: the key of the per-step "group by relation" sort
__global__ void hole_rel_keys_kernel(const int32_t* __restrict__ triples, int64_t B, int64_t tstride,
                                     uint32_t* __restrict__ relkeys) {
  const size_t base = (size_t)blockIdx.y * B;
  const int32_t* tr = triples + (size_t)blockIdx.y * tstride;   // tstride 0: every step shares the batch
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < B;
       i += (int64_t)gridDim.x * blockDim.x)
    relkeys[base + i] = (uint32_t)tr[i * 3 + 2];
}

// For step s and position g of the relation-grouped order: i = perm[g]; draws (or takes) the
// corrupt entity and emits the step's four (row, position) sort keys, position = slot*B + i
// with slots [relation, tail-slot, head-slot, corrupt entity].  K1 gives T consecutive
// positions to one lane group and pre-sums the relation gradient over runs of equal relation
// inside that range, so only the first triple of such a run carries a relation key.
__global__ void hole_plan_keys_kernel(const int32_t* __restrict__ triples, int64_t B, int64_t tstride, int T,
                                      const int32_t* __restrict__ perm,
                                      const int32_t* __restrict__ type_of,
                                      const int64_t* __restrict__ csr_off,
                                      const int32_t* __restrict__ csr_ids, uint64_t seed,
                                      uint64_t first_step, const int32_t* __restrict__ neg_in,
                                      int32_t* __restrict__ neg_out, uint32_t* __restrict__ keys,
                                      uint32_t* __restrict__ seen, uint32_t* __restrict__ dup, int W) {
  const int s = blockIdx.y;
  const uint64_t step = first_step + (uint64_t)s;
  const int side = hole_side_coin(seed, step);
  const int32_t* tr = triples + (size_t)s * tstride;
  const int32_t* pm = perm + (size_t)s * B;
  uint32_t* k = keys + (size_t)s * 4 * B;
  for (int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; g < B;
       g += (int64_t)gridDim.x * blockDim.x) {
    const int i = pm[g];
    const int h = tr[3 * i], t = tr[3 * i + 1], r = tr[3 * i + 2];
    int n;
    if (neg_in != nullptr) {
      n = neg_in[(size_t)s * B + i];
    } else {
      const int ty = type_of[side ? h : t];
      const int64_t lo = csr_off[ty];
      const uint32_t cnt = (uint32_t)(csr_off[ty + 1] - lo);
      n = csr_ids[lo + hole_entity_draw(seed, step, (uint32_t)i, cnt)];
      neg_out[(size_t)s * B + i] = n;
    }
    const bool run_head = (g % T == 0) || (tr[3 * pm[g - 1] + 2] != r);
    k[i] = run_head ? (uint32_t)r : HOLE_KEY_ABSENT;
    k[B + i] = (uint32_t)t;
    k[2 * B + i] = (uint32_t)h;
    k[3 * B + i] = (uint32_t)n;
    // which rows the step uses more than once: a row's second (third, ...) use finds its `seen` bit set
    uint32_t* sn = seen + (size_t)s * W;
    uint32_t* dp = dup + (size_t)s * W;
    auto mark = [&](uint32_t row) {
      const uint32_t m = 1u << (row & 31u);
      if (atomicOr(sn + (row >> 5), m) & m) atomicOr(dp + (row >> 5), m);
    };
    if (run_head) mark((uint32_t)r);
    mark((uint32_t)t);
    mark((uint32_t)h);
    mark((uint32_t)n);
  }
}

// Uses of rows that occur once in the step need no ordering at all (K1 updates them in place): only the
// uses of duplicated rows -- typically ~10 % of the 4B -- go through the sort.  Three small kernels compact
// them stably (in position order): flag + per-block count, per-step scan of the block counts, write.
constexpr int DP_THREADS = 256;
constexpr int DP_ITEMS = 4;
constexpr int DP_TILE = DP_THREADS * DP_ITEMS;

__device__ __forceinline__ bool plan_is_dup(const uint32_t* __restrict__ dp, uint32_t key) {
  return key != HOLE_KEY_ABSENT && ((dp[key >> 5] >> (key & 31u)) & 1u);
}

// gslot[u] = UNIQUE for uses of rows that occur once; blkcnt[s][blk] = duplicated uses in the block's tile
__device__ __forceinline__ void plan_dupscan(int* __restrict__ c, int nblk, int* __restrict__ mdup_s);

__global__ void __launch_bounds__(DP_THREADS)
hole_plan_dupflag_kernel(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ dup, int M, int W,
                         uint32_t* __restrict__ gslot, int* __restrict__ blkcnt, int* __restrict__ mdup,
                         unsigned* __restrict__ done) {
  __shared__ bool s_last;
  const int s = blockIdx.y, nblk = gridDim.x;
  const uint32_t* k = keys + (size_t)s * M;
  const uint32_t* dp = dup + (size_t)s * W;
  int cnt = 0;
#pragma unroll
  for (int i = 0; i < DP_ITEMS; ++i) {
    const int u = blockIdx.x * DP_TILE + i * DP_THREADS + threadIdx.x;
    bool d = false;
    if (u < M) {
      const uint32_t key = k[u];
      d = plan_is_dup(dp, key);
      if (!d && key != HOLE_KEY_ABSENT) gslot[(size_t)s * M + u] = HOLE_SLOT_UNIQUE;
    }
    cnt += __syncthreads_count(d);
  }
  if (threadIdx.x == 0) {
    __stcg(&blkcnt[(size_t)s * (nblk + 1) + blockIdx.x], cnt);
    __threadfence();
    s_last = atomicAdd(done + s, 1u) == (unsigned)nblk - 1u;
  }
  __syncthreads();
  if (!s_last) return;
  // the last block of the step to finish turns the step's block counts into offsets (it used to be a launch
  // of its own: the plan chain is paid per launch)
  if (threadIdx.x == 0) done[s] = 0;
  __threadfence();
  plan_dupscan(blkcnt + (size_t)s * (nblk + 1), nblk, mdup + s);
}

// per step: block counts -> exclusive offsets; the total goes to blkcnt[s][nblk] and mdup[s]
__device__ __forceinline__ void plan_dupscan(int* __restrict__ c, int nblk, int* __restrict__ mdup_s) {
  __shared__ int wsum[8];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int per = (nblk + 255) / 256;
  int tot = 0;
  for (int q = tid * per; q < min(nblk, (tid + 1) * per); ++q) tot += __ldcg(c + q);
  int inc = tot;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int y = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += y;
  }
  if (lane == 31) wsum[w] = inc;
  __syncthreads();
  int base = inc - tot;
  for (int q = 0; q < w; ++q) base += wsum[q];
  for (int q = tid * per; q < min(nblk, (tid + 1) * per); ++q) {
    const int v = __ldcg(c + q);
    c[q] = base;
    base += v;
  }
  if (tid == 255) { c[nblk] = base; *mdup_s = base; }
}

// (key, position) of every duplicated use, in position order
__global__ void __launch_bounds__(DP_THREADS)
hole_plan_compact_kernel(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ dup, int M, int W,
                         const int* __restrict__ blkcnt, uint32_t* __restrict__ ckey, uint32_t* __restrict__ cval) {
  __shared__ int wcnt[DP_THREADS / 32];
  const int s = blockIdx.y, nblk = gridDim.x;
  const uint32_t* k = keys + (size_t)s * M;
  const uint32_t* dp = dup + (size_t)s * W;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int base = blkcnt[(size_t)s * (nblk + 1) + blockIdx.x];
#pragma unroll 1
  for (int i = 0; i < DP_ITEMS; ++i) {
    const int u = blockIdx.x * DP_TILE + i * DP_THREADS + threadIdx.x;
    uint32_t key = HOLE_KEY_ABSENT;
    if (u < M) key = k[u];
    const bool d = u < M && plan_is_dup(dp, key);
    const unsigned bal = __ballot_sync(0xffffffffu, d);
    __syncthreads();                       // wcnt of the previous iteration is consumed
    if (lane == 0) wcnt[w] = __popc(bal);
    __syncthreads();
    int before = 0, all = 0;
#pragma unroll
    for (int q = 0; q < DP_THREADS / 32; ++q) {
      const int c = wcnt[q];
      before += (q < w) ? c : 0;
      all += c;
    }
    if (d) {
      const int dst = base + before + __popc(bal & ((1u << lane) - 1u));
      ckey[(size_t)s * M + dst] = key;
      cval[(size_t)s * M + dst] = (uint32_t)u;
    }
    base += all;
  }
}

// ---------------------------------------------------------------------------------------
// update plan: for every step of a chunk, sort the step's 4B (row, position) pairs by row,
// stably (LSD radix, 8-bit digits), then mark segments.  Integer-only, off the critical
// path (it depends on the triples and the Philox draw, never on the table), so a chunk of
// steps is planned in one batch of launches: grid.y = step, grid.x = tile of the step.
// ---------------------------------------------------------------------------------------
constexpr int ST_THREADS = 256;
constexpr int ST_WARPS = ST_THREADS / 32;
constexpr int ST_SLICE = 512;                    // entries per warp
constexpr int ST_TILE = ST_SLICE * ST_WARPS;     // entries per block

// lanes of the warp whose 8-bit digit equals mine (`ok` lanes only): eight ballots.  (match.any is an order of
// magnitude slower when the 32 digits are all different, and it serialises the warps of an SM: the one-block
// sort kernels spent ~90 % of their time in it -- profiles/r02b_train_full_summary.csv.)
__device__ __forceinline__ uint32_t warp_match_digit(uint32_t d, bool ok) {
  uint32_t peers = __ballot_sync(0xffffffffu, ok);
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const bool bit = (d >> k) & 1u;
    const uint32_t b = __ballot_sync(0xffffffffu, bit);
    peers &= bit ? b : ~b;
  }
  return peers;
}

// per-warp digit histogram of the warp's slice of the tile (wh = this warp's 256 counters)
__device__ __forceinline__ void st_warp_hist(const uint32_t* __restrict__ k, int lo, int hi,
                                             int shift, uint32_t* wh, int lane) {
  for (int j0 = lo; j0 < hi; j0 += 128) {
    uint32_t key[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      int j = j0 + 32 * u + lane;
      key[u] = (j < hi) ? k[j] : 0u;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      int j = j0 + 32 * u + lane;
      bool ok = j < hi;
      uint32_t d = ok ? ((key[u] >> shift) & 255u) : 256u + lane;   // inactive lanes: unique
      uint32_t peers = warp_match_digit(d, ok);
      if (ok && lane == __ffs(peers) - 1) wh[d] += __popc(peers);
      __syncwarp();
    }
  }
}

// One radix pass = two launches.  This one: ghist[(s*256 + digit)*P + p] = number of entries of tile p of
// step s with that digit; the LAST tile block of a step to finish (ticket counter, self-resetting) then
// turns the step's counts into exclusive offsets in (digit-major, tile-minor) order -- the scan that used
// to be a launch of its own.  Only the tiles the step really uses (Ms entries) are scanned: a warp takes
// four digits at a time, its lanes the tiles (coalesced, four independent loads in flight).
__global__ void __launch_bounds__(ST_THREADS)
hole_sort_hist_kernel(const uint32_t* __restrict__ keys, uint32_t* __restrict__ ghist, int M, int P,
                      int shift, const int* __restrict__ mdev, unsigned* __restrict__ done) {
  __shared__ uint32_t wh[ST_WARPS][256];
  __shared__ uint32_t wsum[ST_WARPS];
  __shared__ bool s_last;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int p = blockIdx.x, s = blockIdx.y;
  for (int i = tid; i < ST_WARPS * 256; i += ST_THREADS) (&wh[0][0])[i] = 0;
  __syncthreads();
  const uint32_t* k = keys + (size_t)s * M;               // arrays are M apart, Ms entries of a step are in use
  const int Ms = mdev ? mdev[s] : M;
  const int lo = min(Ms, p * ST_TILE + w * ST_SLICE), hi = min(Ms, lo + ST_SLICE);
  st_warp_hist(k, lo, hi, shift, wh[w], lane);
  __syncthreads();
  uint32_t* gh = ghist + (size_t)s * 256 * P;
  {
    uint32_t tot = 0;
#pragma unroll
    for (int q = 0; q < ST_WARPS; ++q) tot += wh[q][tid];
    gh[(size_t)tid * P + p] = tot;
  }
  __threadfence();
  __syncthreads();
  if (tid == 0) s_last = atomicAdd(done + s, 1u) == (unsigned)P - 1u;
  __syncthreads();
  if (!s_last) return;
  if (tid == 0) done[s] = 0;                              // ready for the next pass
  __threadfence();
  const int Pe = max(1, (Ms + ST_TILE - 1) / ST_TILE);    // tiles that hold entries
  uint32_t* s_tot = &wh[0][0];                            // 256 digit totals (the tile histograms are spent)
  for (int d0 = w * 4; d0 < 256; d0 += ST_WARPS * 4) {
    uint32_t t[4] = {0u, 0u, 0u, 0u};
    for (int q0 = 0; q0 < Pe; q0 += 32) {
      const int q = q0 + lane;
      if (q < Pe) {
#pragma unroll
        for (int u = 0; u < 4; ++u) t[u] += __ldcg(gh + (size_t)(d0 + u) * P + q);
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) t[u] += __shfl_xor_sync(0xffffffffu, t[u], o);
    }
    __syncwarp();
    if (lane < 4) s_tot[d0 + lane] = (lane == 0) ? t[0] : (lane == 1) ? t[1] : (lane == 2) ? t[2] : t[3];
  }
  __syncthreads();
  {
    const uint32_t tot = s_tot[tid];
    uint32_t inc = tot;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      uint32_t y = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += y;
    }
    if (lane == 31) wsum[w] = inc;
    __syncthreads();
    uint32_t base = inc - tot;
    for (int q = 0; q < w; ++q) base += wsum[q];
    s_tot[tid] = base;
  }
  __syncthreads();
  for (int d0 = w * 4; d0 < 256; d0 += ST_WARPS * 4) {
    uint32_t carry[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) carry[u] = s_tot[d0 + u];
    for (int q0 = 0; q0 < Pe; q0 += 32) {
      const int q = q0 + lane;
      uint32_t c[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) c[u] = (q < Pe) ? __ldcg(gh + (size_t)(d0 + u) * P + q) : 0u;
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        uint32_t inc = c[u];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          uint32_t y = __shfl_up_sync(0xffffffffu, inc, o);
          if (lane >= o) inc += y;
        }
        if (q < Pe) gh[(size_t)(d0 + u) * P + q] = carry[u] + inc - c[u];
        carry[u] += __shfl_sync(0xffffffffu, inc, 31);
      }
    }
  }
}

// stable scatter of one tile; vals_in == nullptr means "value = index" (first pass)
__global__ void __launch_bounds__(ST_THREADS)
hole_sort_scatter_kernel(const uint32_t* __restrict__ keys_in, const uint32_t* __restrict__ vals_in,
                         uint32_t* __restrict__ keys_out, uint32_t* __restrict__ vals_out,
                         const uint32_t* __restrict__ ghist, int M, int P, int shift,
                         const int* __restrict__ mdev) {
  __shared__ uint32_t wh[ST_WARPS][256];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int p = blockIdx.x, s = blockIdx.y;
  for (int i = tid; i < ST_WARPS * 256; i += ST_THREADS) (&wh[0][0])[i] = 0;
  __syncthreads();
  const size_t base = (size_t)s * M;
  const uint32_t* k = keys_in + base;
  const uint32_t* v = vals_in ? vals_in + base : nullptr;
  uint32_t* ko = keys_out + base;
  uint32_t* vo = vals_out + base;
  const int Ms = mdev ? mdev[s] : M;
  if (p * ST_TILE >= Ms) return;             // (block-uniform) nothing of this step in my tile
  const int lo = min(Ms, p * ST_TILE + w * ST_SLICE), hi = min(Ms, lo + ST_SLICE);
  st_warp_hist(k, lo, hi, shift, wh[w], lane);
  __syncthreads();
  {   // per digit: exclusive scan over the warps of this tile, on top of the global offset
    uint32_t run = ghist[((size_t)s * 256 + tid) * P + p];
#pragma unroll
    for (int q = 0; q < ST_WARPS; ++q) {
      uint32_t c = wh[q][tid];
      wh[q][tid] = run;
      run += c;
    }
  }
  __syncthreads();
  uint32_t* myh = wh[w];
  for (int j0 = lo; j0 < hi; j0 += 128) {
    uint32_t key[4], val[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      int j = j0 + 32 * u + lane;
      key[u] = (j < hi) ? k[j] : 0u;
      val[u] = (j < hi) ? (v ? v[j] : (uint32_t)j) : 0u;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      int j = j0 + 32 * u + lane;
      bool ok = j < hi;
      uint32_t d = ok ? ((key[u] >> shift) & 255u) : 256u + lane;
      uint32_t peers = warp_match_digit(d, ok);
      uint32_t rank = __popc(peers & ((1u << lane) - 1u));
      if (ok) {
        uint32_t dst = myh[d] + rank;
        ko[dst] = key[u];
        vo[dst] = val[u];
      }
      __syncwarp();
      if (ok && lane == __ffs(peers) - 1) myh[d] += __popc(peers);
      __syncwarp();
    }
  }
}

// Segments of the sorted duplicated uses.  gslot[original position] = the sorted index of that use = the
// row of G its gradient goes to (so K3 reads the gradients of one table row from consecutive G rows);
// uses of rows that occur exactly once were marked HOLE_SLOT_UNIQUE by hole_plan_dupflag_kernel (such
// rows are updated in place by K1; nobody else reads them during the step).
// For rows that occur n >= 2 times, every sorted entry that heads a chunk of C occurrences
// is appended to the step's compact work list heads[] = {sorted index, segment start, n, row}
// (list order is irrelevant: each entry is an independent leaf of the combine tree).
__global__ void __launch_bounds__(256)
hole_plan_segments_kernel(const uint32_t* __restrict__ skey, const uint32_t* __restrict__ spos,
                          uint32_t* __restrict__ gslot, uint4* __restrict__ heads,
                          int* __restrict__ nheads, int Mcap, const int* __restrict__ mdev, int heads_cap) {
  constexpr int C = HOLE_TREE_C;
  const size_t base = (size_t)blockIdx.y * Mcap;
  const uint32_t* k = skey + base;
  const int M = mdev[blockIdx.y];              // the step's duplicated uses, sorted by (row, position)
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < M; j += gridDim.x * blockDim.x) {
    const uint32_t key = k[j];
    const bool head = (j == 0) || (k[j - 1] != key);
    const bool last = (j == M - 1) || (k[j + 1] != key);
    gslot[base + spos[base + j]] = (uint32_t)j;
    if (head && last) continue;                // (cannot happen: every listed row occurs at least twice)
    // segment [s, e) of this row.  Most duplicated rows are used two or three times: look at the
    // neighbours first, and only search (binary, over the whole step) when the run is longer than that.
    int s = j;
    if (!head) {
      if (j < 2 || k[j - 2] != key) s = j - 1;
      else if (j < 3 || k[j - 3] != key) s = j - 2;
      else {              // lower_bound(key) in [0, j - 3)
        int lo = 0, hi = j - 3;
        while (lo < hi) {
          int mid = (lo + hi) >> 1;
          if (k[mid] < key) lo = mid + 1; else hi = mid;
        }
        s = lo;
      }
    }
    if ((j - s) % C != 0) continue;
    int e = j + 1;
    if (!last) {
      if (j + 2 >= M || k[j + 2] != key) e = j + 2;
      else if (j + 3 >= M || k[j + 3] != key) e = j + 3;
      else {              // upper_bound(key) in (j + 3, M)
        int lo = j + 4, hi = M;
        while (lo < hi) {
          int mid = (lo + hi) >> 1;
          if (k[mid] <= key) lo = mid + 1; else hi = mid;
        }
        e = lo;
      }
    }
    const int slot = atomicAdd(&nheads[blockIdx.y], 1);
    heads[(size_t)blockIdx.y * heads_cap + slot] = make_uint4((uint32_t)j, (uint32_t)s, (uint32_t)(e - s), key);
  }
}

// ---------------------------------------------------------------------------------------
// The row sort + segments of a step in ONE launch, one block per step: the same stable LSD passes as
// hole_sort_{hist,scatter}_kernel and the same segment rules as hole_plan_segments_kernel (identical
// output), with the (key, position) pairs in shared memory when the step has at most SS_CAP duplicated
// uses (a typical step of a large table: ~7 % of the 4B uses) and in the global ping-pong buffers
// otherwise (correct but slow: the host only takes this path while the steps it has seen were small).
// Replaces 2 * passes + 1 dependent launches of the plan chain, whose length -- not its work -- is what
// a training call waits for before its first step.
// ---------------------------------------------------------------------------------------
// The per-step "group the triples by relation" sort in ONE launch (it used to be hole_rel_keys_kernel + one
// histogram / scatter pair per pass): one block per step, the B relation ids in shared memory, stable LSD
// passes as in hole_plan_sortseg_small_kernel.  One pass (relation ids < 256) scatters the triple indices
// straight into perm; a second pass goes through a 16-bit index array.  The host takes this kernel when the
// step fits (plan_relsort_smem), else the radix chain.
constexpr int RS_THREADS = 1024;
constexpr int RS_WARPS = RS_THREADS / 32;
constexpr int RS_SMEM_MAX = 227 * 1024 - 1024;   // dynamic + the kernel's static shared memory <= 227 KB

static size_t plan_relsort_smem(int64_t B, int passes) {      // 0: does not fit
  if (passes < 1 || passes > 2 || B > 65536) return 0;
  const size_t need = (size_t)RS_WARPS * 256 * 4 + (size_t)B * 4 + (passes == 2 ? (size_t)B * 2 : 0);
  return need <= (size_t)RS_SMEM_MAX ? need : 0;
}

__global__ void __launch_bounds__(RS_THREADS)
hole_plan_relsort_kernel(const int32_t* __restrict__ triples, int B, int64_t tstride, int passes,
                         int32_t* __restrict__ perm) {
  extern __shared__ uint32_t rs_smem[];
  __shared__ uint32_t s_wsum[RS_WARPS];
  uint32_t (*wh)[256] = reinterpret_cast<uint32_t (*)[256]>(rs_smem);
  uint32_t* keys = rs_smem + RS_WARPS * 256;
  uint16_t* p0 = reinterpret_cast<uint16_t*>(keys + B);           // order after the first of two passes
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int32_t* tr = triples + (size_t)blockIdx.x * tstride;
  int32_t* pm = perm + (size_t)blockIdx.x * B;
  for (int j = tid; j < B; j += RS_THREADS) keys[j] = (uint32_t)tr[3 * (size_t)j + 2];
  const int L = ((B + RS_WARPS - 1) / RS_WARPS + 31) & ~31;       // entries per warp
  const int lo = min(B, w * L), hi = min(B, lo + L);
  for (int pass = 0; pass < passes; ++pass) {
    const int shift = 8 * pass;
    const bool first = pass == 0, last = pass == passes - 1;
    for (int i = tid; i < RS_WARPS * 256; i += RS_THREADS) (&wh[0][0])[i] = 0;
    __syncthreads();
    for (int j0 = lo; j0 < hi; j0 += 32) {
      const int j = j0 + lane;
      const bool ok = j < hi;
      const uint32_t d = ok ? ((keys[first ? j : (int)p0[j]] >> shift) & 255u) : 256u + lane;
      const uint32_t peers = warp_match_digit(d, ok);
      if (ok && lane == __ffs(peers) - 1) wh[w][d] += __popc(peers);
      __syncwarp();
    }
    __syncthreads();
    {   // exclusive scan in (digit-major, warp-minor) order: thread t takes digit t/4, warps 8*(t%4) .. +8
      const int d = tid >> 2, w0 = (tid & 3) * 8;
      uint32_t cnt[8], tot = 0;
#pragma unroll
      for (int q = 0; q < 8; ++q) { cnt[q] = wh[w0 + q][d]; tot += cnt[q]; }
      uint32_t inc = tot;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += y;
      }
      if (lane == 31) s_wsum[w] = inc;
      __syncthreads();
      uint32_t run = inc - tot;
      for (int q = 0; q < w; ++q) run += s_wsum[q];
#pragma unroll
      for (int q = 0; q < 8; ++q) { wh[w0 + q][d] = run; run += cnt[q]; }
    }
    __syncthreads();
    uint32_t* myh = wh[w];
    // two passes: the second reads p0 in order while it ... writes perm (global), so p0 is not overwritten
    for (int j0 = lo; j0 < hi; j0 += 32) {
      const int j = j0 + lane;
      const bool ok = j < hi;
      const int idx = ok ? (first ? j : (int)p0[j]) : 0;
      const uint32_t d = ok ? ((keys[idx] >> shift) & 255u) : 256u + lane;
      const uint32_t peers = warp_match_digit(d, ok);
      const uint32_t rank = __popc(peers & ((1u << lane) - 1u));
      if (ok) {
        const uint32_t dst = myh[d] + rank;
        if (last) pm[dst] = idx; else p0[dst] = (uint16_t)idx;
      }
      __syncwarp();
      if (ok && lane == __ffs(peers) - 1) myh[d] += __popc(peers);
      __syncwarp();
    }
    __syncthreads();
  }
}

// The same sort when the caller has promised few relations (hole_ctx_set_relations, R <= RF_MAX_REL -- 14 in the
// Diffbot-shaped config): a counting sort with one counter per (relation, thread).  Thread t owns P consecutive
// triples; it counts them per relation, the counters are scanned in (relation-major, thread-minor) order, and the
// thread walks its triples again handing out destinations -- stable, no warp votes, ~10x fewer instructions than
// the digit passes above (32 us -> a few us for B = 32768).  Relation ids >= R (a broken promise) are clamped:
// they sort with relation R - 1 instead of corrupting shared memory.
constexpr int RF_THREADS = 1024;
constexpr int RF_MAX_REL = 64;

static int plan_relsort_few_stride(int64_t B) {      // bytes per thread of the staged ids: P rounded up, an odd number of words
  const int P = (int)((B + RF_THREADS - 1) / RF_THREADS);
  int words = (P + 3) / 4 + 1;
  if ((words & 1) == 0) ++words;
  return 4 * words;
}
static size_t plan_relsort_few_smem(int64_t B, int64_t R) {      // 0: not applicable
  if (R < 1 || R > RF_MAX_REL || B < 1 || B > 65535) return 0;
  const size_t need = (size_t)R * RF_THREADS * 2 + (size_t)RF_THREADS * plan_relsort_few_stride(B);
  return need <= (size_t)RS_SMEM_MAX ? need : 0;
}

__global__ void __launch_bounds__(RF_THREADS)
hole_plan_relsort_few_kernel(const int32_t* __restrict__ triples, int B, int64_t tstride, int R, int stride_bytes,
                             int32_t* __restrict__ perm) {
  extern __shared__ uint32_t rf_smem[];
  __shared__ uint32_t s_wsum[RF_THREADS / 32];
  uint16_t* cnt = reinterpret_cast<uint16_t*>(rf_smem);                       // [R][RF_THREADS]
  uint8_t* ids = reinterpret_cast<uint8_t*>(rf_smem) + (size_t)R * RF_THREADS * 2;   // [RF_THREADS][stride_bytes]
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int32_t* tr = triples + (size_t)blockIdx.x * tstride;
  int32_t* pm = perm + (size_t)blockIdx.x * B;
  const int P = (B + RF_THREADS - 1) / RF_THREADS;
  for (int i = tid; i < R * RF_THREADS / 2; i += RF_THREADS) rf_smem[i] = 0u;
  for (int j = tid; j < B; j += RF_THREADS) {
    const int t = j / P;
    ids[(size_t)t * stride_bytes + (j - t * P)] = (uint8_t)min(tr[3 * (size_t)j + 2], R - 1);
  }
  __syncthreads();
  const int j_lo = tid * P, j_hi = min(B, j_lo + P);
  const uint8_t* mine = ids + (size_t)tid * stride_bytes;
  for (int j = j_lo; j < j_hi; ++j) ++cnt[(int)mine[j - j_lo] * RF_THREADS + tid];
  __syncthreads();
  {   // exclusive scan of the R * RF_THREADS counters as they lie (relation-major): thread t takes R in a row
    uint16_t* c = cnt + (size_t)tid * R;
    uint32_t tot = 0;
    for (int q = 0; q < R; ++q) tot += c[q];
    uint32_t inc = tot;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t y = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += y;
    }
    if (lane == 31) s_wsum[w] = inc;
    __syncthreads();
    uint32_t run = inc - tot;
    for (int q = 0; q < w; ++q) run += s_wsum[q];
    for (int q = 0; q < R; ++q) {
      const uint32_t v = c[q];
      c[q] = (uint16_t)run;
      run += v;
    }
  }
  __syncthreads();
  for (int j = j_lo; j < j_hi; ++j) {
    uint16_t* slot = cnt + (int)mine[j - j_lo] * RF_THREADS + tid;
    pm[*slot] = j;
    ++*slot;
  }
}

// max over the plan's steps of their duplicated-use count -> the plan slot's word in mapped host memory
__global__ void hole_plan_dupmax_kernel(const int* __restrict__ mdup, int S, int* __restrict__ out_host) {
  int m = 0;
  for (int s = threadIdx.x; s < S; s += blockDim.x) m = max(m, mdup[s]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  __shared__ int sm[8];
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int q = 1; q < (int)(blockDim.x >> 5); ++q) m = max(m, sm[q]);
    *reinterpret_cast<volatile int*>(out_host) = m;
    __threadfence_system();
  }
}

constexpr int SS_THREADS = 1024;
constexpr int SS_WARPS = SS_THREADS / 32;
constexpr int SS_CAP = 11264;                      // 4 arrays x 4 B x SS_CAP + 32 KB of histograms < 227 KB
constexpr int SS_SMEM = (SS_WARPS * 256 + 4 * SS_CAP) * 4;

__global__ void __launch_bounds__(SS_THREADS)
hole_plan_sortseg_small_kernel(uint32_t* ck, uint32_t* cv, uint32_t* ak, uint32_t* av, uint32_t* skey_out,
                               uint32_t* spos_out, uint32_t* __restrict__ gslot,
                               uint4* __restrict__ heads, int* __restrict__ nheads, int Mcap,
                               const int* __restrict__ mdev, int heads_cap, int passes) {
  extern __shared__ uint32_t ss_smem[];
  __shared__ uint32_t s_wsum[SS_WARPS];
  __shared__ int s_nh;
  constexpr int C = HOLE_TREE_C;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int step = blockIdx.x;
  const int n = mdev[step];
  const size_t base = (size_t)step * Mcap;
  if (tid == 0) s_nh = 0;
  if (n <= 0) { if (tid == 0 && nheads != nullptr) nheads[step] = 0; return; }   // (n < 0: the load-the-module launch)
  uint32_t (*wh)[256] = reinterpret_cast<uint32_t (*)[256]>(ss_smem);
  const bool small = n <= SS_CAP;
  uint32_t *kin, *vin, *kout, *vout;
  if (small) {
    kin = ss_smem + SS_WARPS * 256; vin = kin + SS_CAP; kout = vin + SS_CAP; vout = kout + SS_CAP;
    for (int j0 = tid; j0 < n; j0 += 4 * SS_THREADS) {          // (loads first: the pointers may alias)
      uint32_t a[4], b[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = j0 + u * SS_THREADS;
        a[u] = j < n ? __ldcg(ck + base + j) : 0u;
        b[u] = j < n ? __ldcg(cv + base + j) : 0u;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = j0 + u * SS_THREADS;
        if (j < n) { kin[j] = a[u]; vin[j] = b[u]; }
      }
    }
  } else {
    kin = ck + base; vin = cv + base; kout = ak + base; vout = av + base;
  }
  const int L = ((n + SS_WARPS - 1) / SS_WARPS + 31) & ~31;      // entries per warp
  const int lo = min(n, w * L), hi = min(n, lo + L);
  for (int pass = 0; pass < passes; ++pass) {
    const int shift = 8 * pass;
    for (int i = tid; i < SS_WARPS * 256; i += SS_THREADS) (&wh[0][0])[i] = 0;
    __syncthreads();                                             // (also: the previous pass's scatter is complete)
    for (int j0 = lo; j0 < hi; j0 += 32) {                       // (plain loads: this kernel wrote kin itself)
      const int j = j0 + lane;
      const bool ok = j < hi;
      const uint32_t d = ok ? ((kin[j] >> shift) & 255u) : 256u + lane;
      const uint32_t peers = warp_match_digit(d, ok);
      if (ok && lane == __ffs(peers) - 1) wh[w][d] += __popc(peers);
      __syncwarp();
    }
    __syncthreads();
    {   // exclusive scan in (digit-major, warp-minor) order: thread t takes digit t/4, warps 8*(t%4) .. +8
      const int d = tid >> 2, w0 = (tid & 3) * 8;
      uint32_t cnt[8], tot = 0;
#pragma unroll
      for (int q = 0; q < 8; ++q) { cnt[q] = wh[w0 + q][d]; tot += cnt[q]; }
      uint32_t inc = tot;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += y;
      }
      if (lane == 31) s_wsum[w] = inc;
      __syncthreads();
      uint32_t run = inc - tot;
      for (int q = 0; q < w; ++q) run += s_wsum[q];
#pragma unroll
      for (int q = 0; q < 8; ++q) { wh[w0 + q][d] = run; run += cnt[q]; }
    }
    __syncthreads();
    uint32_t* myh = wh[w];
    for (int j0 = lo; j0 < hi; j0 += 32) {                       // stable scatter of the warp's slice
      const int j = j0 + lane;
      const bool ok = j < hi;
      const uint32_t key = ok ? kin[j] : 0u, val = ok ? vin[j] : 0u;
      const uint32_t d = ok ? ((key >> shift) & 255u) : 256u + lane;
      const uint32_t peers = warp_match_digit(d, ok);
      const uint32_t rank = __popc(peers & ((1u << lane) - 1u));
      if (ok) {
        const uint32_t dst = myh[d] + rank;
        kout[dst] = key;
        vout[dst] = val;
      }
      __syncwarp();
      if (ok && lane == __ffs(peers) - 1) myh[d] += __popc(peers);
      __syncwarp();
    }
    __syncthreads();
    uint32_t* t = kin; kin = kout; kout = t;
    t = vin; vin = vout; vout = t;
  }
  // kin / vin: the step's duplicated uses sorted by (row, position).  Consumers read them from skey_out / spos_out.
  uint32_t* so = skey_out + base;
  uint32_t* po = spos_out + base;
  if (kin != so)
    for (int j = tid; j < n; j += SS_THREADS) { so[j] = kin[j]; po[j] = vin[j]; }
  // segments (hole_plan_segments_kernel's rules)
  const uint32_t* k = kin;
  for (int j = tid; j < n; j += SS_THREADS) {
    const uint32_t key = k[j];
    const bool head = (j == 0) || (k[j - 1] != key);
    const bool last = (j == n - 1) || (k[j + 1] != key);
    gslot[base + vin[j]] = (uint32_t)j;
    if (head && last) continue;
    int sg = j;
    if (!head) {
      if (j < 2 || k[j - 2] != key) sg = j - 1;
      else if (j < 3 || k[j - 3] != key) sg = j - 2;
      else {
        int a = 0, b = j - 3;
        while (a < b) {
          const int mid = (a + b) >> 1;
          if (k[mid] < key) a = mid + 1; else b = mid;
        }
        sg = a;
      }
    }
    if ((j - sg) % C != 0) continue;
    int e = j + 1;
    if (!last) {
      if (j + 2 >= n || k[j + 2] != key) e = j + 2;
      else if (j + 3 >= n || k[j + 3] != key) e = j + 3;
      else {
        int a = j + 4, b = n;
        while (a < b) {
          const int mid = (a + b) >> 1;
          if (k[mid] <= key) a = mid + 1; else b = mid;
        }
        e = a;
      }
    }
    const int slot = atomicAdd(&s_nh, 1);
    heads[(size_t)step * heads_cap + slot] = make_uint4((uint32_t)j, (uint32_t)sg, (uint32_t)(e - sg), key);
  }
  __syncthreads();
  if (tid == 0) nheads[step] = s_nh;
}

// ---------------------------------------------------------------------------------------
// forward only: sigma(score)  (evaluate_triples, holE.py:179-202)
// ---------------------------------------------------------------------------------------
template <int GS, int V>
__global__ void __launch_bounds__(256)
hole_score_kernel(const float* __restrict__ E, const int32_t* __restrict__ triples, int64_t B,
                  int nvec, int stride, float* __restrict__ out) {
  const int lane = threadIdx.x % GS;
  int64_t g = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / GS;
  const bool valid = g < B;
  const int64_t i = valid ? g : B - 1;
  const int h = triples[3 * i], t = triples[3 * i + 1], r = triples[3 * i + 2];
  Row<V> xh, xt, xr;
  row_load<GS, V, true>(xh, E + (size_t)h * stride, lane, nvec);
  row_load<GS, V, true>(xt, E + (size_t)t * stride, lane, nvec);
  row_load<GS, V, true>(xr, E + (size_t)r * stride, lane, nvec);
  float ih = __frsqrt_rn(group_sum<GS>(row_sumsq(xh)));
  float it = __frsqrt_rn(group_sum<GS>(row_sumsq(xt)));
  float ir = __frsqrt_rn(group_sum<GS>(row_sumsq(xr)));
  row_clip(xh, ih); row_clip(xt, it); row_clip(xr, ir);
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < 4 * V; ++k) {
    float a = xh.re[k], b = xh.im[k], c = xr.re[k], d = xr.im[k], e = xt.re[k], f = xt.im[k];
    s += (a * c - b * d) * e + (a * d + b * c) * f;
  }
  s = group_sum<GS>(s);
  if (valid && lane == 0) out[i] = sigmoidf_precise(s);
}

// ---------------------------------------------------------------------------------------
// K3: deterministic sparse SGD (or AdaGrad) update for rows that occur more than once in the step.
// One group per sorted entry; only entries that head a chunk of C consecutive occurrences
// of a row do work.  A row with n occurrences is reduced by a fixed C-ary tree over its
// sorted occurrences (order: slot, then batch index); the last group to finish a node's
// children combines them in child order, so the result does not depend on scheduling.
// Partials reuse the (already consumed) staged gradient row of a node's first occurrence.
// ---------------------------------------------------------------------------------------

// acc = sum over q < cnt (<= C) of the staged rows G[first + q*step], in q order, NB row
// loads in flight at a time.
template <int GS, int V>
__device__ __forceinline__ void sum_rows(Row<V>& acc, const float* __restrict__ G, int64_t first,
                                         int64_t step, int cnt, int stride, int lane, int nvec) {
  constexpr int C = HOLE_TREE_C;
  constexpr int NB = (V == 1) ? 8 : 4;
  row_zero(acc);
#pragma unroll
  for (int q0 = 0; q0 < C; q0 += NB) {
    if (q0 >= cnt) break;          // group-uniform
    Row<V> x[NB];
#pragma unroll
    for (int u = 0; u < NB; ++u) {
      const int q = q0 + u;
      if (q < cnt) row_load<GS, V, false>(x[u], G + (size_t)(first + q * step) * stride, lane, nvec);
      else row_zero(x[u]);
    }
#pragma unroll
    for (int u = 0; u < NB; ++u) row_add(acc, x[u]);
  }
}

// row-sharded step (hole_shard_step): a row's change goes to my slice of its owner's staging buffer
struct hole_k3_shard {
  const int32_t* cuts;      // [world+1] first request-list slot per owner
  int R, me, world;         // world == 0: not sharded
  long long cap;
  hole_peer_ptrs stage;     // PEER: rank o's delta staging [world][cap][stride]
};

// ADA: the root applies the AdaGrad update with the accumulator S (hole_ctx_set_optimizer) instead of SGD
template <int GS, int V, bool ADA>
__device__ __forceinline__ void hole_apply_body(float* __restrict__ E, float* __restrict__ G,
                                                const uint4* __restrict__ heads, const int* __restrict__ nheads,
                                                int* __restrict__ counters, int M, int nvec, int stride, float lr,
                                                float* __restrict__ Dtab, int flags, const hole_k3_shard& sh,
                                                float* __restrict__ S) {
  constexpr int C = HOLE_TREE_C;
  const int lane = threadIdx.x % GS;
  const int gbase = (threadIdx.x % 32) / GS * GS;
  const unsigned gmask = (GS == 32) ? 0xffffffffu : (((1u << GS) - 1u) << gbase);
  // persistent: a fixed grid strides over the step's work list (its length is only known on
  // the device)
  const int nh = *nheads;
  pdl_launch_dependents();    // the next step's K1 may run its (table-independent) prologue
  pdl_wait();                 // K1 of this step has staged every gradient row
  const int64_t gstride = ((int64_t)gridDim.x * blockDim.x) / GS;
  for (int64_t g = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / GS; g < nh; g += gstride) {
    const uint4 hd = heads[g];
    const int j = (int)hd.x, s = (int)hd.y, n = (int)hd.z, row = (int)hd.w;
    const int rel = j - s;
    const int cnt = min(C, n - rel);
    float* erow = E + (size_t)row * stride;
    Row<V> acc, x, s2;
    const bool delta = Dtab != nullptr;   // delta mode: write -lr * sum into Dtab, leave E alone
    const bool single = n <= C && !delta; // this leaf is also the root: fetch the table row alongside
    if (single) row_load<GS, V, false>(x, erow, lane, nvec);
    if constexpr (ADA) { if (single) row_load<GS, V, false>(s2, S + (size_t)row * stride, lane, nvec); }
    sum_rows<GS, V>(acc, G, j, 1, cnt, stride, lane, nvec);
    int level = 0, idx = rel / C, nl = (n + C - 1) / C;
    int64_t span = C;   // sorted entries covered by one node of this level
    while (true) {
      if (nl == 1) {    // root: apply   E[row] -= lr * acc   (holE.py:296)
        if (delta) {
#pragma unroll
          for (int k = 0; k < 4 * V; ++k) { x.re[k] = -lr * acc.re[k]; x.im[k] = -lr * acc.im[k]; }
          float* drow = Dtab + (size_t)row * stride;
          if (sh.world > 0 && row >= sh.R) {     // entity row of a sharded step: the owner's staging buffer
            const int slot = row - sh.R;
            int o = 0;
            while (slot >= sh.cuts[o + 1]) ++o;
            drow = static_cast<float*>(sh.stage.p[o]) +
                   ((size_t)sh.me * (size_t)sh.cap + (size_t)(slot - sh.cuts[o])) * stride;
          }
          if (flags & HOLE_K1_ACCUMULATE) {
            Row<V> o;
            row_load<GS, V, false>(o, drow, lane, nvec);
            row_add(x, o);
          }
          row_store<GS, V>(x, drow, lane, nvec);
          break;
        }
        if (!single) row_load<GS, V, false>(x, erow, lane, nvec);
        if constexpr (ADA) {    // S[row] += acc^2;  E[row] -= lr * acc * rsqrt(S[row])  (SparseApplyAdagrad)
          if (!single) row_load<GS, V, false>(s2, S + (size_t)row * stride, lane, nvec);
#pragma unroll
          for (int k = 0; k < 4 * V; ++k) {
            s2.re[k] = fmaf(acc.re[k], acc.re[k], s2.re[k]);
            s2.im[k] = fmaf(acc.im[k], acc.im[k], s2.im[k]);
            x.re[k] = fmaf(-lr * acc.re[k], __frsqrt_rn(s2.re[k]), x.re[k]);
            x.im[k] = fmaf(-lr * acc.im[k], __frsqrt_rn(s2.im[k]), x.im[k]);
          }
          row_store<GS, V>(s2, S + (size_t)row * stride, lane, nvec);
        } else {
#pragma unroll
          for (int k = 0; k < 4 * V; ++k) {
            x.re[k] -= lr * acc.re[k];
            x.im[k] -= lr * acc.im[k];
          }
        }
        row_store<GS, V>(x, erow, lane, nvec);
        break;
      }
      // partial of node (level, idx) overwrites the (consumed) first gradient row of the node
      row_store<GS, V>(acc, G + (size_t)(s + idx * span) * stride, lane, nvec);
      __threadfence();
      __syncwarp(gmask);
      const int parent = idx / C;
      const int nchild = min(C, nl - parent * C);
      int* ctr = counters + (size_t)level * M + (s + parent * span * C);
      int ticket = 0;
      if (lane == 0) ticket = atomicAdd(ctr, 1);
      ticket = __shfl_sync(gmask, ticket, gbase);
      if (ticket != nchild - 1) break;
      if (lane == 0) *ctr = 0;          // self-reset for the next step
      __threadfence();
      sum_rows<GS, V>(acc, G, s + (parent * (int64_t)C) * span, span, nchild, stride, lane, nvec);
      ++level;
      idx = parent;
      nl = (nl + C - 1) / C;
      span *= C;
    }
  }
  if (sh.world > 0) __threadfence_system();   // delta rows stored to peer memory: see hole_k1_body
}

template <int GS, int V>
__global__ void __launch_bounds__(256)
hole_apply_kernel(float* __restrict__ E, float* __restrict__ G, const uint4* __restrict__ heads,
                  const int* __restrict__ nheads, int* __restrict__ counters, int M, int nvec,
                  int stride, float lr, float* __restrict__ Dtab, int flags, const hole_k3_shard sh) {
  hole_apply_body<GS, V, false>(E, G, heads, nheads, counters, M, nvec, stride, lr, Dtab, flags, sh, nullptr);
}

// K3 of an AdaGrad step: in place on the table E and the accumulator S
template <int GS, int V>
__global__ void __launch_bounds__(256)
hole_adagrad_apply_kernel(float* __restrict__ E, float* __restrict__ G, const uint4* __restrict__ heads,
                          const int* __restrict__ nheads, int* __restrict__ counters, int M, int nvec,
                          int stride, float lr, float* __restrict__ S) {
  const hole_k3_shard sh = {};
  hole_apply_body<GS, V, true>(E, G, heads, nheads, counters, M, nvec, stride, lr, nullptr, 0, sh, S);
}

// ---------------------------------------------------------------------------------------
#include "hole_k1.cuh"
#include "hole_ccorr.cuh"

// table[ids[k]] += rows[k] for UNIQUE ids (multi-GPU: the owner applies one source rank's
// row deltas; ranks are applied one after the other, so the sum order is fixed)
template <int GS, int V>
__global__ void __launch_bounds__(256)
hole_add_rows_kernel(float* __restrict__ E, const int64_t* __restrict__ ids, const float* __restrict__ rows,
                     int64_t n, int64_t id_offset, int nvec, int stride) {
  const int lane = threadIdx.x % GS;
  const int64_t k = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / GS;
  if (k >= n) return;
  float* erow = E + (size_t)(ids[k] + id_offset) * stride;
  Row<V> x, d;
  row_load<GS, V, false>(x, erow, lane, nvec);
  row_load<GS, V, false>(d, rows + (size_t)k * stride, lane, nvec);   // may be peer memory
  row_add(x, d);
  row_store<GS, V>(x, erow, lane, nvec);
}

// dst[k] = table[ids[k] + id_offset] (multi-GPU: the owner pushes the rows a peer asked for
// straight into that peer's step table over NVLink -- dst may be peer memory)
template <int GS, int V>
__global__ void __launch_bounds__(256)
hole_gather_rows_kernel(const float* __restrict__ E, const int64_t* __restrict__ ids, float* __restrict__ dst,
                        int64_t n, int64_t id_offset, int nvec, int stride) {
  const int lane = threadIdx.x % GS;
  const int64_t k = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / GS;
  if (k >= n) return;
  Row<V> x;
  row_load<GS, V, false>(x, E + (size_t)(ids[k] + id_offset) * stride, lane, nvec);
  row_store<GS, V>(x, dst + (size_t)k * stride, lane, nvec);
}

// ---------------------------------------------------------------------------------------
// Multi-GPU step routing (SURVEY 8e).  The table is row-sharded; a rank's step touches the
// entity rows {h, t, corrupt entity} of its B triples.  Everything below runs on the device
// with device-side counts, so that a sharded step never returns to the host:
//   route : dedup the 3B ids (radix sort + tiled scan), sorted unique request list `uniq`,
//           per-owner cut points, triples re-indexed to request-list rows R + slot
//   post  : write each owner's slice of `uniq` into THAT owner's inbox (peer memory)
// The route kernels handle a chunk of steps per launch (grid.y = step of the chunk), like the
// plan kernels: the chain's latency (~30 dependent launches) is paid once per chunk.
// ---------------------------------------------------------------------------------------
__global__ void hole_shard_keys_kernel(const int32_t* __restrict__ pos, const int32_t* __restrict__ neg,
                                       int B, uint32_t* __restrict__ keys) {
  pos += (size_t)blockIdx.y * 3 * B;
  neg += (size_t)blockIdx.y * B;
  keys += (size_t)blockIdx.y * 3 * B;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < B; i += gridDim.x * blockDim.x) {
    keys[i] = (uint32_t)pos[3 * i];
    keys[B + i] = (uint32_t)pos[3 * i + 1];
    keys[2 * B + i] = (uint32_t)neg[i];
  }
}

// Dedup of the sorted keys in two passes over tiles of RT_TILE entries (coalesced):
// count: heads per tile;  assign: slot of every entry = (heads up to and including it) - 1,
// uniq[slot] = id, and the three entity columns of the step-table triples;
// cuts: cuts[o] = first slot owned by rank o, cuts[world] = U.
constexpr int RT_THREADS = 256;
constexpr int RT_ITERS = 8;
constexpr int RT_TILE = RT_THREADS * RT_ITERS;

__global__ void __launch_bounds__(RT_THREADS)
hole_shard_count_kernel(const uint32_t* __restrict__ sk, int M, int* __restrict__ tile_heads,
                        const int32_t* __restrict__ pos, int B, int32_t* __restrict__ pos_w) {
  __shared__ int wsum[RT_THREADS / 32];
  const int tid = threadIdx.x;
  sk += (size_t)blockIdx.y * M;
  tile_heads += (size_t)blockIdx.y * (gridDim.x + 1);       // [tiles] + the step's total
  pos += (size_t)blockIdx.y * 3 * B;
  pos_w += (size_t)blockIdx.y * 3 * B;
  int cnt = 0;
#pragma unroll
  for (int u = 0; u < RT_ITERS; ++u) {
    const int j = blockIdx.x * RT_TILE + u * RT_THREADS + tid;
    cnt += (j < M) && (j == 0 || sk[j] != sk[j - 1]);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if ((tid & 31) == 0) wsum[tid >> 5] = cnt;
  __syncthreads();
  if (tid == 0) {
    int t = 0;
    for (int q = 0; q < RT_THREADS / 32; ++q) t += wsum[q];
    tile_heads[blockIdx.x] = t;
  }
  for (int i = blockIdx.x * RT_THREADS + tid; i < B; i += gridDim.x * RT_THREADS)
    pos_w[3 * i + 2] = pos[3 * i + 2];                    // relation column
}

__global__ void __launch_bounds__(RT_THREADS)
hole_shard_assign_kernel(const uint32_t* __restrict__ sk, const uint32_t* __restrict__ sp, int M, int B,
                         int R, int* __restrict__ tile_heads, int64_t uniq_stride,
                         int32_t* __restrict__ uniq, int32_t* __restrict__ pos_w,
                         int32_t* __restrict__ neg_w) {
  __shared__ int wsum[RT_THREADS / 32];
  __shared__ int base_s;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  sk += (size_t)blockIdx.y * M;
  sp += (size_t)blockIdx.y * M;
  tile_heads += (size_t)blockIdx.y * (gridDim.x + 1);
  int* total = tile_heads + gridDim.x;
  uniq += (size_t)blockIdx.y * uniq_stride;
  pos_w += (size_t)blockIdx.y * 3 * B;
  neg_w += (size_t)blockIdx.y * B;
  if (w == 0) {                                   // heads in the tiles before mine
    int t = 0;
    for (int q = lane; q < (int)blockIdx.x; q += 32) t += tile_heads[q];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (lane == 0) base_s = t;
  }
  __syncthreads();
  int base = base_s;
#pragma unroll 1
  for (int u = 0; u < RT_ITERS; ++u) {
    const int j = blockIdx.x * RT_TILE + u * RT_THREADS + tid;
    const bool ok = j < M;
    const uint32_t key = ok ? sk[j] : 0u;
    const bool head = ok && (j == 0 || key != sk[j - 1]);
    const unsigned bal = __ballot_sync(0xffffffffu, head);
    const int incl = __popc(bal & (0xffffffffu >> (31 - lane)));   // heads in my warp up to me
    __syncthreads();                              // wsum of the previous iteration is consumed
    if (lane == 31) wsum[w] = incl;
    __syncthreads();
    int before = 0, all = 0;
#pragma unroll
    for (int q = 0; q < RT_THREADS / 32; ++q) {
      const int c = wsum[q];
      before += (q < w) ? c : 0;
      all += c;
    }
    if (ok) {
      const int slot = base + before + incl - 1;
      if (head) uniq[slot] = (int32_t)key;
      const int p = (int)sp[j], loc = R + slot;
      if (p < B) pos_w[3 * p] = loc;
      else if (p < 2 * B) pos_w[3 * (p - B) + 1] = loc;
      else neg_w[p - 2 * B] = loc;
    }
    base += all;
  }
  if (blockIdx.x == gridDim.x - 1 && tid == 0) *total = base;
}

__global__ void hole_shard_cuts_kernel(const int32_t* __restrict__ uniq, int64_t uniq_stride,
                                       const int* __restrict__ tile_heads, int tiles,
                                       int R, int64_t rows_per, int world, int32_t* __restrict__ cuts) {
  const int tid = threadIdx.x;
  if (tid > world) return;
  uniq += (size_t)blockIdx.x * uniq_stride;
  cuts += (size_t)blockIdx.x * (HOLE_MAX_RANKS + 1);
  const int U = tile_heads[(size_t)blockIdx.x * (tiles + 1) + tiles];
  const int64_t bound = (int64_t)R + rows_per * tid;     // first row of rank `tid`
  int a = 0, b = U;
  while (a < b) {
    const int mid = (a + b) >> 1;
    if ((int64_t)uniq[mid] < bound) a = mid + 1; else b = mid;
  }
  cuts[tid] = (tid == world) ? U : a;
}

__global__ void hole_shard_post_kernel(const int32_t* __restrict__ uniq, const int32_t* __restrict__ cuts,
                                       int world, int me, int64_t cap, hole_peer_ptrs inbox,
                                       hole_peer_ptrs meta) {
  const int U = cuts[world];
  const int gtid = blockIdx.x * blockDim.x + threadIdx.x;
  for (int j = gtid; j < U; j += gridDim.x * blockDim.x) {
    int o = 0;
    while (j >= cuts[o + 1]) ++o;
    static_cast<int32_t*>(inbox.p[o])[(size_t)me * cap + (j - cuts[o])] = uniq[j];
  }
  if (gtid < world) {
    int32_t* m = static_cast<int32_t*>(meta.p[gtid]);
    m[2 * me] = cuts[gtid + 1] - cuts[gtid];     // how many rows I want from rank gtid
    m[2 * me + 1] = cuts[gtid];                  // where they sit in my step table (after R)
  }
  __threadfence_system();                        // peer stores: visible before a later kernel raises the flag
}

// ---------------------------------------------------------------------------------------
// --log_loss step (holE.py:194-196, 206-220): helpers around the K1/K3 passes
// ---------------------------------------------------------------------------------------
// The L2 term  l2 * tf.nn.l2_loss(embeddings)  sits in every one of the (1+k)B loss rows
// (holE.py:196), so its gradient is dense: E <- E * (1 - lr * (1+k) B l2).  One pass over the
// table applies it and sums x^2 of the OLD table (block partials; hole_l2_finish adds them
// in a fixed order and halves).
__global__ void __launch_bounds__(256)
hole_l2_scale_kernel(float4* __restrict__ E4, size_t n4, float scale, float* __restrict__ partial) {
  __shared__ float sm[256];
  float a = 0.f;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    float4 v = E4[i];
    a += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
    if (scale != 1.0f) {
      v.x *= scale; v.y *= scale; v.z *= scale; v.w *= scale;
      E4[i] = v;
    }
  }
  sm[threadIdx.x] = a;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) sm[threadIdx.x] += sm[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) partial[blockIdx.x] = sm[0];
}

__global__ void __launch_bounds__(256)
hole_l2_finish_kernel(const float* __restrict__ partial, int n, float* __restrict__ out) {
  __shared__ double sm[256];
  double a = 0.0;
  for (int i = threadIdx.x; i < n; i += 256) a += (double)partial[i];
  sm[threadIdx.x] = a;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) sm[threadIdx.x] += sm[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) *out = (float)(0.5 * sm[0]);
}

// E[row] += D[row]; D[row] = 0  for every distinct row of one pass: every use of a row that occurs once,
// and the first sorted entry of every duplicated row.  A row shared by several passes is applied by the
// first and adds zero after.
template <int GS, int V>
__global__ void __launch_bounds__(256)
hole_apply_delta_kernel(float* __restrict__ E, float* __restrict__ D, const uint32_t* __restrict__ keys,
                        const uint32_t* __restrict__ gslot, const uint32_t* __restrict__ skey, int M,
                        int nvec, int stride) {
  const int lane = threadIdx.x % GS;
  const int64_t u = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / GS;
  if (u >= M) return;
  const uint32_t key = keys[u];
  if (key == HOLE_KEY_ABSENT) return;
  const uint32_t j = gslot[u];
  if (j != HOLE_SLOT_UNIQUE && j > 0 && skey[j - 1] == key) return;
  Row<V> x, d, z;
  row_zero(z);
  row_load<GS, V, false>(x, E + (size_t)key * stride, lane, nvec);
  row_load<GS, V, false>(d, D + (size_t)key * stride, lane, nvec);
  row_add(x, d);
  row_store<GS, V>(x, E + (size_t)key * stride, lane, nvec);
  row_store<GS, V>(z, D + (size_t)key * stride, lane, nvec);
}

// deterministic per-step loss sum: one CTA per step, fixed-shape tree
__global__ void __launch_bounds__(256)
hole_loss_sum_kernel(const float* __restrict__ loss, int64_t B, float* __restrict__ out) {
  __shared__ float sm[256];
  const float* l = loss + (size_t)blockIdx.x * B;
  float a = 0.f;
  for (int64_t i = threadIdx.x; i < B; i += 256) a += l[i];
  sm[threadIdx.x] = a;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) sm[threadIdx.x] += sm[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[blockIdx.x] = sm[0];
}

// ---------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------
#define HOLE_DISPATCH(ctx, KERNEL, grid, block, stream, ...)                                 \
  do {                                                                                       \
    if ((ctx)->gs == 8 && (ctx)->v == 1) KERNEL<8, 1><<<grid, block, 0, stream>>>(__VA_ARGS__);          \
    else if ((ctx)->gs == 16 && (ctx)->v == 1) KERNEL<16, 1><<<grid, block, 0, stream>>>(__VA_ARGS__);   \
    else if ((ctx)->gs == 32 && (ctx)->v == 1) KERNEL<32, 1><<<grid, block, 0, stream>>>(__VA_ARGS__);   \
    else if ((ctx)->gs == 32 && (ctx)->v == 2) KERNEL<32, 2><<<grid, block, 0, stream>>>(__VA_ARGS__);   \
    else if ((ctx)->gs == 32 && (ctx)->v == 3) KERNEL<32, 3><<<grid, block, 0, stream>>>(__VA_ARGS__);   \
    else return hole_set_error(HOLE_ERR_UNSUPPORTED, "no kernel variant for gs=%d v=%d",     \
                               (ctx)->gs, (ctx)->v);                                         \
    HOLE_LAUNCHED();                                                                         \
  } while (0)

// same, launched with programmatic stream serialization (see pdl_wait)
#define HOLE_DISPATCH_PDL(ctx, KERNEL, grid_, block_, smem_, stream_, ...)                   \
  do {                                                                                       \
    cudaLaunchConfig_t cfg_ = {};                                                            \
    cfg_.gridDim = dim3(grid_);                                                              \
    cfg_.blockDim = dim3(block_);                                                            \
    cfg_.dynamicSmemBytes = (size_t)(smem_);                                                 \
    cfg_.stream = stream_;                                                                   \
    cudaLaunchAttribute at_[1];                                                              \
    at_[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;                          \
    at_[0].val.programmaticStreamSerializationAllowed = 1;                                   \
    cfg_.attrs = at_;                                                                        \
    cfg_.numAttrs = 1;                                                                       \
    cudaError_t le_ = cudaSuccess;                                                           \
    if ((ctx)->gs == 8 && (ctx)->v == 1) le_ = cudaLaunchKernelEx(&cfg_, KERNEL<8, 1>, __VA_ARGS__);        \
    else if ((ctx)->gs == 16 && (ctx)->v == 1) le_ = cudaLaunchKernelEx(&cfg_, KERNEL<16, 1>, __VA_ARGS__); \
    else if ((ctx)->gs == 32 && (ctx)->v == 1) le_ = cudaLaunchKernelEx(&cfg_, KERNEL<32, 1>, __VA_ARGS__); \
    else if ((ctx)->gs == 32 && (ctx)->v == 2) le_ = cudaLaunchKernelEx(&cfg_, KERNEL<32, 2>, __VA_ARGS__); \
    else if ((ctx)->gs == 32 && (ctx)->v == 3) le_ = cudaLaunchKernelEx(&cfg_, KERNEL<32, 3>, __VA_ARGS__); \
    else return hole_set_error(HOLE_ERR_UNSUPPORTED, "no kernel variant for gs=%d v=%d",     \
                               (ctx)->gs, (ctx)->v);                                         \
    HOLE_CUDA_TRY(le_);                                                                      \
    HOLE_LAUNCHED();                                                                         \
  } while (0)

static inline unsigned grid_for_groups(int64_t groups, int gs, int block = 256) {
  int64_t per_block = block / gs;
  return (unsigned)std::max<int64_t>(1, (groups + per_block - 1) / per_block);
}

extern "C" int hole_abi_version(void) { return HOLE_ABI_VERSION; }
extern "C" const char* hole_last_error(void) { return g_hole_err.c_str(); }
extern "C" int64_t hole_launch_count(void) { return g_hole_launches; }
extern "C" void hole_launch_count_reset(void) { g_hole_launches = 0; }

extern "C" int hole_row_stride(int dim) {
  if (dim <= 0 || (dim & 1)) return HOLE_ERR_ARG;
  return 2 * (((dim / 2) + 3) / 4 * 4);
}

// ---- the archived FFT / tanh score variant (hole_ccorr.cuh)
#define HOLE_CC_DISPATCH(NVNEED, STMT)                                                       \
  do {                                                                                       \
    const int nv_ = (NVNEED);                                                                \
    if (nv_ <= 1) { constexpr int NV = 1; STMT; }                                            \
    else if (nv_ <= 2) { constexpr int NV = 2; STMT; }                                       \
    else if (nv_ <= 3) { constexpr int NV = 3; STMT; }                                       \
    else if (nv_ <= 4) { constexpr int NV = 4; STMT; }                                       \
    else if (nv_ <= 6) { constexpr int NV = 6; STMT; }                                       \
    else if (nv_ <= 8) { constexpr int NV = 8; STMT; }                                       \
    else { constexpr int NV = 12; STMT; }                                                    \
  } while (0)

static int cc_nv(const hole_ctx* c) { return (c->row_stride / 2 + 31) / 32; }

// warps per block such that the block's rows fit the opt-in shared memory
static int cc_warps(int floats_per_warp) {
  return std::max(1, std::min(8, (220 * 1024) / (floats_per_warp * (int)sizeof(float))));
}

static int cc_prepare(hole_ctx* c) {
  if (c->cc_ready) return HOLE_OK;
  const int lim = 227 * 1024;
  cudaError_t e1 = cudaSuccess, e2 = cudaSuccess;
  HOLE_CC_DISPATCH(cc_nv(c),
                   e1 = cudaFuncSetAttribute(hole_ccorr_fwd_bwd_kernel<NV>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim);
                   e2 = cudaFuncSetAttribute(hole_ccorr_score_kernel<NV>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
  HOLE_CUDA_TRY(e1);
  HOLE_CUDA_TRY(e2);
  c->cc_ready = true;
  return HOLE_OK;
}

extern "C" int hole_ctx_set_score_mode(hole_ctx* c, int mode) {
  HOLE_CHECK_ARG(c != nullptr);
  HOLE_CHECK_ARG(mode == HOLE_SCORE_COMPLEX || mode == HOLE_SCORE_CCORR_TANH);
  if (mode == HOLE_SCORE_CCORR_TANH && c->shard_state != nullptr)
    return hole_set_error(HOLE_ERR_UNSUPPORTED, "the archived ccorr/tanh score mode has no row-sharded step");
  c->score_mode = mode;
  return HOLE_OK;
}

extern "C" int hole_ctx_set_optimizer(hole_ctx* c, int optimizer, float* accum) {
  HOLE_CHECK_ARG(c != nullptr);
  HOLE_CHECK_ARG((optimizer == HOLE_OPT_SGD && accum == nullptr) || (optimizer == HOLE_OPT_ADAGRAD && accum != nullptr));
  if (optimizer == HOLE_OPT_ADAGRAD && c->shard_state != nullptr)
    return hole_set_error(HOLE_ERR_UNSUPPORTED, "AdaGrad has no row-sharded step");
  c->optimizer = optimizer;
  c->accum = accum;
  return HOLE_OK;
}

static int ctx_create_streams(hole_ctx* c) {
  HOLE_CUDA_TRY(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
  {   // the plan is small integer work that the next step waits for: highest priority
    int lo = 0, hi = 0;
    HOLE_CUDA_TRY(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    // (for the chunked single-GPU path the priority makes no measurable difference)
    HOLE_CUDA_TRY(cudaStreamCreateWithPriority(&c->plan_stream, cudaStreamNonBlocking, hi));
  }
  HOLE_CUDA_TRY(cudaEventCreateWithFlags(&c->ev_entry, cudaEventDisableTiming));
  HOLE_CUDA_TRY(cudaHostAlloc((void**)&c->dup_max_host, 2 * sizeof(int), cudaHostAllocMapped));   // one word per plan slot
  c->dup_max_host[0] = c->dup_max_host[1] = -1;
  HOLE_CUDA_TRY(cudaHostGetDevicePointer((void**)&c->dup_max_host_dev, c->dup_max_host, 0));
  HOLE_CUDA_TRY(cudaFuncSetAttribute(hole_plan_sortseg_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SS_SMEM));
  HOLE_CUDA_TRY(cudaFuncSetAttribute(hole_plan_relsort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, RS_SMEM_MAX));
  HOLE_CUDA_TRY(cudaFuncSetAttribute(hole_plan_relsort_few_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, RS_SMEM_MAX));
  // The first launch of a kernel loads its module (tens of microseconds with lazy loading).  The one-launch
  // sort is first used by a context's SECOND training call (the first one reports the step sizes), so it
  // is launched once here on nothing: mdev = the mapped word, still -1 -> every thread returns.
  hole_plan_sortseg_small_kernel<<<1, SS_THREADS, SS_SMEM, c->plan_stream>>>(
      nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0, c->dup_max_host_dev, 0, 0);
  HOLE_LAUNCHED();
  --g_hole_launches;      // (not a step's launch)
  for (int k = 0; k < 2; ++k) {
    HOLE_CUDA_TRY(cudaEventCreateWithFlags(&c->ev_copy[k], cudaEventDisableTiming));
    HOLE_CUDA_TRY(cudaEventCreateWithFlags(&c->plan[k].ready, cudaEventDisableTiming));
    HOLE_CUDA_TRY(cudaEventCreateWithFlags(&c->plan[k].released, cudaEventDisableTiming));
  }
  return HOLE_OK;
}

extern "C" int hole_ctx_create(hole_ctx** out, int device, int64_t n_rows, int dim) {
  HOLE_CHECK_ARG(out != nullptr);
  *out = nullptr;
  HOLE_CHECK_ARG(n_rows > 0 && n_rows < (int64_t(1) << 31));
  if (dim <= 0 || (dim & 1))   // holE.py:164-165 splits the row at dim//2
    return hole_set_error(HOLE_ERR_ARG, "embedding_dim must be a positive even number, got %d", dim);
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return hole_set_error(HOLE_ERR_CUDA, "no CUDA device available (%s); libhole_b200 has no CPU fallback",
                          cudaGetErrorString(e));
  HOLE_CHECK_ARG(device >= 0 && device < ndev);
  cudaDeviceProp prop;
  HOLE_CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return hole_set_error(HOLE_ERR_CUDA, "device %d is sm_%d%d; libhole_b200 is built for sm_100a only",
                          device, prop.major, prop.minor);
  HOLE_CUDA_TRY(cudaSetDevice(device));
  hole_ctx* c = new hole_ctx();
  c->device = device;
  c->n_rows = n_rows;
  c->dim = dim;
  c->H = dim / 2;
  c->nvec = (c->H + 3) / 4;
  c->row_stride = 8 * c->nvec;
  c->sm_count = prop.multiProcessorCount;
  if (c->nvec <= 8) { c->gs = 8; c->v = 1; }
  else if (c->nvec <= 16) { c->gs = 16; c->v = 1; }
  else { c->gs = 32; c->v = (c->nvec + 31) / 32; }
  if (c->v > 3) {
    delete c;
    return hole_set_error(HOLE_ERR_UNSUPPORTED, "embedding_dim %d > 768 not built", dim);
  }
  int bits = 1;
  while ((int64_t(1) << bits) < n_rows) ++bits;
  c->key_bits = bits;
  // radix passes: smallest p with 2^(8p) - 1 >= n_rows, so the "absent" key's low bits sort last
  c->row_passes = 1;
  while (((int64_t(1) << (8 * c->row_passes)) - 1) < n_rows) ++c->row_passes;
  c->rel_passes = c->row_passes;
  if (const char* e = getenv("HOLE_HOST_FIRST")) c->host_first = atoi(e);
  if (const char* e = getenv("HOLE_SORT_SMALL")) c->sort_small = atoi(e);   // 0 = always the radix chain, 2 = always one launch
  if (const char* e = getenv("HOLE_PLAN_RAMP")) {     // "first,factor"; "0" disables the ramp
    int a = 0, b = 4;
    if (sscanf(e, "%d,%d", &a, &b) >= 1) { c->ramp_first = a; c->ramp_factor = b < 2 ? 2 : b; }
  }
  int rc = ctx_create_streams(c);
  if (rc != HOLE_OK) {
    hole_ctx_destroy(c);
    return rc;
  }
  *out = c;
  return HOLE_OK;
}

static void plan_free(hole_plan& p) {
  cudaFree(p.keysA); cudaFree(p.keysB); cudaFree(p.keysC); cudaFree(p.valsA); cudaFree(p.valsB);
  cudaFree(p.seen); cudaFree(p.blkcnt); cudaFree(p.mdup); cudaFree(p.done);
  p.keysC = p.seen = p.dup = nullptr;
  p.done = nullptr;
  p.blkcnt = p.mdup = nullptr;
  cudaFree(p.gslot); cudaFree(p.heads); cudaFree(p.nheads); cudaFree(p.neg); cudaFree(p.ghist); cudaFree(p.perm);
  p.perm = nullptr;
  p.keysA = p.keysB = p.valsA = p.valsB = nullptr;
  p.gslot = nullptr; p.heads = nullptr; p.nheads = nullptr; p.neg = nullptr; p.ghist = nullptr;
  p.skey = p.spos = nullptr;
}

static void ws_free(hole_ctx* c) {
  cudaFree(c->G); cudaFree(c->counters); cudaFree(c->loss); cudaFree(c->loss_sum);
  c->G = nullptr; c->counters = nullptr; c->loss = nullptr; c->loss_sum = nullptr;
  plan_free(c->plan[0]);
  plan_free(c->plan[1]);
  c->cap_B = c->cap_S = 0;
}

extern "C" int hole_ctx_set_relations(hole_ctx* c, int64_t n_relations) {
  HOLE_CHECK_ARG(c && n_relations > 0 && n_relations <= c->n_rows);
  c->rel_passes = 1;
  while (((int64_t(1) << (8 * c->rel_passes)) - 1) < n_relations) ++c->rel_passes;
  c->n_rel_hint = n_relations;
  return HOLE_OK;
}

static void shard_free(hole_ctx* c);

extern "C" int hole_ctx_destroy(hole_ctx* c) {
  if (c == nullptr) return HOLE_OK;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  shard_free(c);
  ws_free(c);
  hole_rank_ws_free(c);
  cudaFree(c->route_buf);
  cudaFree(c->route_done);
  cudaFree(c->triples_stage[0]); cudaFree(c->triples_stage[1]);
  if (c->loss_sum_pinned) cudaFreeHost(c->loss_sum_pinned);
  for (int k = 0; k < 2; ++k) {
    if (c->ev_copy[k]) cudaEventDestroy(c->ev_copy[k]);
    if (c->plan[k].ready) cudaEventDestroy(c->plan[k].ready);
    if (c->plan[k].released) cudaEventDestroy(c->plan[k].released);
  }
  if (c->ev_entry) cudaEventDestroy(c->ev_entry);
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  if (c->plan_stream) cudaStreamDestroy(c->plan_stream);
  if (c->dup_max_host) cudaFreeHost(c->dup_max_host);
  for (cudaEvent_t e : c->prof_ev) cudaEventDestroy(e);
  delete c;
  return HOLE_OK;
}

static int k1_prepare(hole_ctx* c);

// Workspace for chunks of S steps of batch B.  Reallocation synchronises the device.
int hole_ws_reserve(hole_ctx* c, int64_t B, int64_t S) {
  hole_rank_cache_invalidate(c);     // every training entry point comes through here
  if (!c->k1_ready) {
    int rc = k1_prepare(c);
    if (rc) return rc;
  }
  if (B <= c->cap_B && S <= c->cap_S) return HOLE_OK;
  HOLE_CUDA_TRY(cudaSetDevice(c->device));
  HOLE_CUDA_TRY(cudaDeviceSynchronize());
  B = std::max(B, c->cap_B);
  S = std::max(S, c->cap_S);
  ws_free(c);
  const size_t M = (size_t)4 * B;
  const size_t tiles = (M + ST_TILE - 1) / ST_TILE;
#define WS_ALLOC(ptr, bytes)                                                             \
  do {                                                                                   \
    if (cudaMalloc((void**)&(ptr), (bytes)) != cudaSuccess) {                            \
      cudaGetLastError();                                                                \
      ws_free(c);                                                                        \
      return hole_set_error(HOLE_ERR_ALLOC, "workspace allocation of %zu bytes failed", (size_t)(bytes)); \
    }                                                                                    \
  } while (0)
  WS_ALLOC(c->G, M * c->row_stride * sizeof(float));
  WS_ALLOC(c->counters, (size_t)HOLE_TREE_LEVELS * M * 4);
  WS_ALLOC(c->loss, (size_t)S * B * 4);
  WS_ALLOC(c->loss_sum, (size_t)S * 4);
  for (int k = 0; k < 2; ++k) {
    hole_plan& p = c->plan[k];
    WS_ALLOC(p.keysA, S * M * 4); WS_ALLOC(p.keysB, S * M * 4); WS_ALLOC(p.keysC, S * M * 4);
    WS_ALLOC(p.valsA, S * M * 4); WS_ALLOC(p.valsB, S * M * 4);
    {
      const size_t W = (size_t)(c->n_rows + 31) / 32;
      p.bitmap_words = (size_t)S * W;
      WS_ALLOC(p.seen, 2 * p.bitmap_words * 4);
      HOLE_CUDA_TRY(cudaMemset(p.seen, 0, 2 * p.bitmap_words * 4));
      p.dup = p.seen + p.bitmap_words;
      WS_ALLOC(p.done, (size_t)S * sizeof(unsigned));
      HOLE_CUDA_TRY(cudaMemset(p.done, 0, (size_t)S * sizeof(unsigned)));
      WS_ALLOC(p.blkcnt, (size_t)S * ((M + DP_TILE - 1) / DP_TILE + 1) * 4);
      WS_ALLOC(p.mdup, (size_t)S * 4);
    }
    WS_ALLOC(p.gslot, S * M * 4);
    WS_ALLOC(p.heads, (size_t)S * (M / 2 + 1) * sizeof(uint4));
    WS_ALLOC(p.nheads, (size_t)S * 4);
    WS_ALLOC(p.neg, (size_t)S * B * 4);
    WS_ALLOC(p.perm, (size_t)S * B * 4);
    WS_ALLOC(p.ghist, (size_t)S * 256 * tiles * 4);
    p.used = false;
  }
#undef WS_ALLOC
  HOLE_CUDA_TRY(cudaMemset(c->counters, 0, (size_t)HOLE_TREE_LEVELS * M * 4));
  c->cap_B = B;
  c->cap_S = S;
  return HOLE_OK;
}

extern "C" int hole_pack_rows(hole_ctx* c, const float* src, float* dst, int64_t n, void* stream) {
  HOLE_CHECK_ARG(c && src && dst && n >= 0);
  if (n == 0) return HOLE_OK;
  HOLE_CUDA_TRY(cudaSetDevice(c->device));
  int64_t total = n * c->row_stride;
  unsigned grid = (unsigned)std::min<int64_t>((total + 255) / 256, (int64_t)c->sm_count * 32);
  hole_pack_rows_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(src, dst, n, c->dim, c->H, c->row_stride / 2);
  HOLE_LAUNCHED();
  return HOLE_OK;
}

extern "C" int hole_unpack_rows(hole_ctx* c, const float* src, float* dst, int64_t n, void* stream) {
  HOLE_CHECK_ARG(c && src && dst && n >= 0);
  if (n == 0) return HOLE_OK;
  HOLE_CUDA_TRY(cudaSetDevice(c->device));
  int64_t total = n * c->dim;
  unsigned grid = (unsigned)std::min<int64_t>((total + 255) / 256, (int64_t)c->sm_count * 32);
  hole_unpack_rows_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(src, dst, n, c->dim, c->H, c->row_stride / 2);
  HOLE_LAUNCHED();
  return HOLE_OK;
}

extern "C" int hole_corrupt_at(hole_ctx* c, const int32_t* triples, int64_t B, const int32_t* type_of,
                               const int64_t* csr_off, const int32_t* csr_ids, uint64_t seed,
                               uint64_t step, uint64_t index_base, int32_t* side_out,
                               int32_t* neg_out, int* side_host, void* stream) {
  HOLE_CHECK_ARG(c && B >= 0);
  if (side_host) *side_host = hole_side_coin(seed, step);
  if (B == 0) return HOLE_OK;
  HOLE_CHECK_ARG(triples && type_of && csr_off && csr_ids && neg_out);
  HOLE_CHECK_ARG(index_base + (uint64_t)B <= (uint64_t(1) << 32));
  HOLE_CUDA_TRY(cudaSetDevice(c->device));
  dim3 grid((unsigned)std::min<int64_t>((B + 255) / 256, 65535), 1);
  hole_corrupt_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(triples, B, 1, type_of, csr_off, csr_ids,
                                                              seed, step, index_base, neg_out, side_out);
  HOLE_LAUNCHED();
  return HOLE_OK;
}

extern "C" int hole_corrupt(hole_ctx* c, const int32_t* triples, int64_t B, const int32_t* type_of,
                            const int64_t* csr_off, const int32_t* csr_ids, uint64_t seed,
                            uint64_t step, int32_t* side_out, int32_t* neg_out, int* side_host,
                            void* stream) {
  return hole_corrupt_at(c, triples, B, type_of, csr_off, csr_ids, seed, step, 0, side_out, neg_out,
                         side_host, stream);
}

extern "C" int hole_score(hole_ctx* c, const float* table, const int32_t* triples, int64_t B,
                          float* out_sigma, void* stream) {
  HOLE_CHECK_ARG(c && B >= 0);
  if (B == 0) return HOLE_OK;
  HOLE_CHECK_ARG(table && triples && out_sigma);
  HOLE_CUDA_TRY(cudaSetDevice(c->device));
  if (c->score_mode == HOLE_SCORE_CCORR_TANH) {       // archived variant: tanh(s) instead of sigma(s)
    int rc = cc_prepare(c);
    if (rc) return rc;
    const int fw = cc_score_warp_floats(c->H), warps = cc_warps(fw);
    const unsigned grid = (unsigned)((B + warps - 1) / warps);
    HOLE_CC_DISPATCH(cc_nv(c), (hole_ccorr_score_kernel<NV><<<grid, 32 * warps, (size_t)warps * fw * sizeof(float),
                                                            (cudaStream_t)stream>>>(table, triples, B, c->H, c->row_stride,
                                                                                    out_sigma)));
    HOLE_CUDA_TRY(cudaGetLastError());
    HOLE_LAUNCHED();
    return HOLE_OK;
  }
  HOLE_DISPATCH(c, hole_score_kernel, grid_for_groups(B, c->gs), 256, (cudaStream_t)stream, table,
                triples, B, c->nvec, c->row_stride, out_sigma);
  return HOLE_OK;
}

// Stable LSD radix sort of S independent arrays of M (key, value = original index) pairs.
// Keys start in kA (destroyed); kB, vA, vB are scratch; the last pass writes the values to
// v_final when given.  Returns where the sorted keys / values ended up.
// v_init: the values travelling with the keys of kA live in vA (else value = index).  mdev: per-array
// element counts on the device (else M); the arrays are M apart either way.  done: S zero-initialised
// ticket counters (left zero).
static int radix_sort(uint32_t* ghist, uint32_t* kA, uint32_t* kB, uint32_t* vA, uint32_t* vB,
                      uint32_t* v_final, int64_t S, int M, int passes, cudaStream_t st,
                      uint32_t** k_out, uint32_t** v_out, unsigned* done, bool v_init = false,
                      const int* mdev = nullptr) {
  const int P = (M + ST_TILE - 1) / ST_TILE;
  uint32_t *kin = kA, *vin = v_init ? vA : nullptr, *kout = kB, *vout = vB;
  dim3 grid((unsigned)P, (unsigned)S);
  for (int pass = 0; pass < passes; ++pass) {
    if (pass == passes - 1 && v_final != nullptr) vout = v_final;
    hole_sort_hist_kernel<<<grid, ST_THREADS, 0, st>>>(kin, ghist, M, P, 8 * pass, mdev, done);
    HOLE_LAUNCHED();
    hole_sort_scatter_kernel<<<grid, ST_THREADS, 0, st>>>(kin, vin, kout, vout, ghist, M, P, 8 * pass, mdev);
    HOLE_LAUNCHED();
    uint32_t* nk = (kout == kB) ? kA : kB;
    uint32_t* nv = (vout == vB) ? vA : vB;
    kin = kout; vin = vout; kout = nk; vout = nv;
  }
  *k_out = kin;
  *v_out = vin;
  return HOLE_OK;
}

typedef void (*hole_k1_fn)(const hole_k1_args, const hole_k1_shard);
template <int DM>
static hole_k1_fn k1_fn(const hole_ctx* c) {
  if (c->gs == 8) return hole_k1_kernel<8, 1, DM>;
  if (c->gs == 16) return hole_k1_kernel<16, 1, DM>;
  if (c->v == 1) return hole_k1_kernel<32, 1, DM>;
  if (c->v == 2) return hole_k1_kernel<32, 2, DM>;
  return hole_k1_kernel<32, 3, DM>;
}
static hole_k1_fn k1_fn_dm(const hole_ctx* c, int dm) {
  return dm == 0 ? k1_fn<0>(c) : dm == 1 ? k1_fn<1>(c) : dm == 2 ? k1_fn<2>(c) : dm == 3 ? k1_fn<3>(c) : k1_fn<4>(c);
}

// Kernel attributes of the training kernels, set on the first training call of a context
// (scoring / ranking contexts never pay for, or fail on, K1's shared-memory request).
static int k1_prepare(hole_ctx* c) {
  if (c->k1_ready) return HOLE_OK;
  // K1V2_STAGES x 3 landing rows + K1V2_STAGES mbarriers per lane group
  c->k1v2_smem = (K1_THREADS / c->gs) * K1V2_STAGES * (3 * c->row_stride * (int)sizeof(float) + 8);
  if (c->k1v2_smem > 227 * 1024)
    return hole_set_error(HOLE_ERR_UNSUPPORTED, "embedding_dim %d: K1 needs %d bytes of shared memory",
                          c->dim, c->k1v2_smem);
  int nb = 1;
  for (int dm = 0; dm < 5; ++dm) {
    HOLE_CUDA_TRY(cudaFuncSetAttribute(k1_fn_dm(c, dm), cudaFuncAttributeMaxDynamicSharedMemorySize, c->k1v2_smem));
  }
  HOLE_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k1_fn<0>(c), K1_THREADS, c->k1v2_smem));
  c->k1_groups = c->sm_count * std::max(nb, 1) * (K1_THREADS / c->gs);
  c->k1_ready = true;
  return HOLE_OK;
}

static int k1_launch(hole_ctx* c, int dm, const hole_k1_args& a, const hole_k1_shard& sh, cudaStream_t st,
                     bool pdl) {
  const int per_block = K1_THREADS / c->gs;
  const int64_t groups = ((int64_t)a.B + a.T - 1) / a.T;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)std::max<int64_t>(1, (groups + per_block - 1) / per_block));
  cfg.blockDim = dim3((unsigned)K1_THREADS);
  cfg.dynamicSmemBytes = (size_t)c->k1v2_smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl ? 1 : 0;
  HOLE_CUDA_TRY(cudaLaunchKernelEx(&cfg, k1_fn_dm(c, dm), a, sh));
  HOLE_LAUNCHED();
  return HOLE_OK;
}

// triples per lane group in K1 (and the run length the plan folds relation keys over)
static int triples_per_group(const hole_ctx* c, int64_t B) {
  const int64_t wmax = c->k1_groups > 0 ? c->k1_groups : (int64_t)c->sm_count * 2 * (256 / c->gs);
  return (int)std::max<int64_t>(1, (B + wmax - 1) / wmax);
}

// The integer plan of S steps, enqueued on `ps` (the plan stream, or the caller's stream):
// group triples by relation -> corruption + row keys -> sort by row -> segments.
// neg_in != nullptr (single-step API): the caller supplies the corruption.
static int plan_steps(hole_ctx* c, hole_plan& pl, const int32_t* triples_dev, int64_t B, int64_t S,
                      const int32_t* type_of, const int64_t* csr_off, const int32_t* csr_ids,
                      uint64_t seed, uint64_t first_step, const int32_t* neg_in, cudaStream_t ps,
                      int64_t tstride = -1) {
  if (tstride < 0) tstride = 3 * B;
  if (pl.used) HOLE_CUDA_TRY(cudaStreamWaitEvent(ps, pl.released, 0));   // last consumer is done
  const int M = (int)(4 * B);
  dim3 grid((unsigned)std::min<int64_t>((B + 255) / 256, 4096), (unsigned)S);
  // 1. perm: triples grouped by relation (stable)
  int rc = HOLE_OK;
  if (const size_t rf_smem = c->sort_small ? plan_relsort_few_smem(B, c->n_rel_hint) : 0) {
    hole_plan_relsort_few_kernel<<<(unsigned)S, RF_THREADS, rf_smem, ps>>>(triples_dev, (int)B, tstride, (int)c->n_rel_hint,
                                                                         plan_relsort_few_stride(B), pl.perm);
    HOLE_LAUNCHED();
  } else if (const size_t rs_smem = c->sort_small ? plan_relsort_smem(B, c->rel_passes) : 0) {
    hole_plan_relsort_kernel<<<(unsigned)S, RS_THREADS, rs_smem, ps>>>(triples_dev, (int)B, tstride, c->rel_passes, pl.perm);
    HOLE_LAUNCHED();
  } else {
    hole_rel_keys_kernel<<<grid, 256, 0, ps>>>(triples_dev, B, tstride, pl.keysA);
    HOLE_LAUNCHED();
    uint32_t *ko, *vo;
    rc = radix_sort(pl.ghist, pl.keysA, pl.keysB, pl.valsA, pl.valsB, reinterpret_cast<uint32_t*>(pl.perm),
                    S, (int)B, c->rel_passes, ps, &ko, &vo, pl.done);
    if (rc) return rc;
  }
  // 2. corruption + the 4B row keys of every step; rows used more than once are marked in the bitmaps
  pl.T = triples_per_group(c, B);
  const int W = (int)((c->n_rows + 31) / 32);
  // (the bitmaps seen | dup are clean here: cleared at allocation and after every plan, off the chain)
  hole_plan_keys_kernel<<<grid, 256, 0, ps>>>(triples_dev, B, tstride, pl.T, pl.perm, type_of, csr_off, csr_ids,
                                              seed, first_step, neg_in, pl.neg, pl.keysA, pl.seen, pl.dup, W);
  HOLE_LAUNCHED();
  // 3. the uses of duplicated rows, compacted in position order (the others are marked UNIQUE)
  const int nblk = (M + DP_TILE - 1) / DP_TILE;
  dim3 dgrid((unsigned)nblk, (unsigned)S);
  hole_plan_dupflag_kernel<<<dgrid, DP_THREADS, 0, ps>>>(pl.keysA, pl.dup, M, W, pl.gslot, pl.blkcnt, pl.mdup, pl.done);
  HOLE_LAUNCHED();
  hole_plan_compact_kernel<<<dgrid, DP_THREADS, 0, ps>>>(pl.keysA, pl.dup, M, W, pl.blkcnt, pl.keysB, pl.valsA);
  HOLE_LAUNCHED();
  // 4. sort them by row (stable: equal rows stay in position order), 5. segments
  pl.heads_cap = M / 2 + 1;
  // How many duplicated uses the steps of the previous plans of this batch size had (read back without
  // waiting: a plan that has not reported yet counts as "unknown").  While they fit the one-launch kernel's
  // shared memory, it replaces the 2 * passes + 1 launches below; it stays correct for a larger step.
  // Every plan overwrites the word of its slot, so the decision follows the last plan of each slot (a window of
  // two chunks), not an all-time maximum: one unusually large step does not switch the context to the chain
  // for good.
  volatile int* rep = c->dup_max_host;
  if (c->dup_seen_B != B) { c->dup_seen_B = B; rep[0] = rep[1] = -1; }
  c->dup_seen_max = std::max(rep[0], rep[1]);
  const bool one_launch = c->sort_small == 2 || (c->sort_small == 1 && c->dup_seen_max >= 0 && c->dup_seen_max <= SS_CAP);
  if (one_launch) {
    const bool odd = (c->row_passes & 1) != 0;
    pl.skey = odd ? pl.keysC : pl.keysB;
    pl.spos = odd ? pl.valsB : pl.valsA;
    hole_plan_sortseg_small_kernel<<<(unsigned)S, SS_THREADS, SS_SMEM, ps>>>(
        pl.keysB, pl.valsA, pl.keysC, pl.valsB, pl.skey, pl.spos, pl.gslot, pl.heads, pl.nheads, M, pl.mdup,
        pl.heads_cap, c->row_passes);
    HOLE_LAUNCHED();
  } else {
    rc = radix_sort(pl.ghist, pl.keysB, pl.keysC, pl.valsA, pl.valsB, nullptr, S, M, c->row_passes, ps,
                    &pl.skey, &pl.spos, pl.done, /*v_init=*/true, pl.mdup);
    if (rc) return rc;
    HOLE_CUDA_TRY(cudaMemsetAsync(pl.nheads, 0, (size_t)S * 4, ps));
    dim3 sgrid((unsigned)std::min<int64_t>((M + 255) / 256, 1024), (unsigned)S);
    hole_plan_segments_kernel<<<sgrid, 256, 0, ps>>>(pl.skey, pl.spos, pl.gslot, pl.heads, pl.nheads, M, pl.mdup,
                                                    pl.heads_cap);
    HOLE_LAUNCHED();
  }
  HOLE_CUDA_TRY(cudaEventRecord(pl.ready, ps));
  // (off the consumer's path) clean bitmaps for the next plan in this slot; report the largest step to the host
  HOLE_CUDA_TRY(cudaMemsetAsync(pl.seen, 0, (size_t)2 * pl.bitmap_words * 4, ps));   // seen | dup (one allocation)
  hole_plan_dupmax_kernel<<<1, 256, 0, ps>>>(pl.mdup, (int)S, c->dup_max_host_dev + (&pl - c->plan));
  HOLE_LAUNCHED();
  return HOLE_OK;
}

// The training calls without an AdaGrad form refuse it here, before they enqueue anything (a refused call
// leaves the context as it was): the delta-table and log-loss steps, the row-sharded steps, and every
// training call in the archived ccorr/tanh score mode.
enum { HOLE_STEP_TABLE, HOLE_STEP_DELTA, HOLE_STEP_LOGLOSS, HOLE_STEP_SHARD };
static int optimizer_refusal(const hole_ctx* c, int kind) {
  if (c->optimizer == HOLE_OPT_SGD) return HOLE_OK;
  if (kind == HOLE_STEP_DELTA)
    return hole_set_error(HOLE_ERR_UNSUPPORTED, "AdaGrad updates the table in place: no delta-table step");
  if (kind == HOLE_STEP_LOGLOSS)
    return hole_set_error(HOLE_ERR_UNSUPPORTED, "AdaGrad has no log-loss step (its L2 gradient is dense)");
  if (kind == HOLE_STEP_SHARD) return hole_set_error(HOLE_ERR_UNSUPPORTED, "AdaGrad has no row-sharded step");
  if (c->score_mode != HOLE_SCORE_COMPLEX)
    return hole_set_error(HOLE_ERR_UNSUPPORTED, "the archived ccorr/tanh score mode has no AdaGrad step");
  return HOLE_OK;
}

// K1 + K3 of one step whose plan is slot `slot` of pl.
// shard != nullptr (hole_shard_step): pos / neg are the step's triples as request-list rows (what the
// plan was built on), shard_tri / shard_neg the same triples as global row ids (what K1 gathers).
static int run_step(hole_ctx* c, hole_plan& pl, float* table, const int32_t* pos, const int32_t* neg,
                    int side, int64_t B, float margin, float lr, float* loss_out, float* sigma_out,
                    int64_t slot, cudaStream_t st, float* delta_out = nullptr, bool k1_follows_k3 = false,
                    int flags = 0, const hole_k1_shard* shard = nullptr, const int32_t* shard_tri = nullptr,
                    const int32_t* shard_neg = nullptr, cudaEvent_t k1_done_mark = nullptr) {
  const int M = (int)(4 * B);
  const size_t off = (size_t)slot * M;
  cudaEvent_t* pe = nullptr;
  if (c->profile) {
    if (c->prof_used + 3 > c->prof_ev.size()) {
      for (int q = 0; q < 3; ++q) {
        cudaEvent_t e;
        HOLE_CUDA_TRY(cudaEventCreate(&e));
        c->prof_ev.push_back(e);
      }
    }
    pe = &c->prof_ev[c->prof_used];
    c->prof_used += 3;
    HOLE_CUDA_TRY(cudaEventRecord(pe[0], st));
  }
  // K1's prologue reads plan data before griddepcontrol.wait: only overlap it with a
  // predecessor that does not write the plan, i.e. the previous step's K3 of the same chunk
  hole_k3_shard k3s = {};
  if (shard != nullptr) {
    k3s.cuts = shard->cuts; k3s.R = shard->R; k3s.me = shard->me; k3s.world = shard->world;
    k3s.cap = shard->cap; k3s.stage = shard->stage;
  }
  if (c->score_mode == HOLE_SCORE_CCORR_TANH) {
    if (shard != nullptr || delta_out != nullptr || (flags & 3) != 0)
      return hole_set_error(HOLE_ERR_UNSUPPORTED, "the archived ccorr/tanh score mode supports the hinge step on one table only");
    int rc = cc_prepare(c);
    if (rc) return rc;
    const int fw = cc_warp_floats(c->H), warps = cc_warps(fw);
    const int64_t groups = (B + pl.T - 1) / pl.T;
    const unsigned grid = (unsigned)((groups + warps - 1) / warps);
    HOLE_CC_DISPATCH(cc_nv(c), (hole_ccorr_fwd_bwd_kernel<NV><<<grid, 32 * warps, (size_t)warps * fw * sizeof(float), st>>>(
                                   table, pos, neg, pl.perm + (size_t)slot * B, pl.gslot + off, side, (int)B, pl.T, c->H,
                                   c->row_stride, margin, lr, c->G, loss_out, sigma_out)));
    HOLE_CUDA_TRY(cudaGetLastError());
    HOLE_LAUNCHED();
  } else {
    hole_k1_args ka = {};
    ka.E = table; ka.tri = shard ? shard_tri : pos; ka.neg = shard ? shard_neg : neg;
    ka.perm = pl.perm + (size_t)slot * B; ka.gslot = pl.gslot + off;
    ka.side = side; ka.B = (int)B; ka.T = pl.T; ka.nvec = c->nvec; ka.stride = c->row_stride;
    ka.margin = margin; ka.lr = lr; ka.G = c->G; ka.sigma = sigma_out; ka.Dtab = delta_out;
    ka.loss = (flags & 3) == 2 ? nullptr : loss_out;       // a log-loss pass without the positive term
    static const hole_k1_shard no_shard = {};
    int dm = (flags & 3) ? 3 : shard ? 2 : (delta_out ? 1 : 0);
    if (c->optimizer == HOLE_OPT_ADAGRAD) {     // (optimizer_refusal: only the in-place step gets here)
      dm = 4;
      ka.Dtab = c->accum;
    }
    int rc = k1_launch(c, dm, ka, shard ? *shard : no_shard, st, k1_follows_k3 && !c->profile);
    if (rc) return rc;
  }
  if (pe) HOLE_CUDA_TRY(cudaEventRecord(pe[1], st));
  if (k1_done_mark) HOLE_CUDA_TRY(cudaEventRecord(k1_done_mark, st));
  const unsigned k3_grid = std::min<unsigned>(grid_for_groups(pl.heads_cap, c->gs), (unsigned)c->sm_count * 4);
  if (c->optimizer == HOLE_OPT_ADAGRAD)
    HOLE_DISPATCH_PDL(c, hole_adagrad_apply_kernel, k3_grid, 256, 0, st, table, c->G,
                      pl.heads + (size_t)slot * pl.heads_cap, pl.nheads + slot, c->counters, M, c->nvec,
                      c->row_stride, lr, c->accum);
  else
    HOLE_DISPATCH_PDL(c, hole_apply_kernel, k3_grid, 256, 0, st, table, c->G,
                  pl.heads + (size_t)slot * pl.heads_cap, pl.nheads + slot, c->counters, M, c->nvec,
                  c->row_stride, lr, delta_out, flags, k3s);
  if (pe) HOLE_CUDA_TRY(cudaEventRecord(pe[2], st));
  return HOLE_OK;
}

extern "C" int hole_profile_enable(hole_ctx* c, int on) {
  HOLE_CHECK_ARG(c != nullptr);
  c->profile = on != 0;
  c->prof_used = 0;
  return HOLE_OK;
}

extern "C" int hole_profile_read(hole_ctx* c, double* k1_ms, double* k3_ms, int64_t* n_steps) {
  HOLE_CHECK_ARG(c && k1_ms && k3_ms && n_steps);
  HOLE_CUDA_TRY(cudaSetDevice(c->device));
  HOLE_CUDA_TRY(cudaDeviceSynchronize());
  double a = 0.0, b = 0.0;
  for (size_t q = 0; q + 2 < c->prof_used && q + 2 < c->prof_ev.size(); q += 3) {
    float t1 = 0.f, t3 = 0.f;
    HOLE_CUDA_TRY(cudaEventElapsedTime(&t1, c->prof_ev[q], c->prof_ev[q + 1]));
    HOLE_CUDA_TRY(cudaEventElapsedTime(&t3, c->prof_ev[q + 1], c->prof_ev[q + 2]));
    a += t1;
    b += t3;
  }
  *k1_ms = a;
  *k3_ms = b;
  *n_steps = (int64_t)(c->prof_used / 3);
  return HOLE_OK;
}

extern "C" int hole_train_step_plan(hole_ctx* c, const int32_t* pos, const int32_t* neg_ent, int64_t B,
                                    void* stream) {
  HOLE_CHECK_ARG(c && B >= 0);
  if (B == 0) return HOLE_OK;
  HOLE_CHECK_ARG(pos && neg_ent && 4 * B < (int64_t(1) << 31));
  HOLE_CUDA_TRY(cudaSetDevice(c->device));
  int rc = hole_ws_reserve(c, B, 1);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  // the plan stream reads pos / neg_ent once the caller's stream has produced them
  HOLE_CUDA_TRY(cudaEventRecord(c->ev_entry, st));
  HOLE_CUDA_TRY(cudaStreamWaitEvent(c->plan_stream, c->ev_entry, 0));
  // alternate between the two plan slots, so that the plan of step s+1 can be built while the
  // kernels of step s still read theirs
  hole_plan& pl = c->plan[c->plan_toggle];
  c->plan_toggle ^= 1;
  rc = plan_steps(c, pl, pos, B, 1, nullptr, nullptr, nullptr, 0, 0, neg_ent, c->plan_stream);
  if (rc) return rc;
  pl.prepared_pos = pos;
  pl.prepared_neg = neg_ent;
  pl.prepared_B = B;
  return HOLE_OK;
}

extern "C" int hole_train_step_ex(hole_ctx* c, float* table, float* delta_out, const int32_t* pos,
                                  const int32_t* neg_ent, int side, int64_t B, float margin, float lr,
                                  float* loss_out, float* sigma_out, void* stream) {
  HOLE_CHECK_ARG(c && B >= 0 && (side == 0 || side == 1));
  int rc = optimizer_refusal(c, delta_out ? HOLE_STEP_DELTA : HOLE_STEP_TABLE);
  if (rc) return rc;
  if (B == 0) return HOLE_OK;   // an empty batch is a no-op
  HOLE_CHECK_ARG(table && pos && neg_ent && loss_out);
  HOLE_CHECK_ARG(4 * B < (int64_t(1) << 31));
  HOLE_CUDA_TRY(cudaSetDevice(c->device));
  rc = hole_ws_reserve(c, B, 1);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  int slot_ix = -1;
  for (int q = 0; q < 2; ++q)
    if (c->plan[q].prepared_B == B && c->plan[q].prepared_pos == pos && c->plan[q].prepared_neg == neg_ent)
      slot_ix = q;
  const bool planned_ahead = slot_ix >= 0;
  if (!planned_ahead) slot_ix = (c->plan[0].prepared_B >= 0 && c->plan[1].prepared_B < 0) ? 1 : 0;
  hole_plan& pl = c->plan[slot_ix];
  if (planned_ahead) {
    HOLE_CUDA_TRY(cudaStreamWaitEvent(st, pl.ready, 0));     // planned ahead by hole_train_step_plan
  } else {
    // the plan's keys do not depend on the side, and the corruption is the caller's
    rc = plan_steps(c, pl, pos, B, 1, nullptr, nullptr, nullptr, 0, 0, neg_ent, st);
    if (rc) return rc;
  }
  pl.prepared_B = -1;
  pl.prepared_pos = pl.prepared_neg = nullptr;
  rc = run_step(c, pl, table, pos, neg_ent, side, B, margin, lr, loss_out, sigma_out, 0, st, delta_out);
  if (rc) return rc;
  pl.used = true;
  HOLE_CUDA_TRY(cudaEventRecord(pl.released, st));
  return HOLE_OK;
}

extern "C" int hole_train_step(hole_ctx* c, float* table, const int32_t* pos, const int32_t* neg_ent,
                               int side, int64_t B, float margin, float lr, float* loss_out,
                               float* sigma_out, void* stream) {
  return hole_train_step_ex(c, table, nullptr, pos, neg_ent, side, B, margin, lr, loss_out, sigma_out,
                            stream);
}

// ---------------------------------------------------------------------------------------
// --log_loss training step (holE.py:194-196, 206-220, 296): k = negative_ratio corrupt
// batches, each with its own side coin and draws (virtual step  step * k + j).  Every term's
// gradient is taken at the OLD table, so the k passes run K1/K3 in accumulate-delta mode on an
// untouched table (pass 0 carries the positive term), then the dense L2 decay and the summed
// deltas are applied.  delta_ws: table-sized, all zero on entry, all zero again on return.
// ---------------------------------------------------------------------------------------
extern "C" int hole_train_step_logloss(hole_ctx* c, float* table, float* delta_ws, const int32_t* triples,
                                       int64_t B, int negative_ratio, const int32_t* type_of,
                                       const int64_t* csr_off, const int32_t* csr_ids, uint64_t seed,
                                       uint64_t step, float lr, float l2, float* loss_out,
                                       float* l2_loss_out, int32_t* neg_out, int32_t* sides_out,
                                       void* stream) {
  HOLE_CHECK_ARG(c && B >= 0 && negative_ratio >= 1 && negative_ratio <= 64);
  if (c->score_mode != HOLE_SCORE_COMPLEX)
    return hole_set_error(HOLE_ERR_UNSUPPORTED, "the archived ccorr/tanh score mode has no log-loss branch");
  int rc = optimizer_refusal(c, HOLE_STEP_LOGLOSS);
  if (rc) return rc;
  if (B == 0) return HOLE_OK;
  HOLE_CHECK_ARG(table && delta_ws && triples && type_of && csr_off && csr_ids && loss_out);
  HOLE_CHECK_ARG(4 * B < (int64_t(1) << 31));
  HOLE_CUDA_TRY(cudaSetDevice(c->device));
  const int k = negative_ratio;
  rc = hole_ws_reserve(c, B, k);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  hole_plan& pl = c->plan[0];
  pl.prepared_B = -1;
  pl.prepared_pos = pl.prepared_neg = nullptr;
  const uint64_t v0 = step * (uint64_t)k;
  rc = plan_steps(c, pl, triples, B, k, type_of, csr_off, csr_ids, seed, v0, nullptr, st, /*tstride=*/0);
  if (rc) return rc;
  for (int j = 0; j < k; ++j) {
    const int side = hole_side_coin(seed, v0 + (uint64_t)j);
    if (sides_out) sides_out[j] = side;
    rc = run_step(c, pl, table, triples, pl.neg + (size_t)j * B, side, B, 0.0f, lr, loss_out,
                  loss_out + (size_t)(1 + j) * B, j, st, delta_ws, false,
                  (j == 0 ? 1 : 2) | HOLE_K1_ACCUMULATE);
    if (rc) return rc;
  }
  if (neg_out)
    HOLE_CUDA_TRY(cudaMemcpyAsync(neg_out, pl.neg, (size_t)k * B * 4, cudaMemcpyDeviceToDevice, st));
  if (l2 != 0.0f || l2_loss_out != nullptr) {
    const float scale = 1.0f - lr * (float)(1 + k) * (float)B * l2;
    const size_t n4 = (size_t)c->n_rows * c->row_stride / 4;
    const int blocks = c->sm_count * 8;
    float* partial = c->G;                 // the gradient staging area is free between steps
    hole_l2_scale_kernel<<<blocks, 256, 0, st>>>(reinterpret_cast<float4*>(table), n4, scale, partial);
    HOLE_LAUNCHED();
    float* out = l2_loss_out ? l2_loss_out : partial + blocks;
    hole_l2_finish_kernel<<<1, 256, 0, st>>>(partial, blocks, out);
    HOLE_LAUNCHED();
  }
  const int M = (int)(4 * B);
  for (int j = 0; j < k; ++j)
    HOLE_DISPATCH(c, hole_apply_delta_kernel, grid_for_groups(M, c->gs), 256, st, table, delta_ws,
                  pl.keysA + (size_t)j * M, pl.gslot + (size_t)j * M, pl.skey + (size_t)j * M, M, c->nvec,
                  c->row_stride);
  pl.used = true;
  HOLE_CUDA_TRY(cudaEventRecord(pl.released, st));
  return HOLE_OK;
}

extern "C" int hole_enable_peer_access(hole_ctx* c, int peer_device) {
  HOLE_CHECK_ARG(c && peer_device >= 0);
  if (peer_device == c->device) return HOLE_OK;
  HOLE_CUDA_TRY(cudaSetDevice(c->device));
  int can = 0;
  HOLE_CUDA_TRY(cudaDeviceCanAccessPeer(&can, c->device, peer_device));
  if (!can) return hole_set_error(HOLE_ERR_CUDA, "device %d cannot access peer %d", c->device, peer_device);
  cudaError_t e = cudaDeviceEnablePeerAccess(peer_device, 0);
  if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); return HOLE_OK; }
  HOLE_CUDA_TRY(e);
  return HOLE_OK;
}

extern "C" int hole_gather_rows(hole_ctx* c, const float* table, const int64_t* ids, int64_t id_offset,
                                float* dst_rows, int64_t n, void* stream) {
  HOLE_CHECK_ARG(c && n >= 0);
  if (n == 0) return HOLE_OK;
  HOLE_CHECK_ARG(table && ids && dst_rows);
  HOLE_CUDA_TRY(cudaSetDevice(c->device));
  HOLE_DISPATCH(c, hole_gather_rows_kernel, grid_for_groups(n, c->gs), 256, (cudaStream_t)stream, table, ids,
                dst_rows, n, id_offset, c->nvec, c->row_stride);
  return HOLE_OK;
}

extern "C" int hole_add_rows(hole_ctx* c, float* table, const int64_t* ids, int64_t id_offset,
                             const float* rows, int64_t n, void* stream) {
  HOLE_CHECK_ARG(c && n >= 0);
  if (n == 0) return HOLE_OK;
  HOLE_CHECK_ARG(table && ids && rows);
  HOLE_CUDA_TRY(cudaSetDevice(c->device));
  HOLE_DISPATCH(c, hole_add_rows_kernel, grid_for_groups(n, c->gs), 256, (cudaStream_t)stream, table, ids,
                rows, n, id_offset, c->nvec, c->row_stride);
  return HOLE_OK;
}

// ---------------------------------------------------------------------------------------
// multi-GPU step routing: host side (see the kernels above)
// ---------------------------------------------------------------------------------------
// scratch of the request routing for chunks of S steps of M = 3B keys
static int route_reserve(hole_ctx* c, int64_t M, int64_t S = 1) {
  if (M * S <= c->route_cap) return HOLE_OK;
  HOLE_CUDA_TRY(cudaDeviceSynchronize());
  cudaFree(c->route_buf);
  c->route_buf = nullptr;
  c->route_cap = 0;
  const size_t tiles = (M + ST_TILE - 1) / ST_TILE;
  const size_t rtiles = (M + RT_TILE - 1) / RT_TILE;
  const size_t words = (size_t)S * (4 * (size_t)M + std::max<size_t>(256 * tiles, rtiles + 1));
  if (cudaMalloc((void**)&c->route_buf, words * 4) != cudaSuccess) {
    cudaGetLastError();
    return hole_set_error(HOLE_ERR_ALLOC, "route workspace allocation failed");
  }
  c->route_cap = M * S;
  // the sort's ticket counters (one per step of a chunk; zero between uses)
  cudaFree(c->route_done);
  c->route_done = nullptr;
  const size_t nd = (size_t)std::max<int64_t>(S, 64);
  if (cudaMalloc((void**)&c->route_done, nd * sizeof(unsigned)) != cudaSuccess) {
    cudaGetLastError();
    return hole_set_error(HOLE_ERR_ALLOC, "route workspace allocation failed");
  }
  HOLE_CUDA_TRY(cudaMemset(c->route_done, 0, nd * sizeof(unsigned)));
  return HOLE_OK;
}

// S steps at once: pos [S][B][3], neg_ent [S][B] -> uniq_out [S][uniq_stride], cuts_out [S][HOLE_MAX_RANKS+1]
// (S == 1: exactly world+1 entries are written), pos_w [S][B][3], neg_w [S][B]
static int shard_route(hole_ctx* c, const int32_t* pos, const int32_t* neg_ent, int64_t B,
                       int64_t n_relations, int64_t n_rows_global, int64_t rows_per_rank,
                       int world, int32_t* uniq_out, int32_t* cuts_out, int32_t* pos_w,
                       int32_t* neg_w, void* stream, int64_t S = 1, int64_t uniq_stride = 0) {
  HOLE_CHECK_ARG(c && pos && neg_ent && uniq_out && cuts_out && pos_w && neg_w);
  HOLE_CHECK_ARG(B > 0 && 3 * B < (int64_t(1) << 31) && world >= 1 && world <= HOLE_MAX_RANKS && S >= 1);
  HOLE_CHECK_ARG(n_relations >= 0 && rows_per_rank > 0 && n_rows_global > n_relations &&
                 n_rows_global <= (int64_t(1) << 31));
  HOLE_CUDA_TRY(cudaSetDevice(c->device));
  const int M = (int)(3 * B);
  if (uniq_stride <= 0) uniq_stride = M;
  int rc = route_reserve(c, M, S);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t SM_ = (size_t)S * M;
  uint32_t *kA = c->route_buf, *kB = kA + SM_, *vA = kB + SM_, *vB = vA + SM_, *ghist = vB + SM_;
  int passes = 1;
  while (passes < 4 && (n_rows_global - 1) >> (8 * passes)) ++passes;
  dim3 kgrid((unsigned)std::min<int64_t>((B + 255) / 256, 1024), (unsigned)S);
  hole_shard_keys_kernel<<<kgrid, 256, 0, st>>>(pos, neg_ent, (int)B, kA);
  HOLE_LAUNCHED();
  uint32_t *sk, *sp;
  rc = radix_sort(ghist, kA, kB, vA, vB, nullptr, S, M, passes, st, &sk, &sp, c->route_done);
  if (rc) return rc;
  // the sort's tile histogram is free again: per step, tile head counts + the total live there
  const int tiles = (M + RT_TILE - 1) / RT_TILE;
  int* tile_heads = reinterpret_cast<int*>(ghist);
  dim3 tgrid((unsigned)tiles, (unsigned)S);
  hole_shard_count_kernel<<<tgrid, RT_THREADS, 0, st>>>(sk, M, tile_heads, pos, (int)B, pos_w);
  HOLE_LAUNCHED();
  hole_shard_assign_kernel<<<tgrid, RT_THREADS, 0, st>>>(sk, sp, M, (int)B, (int)n_relations, tile_heads,
                                                        uniq_stride, uniq_out, pos_w, neg_w);
  HOLE_LAUNCHED();
  hole_shard_cuts_kernel<<<(unsigned)S, 32, 0, st>>>(uniq_out, uniq_stride, tile_heads, tiles, (int)n_relations,
                                                    rows_per_rank, world, cuts_out);
  HOLE_LAUNCHED();
  return HOLE_OK;
}

extern "C" int hole_shard_route(hole_ctx* c, const int32_t* pos, const int32_t* neg_ent, int64_t B,
                                int64_t n_relations, int64_t n_rows_global, int64_t rows_per_rank,
                                int world, int32_t* uniq_out, int32_t* cuts_out, int32_t* pos_w,
                                int32_t* neg_w, void* stream) {
  return shard_route(c, pos, neg_ent, B, n_relations, n_rows_global, rows_per_rank, world, uniq_out, cuts_out,
                     pos_w, neg_w, stream);
}

static int peer_ptrs(hole_peer_ptrs& out, void* const* in, int world) {
  for (int k = 0; k < HOLE_MAX_RANKS; ++k) out.p[k] = nullptr;
  for (int k = 0; k < world; ++k) {
    if (in[k] == nullptr) return hole_set_error(HOLE_ERR_ARG, "peer pointer %d is null", k);
    out.p[k] = in[k];
  }
  return HOLE_OK;
}

extern "C" int hole_shard_post(hole_ctx* c, const int32_t* uniq, const int32_t* cuts, int world, int me,
                               int64_t cap, void* const* peer_inbox, void* const* peer_meta, void* stream) {
  HOLE_CHECK_ARG(c && uniq && cuts && peer_inbox && peer_meta);
  HOLE_CHECK_ARG(world >= 1 && world <= HOLE_MAX_RANKS && me >= 0 && me < world && cap > 0);
  HOLE_CUDA_TRY(cudaSetDevice(c->device));
  hole_peer_ptrs ib, mt;
  int rc = peer_ptrs(ib, peer_inbox, world);
  if (rc) return rc;
  rc = peer_ptrs(mt, peer_meta, world);
  if (rc) return rc;
  hole_shard_post_kernel<<<(unsigned)std::min<int64_t>((cap + 255) / 256, c->sm_count * 4), 256, 0,
                           (cudaStream_t)stream>>>(uniq, cuts, world, me, cap, ib, mt);
  HOLE_LAUNCHED();
  return HOLE_OK;
}

// steps planned per chunk: enough blocks for the plan kernels to fill the GPU, bounded memory
// (a function of B only, so that the workspace is sized once per batch size)
static int64_t plan_chunk(int64_t B) {
  const int64_t M = 4 * B;
  return std::max<int64_t>(32, std::min<int64_t>(256, (int64_t(1) << 23) / M));
}

// Chunk sizes of an n_steps call.  The first chunk's plan cannot overlap anything (nothing is
// training yet), so it is kept short -- ramp_first steps -- and the chunks grow by ramp_factor up to
// plan_chunk(B): every later plan is hidden behind the previous chunk's steps.
// from_host: HOLE_HOST_FIRST=n starts the host-buffer path with a chunk of n steps (its copy is exposed
// too); off by default -- measured slower at every n (profiles/r02_e2e_ab.jsonl: a second plan chain costs
// more than the shorter first copy saves).
static std::vector<int64_t> chunk_sizes(const hole_ctx* c, int64_t B, int64_t n_steps, bool from_host = false) {
  const int64_t S = plan_chunk(B);
  std::vector<int64_t> v;
  int64_t first = c->ramp_first;
  if (from_host && first <= 0 && c->host_first > 0 && n_steps > 2 * c->host_first) first = c->host_first;
  int64_t cur = first > 0 ? std::min<int64_t>(S, first) : S;
  for (int64_t left = n_steps; left > 0;) {
    const int64_t n = std::min(cur, left);
    v.push_back(n);
    left -= n;
    cur = (from_host && c->ramp_first <= 0) ? S : std::min<int64_t>(S, cur * std::max(2, c->ramp_factor));
  }
  return v;
}

// the S steps of one planned chunk on the compute stream
static int run_chunk(hole_ctx* c, hole_plan& pl, float* table, const int32_t* triples_dev, int64_t B,
                     int64_t S, uint64_t seed, uint64_t first_step, float margin, const float* lr_host,
                     float* loss_out, float* loss_sum_dev, cudaStream_t st) {
  HOLE_CUDA_TRY(cudaStreamWaitEvent(st, pl.ready, 0));
  for (int64_t k = 0; k < S; ++k) {
    int side = hole_side_coin(seed, first_step + (uint64_t)k);
    int rc = run_step(c, pl, table, triples_dev + (size_t)k * B * 3, pl.neg + (size_t)k * B, side, B,
                      margin, lr_host[k], loss_out + (size_t)k * B, nullptr, k, st, nullptr, k > 0);
    if (rc) return rc;
  }
  if (loss_sum_dev != nullptr) {
    hole_loss_sum_kernel<<<(unsigned)S, 256, 0, st>>>(loss_out, B, loss_sum_dev);
    HOLE_LAUNCHED();
  }
  pl.used = true;
  HOLE_CUDA_TRY(cudaEventRecord(pl.released, st));
  return HOLE_OK;
}

extern "C" int hole_train_steps(hole_ctx* c, float* table, const int32_t* triples, int64_t B,
                                int64_t n_steps, const int32_t* type_of, const int64_t* csr_off,
                                const int32_t* csr_ids, uint64_t seed, uint64_t first_step,
                                float margin, const float* lr, float* loss_out, float* loss_sum_out,
                                void* stream) {
  HOLE_CHECK_ARG(c && B >= 0 && n_steps >= 0);
  int rc = optimizer_refusal(c, HOLE_STEP_TABLE);
  if (rc) return rc;
  if (B == 0 || n_steps == 0) return HOLE_OK;
  HOLE_CHECK_ARG(table && triples && type_of && csr_off && csr_ids && lr);
  HOLE_CHECK_ARG(4 * B < (int64_t(1) << 31));
  HOLE_CUDA_TRY(cudaSetDevice(c->device));
  const int64_t S = plan_chunk(B);
  rc = hole_ws_reserve(c, B, S);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  // the plan stream may only read the caller's triples once the caller's stream got here
  HOLE_CUDA_TRY(cudaEventRecord(c->ev_entry, st));
  HOLE_CUDA_TRY(cudaStreamWaitEvent(c->plan_stream, c->ev_entry, 0));
  const std::vector<int64_t> sizes = chunk_sizes(c, B, n_steps);
  const int64_t nchunks = (int64_t)sizes.size();
  rc = plan_steps(c, c->plan[0], triples, B, sizes[0], type_of, csr_off, csr_ids, seed,
                  first_step, nullptr, c->plan_stream);
  if (rc) return rc;
  int64_t k0 = 0;
  for (int64_t ci = 0; ci < nchunks; k0 += sizes[ci], ++ci) {
    const int64_t s = sizes[ci];
    if (ci + 1 < nchunks) {   // plan the next chunk while this one trains
      const int64_t k1 = k0 + s, s1 = sizes[ci + 1];
      rc = plan_steps(c, c->plan[(ci + 1) & 1], triples + (size_t)k1 * B * 3, B, s1, type_of, csr_off,
                      csr_ids, seed, first_step + (uint64_t)k1, nullptr, c->plan_stream);
      if (rc) return rc;
    }
    float* lo = loss_out ? loss_out + (size_t)k0 * B : c->loss;
    rc = run_chunk(c, c->plan[ci & 1], table, triples + (size_t)k0 * B * 3, B, s, seed,
                   first_step + (uint64_t)k0, margin, lr + k0, lo,
                   loss_sum_out ? loss_sum_out + k0 : nullptr, st);
    if (rc) return rc;
  }
  return HOLE_OK;
}

extern "C" int hole_train_steps_host(hole_ctx* c, float* table, const int32_t* triples_host, int64_t B,
                                     int64_t n_steps, const int32_t* type_of, const int64_t* csr_off,
                                     const int32_t* csr_ids, uint64_t seed, uint64_t first_step,
                                     float margin, const float* lr, float* loss_sum_host,
                                     void* stream) {
  HOLE_CHECK_ARG(c && B >= 0 && n_steps >= 0);
  int rc = optimizer_refusal(c, HOLE_STEP_TABLE);
  if (rc) return rc;
  if (B == 0 || n_steps == 0) return HOLE_OK;
  HOLE_CHECK_ARG(table && triples_host && type_of && csr_off && csr_ids && lr && loss_sum_host);
  HOLE_CHECK_ARG(4 * B < (int64_t(1) << 31));
  HOLE_CUDA_TRY(cudaSetDevice(c->device));
  const int64_t S = plan_chunk(B);
  rc = hole_ws_reserve(c, B, S);
  if (rc) return rc;
  const int64_t stage_elems = S * B * 3;
  if (stage_elems > c->cap_stage) {
    HOLE_CUDA_TRY(cudaDeviceSynchronize());
    for (int k = 0; k < 2; ++k) {
      cudaFree(c->triples_stage[k]);
      c->triples_stage[k] = nullptr;
      if (cudaMalloc((void**)&c->triples_stage[k], stage_elems * 4) != cudaSuccess) {
        cudaGetLastError();
        c->cap_stage = 0;
        return hole_set_error(HOLE_ERR_ALLOC, "triple staging allocation failed");
      }
    }
    c->cap_stage = stage_elems;
  }
  if (n_steps > c->cap_pinned) {     // (sized generously: a page-locked allocation costs ~a step)
    if (c->loss_sum_pinned) cudaFreeHost(c->loss_sum_pinned);
    c->loss_sum_pinned = nullptr;
    c->cap_pinned = 0;
    const int64_t want = std::max<int64_t>(n_steps, 16384);
    HOLE_CUDA_TRY(cudaMallocHost((void**)&c->loss_sum_pinned, want * sizeof(float)));
    c->cap_pinned = want;
  }
  cudaStream_t st = (cudaStream_t)stream;
  HOLE_CUDA_TRY(cudaEventRecord(c->ev_entry, st));
  HOLE_CUDA_TRY(cudaStreamWaitEvent(c->copy_stream, c->ev_entry, 0));
  const std::vector<int64_t> sizes = chunk_sizes(c, B, n_steps, true);
  const int64_t nchunks = (int64_t)sizes.size();
  std::vector<int64_t> starts(nchunks, 0);
  for (int64_t ci = 1; ci < nchunks; ++ci) starts[ci] = starts[ci - 1] + sizes[ci - 1];
  // chunk ci: H2D copy into staging buffer ci&1 (copy stream) -> plan (plan stream) -> steps
  // (caller's stream).  Staging buffer b is free again when plan[b].released fires.
  auto stage_and_plan = [&](int64_t ci) -> int {
    const int b = (int)(ci & 1);
    const int64_t k0 = starts[ci], s = sizes[ci];
    if (c->plan[b].used) HOLE_CUDA_TRY(cudaStreamWaitEvent(c->copy_stream, c->plan[b].released, 0));
    HOLE_CUDA_TRY(cudaMemcpyAsync(c->triples_stage[b], triples_host + (size_t)k0 * B * 3,
                                  (size_t)s * B * 3 * 4, cudaMemcpyHostToDevice, c->copy_stream));
    HOLE_CUDA_TRY(cudaEventRecord(c->ev_copy[b], c->copy_stream));
    HOLE_CUDA_TRY(cudaStreamWaitEvent(c->plan_stream, c->ev_copy[b], 0));
    return plan_steps(c, c->plan[b], c->triples_stage[b], B, s, type_of, csr_off, csr_ids, seed,
                      first_step + (uint64_t)k0, nullptr, c->plan_stream);
  };
  rc = stage_and_plan(0);
  if (rc) return rc;
  for (int64_t ci = 0; ci < nchunks; ++ci) {
    const int b = (int)(ci & 1);
    const int64_t k0 = starts[ci], s = sizes[ci];
    if (ci + 1 < nchunks) {
      rc = stage_and_plan(ci + 1);
      if (rc) return rc;
    }
    rc = run_chunk(c, c->plan[b], table, c->triples_stage[b], B, s, seed, first_step + (uint64_t)k0,
                   margin, lr + k0, c->loss, c->loss_sum, st);
    if (rc) return rc;
    HOLE_CUDA_TRY(cudaMemcpyAsync(c->loss_sum_pinned + k0, c->loss_sum, (size_t)s * 4,
                                  cudaMemcpyDeviceToHost, st));
    // the next chunk's loss_sum kernel is ordered after this copy on st
  }
  HOLE_CUDA_TRY(cudaStreamSynchronize(st));
  for (int64_t k = 0; k < n_steps; ++k) loss_sum_host[k] = c->loss_sum_pinned[k];
  return HOLE_OK;
}

#include "hole_shard.cuh"

// ---------------------------------------------------------------------------------------
// CRC32C (Castagnoli) for the TF tensor-bundle checkpoint writer (host code; holE.py:359
// saver.save writes a masked crc32c per tensor and per SSTable block).
// ---------------------------------------------------------------------------------------
static uint32_t g_crc32c_table[8][256];
static bool g_crc32c_ready = false;

static void crc32c_init() {
  for (uint32_t i = 0; i < 256; ++i) {
    uint32_t c = i;
    for (int k = 0; k < 8; ++k) c = (c & 1) ? (c >> 1) ^ 0x82F63B78u : (c >> 1);
    g_crc32c_table[0][i] = c;
  }
  for (uint32_t i = 0; i < 256; ++i)
    for (int t = 1; t < 8; ++t)
      g_crc32c_table[t][i] = (g_crc32c_table[t - 1][i] >> 8) ^ g_crc32c_table[0][g_crc32c_table[t - 1][i] & 0xFF];
  g_crc32c_ready = true;
}

extern "C" uint32_t hole_crc32c(uint32_t crc, const void* data, uint64_t n) {
  if (!g_crc32c_ready) crc32c_init();
  const uint8_t* p = static_cast<const uint8_t*>(data);
  uint32_t c = crc ^ 0xFFFFFFFFu;
  while (n >= 8) {   // slice-by-8
    uint32_t lo, hi;
    memcpy(&lo, p, 4);
    memcpy(&hi, p + 4, 4);
    lo ^= c;
    c = g_crc32c_table[7][lo & 0xFF] ^ g_crc32c_table[6][(lo >> 8) & 0xFF] ^
        g_crc32c_table[5][(lo >> 16) & 0xFF] ^ g_crc32c_table[4][lo >> 24] ^
        g_crc32c_table[3][hi & 0xFF] ^ g_crc32c_table[2][(hi >> 8) & 0xFF] ^
        g_crc32c_table[1][(hi >> 16) & 0xFF] ^ g_crc32c_table[0][hi >> 24];
    p += 8;
    n -= 8;
  }
  while (n--) c = (c >> 8) ^ g_crc32c_table[0][(c ^ *p++) & 0xFF];
  return c ^ 0xFFFFFFFFu;
}

// ---------------------------------------------------------------------------------------
// Fast ingestion of the triple files (host code): `head<TAB>tail<TAB>relation\n`, decimal,
// no header (holE.py:76-81).  Replaces TextLineReader + decode_csv (holE.py:72-81) for the
// 30 M-line files of BASELINE config 1, where a Python-level parser takes minutes.
// Returns the number of triples (<= cap are stored), or a negative error.
// ---------------------------------------------------------------------------------------
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

extern "C" int64_t hole_parse_triples(const char* path, int32_t* out, int64_t cap) {
  if (path == nullptr || (out == nullptr && cap > 0)) return hole_set_error(HOLE_ERR_ARG, "hole_parse_triples: bad argument");
  int fd = open(path, O_RDONLY);
  if (fd < 0) return hole_set_error(HOLE_ERR_ARG, "cannot open %s", path);
  struct stat stt;
  if (fstat(fd, &stt) != 0) { close(fd); return hole_set_error(HOLE_ERR_ARG, "cannot stat %s", path); }
  const size_t size = (size_t)stt.st_size;
  if (size == 0) { close(fd); return 0; }
  const char* p = (const char*)mmap(nullptr, size, PROT_READ, MAP_PRIVATE, fd, 0);
  close(fd);
  if (p == MAP_FAILED) return hole_set_error(HOLE_ERR_ALLOC, "cannot map %s", path);
  const char* end = p + size;
  const char* q = p;
  int64_t n = 0, line = 0;
  int64_t rc = 0;
  while (q < end) {
    while (q < end && (*q == '\n' || *q == '\r')) ++q;      // blank lines
    if (q >= end) break;
    ++line;
    int64_t v[3];
    for (int f = 0; f < 3; ++f) {
      if (q >= end || *q < '0' || *q > '9') { rc = -1; break; }
      int64_t x = 0;
      while (q < end && *q >= '0' && *q <= '9') { x = x * 10 + (*q - '0'); if (x > 2147483647LL) { rc = -1; break; } ++q; }
      if (rc) break;
      v[f] = x;
      if (f < 2) { if (q < end && *q == '\t') ++q; else { rc = -1; break; } }
    }
    if (rc) break;
    if (q < end && *q != '\n' && *q != '\r') { rc = -1; break; }
    if (n < cap) { out[3 * n] = (int32_t)v[0]; out[3 * n + 1] = (int32_t)v[1]; out[3 * n + 2] = (int32_t)v[2]; }
    ++n;
  }
  munmap((void*)p, size);
  if (rc) return hole_set_error(HOLE_ERR_ARG, "%s: line %lld is not three tab-separated non-negative int32 values", path, (long long)line);
  return n;
}
