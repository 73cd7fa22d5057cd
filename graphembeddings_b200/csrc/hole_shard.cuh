// Row-sharded training step over NVLink peer memory (SURVEY.md 8e; no counterpart in the
// reference, which is single-device).  Included by hole_train.cu.
//
// Entity rows are partitioned into contiguous blocks, rank o owning rows
// [R + o*rows_per, R + (o+1)*rows_per); the R relation rows are replicated.  Every rank holds
// shard = [relations | its block] and maps (CUDA IPC) every peer's shard, delta staging buffer,
// relation staging buffer, request inbox and flag array.  One step of rank `me` on its slice of
// the global batch:
//
//   side stream (table independent; hole_shard_prepare works one step ahead):
//     Philox corruption keyed on the GLOBAL triple index -> route (dedup the 3B entity ids into
//     the request list `uniq`, per-owner cut points, triples re-indexed to request-list rows)
//     -> integer update plan
//   compute stream:
//     K1      posts my request lists to the owners' inboxes (peer stores, ids only), waits until every
//             peer's shard is current (flag A), GATHERS the rows of its triples
//             straight from the owners' shards (bulk async copies over NVLink), computes, and
//             stores every unique row's delta into my slice of the owner's staging buffer
//             (peer stores) -- the exchange is fused into the compute kernel, tile by tile
//     K3      ordered combine of rows used more than once -> same staging buffers
//     finish  my relation deltas -> every peer's relation staging; then signals flag B
//             ("my deltas and request lists of this step are delivered") to every peer
//     claim   waits for flag B of every peer; indexes the request lists by owned row
//     apply   adds the staged deltas to my shard -- a row
//             requested by several ranks gets its deltas in rank order, and the replicated
//             relation block takes every rank's deltas in rank order, so the result is
//             deterministic and the replicas stay bit-identical -- then signals flag A
//
// AdaGrad (hole_shard_set_optimizer): compute runs unchanged with lr = -1, so the staged rows are gradients;
// the owner's apply (hole_shard_adagrad_apply_kernel) sums a row's gradients in rank order, then updates the
// row and its accumulator row once.  The exchange is byte for byte that of an SGD step.
//
// No NCCL call and no host synchronisation inside a step; two flag waits per step, both at the
// head of a kernel that has work to do anyway.  Flags only grow (epoch = steps completed).
#pragma once

constexpr int SHARD_LOSS_CHUNK = 64;     // steps whose loss rows are kept before they are summed

constexpr int SHARD_PREP_STEPS = 16;     // steps whose table-independent part is built per launch chain

struct hole_shard_prep {                 // table-independent part of a chunk of steps, built ahead
  int32_t* uniq = nullptr;               // [S][cap]     request lists: sorted unique global entity rows
  int32_t* cuts = nullptr;               // [S][HOLE_MAX_RANKS+1]  first request-list slot per owner
  int32_t* pos_w = nullptr;              // [S][B,3]     triples as request-list rows (R + slot), relation kept
  int32_t* neg_w = nullptr;              // [S][B]
  int32_t* neg = nullptr;                // [S][B]       corrupt entity (global row)
  const int32_t* pos = nullptr;          // the triples this was built for: [n_steps][B,3]
  int64_t B = -1, n_steps = 0, consumed = 0;
  uint64_t seed = 0, first_step = 0;
  int plan_slot = 0;
  bool valid = false, used = false;
  cudaEvent_t freed = nullptr;           // recorded when the last step that reads this slot has been enqueued
};

struct hole_shard_state {
  int world = 0, me = 0;
  int64_t R = 0, n_ent = 0, rows_per = 0, max_batch = 0, cap = 0;
  float* shard = nullptr;
  hole_peer_ptrs p_shard, p_stage, p_relstage, p_inbox, p_meta, p_flags;
  int32_t* err = nullptr;
  unsigned long long timeout_ns = 600ull * 1000000000ull;
  const int32_t* type_of = nullptr;
  const int64_t* csr_off = nullptr;
  const int32_t* csr_ids = nullptr;
  float* Drel = nullptr;                 // [R, stride] my relation deltas of the running step (zero between steps)
  unsigned* done = nullptr;              // [2] last-block-done counters (finish, apply)
  unsigned* claim = nullptr;             // [rows_per] owner side: bit k = rank k lists the row this step
  int32_t* slot = nullptr;               // [world][rows_per] where in rank k's list
  float* loss = nullptr;                 // [SHARD_LOSS_CHUNK, max_batch]
  float* loss_sum = nullptr;             // [SHARD_LOSS_CHUNK]
  int32_t* stage_tri = nullptr;          // device staging of hole_shard_steps_host
  int64_t stage_cap = 0;
  float* loss_pinned = nullptr;          // pinned host + device mirrors of a call's loss sums
  float* sums_dev = nullptr;
  int64_t pinned_cap = 0;
  hole_shard_prep prep[2];
  int prep_toggle = 0;
  int epoch = 0;                         // steps completed
  int optimizer = HOLE_OPT_SGD;          // hole_shard_set_optimizer: the optimizer of the following steps
  float* accum = nullptr;                // AdaGrad: accumulator shard [R + rows_per, stride] (caller-owned)
  int step_optimizer = HOLE_OPT_SGD;     // latched by hole_shard_step_compute for the step's apply
  float step_lr = 0.f;
  float* step_accum = nullptr;
  std::vector<cudaEvent_t> prof_ev;      // hole_profile_enable: 6 events per step (phase boundaries)
  size_t prof_used = 0;
};

// ------------------------------------------------------------------------------------ kernels
// relation deltas of this step -> every peer's relation staging [world][R][stride] (slice `me`),
// my delta rows back to zero; the last block to finish signals flag B = epoch to every peer
template <int GS, int V>
__global__ void __launch_bounds__(256)
hole_shard_finish_kernel(float* __restrict__ Drel, int R, int me, int world, hole_peer_ptrs relstage,
                         hole_peer_ptrs flags, int epoch, unsigned* __restrict__ done, int nvec, int stride) {
  __shared__ bool s_last;
  const int lane = threadIdx.x % GS;
  const int gstride = (gridDim.x * blockDim.x) / GS;
  Row<V> z;
  row_zero(z);
  for (int r = (blockIdx.x * blockDim.x + threadIdx.x) / GS; r < R; r += gstride) {
    Row<V> d;
    row_load<GS, V, false>(d, Drel + (size_t)r * stride, lane, nvec);
    row_store<GS, V>(z, Drel + (size_t)r * stride, lane, nvec);
    for (int k = 0; k < world; ++k)
      row_store<GS, V>(d, static_cast<float*>(relstage.p[k]) + ((size_t)me * R + r) * stride, lane, nvec);
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(done, 1u) == gridDim.x - 1;
  __syncthreads();
  if (s_last) {
    if (threadIdx.x == 0) *done = 0;                    // self-reset for the next step
    __threadfence_system();
    if (threadIdx.x < world) {
      int* theirs = static_cast<int*>(flags.p[threadIdx.x]) + world + me;     // flags[1][me] on that rank
      asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(theirs), "r"(epoch) : "memory");
    }
  }
}

// Owner side, pass 1.  Waits for flag B of every peer (their deltas and request lists of this step are
// here), then records for every entry g of every rank k's request list (inbox[k][g], a row of mine):
// claim[row] |= 1 << k and slot[k][row] = g, so that pass 2 finds every rank's delta of a row directly.
__global__ void __launch_bounds__(256)
hole_shard_claim_kernel(const int32_t* __restrict__ inbox, const int32_t* __restrict__ meta, int world,
                        int64_t cap, int64_t row0, int64_t rows_per, unsigned* __restrict__ claim,
                        int32_t* __restrict__ slot, const int* __restrict__ my_flags, int wait_epoch,
                        int* __restrict__ err, unsigned long long timeout_ns) {
  __shared__ int s_pre[HOLE_MAX_RANKS + 1];
  hole_flags_wait(my_flags + world, world, wait_epoch, err, timeout_ns);
  if (threadIdx.x == 0) {
    int pre = 0;
    for (int k = 0; k < world; ++k) { s_pre[k] = pre; pre += meta[2 * k]; }
    s_pre[world] = pre;
  }
  __syncthreads();
  const int total = s_pre[world];
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
    int k = 0;
    while (e >= s_pre[k + 1]) ++k;
    const int g = e - s_pre[k];
    const int64_t row = (int64_t)inbox[(size_t)k * cap + g] - row0;
    atomicOr(claim + row, 1u << k);
    slot[(size_t)k * rows_per + row] = g;
  }
}

// Owner side, pass 2.  Items [0, R): replicated relation rows, shard[r] += relstage[k][r] for
// k = 0..world-1 in order.  Items R + e: entry e of the concatenated request lists; the group of the
// LOWEST rank that lists a row adds the staged deltas of every rank that lists it, in rank order (and
// clears the row's claim word); the other groups of that row do nothing.  The last block signals flag A.
template <int GS, int V>
__global__ void __launch_bounds__(256)
hole_shard_apply_kernel(float* __restrict__ shard, const int32_t* __restrict__ inbox,
                        const int32_t* __restrict__ meta, const float* __restrict__ stage,
                        const float* __restrict__ relstage, int R, int world, int me, int64_t cap,
                        int64_t row0, int64_t rows_per, unsigned* __restrict__ claim,
                        const int32_t* __restrict__ slot, hole_peer_ptrs flags, int signal_epoch,
                        unsigned* __restrict__ done, int nvec, int stride) {
  __shared__ int s_pre[HOLE_MAX_RANKS + 1];
  __shared__ bool s_last;
  if (threadIdx.x == 0) {
    int pre = 0;
    for (int k = 0; k < world; ++k) { s_pre[k] = pre; pre += meta[2 * k]; }
    s_pre[world] = pre;
  }
  __syncthreads();
  const int lane = threadIdx.x % GS;
  const int total = R + s_pre[world];
  const int gstride = (gridDim.x * blockDim.x) / GS;
  for (int item = (blockIdx.x * blockDim.x + threadIdx.x) / GS; item < total; item += gstride) {
    if (item < R) {
      float* erow = shard + (size_t)item * stride;
      Row<V> x, d;
      row_load<GS, V, false>(x, erow, lane, nvec);
      for (int k = 0; k < world; ++k) {
        row_load<GS, V, false>(d, relstage + ((size_t)k * R + item) * stride, lane, nvec);
        row_add(x, d);
      }
      row_store<GS, V>(x, erow, lane, nvec);
      continue;
    }
    const int e = item - R;
    int k = 0;
    while (e >= s_pre[k + 1]) ++k;
    const int64_t row = (int64_t)inbox[(size_t)k * cap + (e - s_pre[k])] - row0;
    unsigned m = __ldcg(claim + row);
    if ((m & (0u - m)) != (1u << k)) continue;           // a lower rank's group owns this row (or it is done)
    float* erow = shard + (size_t)(R + row) * stride;
    Row<V> x, d;
    row_load<GS, V, false>(x, erow, lane, nvec);
    while (m != 0) {
      const int l = __ffs(m) - 1;
      m &= m - 1;
      const int g = __ldcg(slot + (size_t)l * rows_per + row);
      row_load<GS, V, false>(d, stage + ((size_t)l * cap + g) * stride, lane, nvec);
      row_add(x, d);
    }
    row_store<GS, V>(x, erow, lane, nvec);
    if (lane == 0) claim[row] = 0;                       // ready for the next step
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(done, 1u) == gridDim.x - 1;
  __syncthreads();
  if (s_last) {
    if (threadIdx.x == 0) *done = 0;
    __threadfence_system();
    if (threadIdx.x < world) {
      int* theirs = static_cast<int*>(flags.p[threadIdx.x]) + me;             // flags[0][me] on that rank
      asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(theirs), "r"(signal_epoch) : "memory");
    }
  }
}

// Owner side, pass 2 of an AdaGrad step (hole_shard_set_optimizer).  The compute half ran with lr = -1, so the
// staged rows are the ranks' summed gradients (-(-1) * g and 1 * g are exact).  Same items, claim / slot protocol
// and flag A as hole_shard_apply_kernel, but a row's gradients are summed first, then applied once, as
// SparseApplyAdagrad after TF's duplicate-index sum:
//   g = sum_k staged_k[row] (rank order);  A[row] += g^2;  E[row] -= lr * g * rsqrt(A[row])
// with the expressions of the single-GPU step (k1_emit DM 4, the root of hole_apply_body<.., true>).  Relation
// rows (items [0, R)) take g = sum_k relstage[k][r] on every rank, so the table and accumulator replicas stay
// bit-identical.  A row whose gradient is zero everywhere keeps both rows (A + 0 = A, x + (-lr * 0) * s = x).
template <int GS, int V>
__global__ void __launch_bounds__(256)
hole_shard_adagrad_apply_kernel(float* __restrict__ shard, float* __restrict__ accum,
                                const int32_t* __restrict__ inbox, const int32_t* __restrict__ meta,
                                const float* __restrict__ stage, const float* __restrict__ relstage, int R, int world,
                                int me, int64_t cap, int64_t row0, int64_t rows_per, unsigned* __restrict__ claim,
                                const int32_t* __restrict__ slot, hole_peer_ptrs flags, int signal_epoch,
                                unsigned* __restrict__ done, int nvec, int stride, float lr) {
  __shared__ int s_pre[HOLE_MAX_RANKS + 1];
  __shared__ bool s_last;
  if (threadIdx.x == 0) {
    int pre = 0;
    for (int k = 0; k < world; ++k) { s_pre[k] = pre; pre += meta[2 * k]; }
    s_pre[world] = pre;
  }
  __syncthreads();
  const int lane = threadIdx.x % GS;
  const int total = R + s_pre[world];
  const int gstride = (gridDim.x * blockDim.x) / GS;
  for (int item = (blockIdx.x * blockDim.x + threadIdx.x) / GS; item < total; item += gstride) {
    Row<V> g, d;
    size_t r;                                            // shard / accumulator row
    if (item < R) {
      r = (size_t)item;
      row_zero(g);
      for (int k = 0; k < world; ++k) {
        row_load<GS, V, false>(d, relstage + ((size_t)k * R + item) * stride, lane, nvec);
        row_add(g, d);
      }
    } else {
      const int e = item - R;
      int k = 0;
      while (e >= s_pre[k + 1]) ++k;
      const int64_t row = (int64_t)inbox[(size_t)k * cap + (e - s_pre[k])] - row0;
      unsigned m = __ldcg(claim + row);
      if ((m & (0u - m)) != (1u << k)) continue;         // a lower rank's group owns this row (or it is done)
      r = (size_t)(R + row);
      row_zero(g);
      while (m != 0) {
        const int l = __ffs(m) - 1;
        m &= m - 1;
        const int gi = __ldcg(slot + (size_t)l * rows_per + row);
        row_load<GS, V, false>(d, stage + ((size_t)l * cap + gi) * stride, lane, nvec);
        row_add(g, d);
      }
      if (lane == 0) claim[row] = 0;                     // ready for the next step
    }
    float* erow = shard + r * stride;
    float* arow = accum + r * stride;
    Row<V> x, a;
    row_load<GS, V, false>(x, erow, lane, nvec);
    row_load<GS, V, false>(a, arow, lane, nvec);
#pragma unroll
    for (int k = 0; k < 4 * V; ++k) {
      a.re[k] = fmaf(g.re[k], g.re[k], a.re[k]);
      a.im[k] = fmaf(g.im[k], g.im[k], a.im[k]);
      x.re[k] = fmaf(-lr * g.re[k], __frsqrt_rn(a.re[k]), x.re[k]);
      x.im[k] = fmaf(-lr * g.im[k], __frsqrt_rn(a.im[k]), x.im[k]);
    }
    row_store<GS, V>(a, arow, lane, nvec);
    row_store<GS, V>(x, erow, lane, nvec);
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(done, 1u) == gridDim.x - 1;
  __syncthreads();
  if (s_last) {
    if (threadIdx.x == 0) *done = 0;
    __threadfence_system();
    if (threadIdx.x < world) {
      int* theirs = static_cast<int*>(flags.p[threadIdx.x]) + me;             // flags[0][me] on that rank
      asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(theirs), "r"(signal_epoch) : "memory");
    }
  }
}

// ------------------------------------------------------------------------------------ host side
static void shard_free(hole_ctx* c) {
  hole_shard_state* s = c->shard_state;
  if (s == nullptr) return;
  for (int b = 0; b < 2; ++b) {
    cudaFree(s->prep[b].uniq); cudaFree(s->prep[b].cuts); cudaFree(s->prep[b].pos_w);
    cudaFree(s->prep[b].neg_w); cudaFree(s->prep[b].neg);
    if (s->prep[b].freed) cudaEventDestroy(s->prep[b].freed);
  }
  cudaFree(s->claim); cudaFree(s->slot);
  cudaFree(s->Drel); cudaFree(s->done); cudaFree(s->loss); cudaFree(s->loss_sum); cudaFree(s->stage_tri);
  cudaFree(s->sums_dev);
  for (cudaEvent_t e : s->prof_ev) cudaEventDestroy(e);
  if (s->loss_pinned) cudaFreeHost(s->loss_pinned);
  delete s;
  c->shard_state = nullptr;
}

extern "C" int hole_shard_init(hole_ctx* c, int world, int me, int64_t n_relations, int64_t n_entities,
                               int64_t rows_per_rank, int64_t max_batch, float* shard,
                               void* const* peer_shard, void* const* peer_stage, void* const* peer_relstage,
                               void* const* peer_inbox, void* const* peer_meta, void* const* peer_flags,
                               int32_t* err_flag, double timeout_s, const int32_t* type_of,
                               const int64_t* csr_off, const int32_t* csr_ids) {
  HOLE_CHECK_ARG(c && shard && peer_shard && peer_stage && peer_relstage && peer_inbox && peer_meta && peer_flags);
  HOLE_CHECK_ARG(err_flag && type_of && csr_off && csr_ids);
  if (c->score_mode != HOLE_SCORE_COMPLEX)
    return hole_set_error(HOLE_ERR_UNSUPPORTED, "the archived ccorr/tanh score mode has no row-sharded step");
  int rc = optimizer_refusal(c, HOLE_STEP_SHARD);
  if (rc) return rc;
  HOLE_CHECK_ARG(world >= 1 && world <= HOLE_MAX_RANKS && me >= 0 && me < world);
  HOLE_CHECK_ARG(n_relations >= 0 && n_entities > 0 && rows_per_rank > 0 && rows_per_rank * world >= n_entities);
  HOLE_CHECK_ARG(n_relations + rows_per_rank * world < (int64_t(1) << 31));
  HOLE_CHECK_ARG(max_batch > 0 && 4 * max_batch < (int64_t(1) << 31));
  HOLE_CUDA_TRY(cudaSetDevice(c->device));
  shard_free(c);
  // the training kernel of a sharded step is NVLink-bound: keep a few SMs' worth of block slots free so
  // that the side stream's routing / plan kernels of the next chunk run beside it, not after it
  int reserve = 12;
  if (const char* e = getenv("HOLE_SHARD_RESERVE_SMS")) reserve = atoi(e);
  rc = hole_ws_reserve(c, max_batch, SHARD_PREP_STEPS);
  if (rc) return rc;
  if (world > 1 && reserve > 0 && reserve < c->sm_count / 2)
    c->k1_groups = c->k1_groups / c->sm_count * (c->sm_count - reserve);
  hole_shard_state* s = new hole_shard_state();
  c->shard_state = s;
  s->world = world; s->me = me; s->R = n_relations; s->n_ent = n_entities; s->rows_per = rows_per_rank;
  s->max_batch = max_batch; s->cap = 3 * max_batch; s->shard = shard; s->err = err_flag;
  if (timeout_s > 0) s->timeout_ns = (unsigned long long)(timeout_s * 1e9);
  s->type_of = type_of; s->csr_off = csr_off; s->csr_ids = csr_ids;
  if ((rc = peer_ptrs(s->p_shard, peer_shard, world)) || (rc = peer_ptrs(s->p_stage, peer_stage, world)) ||
      (rc = peer_ptrs(s->p_relstage, peer_relstage, world)) || (rc = peer_ptrs(s->p_inbox, peer_inbox, world)) ||
      (rc = peer_ptrs(s->p_meta, peer_meta, world)) || (rc = peer_ptrs(s->p_flags, peer_flags, world))) {
    shard_free(c);
    return rc;
  }
  if (s->p_shard.p[me] != shard) {
    shard_free(c);
    return hole_set_error(HOLE_ERR_ARG, "hole_shard_init: peer_shard[me] must be this rank's shard");
  }
#define SH_ALLOC(ptr, bytes)                                                             \
  do {                                                                                   \
    if (cudaMalloc((void**)&(ptr), (bytes)) != cudaSuccess) {                            \
      cudaGetLastError();                                                                \
      shard_free(c);                                                                     \
      return hole_set_error(HOLE_ERR_ALLOC, "sharded-step allocation of %zu bytes failed", (size_t)(bytes)); \
    }                                                                                    \
  } while (0)
  const size_t rowb = (size_t)c->row_stride * sizeof(float);
  SH_ALLOC(s->Drel, std::max<size_t>(1, (size_t)s->R) * rowb);
  SH_ALLOC(s->done, 2 * sizeof(unsigned));
  SH_ALLOC(s->claim, (size_t)rows_per_rank * sizeof(unsigned));
  SH_ALLOC(s->slot, (size_t)world * rows_per_rank * sizeof(int32_t));
  SH_ALLOC(s->loss, (size_t)SHARD_LOSS_CHUNK * max_batch * 4);
  SH_ALLOC(s->loss_sum, (size_t)SHARD_LOSS_CHUNK * 4);
  for (int b = 0; b < 2; ++b) {
    const size_t S = SHARD_PREP_STEPS;
    SH_ALLOC(s->prep[b].uniq, S * (size_t)s->cap * 4);
    SH_ALLOC(s->prep[b].cuts, S * (size_t)(HOLE_MAX_RANKS + 1) * 4);
    SH_ALLOC(s->prep[b].pos_w, S * (size_t)max_batch * 12);
    SH_ALLOC(s->prep[b].neg_w, S * (size_t)max_batch * 4);
    SH_ALLOC(s->prep[b].neg, S * (size_t)max_batch * 4);
    s->prep[b].plan_slot = b;
    HOLE_CUDA_TRY(cudaEventCreateWithFlags(&s->prep[b].freed, cudaEventDisableTiming));
  }
#undef SH_ALLOC
  HOLE_CUDA_TRY(cudaMemset(s->Drel, 0, std::max<size_t>(1, (size_t)s->R) * rowb));
  HOLE_CUDA_TRY(cudaMemset(s->done, 0, 2 * sizeof(unsigned)));
  HOLE_CUDA_TRY(cudaMemset(s->claim, 0, (size_t)rows_per_rank * sizeof(unsigned)));
  rc = route_reserve(c, 3 * max_batch, SHARD_PREP_STEPS);
  if (rc) { shard_free(c); return rc; }
  HOLE_CUDA_TRY(cudaDeviceSynchronize());
  return HOLE_OK;
}

// The optimizer of the row-sharded steps; it lives in the shard state (hole_shard_init resets it to SGD) and
// leaves the context's own optimizer (hole_ctx_set_optimizer) alone.
extern "C" int hole_shard_set_optimizer(hole_ctx* c, int optimizer, float* accum_shard) {
  HOLE_CHECK_ARG(c != nullptr);
  if (c->shard_state == nullptr) return hole_set_error(HOLE_ERR_ARG, "hole_shard_init has not been called");
  HOLE_CHECK_ARG((optimizer == HOLE_OPT_SGD && accum_shard == nullptr) ||
                 (optimizer == HOLE_OPT_ADAGRAD && accum_shard != nullptr));
  c->shard_state->optimizer = optimizer;
  c->shard_state->accum = accum_shard;
  return HOLE_OK;
}

// Corruption + routing + update plan of n_steps (<= SHARD_PREP_STEPS) consecutive steps on the library's
// side stream; pos = [n_steps][B,3].  wait_caller: the side stream first waits for everything enqueued
// on `st` so far (the triples may have been produced there).
static int shard_prepare(hole_ctx* c, const int32_t* pos, int64_t B, int64_t n_steps, uint64_t seed,
                         uint64_t first_step, cudaStream_t st, bool wait_caller) {
  hole_shard_state* s = c->shard_state;
  hole_shard_prep& p = s->prep[s->prep_toggle];
  s->prep_toggle ^= 1;
  cudaStream_t ps = c->plan_stream;
  if (wait_caller) {
    HOLE_CUDA_TRY(cudaEventRecord(c->ev_entry, st));
    HOLE_CUDA_TRY(cudaStreamWaitEvent(ps, c->ev_entry, 0));
  }
  if (p.used) HOLE_CUDA_TRY(cudaStreamWaitEvent(ps, p.freed, 0));      // its last consumer is done
  p.pos = pos; p.B = B; p.n_steps = n_steps; p.consumed = 0; p.seed = seed; p.first_step = first_step;
  const uint64_t index_base = (uint64_t)s->me * (uint64_t)B;           // my slice of the global batch
  dim3 grid((unsigned)std::min<int64_t>((B + 255) / 256, 65535), (unsigned)n_steps);
  hole_corrupt_kernel<<<grid, 256, 0, ps>>>(pos, B, (int)n_steps, s->type_of, s->csr_off, s->csr_ids, seed,
                                            first_step, index_base, p.neg, nullptr);
  HOLE_LAUNCHED();
  int rc = shard_route(c, pos, p.neg, B, s->R, s->R + s->rows_per * s->world, s->rows_per, s->world, p.uniq, p.cuts,
                       p.pos_w, p.neg_w, ps, n_steps, s->cap);
  if (rc) return rc;
  hole_plan& pl = c->plan[p.plan_slot];
  pl.prepared_B = -1;
  pl.prepared_pos = pl.prepared_neg = nullptr;
  rc = plan_steps(c, pl, p.pos_w, B, n_steps, nullptr, nullptr, nullptr, 0, 0, p.neg_w, ps);
  if (rc) return rc;
  p.valid = true;
  return HOLE_OK;
}

static int shard_check_args(hole_ctx* c, const int32_t* pos, int64_t B) {
  HOLE_CHECK_ARG(c != nullptr);
  int rc = optimizer_refusal(c, HOLE_STEP_SHARD);
  if (rc) return rc;
  if (c->shard_state == nullptr) return hole_set_error(HOLE_ERR_ARG, "hole_shard_init has not been called");
  HOLE_CHECK_ARG(pos != nullptr && B > 0 && B <= c->shard_state->max_batch);
  return HOLE_OK;
}

extern "C" int hole_shard_prepare(hole_ctx* c, const int32_t* pos, int64_t B, uint64_t seed, uint64_t step,
                                  void* stream) {
  int rc = shard_check_args(c, pos, B);
  if (rc) return rc;
  HOLE_CUDA_TRY(cudaSetDevice(c->device));
  return shard_prepare(c, pos, B, 1, seed, step, (cudaStream_t)stream, true);
}

// measurement hook (hole_profile_enable): phase boundary `which` (0..5) of the running step
static int shard_mark(hole_ctx* c, int which, cudaStream_t st) {
  hole_shard_state* s = c->shard_state;
  if (!c->profile) return HOLE_OK;
  if (which == 0) {
    if (s->prof_used + 6 > s->prof_ev.size())
      for (int q = 0; q < 6; ++q) {
        cudaEvent_t e;
        HOLE_CUDA_TRY(cudaEventCreate(&e));
        s->prof_ev.push_back(e);
      }
    s->prof_used += 6;
  }
  HOLE_CUDA_TRY(cudaEventRecord(s->prof_ev[s->prof_used - 6 + which], st));
  return HOLE_OK;
}

// post + K1 + K3 + finish of the step
extern "C" int hole_shard_step_compute(hole_ctx* c, const int32_t* pos, int64_t B, uint64_t seed, uint64_t step,
                                       float margin, float lr, float* loss_out, void* stream) {
  int rc = shard_check_args(c, pos, B);
  if (rc) return rc;
  HOLE_CHECK_ARG(loss_out != nullptr);
  HOLE_CUDA_TRY(cudaSetDevice(c->device));
  hole_shard_state* s = c->shard_state;
  cudaStream_t st = (cudaStream_t)stream;
  // the prepared chunk this step belongs to (its next unconsumed step), else prepare it now
  int pi = -1;
  for (int b = 0; b < 2; ++b) {
    const hole_shard_prep& q = s->prep[b];
    if (q.valid && q.B == B && q.seed == seed && q.consumed < q.n_steps && step == q.first_step + (uint64_t)q.consumed &&
        pos == q.pos + (size_t)q.consumed * B * 3)
      pi = b;
  }
  if (pi < 0) {
    pi = s->prep_toggle;
    rc = shard_prepare(c, pos, B, 1, seed, step, st, true);
    if (rc) return rc;
  }
  hole_shard_prep& p = s->prep[pi];
  const int64_t k = p.consumed;                              // step of the chunk
  const int32_t* p_uniq = p.uniq + (size_t)k * s->cap;
  const int32_t* p_cuts = p.cuts + (size_t)k * (HOLE_MAX_RANKS + 1);
  const int32_t* p_pos_w = p.pos_w + (size_t)k * B * 3;
  const int32_t* p_neg_w = p.neg_w + (size_t)k * B;
  const int32_t* p_neg = p.neg + (size_t)k * B;
  const int side = hole_side_coin(seed, step);
  hole_plan& pl = c->plan[p.plan_slot];
  HOLE_CUDA_TRY(cudaStreamWaitEvent(st, pl.ready, 0));       // corruption, routing and plan are complete
  const int par = s->epoch & 1;
  const int world = s->world, me = s->me;
  // my request lists -> the owners' inboxes of this step's parity
  hole_peer_ptrs ib, mt;
  for (int k = 0; k < HOLE_MAX_RANKS; ++k) {
    ib.p[k] = k < world ? static_cast<int32_t*>(s->p_inbox.p[k]) + (size_t)par * world * s->cap : nullptr;
    mt.p[k] = k < world ? static_cast<int32_t*>(s->p_meta.p[k]) + (size_t)par * world * 2 : nullptr;
  }
  if ((rc = shard_mark(c, 0, st))) return rc;
  if ((rc = shard_mark(c, 1, st))) return rc;
  hole_k1_shard sh = {};
  sh.tri_w = p_pos_w; sh.neg_w = p_neg_w; sh.cuts = p_cuts;
  sh.flags = static_cast<const int*>(s->p_flags.p[me]);
  sh.err = s->err; sh.wait_epoch = s->epoch; sh.R = (int)s->R; sh.rows_per = (int)s->rows_per;
  sh.me = me; sh.world = world; sh.cap = s->cap; sh.timeout_ns = s->timeout_ns;
  sh.shard = s->p_shard; sh.stage = s->p_stage;
  sh.uniq = p_uniq; sh.inbox = ib; sh.meta = mt;          // the request lists are posted by K1 itself
  // AdaGrad: K1 / K3 stage -(-1) * g = g, the ranks' summed gradients, and the owners apply lr (latched here
  // for hole_shard_step_apply)
  const bool ada = s->optimizer == HOLE_OPT_ADAGRAD;
  s->step_optimizer = s->optimizer; s->step_lr = lr; s->step_accum = s->accum;
  rc = run_step(c, pl, s->shard, p_pos_w, p_neg_w, side, B, margin, ada ? -1.0f : lr, loss_out, nullptr, k, st,
                s->Drel, false, 0, &sh, pos, p_neg, c->profile ? s->prof_ev[s->prof_used - 6 + 2] : nullptr);
  if (rc) return rc;
  if ((rc = shard_mark(c, 3, st))) return rc;
  p.consumed += 1;
  if (p.consumed == p.n_steps) {                             // the chunk's buffers and plan are free again
    pl.used = true;
    HOLE_CUDA_TRY(cudaEventRecord(pl.released, st));
    p.used = true;
    p.valid = false;
    HOLE_CUDA_TRY(cudaEventRecord(p.freed, st));
  }
  const unsigned fgrid = (unsigned)std::max<int64_t>(1, std::min<int64_t>((s->R + (256 / c->gs) - 1) / (256 / c->gs), c->sm_count));
  HOLE_DISPATCH(c, hole_shard_finish_kernel, fgrid, 256, st, s->Drel, (int)s->R, me, world, s->p_relstage, s->p_flags,
                s->epoch + 1, s->done, c->nvec, c->row_stride);
  return shard_mark(c, 4, st);
}

// apply of the step: every peer's deltas -> my shard
extern "C" int hole_shard_step_apply(hole_ctx* c, void* stream) {
  HOLE_CHECK_ARG(c != nullptr);
  int rc = optimizer_refusal(c, HOLE_STEP_SHARD);
  if (rc) return rc;
  if (c->shard_state == nullptr) return hole_set_error(HOLE_ERR_ARG, "hole_shard_init has not been called");
  HOLE_CUDA_TRY(cudaSetDevice(c->device));
  hole_shard_state* s = c->shard_state;
  const int par = s->epoch & 1, world = s->world, me = s->me;
  const int32_t* inbox = static_cast<const int32_t*>(s->p_inbox.p[me]) + (size_t)par * world * s->cap;
  const int32_t* meta = static_cast<const int32_t*>(s->p_meta.p[me]) + (size_t)par * world * 2;
  const int64_t row0 = s->R + (int64_t)me * s->rows_per;     // first global row of my block
  cudaStream_t st = (cudaStream_t)stream;
  hole_shard_claim_kernel<<<(unsigned)c->sm_count * 2, 256, 0, st>>>(
      inbox, meta, world, s->cap, row0, s->rows_per, s->claim, s->slot, static_cast<const int*>(s->p_flags.p[me]),
      s->epoch + 1, s->err, s->timeout_ns);
  HOLE_LAUNCHED();
  if (s->step_optimizer == HOLE_OPT_ADAGRAD)                 // the optimizer and lr of the step's compute half
    HOLE_DISPATCH(c, hole_shard_adagrad_apply_kernel, (unsigned)c->sm_count * 16, 256, st, s->shard, s->step_accum,
                  inbox, meta, static_cast<const float*>(s->p_stage.p[me]),
                  static_cast<const float*>(s->p_relstage.p[me]), (int)s->R, world, me, s->cap, row0, s->rows_per,
                  s->claim, s->slot, s->p_flags, s->epoch + 1, s->done + 1, c->nvec, c->row_stride, s->step_lr);
  else
    HOLE_DISPATCH(c, hole_shard_apply_kernel, (unsigned)c->sm_count * 16, 256, st, s->shard, inbox, meta,
                  static_cast<const float*>(s->p_stage.p[me]), static_cast<const float*>(s->p_relstage.p[me]),
                  (int)s->R, world, me, s->cap, row0, s->rows_per, s->claim, s->slot, s->p_flags, s->epoch + 1,
                  s->done + 1, c->nvec, c->row_stride);
  s->epoch += 1;
  return shard_mark(c, 5, (cudaStream_t)stream);
}

// Measurement hook: with hole_profile_enable on, every sharded step records events at its phase
// boundaries; returns the summed milliseconds of [post, K1 (incl. its wait for the peers' shards), K3,
// finish, apply (incl. its wait for the peers' deltas)] and the number of steps since the last enable.
extern "C" int hole_shard_profile_read(hole_ctx* c, double* phase_ms5, int64_t* n_steps) {
  HOLE_CHECK_ARG(c && phase_ms5 && n_steps);
  if (c->shard_state == nullptr) return hole_set_error(HOLE_ERR_ARG, "hole_shard_init has not been called");
  HOLE_CUDA_TRY(cudaSetDevice(c->device));
  HOLE_CUDA_TRY(cudaDeviceSynchronize());
  hole_shard_state* s = c->shard_state;
  for (int q = 0; q < 5; ++q) phase_ms5[q] = 0.0;
  for (size_t b = 0; b + 6 <= s->prof_used; b += 6)
    for (int q = 0; q < 5; ++q) {
      float t = 0.f;
      HOLE_CUDA_TRY(cudaEventElapsedTime(&t, s->prof_ev[b + q], s->prof_ev[b + q + 1]));
      phase_ms5[q] += t;
    }
  *n_steps = (int64_t)(s->prof_used / 6);
  s->prof_used = 0;
  return HOLE_OK;
}

extern "C" int hole_shard_step(hole_ctx* c, const int32_t* pos, int64_t B, uint64_t seed, uint64_t step,
                               float margin, float lr, float* loss_out, void* stream) {
  int rc = hole_shard_step_compute(c, pos, B, seed, step, margin, lr, loss_out, stream);
  if (rc) return rc;
  return hole_shard_step_apply(c, stream);
}

// n_steps consecutive steps on device-resident triples [n_steps*B, 3] (this rank's slices).  The
// table-independent part is built a chunk of SHARD_PREP_STEPS steps at a time, one chunk ahead of the
// chunk that is training.  loss_sum_out: device float32[n_steps].  copy_ready[i] (optional): event that
// marks the arrival of triple chunk i (copy_steps steps each; a multiple of SHARD_PREP_STEPS).
static int shard_steps(hole_ctx* c, const int32_t* triples, int64_t B, int64_t n_steps, uint64_t seed,
                       uint64_t first_step, float margin, const float* lr, float* loss_sum_out,
                       cudaStream_t st, const cudaEvent_t* copy_ready, int64_t copy_steps) {
  hole_shard_state* s = c->shard_state;
  const int64_t PS = SHARD_PREP_STEPS;
  int rc;
  auto prepare_chunk = [&](int64_t k0, bool first) -> int {
    const int64_t n = std::min<int64_t>(PS, n_steps - k0);
    if (copy_ready && k0 % copy_steps == 0)
      HOLE_CUDA_TRY(cudaStreamWaitEvent(c->plan_stream, copy_ready[k0 / copy_steps], 0));
    return shard_prepare(c, triples + (size_t)k0 * B * 3, B, n, seed, first_step + (uint64_t)k0, st, first);
  };
  rc = prepare_chunk(0, true);
  if (rc) return rc;
  for (int64_t k = 0; k < n_steps; ++k) {
    if (k % PS == 0 && k + PS < n_steps) {                   // next chunk, while this one trains
      rc = prepare_chunk(k + PS, false);
      if (rc) return rc;
    }
    const int64_t l0 = k / SHARD_LOSS_CHUNK * SHARD_LOSS_CHUNK;
    rc = hole_shard_step(c, triples + (size_t)k * B * 3, B, seed, first_step + (uint64_t)k, margin, lr[k],
                         s->loss + (size_t)(k - l0) * B, st);
    if (rc) return rc;
    if (loss_sum_out != nullptr && (k + 1 == n_steps || (k + 1) % SHARD_LOSS_CHUNK == 0)) {
      hole_loss_sum_kernel<<<(unsigned)(k + 1 - l0), 256, 0, st>>>(s->loss, B, loss_sum_out + l0);
      HOLE_LAUNCHED();
    }
  }
  return HOLE_OK;
}

extern "C" int hole_shard_steps(hole_ctx* c, const int32_t* triples, int64_t B, int64_t n_steps, uint64_t seed,
                                uint64_t first_step, float margin, const float* lr, float* loss_sum_out,
                                void* stream) {
  if (n_steps == 0) return HOLE_OK;
  int rc = shard_check_args(c, triples, B);
  if (rc) return rc;
  HOLE_CHECK_ARG(n_steps > 0 && lr != nullptr);
  HOLE_CUDA_TRY(cudaSetDevice(c->device));
  return shard_steps(c, triples, B, n_steps, seed, first_step, margin, lr, loss_sum_out, (cudaStream_t)stream,
                     nullptr, 0);
}

// Same, end to end from HOST triples (pinned or pageable): copied to the device in chunks that overlap
// the steps, per-step loss sums copied back; blocks until they are on the host.
extern "C" int hole_shard_steps_host(hole_ctx* c, const int32_t* triples_host, int64_t B, int64_t n_steps,
                                     uint64_t seed, uint64_t first_step, float margin, const float* lr,
                                     float* loss_sum_host, void* stream) {
  if (n_steps == 0) return HOLE_OK;
  int rc = shard_check_args(c, triples_host, B);
  if (rc) return rc;
  HOLE_CHECK_ARG(n_steps > 0 && lr != nullptr && loss_sum_host != nullptr);
  HOLE_CUDA_TRY(cudaSetDevice(c->device));
  hole_shard_state* s = c->shard_state;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t elems = n_steps * B * 3;
  if (elems > s->stage_cap) {
    HOLE_CUDA_TRY(cudaDeviceSynchronize());
    cudaFree(s->stage_tri);
    s->stage_tri = nullptr;
    s->stage_cap = 0;
    if (cudaMalloc((void**)&s->stage_tri, (size_t)elems * 4) != cudaSuccess) {
      cudaGetLastError();
      return hole_set_error(HOLE_ERR_ALLOC, "triple staging allocation failed");
    }
    s->stage_cap = elems;
  }
  if (n_steps > s->pinned_cap) {
    HOLE_CUDA_TRY(cudaDeviceSynchronize());
    if (s->loss_pinned) cudaFreeHost(s->loss_pinned);
    cudaFree(s->sums_dev);
  for (cudaEvent_t e : s->prof_ev) cudaEventDestroy(e);
    s->loss_pinned = nullptr;
    s->sums_dev = nullptr;
    s->pinned_cap = 0;
    HOLE_CUDA_TRY(cudaMallocHost((void**)&s->loss_pinned, (size_t)n_steps * sizeof(float)));
    HOLE_CUDA_TRY(cudaMalloc((void**)&s->sums_dev, (size_t)n_steps * sizeof(float)));
    s->pinned_cap = n_steps;
  }
  float* sums = s->sums_dev;
  // H2D in chunks of SHARD_PREP_STEPS steps on the copy stream; a chunk's preparation waits for its copy only
  const int64_t CS = SHARD_PREP_STEPS, nchunks = (n_steps + CS - 1) / CS;
  std::vector<cudaEvent_t> ready((size_t)nchunks);
  HOLE_CUDA_TRY(cudaEventRecord(c->ev_entry, st));
  HOLE_CUDA_TRY(cudaStreamWaitEvent(c->copy_stream, c->ev_entry, 0));   // the staging buffer's last readers are done
  for (int64_t ci = 0; ci < nchunks; ++ci) {
    const int64_t k0 = ci * CS, n = std::min(CS, n_steps - k0);
    HOLE_CUDA_TRY(cudaMemcpyAsync(s->stage_tri + (size_t)k0 * B * 3, triples_host + (size_t)k0 * B * 3,
                                  (size_t)n * B * 12, cudaMemcpyHostToDevice, c->copy_stream));
    HOLE_CUDA_TRY(cudaEventCreateWithFlags(&ready[ci], cudaEventDisableTiming));
    HOLE_CUDA_TRY(cudaEventRecord(ready[ci], c->copy_stream));
  }
  rc = shard_steps(c, s->stage_tri, B, n_steps, seed, first_step, margin, lr, sums, st, ready.data(), CS);
  if (rc == HOLE_OK) {
    cudaError_t e = cudaMemcpyAsync(s->loss_pinned, sums, (size_t)n_steps * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) rc = hole_set_error(HOLE_ERR_CUDA, "hole_shard_steps_host: %s", cudaGetErrorString(e));
  } else {
    cudaStreamSynchronize(st);
  }
  for (cudaEvent_t e : ready) cudaEventDestroy(e);
  if (rc) return rc;
  for (int64_t k = 0; k < n_steps; ++k) loss_sum_host[k] = s->loss_pinned[k];
  return HOLE_OK;
}

// Host check of the flag time-out (synchronises the stream): nonzero *timed_out means a peer never
// arrived and the tables are no longer consistent -- stop.
extern "C" int hole_shard_poll(hole_ctx* c, int* timed_out, void* stream) {
  HOLE_CHECK_ARG(c && timed_out);
  if (c->shard_state == nullptr) return hole_set_error(HOLE_ERR_ARG, "hole_shard_init has not been called");
  HOLE_CUDA_TRY(cudaSetDevice(c->device));
  int32_t v = 0;
  HOLE_CUDA_TRY(cudaMemcpyAsync(&v, c->shard_state->err, 4, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  HOLE_CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
  *timed_out = v;
  return HOLE_OK;
}
