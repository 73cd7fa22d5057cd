// K1: fused gather + norm clip + Hermitian score + sigmoid + loss + backward of one batch
// (holE.py:161-168, 191-192, 194-198, 231 and the backward TF derives for 296).
// Included by hole_train.cu (uses its Row<> helpers).
//
// A group of GS lanes walks T consecutive triples of the step's relation-grouped order (perm),
// software-pipelined: the rows of the next two triples are in flight while the current one is
// computed; the relation row is loaded once per run of equal relation and its gradient is summed
// over the run in registers.  A row that occurs exactly once in the step (gslot == UNIQUE) is
// read by nobody else during the step, so its change is written directly (see DM below);
// otherwise its gradient is staged in G (for a relation run at the run's first triple) for K3.
//   * rows are fetched with ONE 1-D bulk async copy per row (cp.async.bulk + mbarrier
//     complete_tx, SASS UBLKCP) issued by one elected lane of the lane group;
//   * rows stay UNSCALED in registers; the norm clip is carried as four scalars.  The score is
//     trilinear, so s(y) = sc_h sc_r sc_t s(x): the three sums of squares and the two raw scores
//     are reduced across the group in ONE round of shuffles;
//   * Euler's identity for a function linear in a row,  y . ds/dy = s,  gives the projection
//     term of the clip backward  dx = (dy - y (y.dy)) / |x|  as  g * s  -- no reduction;
//   * the gradients share their complex products: with U = g+ y_t + g- y_n (tail side) the head
//     and relation gradients are conj(r) o U and conj(h) o U (24 multiply-adds per complex
//     element for all four rows);
//   * DM selects where the step's row changes go: 0 in place on the table (single GPU),
//     1 into a local delta table (hole_train_step_ex), 2 row-sharded: rows are gathered straight
//     from their owners' shards over NVLink and every unique row's delta is stored into the
//     owner's staging buffer (peer memory), fused into this kernel (hole_shard_step);
//     3 is a --log_loss pass (hole_train_step_logloss): the table is read only and every unique
//     row's delta is ADDED to the delta table, which sums the passes over one old table.  The
//     loss is the only other difference; `loss` is null on the passes without the positive term.
//     4 is DM 0 with AdaGrad (hole_ctx_set_optimizer): a unique row also reads and writes its row
//     of the accumulator (carried in Dtab), with plain vector loads where the row is applied.
#pragma once

constexpr int K1_THREADS = 256;  // threads per block; at dim 768 their landing rows take 221,376 B of 227 KB

constexpr int K1V2_STAGES = 3;   // landing buffers per lane group: the triple being computed + 2 in flight

__device__ __forceinline__ uint32_t k1_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void k1_mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(k1_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void k1_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(k1_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void k1_mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "K1_WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra K1_WAIT_DONE;\n\t"
      "bra K1_WAIT_LOOP;\n\t"
      "K1_WAIT_DONE:\n\t"
      "}" ::"r"(k1_smem_u32(bar)), "r"(parity)
      : "memory");
}
// 1-D bulk async copy global -> shared, completion counted in bytes on an mbarrier
__device__ __forceinline__ void k1_bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   k1_smem_u32(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"(k1_smem_u32(bar))
               : "memory");
}

struct hole_k1_args {
  float* E;                 // table (DM 0: updated in place; DM 1/3: read only; DM 2: unused)
  const int32_t* tri;       // [B,3] (head, tail, relation): rows to GATHER (DM 2: global row ids)
  const int32_t* neg;       // [B]   corrupt entity per triple
  const int32_t* perm;      // [B]   processing order (triples grouped by relation)
  const uint32_t* gslot;    // [4B]  per use: HOLE_SLOT_UNIQUE or the row of G its gradient goes to
  int side, B, T, nvec, stride;
  float margin, lr;
  float* G;                 // staged gradient rows (rows used more than once in the step)
  float* loss;              // [B]  (DM 3: log loss of the positives, null on the passes without them)
  float* sigma;             // [2B] or null  (DM 3: [B] log loss of the pass's negatives)
  float* Dtab;              // DM 1/3: delta table; DM 2: local delta rows of the replicated relation block;
                            // DM 4: the AdaGrad accumulator [n_rows, stride]
};

// DM 2 (row-sharded step): where rows live and where their deltas go
struct hole_k1_shard {
  const int32_t* tri_w;     // [B,3] the same triples as rows of the requester's request list: R + slot
  const int32_t* neg_w;     // [B]
  const int32_t* cuts;      // [world+1] first request-list slot per owner
  const int* flags;         // my barrier flags [2][world] (local memory, written by the peers)
  int* err;                 // barrier time-out flag
  int wait_epoch;           // shards are current once flags[0][k] >= wait_epoch for every peer k
  int R, rows_per, me, world;
  long long cap;            // rows per (owner, requester) staging slice
  unsigned long long timeout_ns;
  hole_peer_ptrs shard;     // PEER: rank o's shard [R + rows_per, stride]
  hole_peer_ptrs stage;     // PEER: rank o's delta staging [world][cap][stride]
  // the step's request lists are posted by this kernel too: uniq[cuts[o]..cuts[o+1]) -> rank o's inbox
  const int32_t* uniq;      // [U] my request list (sorted unique global rows)
  hole_peer_ptrs inbox;     // PEER: rank o's inbox of this step's parity, int32 [world][cap] (row `me` is mine)
  hole_peer_ptrs meta;      // PEER: rank o's meta of this step's parity, int32 [world][2]
};

// wait until every peer's flag (written into MY memory) reaches `epoch`
__device__ __forceinline__ void hole_flags_wait(const int* flags, int world, int epoch, int* err,
                                                unsigned long long timeout_ns) {
  if (threadIdx.x < world) {
    const int* f = flags + threadIdx.x;
    unsigned long long t0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    while (true) {
      int v;
      asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
      if (v - epoch >= 0) break;
      if (*reinterpret_cast<volatile int*>(err) != 0) break;      // the run is already lost: drain
      unsigned long long t1;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
      if (t1 - t0 > timeout_ns) { atomicExch(err, 1); break; }
    }
  }
  __syncthreads();
}

template <int GS, int V, bool FULL>
__device__ __forceinline__ void k1_row_from_smem(Row<V>& x, const float4* ssrc, int lane, int nvec) {
#pragma unroll
  for (int v = 0; v < V; ++v) {
    const int idx = lane + v * GS;
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
    if (FULL || idx < nvec) { a = ssrc[idx]; b = ssrc[nvec + idx]; }
    x.re[4 * v + 0] = a.x; x.re[4 * v + 1] = a.y; x.re[4 * v + 2] = a.z; x.re[4 * v + 3] = a.w;
    x.im[4 * v + 0] = b.x; x.im[4 * v + 1] = b.y; x.im[4 * v + 2] = b.z; x.im[4 * v + 3] = b.w;
  }
}

// One row of the step: dx = A * d - Bc * x  (d = the row's score gradient in raw-row form, A and Bc
// carry the clip scales and the clip-backward projection), then
//   unique row : DM 0  E[row] = x - lr dx   (skipped for an inactive hinge: dx == 0)
//                DM 1/2  out[row] = -lr dx   (always written: the consumer adds every listed row)
//                DM 3    out[row] += -lr dx
//                DM 4    S[row] += dx^2,  E[row] = x - lr dx rsqrt(S[row])  (S: the accumulator row
//                        s_row; skipped for an inactive hinge)
//   otherwise  : G[gslot] = dx  for K3's ordered combine
template <int GS, int V, bool FULL, int DM>
__device__ __forceinline__ void k1_emit(const Row<V>& d, const Row<V>& x, float A, float Bc, bool uniq,
                                        bool act, float lr, float* out_row, float* g_row, int lane, int nvec,
                                        float* s_row = nullptr) {
  Row<V> o;
  if (uniq) {
    if constexpr (DM == 4) {
      if (!act) return;
      Row<V> acc;
      row_load<GS, V, false>(acc, s_row, lane, nvec);
#pragma unroll
      for (int k = 0; k < 4 * V; ++k) {
        const float gr = fmaf(A, d.re[k], -Bc * x.re[k]), gi = fmaf(A, d.im[k], -Bc * x.im[k]);
        acc.re[k] = fmaf(gr, gr, acc.re[k]);
        acc.im[k] = fmaf(gi, gi, acc.im[k]);
        o.re[k] = fmaf(-lr * gr, __frsqrt_rn(acc.re[k]), x.re[k]);
        o.im[k] = fmaf(-lr * gi, __frsqrt_rn(acc.im[k]), x.im[k]);
      }
      row_store<GS, V, FULL>(acc, s_row, lane, nvec);
    } else if (DM == 0) {
      if (!act) return;
#pragma unroll
      for (int k = 0; k < 4 * V; ++k) {
        o.re[k] = fmaf(-lr, fmaf(A, d.re[k], -Bc * x.re[k]), x.re[k]);
        o.im[k] = fmaf(-lr, fmaf(A, d.im[k], -Bc * x.im[k]), x.im[k]);
      }
    } else {
#pragma unroll
      for (int k = 0; k < 4 * V; ++k) {
        o.re[k] = -lr * fmaf(A, d.re[k], -Bc * x.re[k]);
        o.im[k] = -lr * fmaf(A, d.im[k], -Bc * x.im[k]);
      }
      if (DM == 3) {
        Row<V> p;
        row_load<GS, V, false>(p, out_row, lane, nvec);
        row_add(o, p);
      }
    }
    row_store<GS, V, FULL>(o, out_row, lane, nvec);
  } else {
#pragma unroll
    for (int k = 0; k < 4 * V; ++k) {
      o.re[k] = fmaf(A, d.re[k], -Bc * x.re[k]);
      o.im[k] = fmaf(A, d.im[k], -Bc * x.im[k]);
    }
    row_store<GS, V, FULL>(o, g_row, lane, nvec);
  }
}

struct K1Ids { int i, h, t, r, n, hw, tw, nw; };

template <int DM>
__device__ __forceinline__ K1Ids k1_load_ids(const hole_k1_args& a, const hole_k1_shard& sh, int g) {
  K1Ids d;
  d.i = a.perm[g];
  d.h = a.tri[3 * d.i]; d.t = a.tri[3 * d.i + 1]; d.r = a.tri[3 * d.i + 2];
  d.n = a.neg[d.i];
  if (DM == 2) { d.hw = sh.tri_w[3 * d.i]; d.tw = sh.tri_w[3 * d.i + 1]; d.nw = sh.neg_w[d.i]; }
  else { d.hw = d.h; d.tw = d.t; d.nw = d.n; }
  return d;
}

template <int GS, int V, int side, bool FULL, int DM>
__device__ __forceinline__ void hole_k1_body(const hole_k1_args& a, const hole_k1_shard& sh) {
  extern __shared__ float4 k1_smem[];
  const int lane = threadIdx.x % GS;
  const int grp = threadIdx.x / GS;
  const int ngrp = blockDim.x / GS;
  const int gbase = (threadIdx.x % 32) / GS * GS;
  const unsigned gmask = (GS == 32) ? 0xffffffffu : (((1u << GS) - 1u) << gbase);
  const int nvec = a.nvec, stride = a.stride, B = a.B;
  const int row4 = 2 * nvec;                                   // float4s per row
  const uint32_t row_bytes = (uint32_t)stride * 4u;
  // per lane group: K1V2_STAGES x {h, t, n} landing rows; the groups' mbarriers follow the rows
  float4* my_smem = k1_smem + (size_t)grp * (K1V2_STAGES * 3) * row4;
  uint64_t* bars = reinterpret_cast<uint64_t*>(k1_smem + (size_t)ngrp * (K1V2_STAGES * 3) * row4) + grp * K1V2_STAGES;
  if (lane == 0) {
#pragma unroll
    for (int s = 0; s < K1V2_STAGES; ++s) k1_mbar_init(bars + s, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __shared__ int s_cuts[HOLE_MAX_RANKS + 1];
  if (DM == 2 && threadIdx.x <= sh.world) s_cuts[threadIdx.x] = sh.cuts[threadIdx.x];
  __syncthreads();

  if (DM == 2) {
    // post my request lists: slice o of `uniq` goes to rank o's inbox, (count, offset) to its meta.
    // (The inbox is double buffered by step parity, so this needs no flag; the fence at the end of the
    // kernel makes it visible before the step's "delivered" flag is raised.)
    const int U = s_cuts[sh.world];
    const int gtid = blockIdx.x * blockDim.x + threadIdx.x;
    for (int j = gtid; j < U; j += gridDim.x * blockDim.x) {
      int o = 0;
      while (j >= s_cuts[o + 1]) ++o;
      static_cast<int32_t*>(sh.inbox.p[o])[(size_t)sh.me * sh.cap + (j - s_cuts[o])] = sh.uniq[j];
    }
    if (gtid < sh.world) {
      int32_t* m = static_cast<int32_t*>(sh.meta.p[gtid]);
      m[2 * sh.me] = s_cuts[gtid + 1] - s_cuts[gtid];
      m[2 * sh.me + 1] = s_cuts[gtid];
    }
  }
  const int64_t w = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / GS;
  const int64_t g0l = w * a.T;
  const bool have = g0l < B;
  const int g0 = have ? (int)g0l : 0, g1 = have ? min(B, g0 + a.T) : 0;

  // where a row lives (DM 2: its owner's shard, over NVLink unless it is mine)
  auto row_src = [&](int id) -> const float* {
    if (DM == 2) {
      if (id < sh.R) return static_cast<const float*>(sh.shard.p[sh.me]) + (size_t)id * stride;
      const int o = (id - sh.R) / sh.rows_per;
      return static_cast<const float*>(sh.shard.p[o]) + (size_t)(id - o * sh.rows_per) * stride;
    }
    return a.E + (size_t)id * stride;
  };
  // where a unique row's change goes: the table / delta table row, or (DM 2) slot (wrow - R - cuts[o])
  // of my slice of the owner's staging buffer
  auto row_dst = [&](int id, int wrow) -> float* {
    if (DM == 2) {
      const int o = (id - sh.R) / sh.rows_per;
      return static_cast<float*>(sh.stage.p[o]) +
             ((size_t)sh.me * (size_t)sh.cap + (size_t)(wrow - sh.R - s_cuts[o])) * stride;
    }
    return (DM == 0 || DM == 4 ? a.E : a.Dtab) + (size_t)id * stride;
  };
  auto fetch = [&](const K1Ids& d, int stage) {
    if (lane == 0) {
      float4* sb = my_smem + (size_t)stage * 3 * row4;
      k1_mbar_expect_tx(bars + stage, 3u * row_bytes);
      k1_bulk_g2s(sb, row_src(d.h), row_bytes, bars + stage);
      k1_bulk_g2s(sb + row4, row_src(d.t), row_bytes, bars + stage);
      k1_bulk_g2s(sb + 2 * row4, row_src(d.n), row_bytes, bars + stage);
    }
  };

  K1Ids c, n1, n2;
  if (have) {
    c = k1_load_ids<DM>(a, sh, g0);
    n1 = (g0 + 1 < g1) ? k1_load_ids<DM>(a, sh, g0 + 1) : c;
    n2 = (g0 + 2 < g1) ? k1_load_ids<DM>(a, sh, g0 + 2) : c;
  }
  pdl_wait();                 // the previous step's K3 has finished updating the table
  if (DM == 2) hole_flags_wait(sh.flags, sh.world, sh.wait_epoch, sh.err, sh.timeout_ns);   // every shard is current
  if (!have) {
    if (DM == 2) __threadfence_system();      // this thread may have posted request-list entries
    return;
  }
  fetch(c, 0);
  if (g0 + 1 < g1) fetch(n1, 1);

  Row<V> xr, acc;             // relation row of the current run (raw) and its summed gradient (y-space)
  row_zero(xr);
  row_zero(acc);
  int r_cur = -1, run_i = 0;
  float inv_r = 0.f, sc_r = 1.f, proj_r = 0.f;
  bool run_act = false;
  float* const rel_out = (DM == 0 || DM == 4) ? a.E : a.Dtab;

  // end of a run of equal relation: clip backward of the summed gradient, then apply / stage
  auto flush_relation = [&]() {
    const uint32_t sl = a.gslot[run_i];
    const bool cl = inv_r <= 1.0f;
    k1_emit<GS, V, FULL, DM>(acc, xr, cl ? inv_r : 1.0f, cl ? sc_r * proj_r * inv_r : 0.0f,
                             sl == HOLE_SLOT_UNIQUE, run_act, a.lr, rel_out + (size_t)r_cur * stride,
                             a.G + (size_t)sl * stride, lane, nvec, a.Dtab + (size_t)r_cur * stride);
  };

  int stage = 0;
  uint32_t parity = 0;        // bit s = phase parity of stage s's barrier
  for (int g = g0; g < g1; ++g) {
    K1Ids n3 = n2;
    if (g + 3 < g1) n3 = k1_load_ids<DM>(a, sh, g + 3);          // ids three ahead
    __syncwarp(gmask);        // every lane is done reading the landing buffer that is refilled next
    if (g + 2 < g1) fetch(n2, (stage + 2) % K1V2_STAGES);         // rows two ahead
    const int i = c.i;
    const uint32_t sl_t = a.gslot[B + i], sl_h = a.gslot[2 * B + i], sl_n = a.gslot[3 * B + i];
    float* const sr_h = DM == 4 ? a.Dtab + (size_t)c.h * stride : nullptr;     // DM 4: accumulator rows
    float* const sr_t = DM == 4 ? a.Dtab + (size_t)c.t * stride : nullptr;
    float* const sr_n = DM == 4 ? a.Dtab + (size_t)c.n * stride : nullptr;
    if (c.r != r_cur) {                      // group-uniform
      if (r_cur >= 0) flush_relation();
      // the relation row: once per run, straight from L2 (DM 2: my replica)
      row_load<GS, V, false>(xr, row_src(c.r), lane, nvec);
      r_cur = c.r;
      run_i = i;
      run_act = false;
      proj_r = 0.f;
      row_zero(acc);
      inv_r = -1.f;           // norm folded into this triple's reduction round
    }
    k1_mbar_wait(bars + stage, (parity >> stage) & 1u);           // rows of triple g have landed
    parity ^= 1u << stage;
    const float4* sb = my_smem + (size_t)stage * 3 * row4;
    Row<V> xh, xt, xn, P;
    k1_row_from_smem<GS, V, FULL>(xh, sb, lane, nvec);
    k1_row_from_smem<GS, V, FULL>(xt, sb + row4, lane, nvec);
    k1_row_from_smem<GS, V, FULL>(xn, sb + 2 * row4, lane, nvec);

    // raw sums: |h|^2 |t|^2 |n|^2 (|r|^2 on the first triple of a run) and the two raw scores.
    // side 0 (negative = (h, n, r)): P = h r;            s+ = sum P.t, s- = sum P.n
    // side 1 (negative = (n, t, r)): P = r conj(t)~;     s+ = sum h.P, s- = sum n.P      (App. A.4)
    float ssh = 0.f, sst = 0.f, ssn = 0.f, Sp = 0.f, Sn = 0.f, ssr = 0.f;
#pragma unroll
    for (int k = 0; k < 4 * V; ++k) {
      const float ha = xh.re[k], hb = xh.im[k], rc = xr.re[k], rd = xr.im[k], te = xt.re[k], tf = xt.im[k];
      const float nr = xn.re[k], ni = xn.im[k];
      ssh = fmaf(ha, ha, fmaf(hb, hb, ssh));
      sst = fmaf(te, te, fmaf(tf, tf, sst));
      ssn = fmaf(nr, nr, fmaf(ni, ni, ssn));
      if (side == 0) {
        P.re[k] = ha * rc - hb * rd;
        P.im[k] = ha * rd + hb * rc;
        Sp = fmaf(P.re[k], te, fmaf(P.im[k], tf, Sp));
        Sn = fmaf(P.re[k], nr, fmaf(P.im[k], ni, Sn));
      } else {
        P.re[k] = rc * te + rd * tf;
        P.im[k] = rc * tf - rd * te;
        Sp = fmaf(ha, P.re[k], fmaf(hb, P.im[k], Sp));
        Sn = fmaf(nr, P.re[k], fmaf(ni, P.im[k], Sn));
      }
    }
    const bool new_run = inv_r < 0.f;        // group-uniform
    if (new_run) ssr = row_sumsq(xr);
#pragma unroll
    for (int o = GS / 2; o > 0; o >>= 1) {
      ssh += __shfl_xor_sync(gmask, ssh, o);
      sst += __shfl_xor_sync(gmask, sst, o);
      ssn += __shfl_xor_sync(gmask, ssn, o);
      Sp += __shfl_xor_sync(gmask, Sp, o);
      Sn += __shfl_xor_sync(gmask, Sn, o);
      if (new_run) ssr += __shfl_xor_sync(gmask, ssr, o);
    }
    if (new_run) { inv_r = __frsqrt_rn(ssr); sc_r = fminf(inv_r, 1.0f); }
    // clip_by_norm(row, 1): y = x * min(rsqrt(sum x^2), 1)  (App. B)
    const float inv_h = __frsqrt_rn(ssh), inv_t = __frsqrt_rn(sst), inv_n = __frsqrt_rn(ssn);
    const float sc_h = fminf(inv_h, 1.0f), sc_t = fminf(inv_t, 1.0f), sc_n = fminf(inv_n, 1.0f);
    const bool cl_h = inv_h <= 1.0f, cl_t = inv_t <= 1.0f, cl_n = inv_n <= 1.0f;
    const float sp = Sp * (sc_h * sc_r * sc_t);
    const float sn = Sn * (side == 0 ? (sc_h * sc_r * sc_n) : (sc_n * sc_r * sc_t));
    const float vp = sigmoidf_precise(sp), vn = sigmoidf_precise(sn);
    bool act;
    float gp, gn;
    if constexpr (DM == 3) {  // (a plain `if` reorders DM 0-2's loop registers)
      // --log_loss (holE.py:194-195): loss = log(1 + exp(-label * s)), d/ds = -label * sigmoid(-label * s)
      act = true;
      gp = (a.loss != nullptr) ? vp - 1.0f : 0.0f;
      gn = vn;
      if (lane == 0) {
        if (a.loss != nullptr) a.loss[i] = logf(1.0f + expf(-sp));
        a.sigma[i] = logf(1.0f + expf(sn));
      }
    } else {
      const float pre = vp - vn + a.margin;
      act = pre >= 0.0f;                                           // TF Maximum grad: GreaterEqual
      gp = act ? vp * (1.0f - vp) : 0.0f;
      gn = act ? -(vn * (1.0f - vn)) : 0.0f;
      if (lane == 0) {
        a.loss[i] = fmaxf(pre, 0.0f);
        if (a.sigma != nullptr) { a.sigma[i] = vp; a.sigma[B + i] = vn; }
      }
    }
    run_act = run_act || act;
    const float gs_p = gp * sp, gs_n = gn * sn, gs_b = gs_p + gs_n;   // y . dy of a row = g * s (Euler)
    proj_r += gs_b;

    // the two rows whose gradient is a multiple of P; the "shared" entity row and the relation take
    // U = g+ y_a + g- y_n  with a = tail (side 0) or head (side 1)
    float *dst_t = nullptr, *dst_h = nullptr, *dst_n = nullptr;
    if (sl_t == HOLE_SLOT_UNIQUE) dst_t = row_dst(c.t, c.tw);
    if (sl_h == HOLE_SLOT_UNIQUE) dst_h = row_dst(c.h, c.hw);
    if (sl_n == HOLE_SLOT_UNIQUE) dst_n = row_dst(c.n, c.nw);
    const float lr = a.lr;
    if (side == 0) {
      const float hr = sc_h * sc_r;
      k1_emit<GS, V, FULL, DM>(P, xt, gp * hr * (cl_t ? inv_t : 1.0f), cl_t ? sc_t * gs_p * inv_t : 0.0f,
                               sl_t == HOLE_SLOT_UNIQUE, act, lr, dst_t, a.G + (size_t)sl_t * stride, lane, nvec,
                               sr_t);
      k1_emit<GS, V, FULL, DM>(P, xn, gn * hr * (cl_n ? inv_n : 1.0f), cl_n ? sc_n * gs_n * inv_n : 0.0f,
                               sl_n == HOLE_SLOT_UNIQUE, act, lr, dst_n, a.G + (size_t)sl_n * stride, lane, nvec,
                               sr_n);
      const float bt = gp * sc_t, bn = gn * sc_n;
      Row<V> d;
#pragma unroll
      for (int k = 0; k < 4 * V; ++k) {
        const float u = fmaf(bt, xt.re[k], bn * xn.re[k]), wv = fmaf(bt, xt.im[k], bn * xn.im[k]);
        const float rc = xr.re[k], rd = xr.im[k], ha = xh.re[k], hb = xh.im[k];
        d.re[k] = fmaf(rc, u, rd * wv);                  // dh = conj(r) o U
        d.im[k] = fmaf(rc, wv, -rd * u);
        const float us = sc_h * u, ws = sc_h * wv;       // dr += conj(h_y) o U
        acc.re[k] += fmaf(ha, us, hb * ws);
        acc.im[k] += fmaf(ha, ws, -hb * us);
      }
      k1_emit<GS, V, FULL, DM>(d, xh, sc_r * (cl_h ? inv_h : 1.0f), cl_h ? sc_h * gs_b * inv_h : 0.0f,
                               sl_h == HOLE_SLOT_UNIQUE, act, lr, dst_h, a.G + (size_t)sl_h * stride, lane, nvec,
                               sr_h);
    } else {
      const float rt = sc_r * sc_t;
      k1_emit<GS, V, FULL, DM>(P, xh, gp * rt * (cl_h ? inv_h : 1.0f), cl_h ? sc_h * gs_p * inv_h : 0.0f,
                               sl_h == HOLE_SLOT_UNIQUE, act, lr, dst_h, a.G + (size_t)sl_h * stride, lane, nvec,
                               sr_h);
      k1_emit<GS, V, FULL, DM>(P, xn, gn * rt * (cl_n ? inv_n : 1.0f), cl_n ? sc_n * gs_n * inv_n : 0.0f,
                               sl_n == HOLE_SLOT_UNIQUE, act, lr, dst_n, a.G + (size_t)sl_n * stride, lane, nvec,
                               sr_n);
      const float bh = gp * sc_h, bn = gn * sc_n;
      Row<V> d;
#pragma unroll
      for (int k = 0; k < 4 * V; ++k) {
        const float u = fmaf(bh, xh.re[k], bn * xn.re[k]), wv = fmaf(bh, xh.im[k], bn * xn.im[k]);
        const float rc = xr.re[k], rd = xr.im[k], te = xt.re[k], tf = xt.im[k];
        d.re[k] = fmaf(u, rc, -wv * rd);                 // dt = U o r
        d.im[k] = fmaf(u, rd, wv * rc);
        const float us = sc_t * u, ws = sc_t * wv;       // dr += U o conj(t_y)~
        acc.re[k] += fmaf(us, te, ws * tf);
        acc.im[k] += fmaf(us, tf, -ws * te);
      }
      k1_emit<GS, V, FULL, DM>(d, xt, sc_r * (cl_t ? inv_t : 1.0f), cl_t ? sc_t * gs_b * inv_t : 0.0f,
                               sl_t == HOLE_SLOT_UNIQUE, act, lr, dst_t, a.G + (size_t)sl_t * stride, lane, nvec,
                               sr_t);
    }
    c = n1;
    n1 = n2;
    n2 = n3;
    stage = (stage + 1) % K1V2_STAGES;
  }
  pdl_launch_dependents();    // K3 of this step may start its prologue
  flush_relation();
  // DM 2: this thread's delta rows went to peer memory with plain stores; the "delivered" flag is raised
  // by a later kernel from ONE thread, whose fence does not cover stores other SMs still have in flight on
  // NVLink -- every writer makes its own stores visible system-wide before the kernel ends
  if (DM == 2) __threadfence_system();
}

// DM 3 at V 1 is held to two blocks per SM (128 registers, no spills), the occupancy DM 0 has there:
// left free it takes 135 registers and one block per SM, and a log-loss step at d = 256 is 5-20 % slower.
// DM 4 at V 1 likewise (128 registers, no spills; DESIGN §7c)
template <int GS, int V, int DM>
__global__ void __launch_bounds__(K1_THREADS, ((DM == 3 || DM == 4) && V == 1) ? 2 : 1)
hole_k1_kernel(const hole_k1_args a, const hole_k1_shard sh) {
  // specialise on the corruption side and on "every lane owns valid float4s" (nvec == GS*V)
  const bool full = (a.nvec == GS * V);
  if (a.side) { if (full) hole_k1_body<GS, V, 1, true, DM>(a, sh); else hole_k1_body<GS, V, 1, false, DM>(a, sh); }
  else        { if (full) hole_k1_body<GS, V, 0, true, DM>(a, sh); else hole_k1_body<GS, V, 0, false, DM>(a, sh); }
}
