/* hole_b200.h -- C ABI of the B200-native HolE hot path (libhole_b200.so).
 *
 * Drop-in boundary for holE.py's training step and link-prediction ranking
 * (greysun/GraphEmbeddings).  The reference has no FFI around this path (it is inline
 * TensorFlow graph code); each entry point below names the holE.py seam it replaces, and
 * the calling convention follows the repository's only C-ABI precedent, init.cpp + ctypes
 * (init.cpp:47,129-142,223-246; transE.py:95-112): extern "C", plain ints and raw
 * caller-owned buffers.  Two departures from that precedent, both deliberate:
 *   - every call returns int (0 = ok, negative = error) and hole_last_error() gives a
 *     thread-local message (init.cpp reports nothing, e.g. unchecked fopen at init.cpp:53);
 *   - no process-global state (init.cpp:145-150 keeps a global, racy RNG): everything
 *     lives in an opaque hole_ctx, and the sampler is counter-based.
 *
 * Unless a parameter is marked [host], every pointer is a DEVICE pointer owned by the
 * caller (e.g. a torch tensor's data_ptr()).  Every call is asynchronous on `stream`
 * (a cudaStream_t passed as void*; NULL = legacy default stream) unless it says otherwise.
 * There is no CPU fallback: every entry point fails with HOLE_ERR_CUDA when no sm_100
 * device is present.
 *
 * Layouts
 *   triples  int32 [B,3], columns (head, tail, relation)            -- holE.py:80-81
 *   table    float32 [N, row_stride]; a row is [Re(0..H-1) pad | Im(0..H-1) pad] with
 *            H = dim/2 and each half zero-padded to a multiple of 4 floats, so that
 *            row_stride = hole_row_stride(dim) and every half starts 16-byte aligned.
 *            hole_pack_rows / hole_unpack_rows convert from/to the checkpoint layout
 *            float32 [N, dim] = [Re | Im] (holE.py:164-165).
 */
#ifndef HOLE_B200_H
#define HOLE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct hole_ctx hole_ctx;

#if defined(__GNUC__)
#define HOLE_API __attribute__((visibility("default")))
#else
#define HOLE_API
#endif

#define HOLE_OK            0
#define HOLE_ERR_ARG      (-1)   /* bad argument (odd dim, negative size, null pointer) */
#define HOLE_ERR_CUDA     (-2)   /* CUDA runtime/driver error, or no sm_100 device      */
#define HOLE_ERR_ALLOC    (-3)   /* workspace allocation failed                          */
#define HOLE_ERR_UNSUPPORTED (-4)/* shape outside what the kernels are built for         */

#define HOLE_SIDE_TAIL 0         /* corrupt / rank tails */
#define HOLE_SIDE_HEAD 1         /* corrupt / rank heads */
#define HOLE_SIDE_BOTH 2         /* hole_rank / hole_topk only: tails then heads in one pass */
#define HOLE_SIDE_RELATION 3     /* hole_rank / hole_topk only: rank relations (h, ?, t); not part of BOTH */

/* Operand precision of the tensor-core ranking contraction. */
#define HOLE_RANK_BF16   0       /* bf16 operands, fp32 accumulate; dim <= 640           */
#define HOLE_RANK_BF16X3 1       /* split-bf16 (hi*hi + lo*hi + hi*lo): ranks match fp32 except within ~3e-5 of a tie; dim <= 320 */

/* ABI version of this header; hole_abi_version() returns the library's. */
#define HOLE_ABI_VERSION 7
HOLE_API int hole_abi_version(void);

/* Thread-local message of the last failing call on this thread ("" if none). */
HOLE_API const char* hole_last_error(void);

/* floats per device row for an (even) embedding_dim: 2 * round_up(dim/2, 4). */
HOLE_API int hole_row_stride(int dim);

/* Create / destroy a context bound to CUDA device `device` for a table of n_rows x dim
 * (holE.py:263-264: one shared table for relations and entities).  Synchronous.
 * dim <= 768; a larger dim returns HOLE_ERR_UNSUPPORTED.  A call outside the limits of its own path
 * (ranking / top-k above) returns HOLE_ERR_UNSUPPORTED before it launches anything or writes any
 * output, and the context stays usable. */
HOLE_API int hole_ctx_create(hole_ctx** out, int device, int64_t n_rows, int dim);
HOLE_API int hole_ctx_destroy(hole_ctx* ctx);

/* Optional hint: relation ids are < n_relations (holE.py:52 counts relation_ids.txt), which
 * shortens the per-step "group triples by relation" sort (one 8-bit pass below 256 relations, a
 * per-thread counting sort up to 64).  Default: n_rows.  The grouping is a processing order only:
 * an id >= n_relations is grouped with other relations (slower), never mis-trained. */
HOLE_API int hole_ctx_set_relations(hole_ctx* ctx, int64_t n_relations);

/* Score variant.  HOLE_SCORE_COMPLEX (default) is the live holE.py:191-198:
 * sigma(sum_k Re(h_k r_k conj(t_k))).  HOLE_SCORE_CCORR_TANH is the ARCHIVED variant of the run
 * directory holE-20170724 (graph.pbtxt:6221-6521): tanh(sum_k Re(m_k) + Im(m_k)),
 * m = r * ifft(conj(fft(h)) * fft(t)), with the loss max(tanh(s+) - tanh(s-) + margin, 0)
 * (graph.pbtxt:15874-15988; margin 1.0 in that run).  In that mode hole_score returns tanh(s) and
 * hole_train_step / hole_train_steps[_host] run the direct-correlation kernel; hole_rank* rank on the
 * raw score s (tanh is monotone; s is linear in the candidate entity, so the same tensor-core
 * contraction runs on another query vector); the log-loss branch, the delta-table step and the
 * row-sharded step return HOLE_ERR_UNSUPPORTED. */
#define HOLE_SCORE_COMPLEX 0
#define HOLE_SCORE_CCORR_TANH 1
HOLE_API int hole_ctx_set_score_mode(hole_ctx* ctx, int mode);

/* Optimizer of the training step.  HOLE_OPT_SGD (default; accum must be NULL) is holE.py:296's
 * GradientDescentOptimizer: table[i] -= lr * g_i.  HOLE_OPT_ADAGRAD is TF 1.2's AdagradOptimizer in its place
 * (SparseApplyAdagrad after the duplicate indices are summed), per touched row i and element, in fp32:
 *     accum[i] += g_i^2;   table[i] -= lr * g_i * rsqrt(accum[i])
 * with the NEW accumulator and no epsilon; g_i is the gradient the SGD step applies (duplicates summed in the
 * same fixed order), and a row whose hinge is inactive (g_i = 0) keeps its table and accumulator rows.
 *   accum  float32 [n_rows, row_stride], the table's row layout, caller-owned and kept by reference (like the
 *          type tables of hole_corrupt) until the next hole_ctx_set_optimizer call.  EVERY element must be
 *          > 0, the pad columns included (TF starts it at initial_accumulator_value, 0.1 by default): a zero
 *          pad element would make the pad column 0 * rsqrt(0) = NaN instead of keeping it zero.
 * In AdaGrad mode hole_train_step, hole_train_steps and hole_train_steps_host update the table and the
 * accumulator.  hole_train_step_ex with a delta_out, hole_train_step_logloss, every hole_shard_* call, and
 * every training call in HOLE_SCORE_CCORR_TANH mode return HOLE_ERR_UNSUPPORTED before they launch anything
 * or write anything, and the context stays usable.  AdaGrad on a context bound by hole_shard_init is
 * HOLE_ERR_UNSUPPORTED too.  Switching back to HOLE_OPT_SGD restores the SGD step exactly.
 * This call sets the optimizer of the single-table steps only.  The row-sharded steps have their own,
 * hole_shard_set_optimizer below, which this call neither reads nor changes. */
#define HOLE_OPT_SGD 0
#define HOLE_OPT_ADAGRAD 1
HOLE_API int hole_ctx_set_optimizer(hole_ctx* ctx, int optimizer, float* accum);

/* Checkpoint layout [n, dim] <-> device layout [n, row_stride]. */
HOLE_API int hole_pack_rows(hole_ctx* ctx, const float* src_nd, float* dst_padded, int64_t n, void* stream);
HOLE_API int hole_unpack_rows(hole_ctx* ctx, const float* src_padded, float* dst_nd, int64_t n, void* stream);

/* ---- corruption: replaces corrupt_batch (holE.py:97-158) and the per-step host
 * subsample + table insert (holE.py:343-347).
 * One Philox coin per (seed, step) picks the side for the whole batch (holE.py:137-140);
 * triple i's replacement is csr_ids[csr_off[ty] + mulhi64(philox(seed, step, i), cnt[ty])]
 * with ty = type_of[replaced entity].  The stream is specified in oracle/philox.py.
 *   side_out  int32[1] (may be NULL)   neg_out  int32[B]
 * Returns the side also through *side_host [host] when non-NULL (it depends on
 * (seed, step) only and is computed on the host). */
HOLE_API int hole_corrupt(hole_ctx* ctx, const int32_t* triples, int64_t B,
                 const int32_t* type_of, const int64_t* csr_off, const int32_t* csr_ids,
                 uint64_t seed, uint64_t step,
                 int32_t* side_out, int32_t* neg_out, int* side_host, void* stream);

/* Same draw for a batch that is a slice of a larger (multi-GPU) batch: triple i of this call
 * is triple index_base + i of the global batch, so the result does not depend on how the
 * global batch is split over ranks. */
HOLE_API int hole_corrupt_at(hole_ctx* ctx, const int32_t* triples, int64_t B,
                 const int32_t* type_of, const int64_t* csr_off, const int32_t* csr_ids,
                 uint64_t seed, uint64_t step, uint64_t index_base,
                 int32_t* side_out, int32_t* neg_out, int* side_host, void* stream);

/* ---- forward: replaces evaluate_triples (holE.py:179-202): out_sigma[i] =
 * sigmoid(sum_k Re(h_k * r_k * conj(t_k))) on norm-clipped rows (holE.py:161-168). */
HOLE_API int hole_score(hole_ctx* ctx, const float* table, const int32_t* triples, int64_t B,
               float* out_sigma, void* stream);

/* ---- one training step: replaces evaluate_batch's hinge branch (holE.py:222-234) plus
 * GradientDescentOptimizer.minimize (holE.py:296) -- forward, backward and the sparse
 * update table[idx] -= lr * g with duplicates accumulated in a fixed order (or the AdaGrad
 * update, see hole_ctx_set_optimizer).
 *   neg_ent int32[B]: replacement entity per triple; side: HOLE_SIDE_*.
 *   loss_out float32[B] (hinge per triple); sigma_out float32[2B] or NULL
 *   (sigma+ then sigma-, the tensors holE.py:200 summarises). */
HOLE_API int hole_train_step(hole_ctx* ctx, float* table, const int32_t* pos, const int32_t* neg_ent,
                    int side, int64_t B, float margin, float lr,
                    float* loss_out, float* sigma_out, void* stream);

/* Multi-GPU building blocks (graphembeddings_b200/sharded.py).
 * hole_train_step_ex: as hole_train_step; when delta_out != NULL the table is left untouched
 * and every row a step would change receives its change (-lr * summed gradient) at the same
 * row of delta_out (float32 [n_rows, row_stride], zero-initialised by the caller).
 * hole_train_step_plan: optionally builds the integer update plan for the next
 * hole_train_step(_ex) call with the same pos / neg_ent / B on a side stream, so that it
 * overlaps whatever the caller enqueues in between (e.g. the row exchange).
 * hole_add_rows: table[ids[k] + id_offset] += rows[k] for k < n, ids unique within a call.
 * hole_gather_rows: dst_rows[k] = table[ids[k] + id_offset].  For both, the row buffer may be
 * PEER device memory (an IPC-mapped buffer of another rank).  These serve the generic
 * (NCCL / gloo all-to-all) sharded trainer; the NVLink path is hole_shard_step below. */
HOLE_API int hole_train_step_ex(hole_ctx* ctx, float* table, float* delta_out, const int32_t* pos,
                       const int32_t* neg_ent, int side, int64_t B, float margin, float lr,
                       float* loss_out, float* sigma_out, void* stream);
HOLE_API int hole_train_step_plan(hole_ctx* ctx, const int32_t* pos, const int32_t* neg_ent, int64_t B,
                         void* stream);
/* ---- the --log_loss branch of evaluate_batch (holE.py:194-196, 206-220) + minimize (296).
 * loss rows: B positives with label +1, then negative_ratio corrupt batches with label -1,
 * each its own corrupt_batch call (own head/tail coin and draws: virtual step
 * step * negative_ratio + j of the Philox stream).  Row loss = log(1 + exp(-label * score))
 * (+ l2 * l2_loss(embeddings), the same scalar in every row -- returned separately).
 * Update: E -= lr * d(sum of all rows)/dE, i.e. the sparse score gradients taken at the old
 * table plus the dense decay  E * lr * (1 + negative_ratio) * B * l2.
 *   delta_ws     [n_rows, row_stride] device scratch, all zero on entry and on return
 *   loss_out     [(1 + negative_ratio) * B] device: positives, then each corrupt batch
 *   l2_loss_out  device scalar = sum(E_old^2) / 2 (tf.nn.l2_loss), or NULL
 *   neg_out      [negative_ratio * B] device int32 replacement entities, or NULL
 *   sides_out    [negative_ratio] HOST int32 (1 = heads replaced), or NULL */
HOLE_API int hole_train_step_logloss(hole_ctx* ctx, float* table, float* delta_ws, const int32_t* triples,
                                     int64_t B, int negative_ratio, const int32_t* type_of,
                                     const int64_t* csr_off, const int32_t* csr_ids, uint64_t seed,
                                     uint64_t step, float lr, float l2, float* loss_out, float* l2_loss_out,
                                     int32_t* neg_out, int32_t* sides_out, void* stream);

/* ---- row-sharded training over NVLink peer memory (no counterpart in the reference, which is
 * single-device; SURVEY.md 8e).  One process per GPU.  Rank o owns entity rows
 * [n_relations + o*rows_per_rank, +rows_per_rank); the relation rows are replicated:
 *   shard     float32 [n_relations + rows_per_rank, row_stride]  = [relations | my block]
 * Buffers marked PEER live on every rank and are mapped on all of them (CUDA IPC after
 * hole_enable_peer_access); the arrays below hold rank k's buffer at index k (index `me` = mine):
 *   peer_shard     PEER  the shards (rows are GATHERED from them by the training kernel)
 *   peer_stage     PEER  float32 [world][3*max_batch][row_stride]  row deltas, slice k written by rank k
 *   peer_relstage  PEER  float32 [world][n_relations][row_stride]  relation deltas, slice k by rank k
 *   peer_inbox     PEER  int32 [2][world][3*max_batch]             request lists (double buffered)
 *   peer_meta      PEER  int32 [2][world][2]                       (count, offset) of each list
 *   peer_flags     PEER  int32 [2][world], zero-initialised        epochs: [0] shard current, [1] deltas delivered
 *   err_flag       device int32, zero: set when a peer does not arrive within timeout_s (<= 0: 600 s)
 * type_of / csr_off / csr_ids: the type tables of hole_corrupt (kept by reference).
 *
 * hole_shard_step: one batch-synchronous step of the GLOBAL batch = concatenation over ranks of the
 *   ranks' `pos` slices (B triples each, global row ids, device): Philox corruption keyed on the
 *   global triple index me*B + i (so the result does not depend on `world`), rows gathered from their
 *   owners' shards over NVLink inside the training kernel, which also stores every row's delta into
 *   its owner's staging buffer; owners then add the staged deltas in rank order (deterministic; the
 *   relation replicas stay bit-identical).  No host synchronisation, no NCCL.  Every rank must call
 *   it with the same (B, seed, step) sequence.  loss_out float32[B] (hinge of my slice).
 * hole_shard_prepare: optional; builds the table-independent part (corruption, request routing,
 *   update plan) of a later hole_shard_step call with the same (pos, B, seed, step) on a side stream,
 *   so that it overlaps the step before it.
 * hole_shard_step_compute / _apply: the two halves of hole_shard_step (test hook: with several
 *   virtual ranks on one GPU, run compute on every rank, then apply on every rank).
 * hole_shard_steps / hole_shard_steps_host: n_steps consecutive steps from device / host triples
 *   [n_steps*B, 3] (this rank's slices), one step prepared ahead; lr [host] float32[n_steps];
 *   loss sums of my slices to loss_sum_out (device) / loss_sum_host (blocks until they are there).
 * hole_shard_poll: synchronises `stream` and reports whether a flag wait has timed out; the tables
 *   are then inconsistent and the caller must stop.
 * hole_shard_set_optimizer: the optimizer of the following sharded steps (after hole_shard_init, which resets
 *   it to HOLE_OPT_SGD; before it, HOLE_ERR_ARG).  HOLE_OPT_SGD needs accum_shard == NULL, HOLE_OPT_ADAGRAD a
 *   non-NULL one; any other id is HOLE_ERR_ARG.  A refused call changes nothing.
 *     accum_shard  float32 [n_relations + rows_per_rank, row_stride], the shard's layout (replicated relation
 *                  rows, then my block), caller-owned and kept by reference.  EVERY element must be > 0, the pad
 *                  columns and the unused trailing rows of the last rank's block included (see
 *                  hole_ctx_set_optimizer).
 *   AdaGrad step, per row i listed by ranks k1 < k2 < ... and per element, in fp32:
 *     g_i = sum_k staged_k[i] (rank order);  A[i] += g_i^2;  E[i] -= lr * g_i * rsqrt(A[i])
 *   with staged_k[i] rank k's summed gradient of row i; a relation row r takes g_r = sum over every rank's
 *   relation gradient in rank order, applied by every rank to its replicas of the table and the accumulator,
 *   which stay bit-identical.  A row whose gradient is zero on every rank keeps both rows.  The NVLink exchange
 *   is that of an SGD step.  hole_shard_step_compute latches the optimizer and lr of a step and
 *   hole_shard_step_apply applies with them; hole_shard_step(s)(_host) do both per step.  Every rank must set
 *   the same optimizer before the same step (like the (B, seed, step) sequence).  The context's own optimizer
 *   (hole_ctx_set_optimizer) is separate: it must stay HOLE_OPT_SGD on a sharded context, and the single-table
 *   calls on such a context keep their behaviour. */
#define HOLE_MAX_RANKS 16
HOLE_API int hole_shard_init(hole_ctx* ctx, int world, int me, int64_t n_relations, int64_t n_entities,
                             int64_t rows_per_rank, int64_t max_batch, float* shard,
                             void* const* peer_shard, void* const* peer_stage, void* const* peer_relstage,
                             void* const* peer_inbox, void* const* peer_meta, void* const* peer_flags,
                             int32_t* err_flag, double timeout_s, const int32_t* type_of,
                             const int64_t* csr_off, const int32_t* csr_ids);
HOLE_API int hole_shard_prepare(hole_ctx* ctx, const int32_t* pos, int64_t B, uint64_t seed, uint64_t step,
                                void* stream);
HOLE_API int hole_shard_step(hole_ctx* ctx, const int32_t* pos, int64_t B, uint64_t seed, uint64_t step,
                             float margin, float lr, float* loss_out, void* stream);
HOLE_API int hole_shard_step_compute(hole_ctx* ctx, const int32_t* pos, int64_t B, uint64_t seed, uint64_t step,
                                     float margin, float lr, float* loss_out, void* stream);
HOLE_API int hole_shard_step_apply(hole_ctx* ctx, void* stream);
HOLE_API int hole_shard_steps(hole_ctx* ctx, const int32_t* triples, int64_t B, int64_t n_steps, uint64_t seed,
                              uint64_t first_step, float margin, const float* lr, float* loss_sum_out,
                              void* stream);
HOLE_API int hole_shard_steps_host(hole_ctx* ctx, const int32_t* triples_host, int64_t B, int64_t n_steps,
                                   uint64_t seed, uint64_t first_step, float margin, const float* lr,
                                   float* loss_sum_host, void* stream);
HOLE_API int hole_shard_poll(hole_ctx* ctx, int* timed_out, void* stream);
HOLE_API int hole_shard_set_optimizer(hole_ctx* ctx, int optimizer, float* accum_shard);
/* Measurement hook: with hole_profile_enable on, summed milliseconds of the step's phases
 * [post, K1 (incl. its wait for the peers' shards), K3, finish, apply (incl. its wait for the peers'
 * deltas)] -> phase_ms5 [host, double[5]], and the number of steps measured since the last read. */
HOLE_API int hole_shard_profile_read(hole_ctx* ctx, double* phase_ms5, int64_t* n_steps);

/* Building blocks of the step, exported for tests.
 * hole_shard_route: dedup the 3B entity rows {head, tail, corrupt entity} of this rank's B
 *   triples (global row ids).  uniq_out[0..U) ascending, cuts_out[o] = first slot owned by rank
 *   o, cuts_out[world] = U; pos_w / neg_w = the triples re-indexed to request-list rows
 *   n_relations + slot (relation column copied).  uniq_out needs 3B entries, cuts_out world+1.
 * hole_shard_post: writes uniq[cuts[o]..cuts[o+1]) to rank o's inbox (PEER int32 [world][cap],
 *   row `me`) and (count, cuts[o]) to rank o's meta (PEER int32 [world][2], row `me`). */
HOLE_API int hole_shard_route(hole_ctx* ctx, const int32_t* pos, const int32_t* neg_ent, int64_t B,
                              int64_t n_relations, int64_t n_rows_global, int64_t rows_per_rank, int world,
                              int32_t* uniq_out, int32_t* cuts_out, int32_t* pos_w, int32_t* neg_w,
                              void* stream);
HOLE_API int hole_shard_post(hole_ctx* ctx, const int32_t* uniq, const int32_t* cuts, int world, int me,
                             int64_t cap, void* const* peer_inbox, void* const* peer_meta, void* stream);

/* Enable loads/stores from ctx's device to memory of `peer_device` (no-op if already on). */
HOLE_API int hole_enable_peer_access(hole_ctx* ctx, int peer_device);
HOLE_API int hole_gather_rows(hole_ctx* ctx, const float* table, const int64_t* ids, int64_t id_offset,
                     float* dst_rows, int64_t n, void* stream);
HOLE_API int hole_add_rows(hole_ctx* ctx, float* table, const int64_t* ids, int64_t id_offset,
                  const float* rows, int64_t n, void* stream);

/* ---- the training loop body for n_steps consecutive batches: replaces
 * `for batch in range(1, batch_count): sess.run([optimizer])` (holE.py:340-362) without
 * returning to the host between steps.  Step k uses triples[k*B .. (k+1)*B), draws its
 * corruption with (seed, first_step + k) and learning rate lr[k] [host, float32[n_steps]]
 * (the caller evaluates inverse_time_decay, holE.py:292-294).
 *   loss_out float32[n_steps*B] or NULL; loss_sum_out float32[n_steps] or NULL. */
HOLE_API int hole_train_steps(hole_ctx* ctx, float* table, const int32_t* triples, int64_t B,
                     int64_t n_steps, const int32_t* type_of, const int64_t* csr_off,
                     const int32_t* csr_ids, uint64_t seed, uint64_t first_step,
                     float margin, const float* lr, float* loss_out, float* loss_sum_out,
                     void* stream);

/* Same, end to end from HOST buffers: triples_host [host] int32[n_steps*B,3] (pinned or
 * pageable) is copied to the device in chunks overlapped with compute, and the per-step
 * loss sums are copied back to loss_sum_host [host] float32[n_steps].  Blocks until the
 * losses are on the host.  This is the call bench.py times for its "e2e" figure. */
HOLE_API int hole_train_steps_host(hole_ctx* ctx, float* table, const int32_t* triples_host, int64_t B,
                          int64_t n_steps, const int32_t* type_of, const int64_t* csr_off,
                          const int32_t* csr_ids, uint64_t seed, uint64_t first_step,
                          float margin, const float* lr, float* loss_sum_host, void* stream);

/* ---- ranking: replaces the scoring loop of infer_triples (holE.py:564-573) and the heap
 * of eval_link_prediction (holE.py:427-469) with a dense contraction on tcgen05 tensor
 * cores.  For query q = (h, t, r) and side:
 *   TAIL: candidates j in [ent_begin, ent_end) scored s_j = clip(E_j) . (h * r)
 *   HEAD: candidates j scored s_j = clip(E_j) . (r * conj(t))~        (SURVEY App. A.4)
 *   RELATION: candidates j scored s_j = clip(E_j) . (h * conj(t))~, i.e. [Re w ; -Im w] with
 *         w = clip(h) o conj(clip(t)) (ds/dy_r of SURVEY App. A.3).  The caller passes the relation
 *         rows, [ent_begin, ent_end) = [0, n_relations), as it passes the entity rows for TAIL / HEAD;
 *         the true candidate is column 2 (r), a query's filter slice lists the known relations of
 *         (h, t), ties go to the smaller relation id, and every per-query array has Q rows.
 *         In HOLE_SCORE_CCORR_TANH mode the query vector is ds/dr = [Re c + Im c ; Re c - Im c] with
 *         c_k = sum_j conj(h_j) t_{j+k} (rows clipped).  hole_rank_ex's query_table supplies h and t.
 *         A relation call over another range than a hole_rank_prepare'd one re-packs the candidate
 *         operand and drops the prepared one (the cache holds one range).
 *   (~: imaginary half negated)
 * raw_before[q]  = #{j : (s_j, j) < (s_true, true_id)}  (ascending: lower is better,
 *                  holE.py:231, 446-453; ties by smaller candidate id, holE.py:434)
 * filt_before[q] = raw_before[q] - #{f in filter[q], f in range : (s_f, f) < (s_true, true_id)}
 *                  (train/valid-true candidates do not advance the filtered rank,
 *                  holE.py:454-463), with s_f the very score raw_before was counted with: a filtered
 *                  candidate is subtracted exactly when it was counted.  With compute_true != 0 the true
 *                  candidate never counts (it is not before itself); with compute_true == 0 its column is an
 *                  ordinary candidate against the given threshold.  rank = 1 + count.
 * filter_off int64[Q+1] / filter_ids int32[.] may be NULL (no filtering); the ids of each slice must be
 * ASCENDING (the count epilogue merge-joins them with its columns; data.build_filter_csr produces them so).
 * A slice is a set: an id listed twice is subtracted once.  Ids outside [ent_begin, ent_end) are ignored.
 * true_score_io float32[Q]: if compute_true != 0 it is written for queries whose true
 * candidate lies in [ent_begin, ent_end) and left untouched otherwise (so candidate shards
 * on several GPUs can be combined by the caller); if compute_true == 0 it is read.
 * Counts are ADDED to raw_before / filt_before (caller zeroes them), so shards accumulate.
 * side == HOLE_SIDE_BOTH ranks both sides in one pass (candidates packed once): every
 * per-query array (true_score_io, raw_before, filt_before, and filter_off with 2Q+1 entries)
 * then has 2Q rows -- rows [0,Q) are the tail ranks, rows [Q,2Q) the head ranks.  BOTH does not include
 * relations; there is no three-side mode. */
HOLE_API int hole_rank(hole_ctx* ctx, const float* table, int64_t ent_begin, int64_t ent_end,
              const int32_t* queries, int64_t Q, int side, int precision,
              const int64_t* filter_off, const int32_t* filter_ids,
              float* true_score_io, int compute_true,
              int32_t* raw_before, int32_t* filt_before, void* stream);

/* hole_rank_ex: as hole_rank, with two extensions used by the candidate-sharded ranking:
 *   query_table  when non-NULL, the rows of a query's OTHER entity and of its relation are read from this
 *                table (same row layout) instead of `table`; the query's true-candidate column is then only
 *                an index into [ent_begin, ent_end) of `table` (it may lie outside: not in this shard);
 *   raw_before == filt_before == NULL (with compute_true != 0): true scores only, no counting pass.
 * hole_rank_prepare packs the candidate operand of [ent_begin, ent_end) once; later hole_rank / hole_rank_ex
 * calls on the same (table, range, precision) reuse it instead of re-packing, until hole_rank_invalidate, a
 * training call on this context, or a call with another table / range -- a HOLE_SIDE_RELATION call over the
 * relation rows included: the cache has a single slot, so the next entity call re-packs.  The caller must
 * invalidate after changing the table by any other means. */
HOLE_API int hole_rank_ex(hole_ctx* ctx, const float* table, int64_t ent_begin, int64_t ent_end,
                 const float* query_table, const int32_t* queries, int64_t Q, int side, int precision,
                 const int64_t* filter_off, const int32_t* filter_ids,
                 float* true_score_io, int compute_true,
                 int32_t* raw_before, int32_t* filt_before, void* stream);
HOLE_API int hole_rank_prepare(hole_ctx* ctx, const float* table, int64_t ent_begin, int64_t ent_end,
                      int precision, void* stream);
HOLE_API int hole_rank_invalidate(hole_ctx* ctx);

/* ---- top-k link prediction: the entities the model puts first for (h, r, ?) or (?, r, t), or with
 * HOLE_SIDE_RELATION the relations it puts first for (h, ?, t) over [ent_begin, ent_end) = [0, n_relations).  Replaces the pop
 * loop of eval_link_prediction (holE.py:427-472: candidates popped in ascending order, at most
 * InferenceCandidates.max_triples of them) over ALL candidates [ent_begin, ent_end), on the same tensor-core
 * contraction as hole_rank (same operand packing, same hole_rank_prepare cache and invalidation rules).
 * For query q = (h, t, r) the candidate scores s_j are hole_rank's (TAIL / HEAD, or the HOLE_SCORE_CCORR_TANH
 * query vector in that mode); the id being predicted (t for TAIL, h for HEAD, r for RELATION) is ignored.
 * Row q of the output holds the k candidates first in ascending (s, id) order (lower is better, ties to the
 * smaller id: the heap's order, holE.py:231, 434, 446-453), skipping the ids of q's filter slice:
 *   ids_out    int32 [Q', k]  global row ids, sorted by (score, id)
 *   scores_out float32 [Q', k] raw s of each id
 * with Q' = Q, or 2Q for HOLE_SIDE_BOTH (rows [0,Q) tails, [Q,2Q) heads, filter_off then has 2Q+1 entries).
 * filter_off int64[Q'+1] / filter_ids int32[.] may be NULL; the ids of each slice must be ASCENDING (binary
 * search; data.build_filter_csr produces them so).  Fewer than k remaining candidates: the row is padded with
 * id -1, score +inf.
 * Precision: the selection runs at the contraction's operand precision (HOLE_RANK_BF16 / _BF16X3); the
 * returned scores are recomputed in fp32 from the fp32 table (clipped candidate row . fp32 query vector), so
 * the id set is the exact top-k except for candidates within the precision's near-tie band of the k-th score.
 * 1 <= k <= 128, else HOLE_ERR_ARG.  HOLE_ERR_ALLOC when the workspace ([Q'][work items][2][k] 8-byte keys)
 * cannot be allocated: split Q.  hole_rank_debug_operands returns the operands of the last hole_rank or
 * hole_topk call. */
HOLE_API int hole_topk(hole_ctx* ctx, const float* table, int64_t ent_begin, int64_t ent_end,
                       const int32_t* queries, int64_t Q, int side, int precision, int k,
                       const int64_t* filter_off, const int32_t* filter_ids,
                       int32_t* ids_out, float* scores_out, void* stream);

/* ---- nearest neighbours: the rows of [ent_begin, ent_end) whose embeddings are most similar to row ids[q]
 * (what holE.py leaves to the TensorBoard projector it configures, holE.py:334-337), on hole_topk's tensor-core
 * contraction, top-k epilogue and merge.  Similarity is the cosine over the whole stored row as one real vector
 * of dim components, cos(q, j) = E_q . E_j / (|E_q| |E_j|) = Re sum_k q_k conj(j_k); neither the norm clip nor
 * the score mode enters it (HOLE_SCORE_COMPLEX and HOLE_SCORE_CCORR_TANH give the same result).  A row of zero
 * norm has similarity exactly 0 with every row, as query and as candidate.
 *   ids        int32 [Q]     query rows; the caller guarantees 0 <= ids[q] < n_rows (they may lie outside the range,
 *                            e.g. an entity queried against the relation rows [0, n_relations))
 *   ids_out    int32 [Q, k]  global row ids, by descending similarity, ties to the smaller id
 *   sim_out    float32 [Q, k] their similarities, recomputed in fp32 from the fp32 table
 * Row ids[q] itself is never returned; other rows with an identical embedding are.  The ids of q's filter slice
 * (filter_off int64[Q+1] / filter_ids int32[.], may be NULL, ids ASCENDING within a slice) are skipped.  Fewer
 * than k candidates left: the row is padded with id -1, similarity -inf.
 * Precision, limits and errors as hole_topk: the id set is exact except within the precision's near-tie band of
 * the k-th similarity (3e-5 for HOLE_RANK_BF16X3, 4e-3 for HOLE_RANK_BF16: both operands have unit norm);
 * 1 <= k <= 128, else HOLE_ERR_ARG; dim <= 640 (bf16) / 320 (bf16x3), else HOLE_ERR_UNSUPPORTED before any launch
 * or write -- except that an empty range (ent_begin == ent_end), which has no candidate to score, writes its
 * all-padding rows and returns HOLE_OK at any dim, as hole_topk does; HOLE_ERR_ALLOC when the workspace does not
 * fit: split Q.
 * Operand cache: the call packs its own (unit-normalised) candidate operand into the single cache slot and drops a
 * hole_rank_prepare'd one, which a later hole_rank / hole_topk call therefore re-packs.  A prepared (clipped)
 * operand is never used for cosine, and a normalised one never for ranking.  hole_rank_debug_operands returns
 * the operands of the last hole_neighbors call as it does for hole_rank / hole_topk.
 * Row-sharded tables: gather the whole table onto one GPU first (gather_embeddings() of the sharded trainer). */
HOLE_API int hole_neighbors(hole_ctx* ctx, const float* table, int64_t ent_begin, int64_t ent_end,
                            const int32_t* ids, int64_t Q, int precision, int k,
                            const int64_t* filter_off, const int32_t* filter_ids,
                            int32_t* ids_out, float* sim_out, void* stream);

/* Test hook: copy the bf16 operands the last hole_rank call packed (device to device).
 * cand_out [n_pad, K] / query_out [q_pad, K] may be NULL to query the shapes only. */
HOLE_API int hole_rank_debug_operands(hole_ctx* ctx, void* cand_out, void* query_out,
                             int64_t* n_pad, int64_t* q_pad, int* K, void* stream);

/* ---- measurement hooks (bench.py's roofline figure).  With profiling enabled every
 * training step records CUDA events on `stream` around its two hot kernels (K1 =
 * hole_k1_kernel, K3 = hole_apply_kernel or, with AdaGrad, hole_adagrad_apply_kernel).  hole_profile_read synchronises and
 * returns the summed kernel times in milliseconds and the number of steps measured since
 * the last hole_profile_enable call. */
HOLE_API int hole_profile_enable(hole_ctx* ctx, int on);
HOLE_API int hole_profile_read(hole_ctx* ctx, double* k1_ms, double* k3_ms, int64_t* n_steps);

/* Host helper: parse a triple file (`head<TAB>tail<TAB>relation` per line, holE.py:76-81) into
 * out [host] int32[cap,3].  Returns the number of triples in the file (call with cap = 0 to
 * size the buffer), or a negative error code. */
HOLE_API int64_t hole_parse_triples(const char* path, int32_t* out_host, int64_t cap);

/* Host helper for the checkpoint writer: CRC32C (Castagnoli) of a HOST buffer, continuing
 * from `crc` (0 to start).  TF's tensor bundle stores it masked (holE.py:359 saver.save). */
HOLE_API uint32_t hole_crc32c(uint32_t crc, const void* data_host, uint64_t n);

/* Number of kernels this library has launched on this thread's contexts since the last
 * reset (bench.py's "gpu_launches"). */
HOLE_API int64_t hole_launch_count(void);
HOLE_API void hole_launch_count_reset(void);

#ifdef __cplusplus
}
#endif
#endif /* HOLE_B200_H */
