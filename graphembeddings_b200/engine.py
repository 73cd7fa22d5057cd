"""Device engine: owns the embedding table in HBM and calls libhole_b200 through ctypes.

PyTorch is plumbing here (device memory, streams, torch.distributed); every numerical
operation is a kernel of libhole_b200.so.  Method names follow the holE.py functions they
replace (corrupt_batch holE.py:152, evaluate_triples holE.py:179, evaluate_batch
holE.py:205 + minimize holE.py:296, eval_link_prediction holE.py:427).
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import (HOLE_RANK_BF16, HOLE_RANK_BF16X3, HOLE_SIDE_BOTH, HOLE_SIDE_HEAD, HOLE_SIDE_RELATION,
                   HOLE_SIDE_TAIL, HoleError, check)

__all__ = ["HoleEngine", "HoleError", "inverse_time_decay", "HOLE_SIDE_TAIL", "HOLE_SIDE_HEAD", "HOLE_SIDE_BOTH",
           "HOLE_SIDE_RELATION", "HOLE_RANK_BF16", "HOLE_RANK_BF16X3"]


def inverse_time_decay(lr0, step, decay_steps, decay_rate):
    """tf.train.inverse_time_decay evaluated in fp32 (holE.py:292-294; App. B)."""
    f = np.float32
    return f(lr0) / (f(1.0) + f(decay_rate) * (f(step) / f(decay_steps)))


def _ptr(t):
    return C.c_void_p(0) if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class HoleEngine:
    """One GPU's share of the HolE model: the shared relation+entity table
    (holE.py:263-264) in the padded device layout, plus the device-resident type tables
    that replace holE.py's two MutableHashTables (holE.py:267-277)."""

    def __init__(self, n_rows, dim, device=0):
        if not torch.cuda.is_available():
            raise HoleError("no CUDA device: libhole_b200 has no CPU fallback")
        self.lib = _lib.load()
        self.device = torch.device("cuda", device)
        self.n_rows, self.dim = int(n_rows), int(dim)
        stride = self.lib.hole_row_stride(self.dim)
        if stride < 0:
            raise HoleError(f"embedding_dim must be a positive even number, got {dim}")
        self.row_stride = stride
        h = C.c_void_p()
        check(self.lib.hole_ctx_create(C.byref(h), device, self.n_rows, self.dim))
        self._ctx = h
        self.table = None
        self.accum = None          # AdaGrad accumulator (set_optimizer)
        self.type_of = self.csr_off = self.csr_ids = None

    def set_relation_count(self, n_relations):
        """holE.py:52 relation_count: relation ids are < n_relations (plan-sort hint)."""
        check(self.lib.hole_ctx_set_relations(self._ctx, int(n_relations)))
        return self

    def set_score_mode(self, mode):
        """"complex" (live holE.py:191-198, sigma of the Hermitian product) or "ccorr_tanh" (the archived
        variant of holE-20170724/graph.pbtxt:6221-6521: tanh of r-weighted circular correlation)."""
        code = {"complex": 0, "ccorr_tanh": 1}.get(mode, mode)      # HOLE_SCORE_COMPLEX / HOLE_SCORE_CCORR_TANH
        check(self.lib.hole_ctx_set_score_mode(self._ctx, int(code)))
        return self

    def set_optimizer(self, optimizer, initial_accumulator=0.1):
        """"sgd" (holE.py:296's GradientDescentOptimizer, the default) or "adagrad" (TF's
        AdagradOptimizer(lr, initial_accumulator_value) in its place).  "adagrad" allocates the accumulator
        [n_rows, row_stride] and fills all of it, pad columns included, with initial_accumulator (> 0);
        "sgd" drops it.  AdaGrad trains through train_step / train_steps / train_steps_host only."""
        if optimizer == "sgd":
            check(self.lib.hole_ctx_set_optimizer(self._ctx, _lib.HOLE_OPT_SGD, None))
            self.accum = None
            return self
        if optimizer != "adagrad":
            raise HoleError(f"unknown optimizer {optimizer!r}: 'sgd' or 'adagrad'")
        if not float(initial_accumulator) > 0.0:
            raise HoleError(f"initial_accumulator must be > 0, got {initial_accumulator}")
        accum = torch.full((self.n_rows, self.row_stride), float(initial_accumulator), dtype=torch.float32,
                           device=self.device)
        check(self.lib.hole_ctx_set_optimizer(self._ctx, _lib.HOLE_OPT_ADAGRAD, _ptr(accum)))
        self.accum, self.initial_accumulator = accum, float(initial_accumulator)
        return self

    def accumulator(self):
        """The AdaGrad accumulator as a [N, dim] float32 CUDA tensor (checkpoint layout, the slot
        `embeddings/Adagrad`)."""
        if getattr(self, "accum", None) is None:
            raise HoleError("the optimizer is not adagrad: there is no accumulator")
        out = torch.empty((self.n_rows, self.dim), dtype=torch.float32, device=self.device)
        check(self.lib.hole_unpack_rows(self._ctx, _ptr(self.accum), _ptr(out), self.n_rows, _stream()))
        return out

    def set_accumulator(self, A):
        """A: [N, dim] float32 (checkpoint layout), every element > 0.  The pad columns of the device layout
        are refilled with the initial value (packing writes zeros there)."""
        if getattr(self, "accum", None) is None:
            raise HoleError("the optimizer is not adagrad: there is no accumulator")
        A = torch.as_tensor(A, dtype=torch.float32)
        assert A.shape == (self.n_rows, self.dim), A.shape
        src = A.to(self.device).contiguous()
        if not bool((src > 0).all()):
            raise HoleError("every accumulator element must be > 0")
        check(self.lib.hole_pack_rows(self._ctx, _ptr(src), _ptr(self.accum), self.n_rows, _stream()))
        half, H = self.row_stride // 2, self.dim // 2
        if H < half:
            self.accum[:, H:half] = self.initial_accumulator
            self.accum[:, half + H:] = self.initial_accumulator
        torch.cuda.current_stream().synchronize()   # src may be freed by the caller
        return self

    def close(self):
        if getattr(self, "_ctx", None):
            self.lib.hole_ctx_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ table
    def set_embeddings(self, E):
        """E: [N, dim] float32 (numpy or torch, checkpoint layout [Re | Im])."""
        E = torch.as_tensor(E, dtype=torch.float32)
        assert E.shape == (self.n_rows, self.dim), E.shape
        src = E.to(self.device).contiguous()
        if self.table is None:
            self.table = torch.empty((self.n_rows, self.row_stride), dtype=torch.float32,
                                     device=self.device)
        check(self.lib.hole_pack_rows(self._ctx, _ptr(src), _ptr(self.table), self.n_rows, _stream()))
        torch.cuda.current_stream().synchronize()   # src may be freed by the caller
        return self

    def embeddings(self):
        """Current table as a [N, dim] float32 CUDA tensor (checkpoint layout)."""
        out = torch.empty((self.n_rows, self.dim), dtype=torch.float32, device=self.device)
        check(self.lib.hole_unpack_rows(self._ctx, _ptr(self.table), _ptr(out), self.n_rows, _stream()))
        return out

    def set_types(self, type_of, csr_off, csr_ids):
        """Device-resident type -> entity CSR (replaces holE.py:267-277, 343-347)."""
        self.type_of = torch.as_tensor(np.asarray(type_of), dtype=torch.int32).to(self.device)
        self.csr_off = torch.as_tensor(np.asarray(csr_off), dtype=torch.int64).to(self.device)
        self.csr_ids = torch.as_tensor(np.asarray(csr_ids), dtype=torch.int32).to(self.device)
        return self

    def _triples(self, triples):
        t = torch.as_tensor(triples)
        if t.dtype != torch.int32:
            t = t.to(torch.int32)
        t = t.to(self.device).contiguous()
        assert t.dim() == 2 and t.shape[1] == 3, t.shape
        return t

    # ------------------------------------------------------------------ hot path
    def corrupt_batch(self, triples, seed, step, index_base=0):
        """holE.py:152 corrupt_batch -> (side, neg_ent int32[B] on device).  index_base: position
        of triples[0] inside the global (multi-GPU) batch."""
        t = self._triples(triples)
        B = t.shape[0]
        neg = torch.empty(B, dtype=torch.int32, device=self.device)
        side = C.c_int(0)
        check(self.lib.hole_corrupt_at(self._ctx, _ptr(t), B, _ptr(self.type_of), _ptr(self.csr_off),
                                       _ptr(self.csr_ids), seed, step, int(index_base), None, _ptr(neg),
                                       C.byref(side), _stream()))
        return int(side.value), neg

    def evaluate_triples(self, triples):
        """holE.py:179 evaluate_triples -> sigma(score) float32[B] on device."""
        t = self._triples(triples)
        out = torch.empty(t.shape[0], dtype=torch.float32, device=self.device)
        check(self.lib.hole_score(self._ctx, _ptr(self.table), _ptr(t), t.shape[0], _ptr(out), _stream()))
        return out

    def train_step(self, pos, neg_ent, side, margin, lr, return_sigma=False):
        """One step: evaluate_batch hinge branch (holE.py:222-234) + minimize (holE.py:296),
        with caller-supplied corruption.  Returns loss float32[B] (and sigma+/-)."""
        p = self._triples(pos)
        B = p.shape[0]
        n = torch.as_tensor(neg_ent).to(torch.int32).to(self.device).contiguous()
        loss = torch.empty(B, dtype=torch.float32, device=self.device)
        sig = torch.empty(2 * B, dtype=torch.float32, device=self.device) if return_sigma else None
        check(self.lib.hole_train_step(self._ctx, _ptr(self.table), _ptr(p), _ptr(n), int(side), B,
                                       float(margin), float(lr), _ptr(loss), _ptr(sig), _stream()))
        if return_sigma:
            return loss, sig[:B], sig[B:]
        return loss

    def train_step_plan(self, pos_i32, neg_i32):
        """Build the update plan of the next train_step_delta call (same tensors) on a side
        stream, overlapping whatever is enqueued in between."""
        check(self.lib.hole_train_step_plan(self._ctx, _ptr(pos_i32), _ptr(neg_i32), pos_i32.shape[0], _stream()))

    def train_step_delta(self, pos_i32, neg_i32, side, margin, lr, delta_out):
        """One step that leaves the table untouched and writes every row's change into
        delta_out [n_rows, row_stride].  Every row the step uses is written; rows it does not
        use (relations absent from the batch) keep their content, so the caller clears the
        relation block.  pos/neg: int32 CUDA tensors."""
        B = pos_i32.shape[0]
        loss = torch.empty(B, dtype=torch.float32, device=self.device)
        check(self.lib.hole_train_step_ex(self._ctx, _ptr(self.table), _ptr(delta_out), _ptr(pos_i32),
                                          _ptr(neg_i32), int(side), B, float(margin), float(lr),
                                          _ptr(loss), None, _stream()))
        return loss

    def train_step_logloss(self, triples, seed, step, lr, l2=0.0, negative_ratio=1, want_corruption=False,
                           want_l2_loss=None):
        """The --log_loss step (holE.py:194-196, 206-220, 296).  Returns (loss [(1+k), B] device,
        l2_loss device scalar = sum(E_old^2)/2) -- the reference's per-row loss is
        loss + l2 * l2_loss -- and, with want_corruption, also (sides list, neg [k, B] device).
        The scalar costs a pass over the whole table: by default it is only computed when
        l2 != 0 (it is zero otherwise); want_l2_loss=True forces it."""
        t = self._triples(triples)
        B, k = t.shape[0], int(negative_ratio)
        if getattr(self, "_delta_ws", None) is None or self._delta_ws.shape != self.table.shape:
            self._delta_ws = torch.zeros_like(self.table)
        loss = torch.empty((1 + k, B), dtype=torch.float32, device=self.device)
        l2_loss = torch.zeros((), dtype=torch.float32, device=self.device)
        neg = torch.empty((k, B), dtype=torch.int32, device=self.device) if want_corruption else None
        sides = (C.c_int32 * k)()
        check(self.lib.hole_train_step_logloss(
            self._ctx, _ptr(self.table), _ptr(self._delta_ws), _ptr(t), B, k, _ptr(self.type_of),
            _ptr(self.csr_off), _ptr(self.csr_ids), int(seed), int(step), float(lr), float(l2), _ptr(loss),
            _ptr(l2_loss) if (want_l2_loss or (want_l2_loss is None and l2 != 0.0)) else None,
            None if neg is None else _ptr(neg), sides, _stream()))
        if want_corruption:
            return loss, l2_loss, list(sides), neg
        return loss, l2_loss

    # ---- multi-GPU step routing (include/hole_b200.h, "multi-GPU step routing") ----
    @staticmethod
    def peer_array(tensors):
        """ctypes void*[world] of the tensors' device addresses (keep the tensors alive)."""
        return (C.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])

    def shard_route(self, pos_i32, neg_i32, n_relations, n_rows_global, rows_per_rank, world,
                    uniq, cuts, pos_w, neg_w):
        check(self.lib.hole_shard_route(self._ctx, _ptr(pos_i32), _ptr(neg_i32), pos_i32.shape[0],
                                        int(n_relations), int(n_rows_global), int(rows_per_rank), int(world),
                                        _ptr(uniq), _ptr(cuts), _ptr(pos_w), _ptr(neg_w), _stream()))

    def shard_post(self, uniq, cuts, world, me, cap, peer_inbox, peer_meta):
        check(self.lib.hole_shard_post(self._ctx, _ptr(uniq), _ptr(cuts), int(world), int(me), int(cap),
                                       peer_inbox, peer_meta, _stream()))

    def shard_init(self, world, me, n_relations, n_entities, rows_per_rank, max_batch, shard, peer_shard,
                   peer_stage, peer_relstage, peer_inbox, peer_meta, peer_flags, err_flag, timeout_s=0.0):
        """hole_shard_init: bind this context to a row-sharded table (peer_* = ctypes void*[world] of the
        IPC-mapped buffers, see include/hole_b200.h).  The type tables must have been set."""
        self._shard_keep = (shard, err_flag)
        check(self.lib.hole_shard_init(self._ctx, int(world), int(me), int(n_relations), int(n_entities),
                                       int(rows_per_rank), int(max_batch), _ptr(shard), peer_shard, peer_stage,
                                       peer_relstage, peer_inbox, peer_meta, peer_flags, _ptr(err_flag),
                                       float(timeout_s), _ptr(self.type_of), _ptr(self.csr_off), _ptr(self.csr_ids)))

    def shard_set_optimizer(self, optimizer, accum_shard=None):
        """hole_shard_set_optimizer: the optimizer of the following sharded steps ("sgd" with no accumulator,
        "adagrad" with accum_shard = float32 CUDA [n_relations + rows_per_rank, row_stride], every element > 0,
        kept alive here while bound).  Call after shard_init, on every rank before the same step."""
        code = {"sgd": _lib.HOLE_OPT_SGD, "adagrad": _lib.HOLE_OPT_ADAGRAD}.get(optimizer, optimizer)
        check(self.lib.hole_shard_set_optimizer(self._ctx, int(code), _ptr(accum_shard)))
        self._shard_accum = accum_shard
        return self

    def shard_prepare(self, pos_i32, seed, step):
        check(self.lib.hole_shard_prepare(self._ctx, _ptr(pos_i32), pos_i32.shape[0], int(seed), int(step), _stream()))

    def shard_step(self, pos_i32, seed, step, margin, lr, loss_out=None, phase=None):
        """One row-sharded step on this rank's slice (int32 CUDA [B,3], global row ids).  phase:
        None = whole step, "compute" / "apply" = its halves (virtual-rank tests)."""
        if phase == "apply":
            check(self.lib.hole_shard_step_apply(self._ctx, _stream()))
            return None
        B = pos_i32.shape[0]
        if loss_out is None:
            loss_out = torch.empty(B, dtype=torch.float32, device=self.device)
        fn = self.lib.hole_shard_step if phase is None else self.lib.hole_shard_step_compute
        check(fn(self._ctx, _ptr(pos_i32), B, int(seed), int(step), float(margin), float(lr), _ptr(loss_out), _stream()))
        return loss_out

    def shard_steps(self, triples_i32, batch_size, seed, first_step, margin, lrs):
        """n_steps consecutive sharded steps on device-resident slices [n_steps*B, 3]; returns the
        per-step loss sums of this rank's slices (device float32)."""
        n_steps = triples_i32.shape[0] // batch_size
        lrs = np.ascontiguousarray(np.asarray(lrs, dtype=np.float32))
        assert len(lrs) >= n_steps
        sums = torch.empty(n_steps, dtype=torch.float32, device=self.device)
        check(self.lib.hole_shard_steps(self._ctx, _ptr(triples_i32), batch_size, n_steps, int(seed), int(first_step),
                                        float(margin), lrs.ctypes.data_as(C.c_void_p), _ptr(sums), _stream()))
        return sums

    def shard_steps_host(self, triples_host, batch_size, seed, first_step, margin, lrs):
        """Same from a HOST int32 [n,3] tensor (pinned) / array; copies inside; returns numpy loss sums."""
        if isinstance(triples_host, torch.Tensor):
            assert triples_host.device.type == "cpu" and triples_host.dtype == torch.int32 and triples_host.is_contiguous()
            n, ptr = triples_host.shape[0], C.c_void_p(triples_host.data_ptr())
        else:
            triples_host = np.ascontiguousarray(triples_host, dtype=np.int32)
            n, ptr = triples_host.shape[0], triples_host.ctypes.data_as(C.c_void_p)
        n_steps = n // batch_size
        lrs = np.ascontiguousarray(np.asarray(lrs, dtype=np.float32))
        out = np.empty(n_steps, dtype=np.float32)
        check(self.lib.hole_shard_steps_host(self._ctx, ptr, batch_size, n_steps, int(seed), int(first_step),
                                             float(margin), lrs.ctypes.data_as(C.c_void_p),
                                             out.ctypes.data_as(C.c_void_p), _stream()))
        return out

    def shard_profile_read(self):
        """-> ({phase: ms per step}, n_steps) of the sharded steps since profile(True)."""
        ms = (C.c_double * 5)()
        n = C.c_int64(0)
        check(self.lib.hole_shard_profile_read(self._ctx, ms, C.byref(n)))
        k = max(int(n.value), 1)
        return {nm: ms[i] / k for i, nm in enumerate(("post", "k1", "k3", "finish", "apply"))}, int(n.value)

    def shard_poll(self):
        """True if a peer failed to arrive at a step barrier (synchronises the stream)."""
        v = C.c_int(0)
        check(self.lib.hole_shard_poll(self._ctx, C.byref(v), _stream()))
        return v.value != 0

    def enable_peer_access(self, peer_device):
        check(self.lib.hole_enable_peer_access(self._ctx, int(peer_device)))

    def gather_rows(self, table, ids_i64, id_offset, dst_rows):
        """dst_rows[k] = table[ids[k] + id_offset]; dst_rows may be a peer GPU's (IPC) buffer."""
        check(self.lib.hole_gather_rows(self._ctx, _ptr(table), _ptr(ids_i64), int(id_offset), _ptr(dst_rows),
                                        ids_i64.shape[0], _stream()))

    def add_rows(self, table, ids_i64, id_offset, rows):
        """table[ids + id_offset] += rows, ids unique (the owner applies one rank's deltas)."""
        check(self.lib.hole_add_rows(self._ctx, _ptr(table), _ptr(ids_i64), int(id_offset), _ptr(rows),
                                     ids_i64.shape[0], _stream()))

    def train_steps(self, triples, batch_size, seed, first_step, margin, lrs, want_loss=False):
        """n_steps = len(triples) // batch_size consecutive steps on device-resident triples
        (the loop body holE.py:340-362).  Returns per-step loss sums (device float32)."""
        t = self._triples(triples)
        n_steps = t.shape[0] // batch_size
        lrs = np.ascontiguousarray(np.asarray(lrs, dtype=np.float32))
        assert len(lrs) >= n_steps
        sums = torch.empty(n_steps, dtype=torch.float32, device=self.device)
        loss = (torch.empty(n_steps * batch_size, dtype=torch.float32, device=self.device)
                if want_loss else None)
        check(self.lib.hole_train_steps(self._ctx, _ptr(self.table), _ptr(t), batch_size, n_steps,
                                        _ptr(self.type_of), _ptr(self.csr_off), _ptr(self.csr_ids),
                                        seed, first_step, float(margin),
                                        lrs.ctypes.data_as(C.c_void_p), _ptr(loss), _ptr(sums),
                                        _stream()))
        return (sums, loss) if want_loss else sums

    def train_steps_host(self, triples_host, batch_size, seed, first_step, margin, lrs):
        """Same from a HOST int32 [n,3] array (numpy or pinned torch tensor); host<->device
        copies happen inside the call.  Returns per-step loss sums as a numpy array."""
        if isinstance(triples_host, torch.Tensor):
            assert triples_host.device.type == "cpu" and triples_host.dtype == torch.int32
            assert triples_host.is_contiguous()
            n, ptr = triples_host.shape[0], C.c_void_p(triples_host.data_ptr())
        else:
            triples_host = np.ascontiguousarray(triples_host, dtype=np.int32)
            n, ptr = triples_host.shape[0], triples_host.ctypes.data_as(C.c_void_p)
        n_steps = n // batch_size
        lrs = np.ascontiguousarray(np.asarray(lrs, dtype=np.float32))
        out = np.empty(n_steps, dtype=np.float32)
        check(self.lib.hole_train_steps_host(self._ctx, _ptr(self.table), ptr, batch_size, n_steps,
                                             _ptr(self.type_of), _ptr(self.csr_off),
                                             _ptr(self.csr_ids), seed, first_step, float(margin),
                                             lrs.ctypes.data_as(C.c_void_p),
                                             out.ctypes.data_as(C.c_void_p), _stream()))
        return out

    # ------------------------------------------------------------------ ranking
    def rank(self, queries, side, ent_begin, ent_end, filter_off=None, filter_ids=None,
             precision=HOLE_RANK_BF16, true_score=None, compute_true=True,
             raw_before=None, filt_before=None):
        """All-candidate ranking of queries [Q,3] over candidate rows [ent_begin, ent_end)
        (eval_link_prediction holE.py:427-469 as a tensor-core contraction).  Returns
        (raw_before int32[Q], filt_before int32[Q], true_score float32[Q]); rank = 1 + count.
        Counts are accumulated into raw_before / filt_before when given (candidate shards).
        HOLE_SIDE_RELATION ranks each query's relation (column 2) over relation rows [ent_begin, ent_end),
        normally [0, n_relations)."""
        q = self._triples(queries)
        Q = q.shape[0]
        nq = Q
        if int(side) == HOLE_SIDE_BOTH:
            Q = 2 * Q          # rows [0,nq) tail ranks, [nq,2nq) head ranks
        if raw_before is None:
            raw_before = torch.zeros(Q, dtype=torch.int32, device=self.device)
        if filt_before is None:
            filt_before = torch.zeros(Q, dtype=torch.int32, device=self.device)
        if true_score is None:
            true_score = torch.zeros(Q, dtype=torch.float32, device=self.device)
        fo = fi = None
        if filter_off is not None and len(filter_ids) > 0:      # no ids: nothing to filter (and no device pointer)
            fo = torch.as_tensor(filter_off).to(torch.int64).to(self.device).contiguous()
            fi = torch.as_tensor(filter_ids).to(torch.int32).to(self.device).contiguous()
        check(self.lib.hole_rank(self._ctx, _ptr(self.table), int(ent_begin), int(ent_end), _ptr(q),
                                 nq, int(side), int(precision), _ptr(fo), _ptr(fi), _ptr(true_score),
                                 1 if compute_true else 0, _ptr(raw_before), _ptr(filt_before),
                                 _stream()))
        return raw_before, filt_before, true_score

    def topk(self, queries, side, ent_begin, ent_end, k, filter_off=None, filter_ids=None,
             precision=HOLE_RANK_BF16X3):
        """Top-k link prediction (the pop loop of eval_link_prediction, holE.py:427-472, over all candidates
        [ent_begin, ent_end)): for every query row the k candidates first in ascending (score, id) order,
        skipping its filter slice.  Returns (ids int32[Q', k], scores float32[Q', k]) on the device, Q' = Q or
        2Q for HOLE_SIDE_BOTH; padding is id -1 / score +inf.  Each filter slice must be ascending.
        HOLE_SIDE_RELATION predicts the relations of (h, ?, t) over relation rows [ent_begin, ent_end)."""
        q = self._triples(queries)
        rows = q.shape[0] * (2 if int(side) == HOLE_SIDE_BOTH else 1)
        fo, fi = self._filter_csr(filter_off, filter_ids, rows)
        ids_out = torch.empty((rows, int(k)), dtype=torch.int32, device=self.device)
        scores = torch.empty((rows, int(k)), dtype=torch.float32, device=self.device)
        check(self.lib.hole_topk(self._ctx, _ptr(self.table), int(ent_begin), int(ent_end), _ptr(q), q.shape[0],
                                 int(side), int(precision), int(k), _ptr(fo), _ptr(fi), _ptr(ids_out), _ptr(scores),
                                 _stream()))
        return ids_out, scores

    def neighbors(self, ids, k, ent_begin, ent_end, filter_off=None, filter_ids=None, precision=HOLE_RANK_BF16X3):
        """Nearest neighbours by cosine similarity of the whole stored rows: for every row ids[q], the k rows of
        [ent_begin, ent_end) most similar to it, itself excluded, skipping its filter slice (ascending ids).
        Returns (ids int32[Q, k], sims float32[Q, k]) on the device, by descending similarity with ties to the
        smaller id; padding is id -1 / similarity -inf.  Independent of the score mode."""
        q = torch.as_tensor(ids).reshape(-1)
        if q.numel() and (int(q.min()) < 0 or int(q.max()) >= self.n_rows):
            raise HoleError(f"neighbour query ids must lie in [0, {self.n_rows})")
        q = q.to(torch.int32).to(self.device).contiguous()
        rows = q.shape[0]
        fo, fi = self._filter_csr(filter_off, filter_ids, rows)
        ids_out = torch.empty((rows, int(k)), dtype=torch.int32, device=self.device)
        sims = torch.empty((rows, int(k)), dtype=torch.float32, device=self.device)
        check(self.lib.hole_neighbors(self._ctx, _ptr(self.table), int(ent_begin), int(ent_end), _ptr(q), rows,
                                      int(precision), int(k), _ptr(fo), _ptr(fi), _ptr(ids_out), _ptr(sims),
                                      _stream()))
        return ids_out, sims

    def _filter_csr(self, filter_off, filter_ids, rows):
        """Checks a filter CSR of `rows` slices (ascending ids within each) and returns it as device tensors
        (int64 offsets, int32 ids), or (None, None) for no filter or one without ids."""
        if filter_off is None:
            return None, None
        off = np.asarray(filter_off.cpu() if isinstance(filter_off, torch.Tensor) else filter_off, dtype=np.int64)
        ids = np.asarray(filter_ids.cpu() if isinstance(filter_ids, torch.Tensor) else filter_ids, dtype=np.int64)
        if off.shape != (rows + 1,) or off[0] != 0 or off[-1] != len(ids) or np.any(np.diff(off) < 0):
            raise HoleError(f"filter_off must be a CSR offset array of {rows + 1} entries over {len(ids)} ids")
        desc = np.diff(ids) < 0                    # descending step inside one slice
        starts = off[1:-1]
        desc[starts[(starts > 0) & (starts < len(ids))] - 1] = False
        if desc.any():
            raise HoleError("filter ids must be ascending within each query's slice")
        if len(ids) == 0:                          # no ids: nothing to filter (and no device pointer)
            return None, None
        return (torch.as_tensor(off).to(self.device).contiguous(),
                torch.as_tensor(ids.astype(np.int32)).to(self.device).contiguous())

    def rank_prepare(self, ent_begin, ent_end, precision=HOLE_RANK_BF16):
        """Pack the candidate operand of [ent_begin, ent_end) once; later rank() calls on the same table /
        range reuse it (until a training call on this engine or rank_invalidate())."""
        check(self.lib.hole_rank_prepare(self._ctx, _ptr(self.table), int(ent_begin), int(ent_end), int(precision),
                                         _stream()))

    def rank_invalidate(self):
        check(self.lib.hole_rank_invalidate(self._ctx))

    def rank_ex(self, queries_i32, side, ent_begin, ent_end, query_table=None, filter_off=None, filter_ids=None,
                precision=HOLE_RANK_BF16, true_score=None, compute_true=True, raw_before=None, filt_before=None):
        """hole_rank_ex on device tensors as they are (no conversions): queries int32 [Q,3]; query_table = the
        table the queries' other-entity / relation rows are read from (None: self.table); raw_before /
        filt_before None = true scores only."""
        check(self.lib.hole_rank_ex(self._ctx, _ptr(self.table), int(ent_begin), int(ent_end), _ptr(query_table),
                                    _ptr(queries_i32), queries_i32.shape[0], int(side), int(precision),
                                    _ptr(filter_off), _ptr(filter_ids), _ptr(true_score), 1 if compute_true else 0,
                                    _ptr(raw_before), _ptr(filt_before), _stream()))

    def rank_debug_operands(self):
        """(candidate operand [n_pad, K], query operand [q_pad, K]) of the last rank() call as
        bf16 CUDA tensors -- test hook."""
        n, q, k = C.c_int64(0), C.c_int64(0), C.c_int(0)
        check(self.lib.hole_rank_debug_operands(self._ctx, None, None, C.byref(n), C.byref(q),
                                                C.byref(k), _stream()))
        cand = torch.empty((n.value, k.value), dtype=torch.bfloat16, device=self.device)
        qp = torch.empty((q.value, k.value), dtype=torch.bfloat16, device=self.device)
        check(self.lib.hole_rank_debug_operands(self._ctx, _ptr(cand), _ptr(qp), C.byref(n),
                                                C.byref(q), C.byref(k), _stream()))
        return cand, qp

    def profile(self, on):
        """Record CUDA events around K1/K3 of every following step (bench.py roofline)."""
        check(self.lib.hole_profile_enable(self._ctx, 1 if on else 0))

    def profile_read(self):
        """-> (k1_ms_total, k3_ms_total, n_steps) since profile(True)."""
        a, b, n = C.c_double(0), C.c_double(0), C.c_int64(0)
        check(self.lib.hole_profile_read(self._ctx, C.byref(a), C.byref(b), C.byref(n)))
        return a.value, b.value, n.value

    def launch_count(self):
        return int(self.lib.hole_launch_count())

    def reset_launch_count(self):
        self.lib.hole_launch_count_reset()
