"""Multi-GPU HolE: entity table row-sharded over the ranks of one node (SURVEY.md section 8e).

One process per GPU (torch.distributed for rendezvous; gloo in the CPU tests).

Training is batch-synchronous and gives the same result as one GPU on the concatenated batch up to
fp32 summation order: every rank corrupts its slice of the global batch (Philox keyed on the
GLOBAL triple index, so the draw does not depend on the number of ranks), the rows a rank's
triples touch come from their owners, the rank runs the step kernels on them, and every row's
change travels back to its owner, who adds the changes in rank order (deterministic).  Relation
rows are replicated and take every rank's change in the same rank order.

Two trainers implement this:
  * P2PRowShardedTrainer (GPUs with peer access; the default) -- one library call per step
    (hole_shard_step): the training kernel gathers rows straight from the owners' shards over
    NVLink and stores the row deltas into the owners' staging buffers; no NCCL, no host
    synchronisation inside a step (include/hole_b200.h, csrc/hole_shard.cuh);
  * RowShardedTrainer -- generic all-to-all version (NCCL or gloo) with a pluggable local
    backend, which is what the CPU tests drive against the oracle.
Ranking: candidates are sharded by row block; the true candidate's score comes from its owner
(all-reduce of a zero-initialised vector), the int32 counts are all-reduced.
"""
import json
import os
import sys
import time

import numpy as np

import torch


TIMING = None      # set to a dict to collect a per-section breakdown (tools/sharded_breakdown.py)
EVENTS = None      # set to a list to collect (name, start, end) CUDA events without synchronising


class _Section:
    """Section timer: synchronising wall-clock when sharded.TIMING is a dict, stream events
    (no synchronisation, the GPU timeline as it runs) when sharded.EVENTS is a list."""

    def __init__(self, name):
        self.name = name

    def __enter__(self):
        if TIMING is not None:
            torch.cuda.synchronize()
            self.t0 = time.perf_counter()
        elif EVENTS is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e0.record()

    def __exit__(self, *a):
        if TIMING is not None:
            torch.cuda.synchronize()
            TIMING[self.name] = TIMING.get(self.name, 0.0) + (time.perf_counter() - self.t0) * 1e3
        elif EVENTS is not None:
            e1 = torch.cuda.Event(enable_timing=True)
            e1.record()
            EVENTS.append((self.name, self.e0, e1))


def row_partition(n_entities, world):
    """Contiguous blocks of entity rows; returns rows_per_rank."""
    return (n_entities + world - 1) // world


class CudaBackend:
    """libhole_b200 on this rank's GPU.  The engine's table is the step table W."""

    def __init__(self, n_relations, dim, max_batch, device_index, type_of=None, csr_off=None, csr_ids=None):
        from .engine import HoleEngine
        self.R = n_relations
        self.eng = HoleEngine(n_relations + 3 * max_batch, dim, device_index)
        self.eng.set_relation_count(n_relations)
        self.width = self.eng.row_stride
        self.dim = dim
        self.device = self.eng.device
        self.max_batch = int(max_batch)
        self._W = self._D = None
        if type_of is not None:
            self.eng.set_types(type_of, csr_off, csr_ids)

    @property
    def W(self):
        """Step table [relations | fetched rows] of the generic trainer (allocated on first use)."""
        if self._W is None:
            self._W = torch.zeros((self.R + 3 * self.max_batch, self.width), dtype=torch.float32, device=self.device)
            self.eng.table = self._W
        return self._W

    @property
    def D(self):
        """Row deltas of one step (delta-mode kernels) of the generic trainer."""
        if self._D is None:
            self._D = torch.zeros_like(self.W)
        return self._D

    def pad_rows(self, E):
        """checkpoint layout [n, dim] -> device layout [n, width]"""
        E = torch.as_tensor(E, dtype=torch.float32, device=self.device)
        H, Hp = self.dim // 2, self.width // 2
        out = torch.zeros((E.shape[0], self.width), dtype=torch.float32, device=self.device)
        out[:, :H] = E[:, :H]
        out[:, Hp:Hp + H] = E[:, H:]
        return out

    def unpad_rows(self, P):
        H, Hp = self.dim // 2, self.width // 2
        return torch.cat([P[:, :H], P[:, Hp:Hp + H]], dim=1)

    def corrupt(self, triples, seed, step, index_base):
        side, neg = self.eng.corrupt_batch(triples, seed, step, index_base)
        return side, neg.long()

    def step(self, n_rows, pos, neg, side, margin, lr):
        self.W                                   # the engine's table is the step table
        return self.eng.train_step(pos.to(torch.int32), neg.to(torch.int32), side, margin, lr)

    # fast path: plan on a side stream, deltas written by the kernels, owner-side row adds
    def plan(self, pos_i32, neg_i32):
        self.eng.train_step_plan(pos_i32, neg_i32)

    def step_delta(self, n_rows, pos_i32, neg_i32, side, margin, lr):
        self.W
        self.D[:n_rows].zero_()
        return self.eng.train_step_delta(pos_i32, neg_i32, side, margin, lr, self.D)

    def add_rows(self, table, ids, id_offset, rows):
        self.eng.add_rows(table, ids.contiguous(), id_offset, rows.contiguous())

    def reserve_step_rows(self, max_batch):
        """Room for R + 3 * max_batch step-table rows in the engine's context (a row-sharded log-loss step with k
        negatives lists up to (2 + k) B rows): replaces the engine by a larger one if it is smaller.  Call before
        anything is bound to the engine."""
        if self.R + 3 * int(max_batch) <= self.eng.n_rows:
            return self
        from .engine import HoleEngine
        old = self.eng
        eng = HoleEngine(self.R + 3 * int(max_batch), self.dim, self.device.index or 0)
        eng.set_relation_count(self.R)
        eng.type_of, eng.csr_off, eng.csr_ids = old.type_of, old.csr_off, old.csr_ids
        old.close()
        self.eng = eng
        return self


class RowShardedTrainer:
    def __init__(self, n_relations, n_entities, dim, backend, dist=None, max_batch=None):
        self.R, self.n_ent, self.dim = int(n_relations), int(n_entities), int(dim)
        self.dist = dist
        self.my_rank = dist.get_rank() if dist is not None else 0
        self.world = dist.get_world_size() if dist is not None else 1
        self.rows_per = row_partition(self.n_ent, self.world)
        self.begin = self.R + self.my_rank * self.rows_per                   # first global row I own
        self.end = min(self.R + self.n_ent, self.begin + self.rows_per)
        self.be = backend
        self.shard = None          # [R + n_mine, width]: replicated relations, then my block

    # ------------------------------------------------------------------ table
    def load_embeddings(self, E):
        """E: full [N, dim] table (checkpoint layout) available on every rank; keeps my part."""
        E = torch.as_tensor(E)
        mine = torch.cat([E[: self.R], E[self.begin:self.end]], dim=0)
        self.shard = self.be.pad_rows(mine)
        return self

    def set_optimizer(self, optimizer, initial_accumulator=0.1):
        """This all-to-all trainer trains with SGD only; AdaGrad runs on P2PRowShardedTrainer."""
        if optimizer == "sgd":
            return self
        from ._lib import HoleError
        raise HoleError(f"{type(self).__name__} (the all-to-all row-sharded trainer) trains with 'sgd' only; "
                        f"optimizer {optimizer!r} on several GPUs needs P2PRowShardedTrainer (NVLink peer memory)")

    def train_step_logloss(self, pos_local, seed, step, lr, l2, negative_ratio):
        """This all-to-all trainer has no --log_loss step; it runs on P2PRowShardedTrainer."""
        from ._lib import HoleError
        raise HoleError(f"{type(self).__name__} (the all-to-all row-sharded trainer) has no log-loss step; "
                        f"--log_loss on several GPUs needs P2PRowShardedTrainer (NVLink peer memory)")

    def gather_embeddings(self):
        """Full [N, dim] table on every rank (tests / checkpointing)."""
        return self._gather(self.shard)

    def _gather(self, P):
        """Full [N, dim] array on every rank from every rank's [relations | block] rows P (device layout)."""
        mine = self.be.unpad_rows(P[self.R:]).contiguous()
        if self.world == 1:
            ents = mine
        else:
            pad = torch.zeros((self.rows_per - mine.shape[0], mine.shape[1]), dtype=mine.dtype, device=mine.device)
            buf = torch.cat([mine, pad], dim=0)
            out = [torch.empty_like(buf) for _ in range(self.world)]
            self.dist.all_gather(out, buf)
            ents = torch.cat(out, dim=0)[: self.n_ent]
        return torch.cat([self.be.unpad_rows(P[: self.R]), ents], dim=0)

    # ------------------------------------------------------------------ exchange helpers
    def _a2a(self, send, send_counts, recv_counts, out=None):
        if self.world == 1:
            if out is not None:
                out.copy_(send)
                return out
            return send
        shape = (int(sum(recv_counts)),) + tuple(send.shape[1:])
        recv = out if out is not None else torch.empty(shape, dtype=send.dtype, device=send.device)
        self.dist.all_to_all_single(recv, send.contiguous(), output_split_sizes=list(recv_counts),
                                    input_split_sizes=list(send_counts))
        return recv

    def _route(self, uniq):
        """uniq: sorted unique global entity rows I need.  -> (send_counts, recv_counts) lists."""
        dev = uniq.device
        bounds = self.R + self.rows_per * torch.arange(1, self.world + 1, device=dev)
        cut = torch.searchsorted(uniq, bounds)
        send = torch.diff(cut, prepend=torch.zeros(1, dtype=cut.dtype, device=dev))
        if self.world == 1:
            sc = [int(send[0])]
            return sc, sc
        recv = torch.empty_like(send)
        self.dist.all_to_all_single(recv, send)
        both = torch.stack([send, recv]).tolist()          # one host synchronisation
        return [int(x) for x in both[0]], [int(x) for x in both[1]]

    # ------------------------------------------------------------------ training
    def train_step(self, pos_local, seed, step, margin, lr, next_pos=None):
        """pos_local: this rank's [B,3] slice (global row ids) of the global batch of
        world*B triples.  Returns the per-triple hinge loss of the slice.  (next_pos is used by
        the peer-memory trainer to work one step ahead; ignored here.)"""
        dev = self.shard.device
        pos = torch.as_tensor(pos_local).to(dev).long()
        B, R = pos.shape[0], self.R
        with _Section("corrupt"):
            side, neg = self.be.corrupt(pos.to(torch.int32), seed, step, self.my_rank * B)
            neg = neg.to(dev)
        with _Section("unique"):
            ents = torch.cat([pos[:, 0], pos[:, 1], neg]).to(torch.int32)    # 32-bit keys sort faster
            uniq, inv = torch.unique(ents, return_inverse=True)
            uniq = uniq.long()
            U = uniq.shape[0]
        with _Section("route (counts, host sync)"):
            send_counts, recv_counts = self._route(uniq)
        with _Section("a2a ids"):
            ids_in = self._a2a(uniq, send_counts, recv_counts)              # rows others want from me
        fast = hasattr(self.be, "step_delta")
        if fast:
            with _Section("plan (side stream)"):
                pos_w = torch.stack([R + inv[:B], R + inv[B:2 * B], pos[:, 2]], dim=1).to(torch.int32)
                neg_w = (R + inv[2 * B:]).to(torch.int32)
                self.be.plan(pos_w, neg_w)        # overlaps the row exchange below
        with _Section("gather rows"):
            rows_out = self.shard.index_select(0, ids_in - self.begin + R)
        W = self.be.W
        if fast:
            with _Section("a2a rows"):
                self._a2a(rows_out, recv_counts, send_counts, out=W[R:R + U])   # lands in the step table
                W[:R].copy_(self.shard[:R])
            with _Section("local step (K1+K3, delta mode)"):
                loss = self.be.step_delta(R + U, pos_w, neg_w, side, margin, lr)
                delta = self.be.D
        else:
            with _Section("a2a rows"):
                rows_in = self._a2a(rows_out, recv_counts, send_counts)         # in `uniq` order
            with _Section("assemble W, W0"):
                W[:R].copy_(self.shard[:R])
                W[R:R + U].copy_(rows_in)
                W0 = W[: R + U].clone()
                pos_w = torch.stack([R + inv[:B], R + inv[B:2 * B], pos[:, 2]], dim=1)
                neg_w = R + inv[2 * B:]
            with _Section("local step (plan+K1+K3)"):
                loss = self.be.step(R + U, pos_w, neg_w, side, margin, lr)
            with _Section("delta"):
                delta = W[: R + U] - W0
        with _Section("allreduce relations"):
            d_rel = delta[:R].contiguous()
            if self.world > 1:
                self.dist.all_reduce(d_rel)
            self.shard[:R] += d_rel
        with _Section("a2a deltas"):
            d_in = self._a2a(delta[R:R + U], send_counts, recv_counts)      # grouped by source rank
        with _Section("apply deltas"):
            off = 0
            for k in range(self.world):                                     # rank order: deterministic
                n_k = recv_counts[k]
                if n_k:
                    if fast:
                        self.be.add_rows(self.shard, ids_in[off:off + n_k], R - self.begin, d_in[off:off + n_k])
                    else:
                        self.shard.index_add_(0, ids_in[off:off + n_k] - self.begin + R, d_in[off:off + n_k])
                off += n_k
        return loss

    def train_steps(self, triples_i32, batch_size, seed, first_step, margin, lrs):
        """n_steps consecutive train_step calls on device-resident slices [n_steps*B, 3] (lrs: at least n_steps
        rates).  Returns this rank's per-step loss sums (device)."""
        n_steps = triples_i32.shape[0] // batch_size
        sums = torch.empty(n_steps, dtype=torch.float32, device=triples_i32.device)
        for k in range(n_steps):
            sums[k] = self.train_step(triples_i32[k * batch_size:(k + 1) * batch_size], seed, first_step + k, margin,
                                      lrs[k]).sum()
        return sums

    def check_barriers(self):
        """Nothing to check: the all-to-all trainer has no step barriers of its own."""

    def close(self):
        """Releases the ranking context of rank()."""
        if getattr(self, "_rank_eng", None) is not None:
            self._rank_eng.close()
            self._rank_eng = None

    # ------------------------------------------------------------------ scoring
    def score(self, triples):
        """sigma (hole_score) of this rank's triples [n,3] (global row ids) on the sharded table.  Collective: every
        rank calls it with its own triples (possibly none).  The rows of the heads and tails come from their owners
        by all-to-all into a side table [relations | fetched rows], as in rank()."""
        dev = self.shard.device
        t = torch.as_tensor(triples).to(dev).long()
        n, R = t.shape[0], self.R
        uniq, inv = torch.unique(t[:, :2].reshape(-1), return_inverse=True)
        send_counts, recv_counts = self._route(uniq)
        ids_in = self._a2a(uniq, send_counts, recv_counts)
        rows_in = self._a2a(self.shard.index_select(0, ids_in - self.begin + R), recv_counts, send_counts)
        side = torch.cat([self.shard[:R], rows_in], dim=0)
        return self.be.eng.evaluate_triples(_side_triples(t, inv, R), table=side)

    # ------------------------------------------------------------------ ranking
    def rank(self, queries, side, filter_off=None, filter_ids=None, precision=None):
        """All-entity ranking of (replicated) queries [Q,3] with candidates sharded by row block.
        Returns (raw_before, filt_before) int32[Q], identical on every rank.

        The candidate operand is my block of the shard as it lies (packed once per call); the rows of the
        queries' other entities come from their owners into a small side table [relations | fetched rows].
        Phase 1 computes only the true candidates' scores (each by its owner), phase 2 counts."""
        from .engine import HOLE_RANK_BF16, HOLE_SIDE_HEAD, HOLE_SIDE_TAIL, HoleEngine, HoleError
        if side not in (HOLE_SIDE_TAIL, HOLE_SIDE_HEAD):
            raise HoleError(f"sharded ranking supports the tail and head sides only, got side {side}; the relation "
                            "rows are replicated, so rank relations on one GPU: HoleEngine.rank(..., "
                            "HOLE_SIDE_RELATION, 0, n_relations) on a table from gather_embeddings()")
        precision = HOLE_RANK_BF16 if precision is None else precision
        dev = self.shard.device
        q = torch.as_tensor(queries).to(dev).long()
        Q, R = q.shape[0], self.R
        other_col, true_col = (0, 1) if side == HOLE_SIDE_TAIL else (1, 0)
        uniq, inv = torch.unique(q[:, other_col], return_inverse=True)
        send_counts, recv_counts = self._route(uniq)
        ids_in = self._a2a(uniq, send_counts, recv_counts)
        rows_in = self._a2a(self.shard.index_select(0, ids_in - self.begin + R), recv_counts, send_counts)
        n_mine = self.end - self.begin                                  # (the last shard may carry padding rows)
        qtab = torch.cat([self.shard[:R], rows_in], dim=0)              # [relations | fetched rows]: small
        tr = q[:, true_col]
        # true candidate: shard-local row if mine, else below / above my candidate range
        tr_loc = torch.where(tr < self.begin, torch.zeros_like(tr) - 1 + R,       # < ent_begin
                             torch.where(tr >= self.end, torch.full_like(tr, R + n_mine + 1),
                                         tr - self.begin + R))
        ql = torch.empty((Q, 3), dtype=torch.int32, device=dev)
        ql[:, other_col] = (R + inv).to(torch.int32)                    # row of the side table
        ql[:, true_col] = tr_loc.to(torch.int32)                        # index into my candidate range only
        ql[:, 2] = q[:, 2].to(torch.int32)
        fo = fi = None
        if filter_off is not None:
            fo = torch.as_tensor(filter_off).to(dev).to(torch.int64).contiguous()
            fi = (torch.as_tensor(filter_ids).to(dev).long() - self.begin + R).to(torch.int32).contiguous()
        # a ranking context over my shard
        eng = getattr(self, "_rank_eng", None)
        if eng is None or eng.n_rows != self.shard.shape[0]:
            if eng is not None:
                eng.close()
            eng = self._rank_eng = HoleEngine(int(self.shard.shape[0]), self.dim, dev.index or 0)
        eng.table = self.shard
        try:
            eng.rank_invalidate()                                       # the shard has been trained since
            eng.rank_prepare(R, R + n_mine, precision)
            ts = torch.zeros(Q, dtype=torch.float32, device=dev)
            eng.rank_ex(ql, side, R, R + n_mine, query_table=qtab, precision=precision, true_score=ts,
                        compute_true=True)
            if self.world > 1:
                self.dist.all_reduce(ts)          # exactly one owner wrote each entry, others hold 0
            cnt = torch.zeros((2, Q), dtype=torch.int32, device=dev)
            eng.rank_ex(ql, side, R, R + n_mine, query_table=qtab, filter_off=fo, filter_ids=fi,
                        precision=precision, true_score=ts, compute_true=False, raw_before=cnt[0],
                        filt_before=cnt[1])
            if self.world > 1:
                self.dist.all_reduce(cnt)
        finally:
            eng.table = None
        return cnt[0], cnt[1]


def _side_triples(t, inv, n_relations):
    """triples t [n,3] re-indexed to a side table [relations | fetched rows] (inv: torch.unique's inverse of
    t[:, :2].reshape(-1))."""
    q = torch.empty((t.shape[0], 3), dtype=torch.int32, device=t.device)
    q[:, :2] = (n_relations + inv.view(-1, 2)).to(torch.int32)
    q[:, 2] = t[:, 2].to(torch.int32)
    return q


def score_on_shards(eng, peer_shards, me, n_relations, rows_per, triples):
    """sigma (hole_score) of triples [n,3] (global row ids) on a row-sharded table read in place.  peer_shards[k] is
    rank k's shard [relations | entity rows n_relations + k*rows_per, ...], possibly another GPU's memory mapped into
    eng's device; me: the caller's rank, whose replica of the relation rows is read.  The relation rows and the rows of
    the heads and tails are copied (hole_gather_rows) into a side table [relations | fetched rows], the triples
    re-indexed to it and scored there, so sigma is bit for bit that of hole_score on the whole table.  eng: any context
    of the table's dim on this device.  The caller orders the reads after the owners' last update and before their
    next one (P2PRowShardedTrainer.score)."""
    dev = eng.device
    t = torch.as_tensor(triples).to(dev).long()
    n, R, world = t.shape[0], int(n_relations), len(peer_shards)
    if n == 0:
        return torch.empty(0, dtype=torch.float32, device=dev)
    uniq, inv = torch.unique(t[:, :2].reshape(-1), return_inverse=True)       # ascending: one run per owner
    bounds = R + rows_per * torch.arange(1, world + 1, device=dev)
    cuts = [0] + torch.searchsorted(uniq, bounds).tolist()
    side = torch.zeros((R + uniq.shape[0], eng.row_stride), dtype=torch.float32, device=dev)
    if R:          # the relation replicas are bit-identical on every rank: read the local one
        eng.gather_rows(peer_shards[me], torch.arange(R, device=dev), 0, side[:R])
    for k in range(world):
        a, b = cuts[k], cuts[k + 1]
        if b > a:      # global row g lies at row g - k*rows_per of rank k's shard
            eng.gather_rows(peer_shards[k], uniq[a:b].contiguous(), -k * rows_per, side[R + a:R + b])
    return eng.evaluate_triples(_side_triples(t, inv, R), table=side)


class PeerMemoryUnavailable(RuntimeError):
    """The GPUs of this job cannot map each other's memory (no P2P / CUDA IPC)."""


def make_trainer(n_relations, n_entities, dim, backend, dist, log=None):
    """P2PRowShardedTrainer when every rank can map every other rank's buffers, else (all ranks
    together) the NCCL all-to-all RowShardedTrainer.  HOLE_SHARDED_NCCL=1 forces the latter."""
    if os.environ.get("HOLE_SHARDED_NCCL") != "1" and hasattr(backend, "eng"):
        try:
            return P2PRowShardedTrainer(n_relations, n_entities, dim, backend, dist)
        except PeerMemoryUnavailable as e:
            if log:
                log(f"peer memory unavailable, using NCCL all-to-alls: {e}")
    return RowShardedTrainer(n_relations, n_entities, dim, backend, dist)


class P2PRowShardedTrainer(RowShardedTrainer):
    """Row-sharded training with the exchange fused into the training kernel over NVLink peer
    memory: one library call per step (hole_shard_step, csrc/hole_shard.cuh).  Every rank maps
    (CUDA IPC) every other rank's shard, delta staging, relation staging, request inbox and flags.

      side stream, one step ahead (pass `next_pos`):  Philox corruption -> request routing -> update plan
      compute stream:  post request lists -> K1 gathers rows from the owners' shards and stores row
                       deltas into the owners' staging buffers -> K3 -> relation deltas + "delivered"
                       flag -> owner adds the staged deltas in rank order + "current" flag

    No NCCL call and no host synchronisation inside a step."""

    def __init__(self, n_relations, n_entities, dim, backend, dist, timeout_s=0.0, check_every=256,
                 negative_ratio=1):
        """negative_ratio: the largest k of the train_step_logloss calls to come.  A log-loss step lists up to
        (2 + k) B rows of B = backend.max_batch triples, so the staging buffers and inboxes hold
        3 * max(B, ceil((2 + k) B / 3)) rows."""
        super().__init__(n_relations, n_entities, dim, backend, dist)
        from torch.multiprocessing.reductions import reduce_tensor
        dev, G, R = backend.device, self.world, self.R
        if backend.eng.type_of is None:
            raise ValueError("the backend needs the type tables (type_of, csr_off, csr_ids) for the corruption")
        B = backend.max_batch
        self.max_batch = max(B, -(-(2 + int(negative_ratio)) * B // 3))
        eng = backend.reserve_step_rows(self.max_batch).eng
        self.cap = 3 * self.max_batch
        width = backend.width
        self.shard = torch.zeros((R + self.rows_per, width), dtype=torch.float32, device=dev)
        self.stage = torch.zeros((G, self.cap, width), dtype=torch.float32, device=dev)
        self.relstage = torch.zeros((G, max(R, 1), width), dtype=torch.float32, device=dev)
        self.inbox = torch.zeros((2, G, self.cap), dtype=torch.int32, device=dev)
        self.meta = torch.zeros((2, G, 2), dtype=torch.int32, device=dev)
        self.flags = torch.zeros((2, G), dtype=torch.int32, device=dev)
        self.barrier_err = torch.zeros(1, dtype=torch.int32, device=dev)
        self.accum = None          # AdaGrad accumulator shard (set_optimizer), the layout of self.shard
        mine = [self.shard, self.stage, self.relstage, self.inbox, self.meta, self.flags]
        if G == 1:
            peers = [mine]
        else:
            everyone = [None] * G
            dist.all_gather_object(everyone, ([reduce_tensor(t) for t in mine], dev.index))
            peers, failure = [], None
            for k, (handles, dev_k) in enumerate(everyone):
                if k == self.my_rank:
                    peers.append(mine)
                    continue
                # Open the peer's allocation in MY device's address space (argument 6 of torch's
                # rebuild is the device the IPC handle is opened on): the tensor then reads as
                # local to torch while its pages live on GPU k -- kernels launched on my device
                # reach it over NVLink.
                try:
                    eng.enable_peer_access(dev_k)
                    peers.append([fn(*(list(a[:6]) + [dev.index] + list(a[7:]))) for fn, a in handles])
                except Exception as e:                       # no P2P / IPC between these two GPUs
                    failure = f"rank {self.my_rank} cannot map rank {k}'s buffers: {e}"
                    break
            # every rank must reach the same verdict, or the first flag wait would spin
            verdicts = [None] * G
            dist.all_gather_object(verdicts, failure)
            bad = [v for v in verdicts if v]
            if bad:
                raise PeerMemoryUnavailable("; ".join(bad))
        self._bind(peers, timeout_s)
        self.check_every = int(check_every)
        self._since_check = 0
        if G > 1:
            torch.cuda.synchronize()
            dist.barrier()

    def _bind(self, peers, timeout_s=0.0):
        self._peers = peers                                         # keeps the mappings alive
        pa = self.be.eng.peer_array
        self.be.eng.shard_init(self.world, self.my_rank, self.R, self.n_ent, self.rows_per, self.max_batch,
                               self.shard, *[pa([p[i] for p in peers]) for i in range(6)], self.barrier_err,
                               timeout_s)

    def close(self):
        """Collective: drop the mappings of the peers' buffers on every rank BEFORE anybody frees the
        memory behind them (CUDA IPC: the exporter must outlive every importer's mapping)."""
        if getattr(self, "_peers", None) is None:
            return
        torch.cuda.synchronize()
        self._peers = None
        super().close()
        if self.world > 1:
            self.dist.barrier()
        self.shard = self.stage = self.relstage = self.inbox = self.meta = self.flags = None
        self.accum = None

    def set_optimizer(self, optimizer, initial_accumulator=0.1):
        """"sgd" (the default) or "adagrad" (TF's AdagradOptimizer(lr, initial_accumulator_value), applied by each
        row's owner to the gradient summed over every rank that uses the row; hole_shard_set_optimizer).
        "adagrad" allocates this rank's accumulator shard [relations | my block] and fills all of it, pad columns
        and the unused trailing rows included, with initial_accumulator (> 0); "sgd" drops it.  Every rank must
        make the same call before the same step."""
        from ._lib import HoleError
        eng = self.be.eng
        if optimizer == "sgd":
            eng.shard_set_optimizer("sgd", None)
            self.accum = None
            return self
        if optimizer != "adagrad":
            raise HoleError(f"unknown optimizer {optimizer!r}: 'sgd' or 'adagrad'")
        if not float(initial_accumulator) > 0.0:
            raise HoleError(f"initial_accumulator must be > 0, got {initial_accumulator}")
        accum = torch.full_like(self.shard, float(initial_accumulator))
        eng.shard_set_optimizer("adagrad", accum)
        self.accum, self.initial_accumulator = accum, float(initial_accumulator)
        return self

    def load_accumulator(self, A):
        """A: the full [N, dim] AdaGrad accumulator (checkpoint layout, the slot `embeddings/Adagrad`), every element
        > 0, available on every rank; keeps this rank's part.  The pad columns and unused rows keep the initial
        value."""
        from ._lib import HoleError
        if getattr(self, "accum", None) is None:
            raise HoleError("the optimizer is not adagrad: there is no accumulator")
        A = torch.as_tensor(A, dtype=torch.float32)
        assert A.shape == (self.R + self.n_ent, self.dim), A.shape
        mine = torch.cat([A[: self.R], A[self.begin:self.end]], dim=0).to(self.accum.device)
        if not bool((mine > 0).all()):
            raise HoleError("every accumulator element must be > 0")
        H, Hp = self.dim // 2, self.be.width // 2
        self.accum.fill_(self.initial_accumulator)
        self.accum[: mine.shape[0], :H] = mine[:, :H]
        self.accum[: mine.shape[0], Hp:Hp + H] = mine[:, H:]
        torch.cuda.current_stream().synchronize()   # A may be freed by the caller
        return self

    def gather_accumulator(self):
        """Full [N, dim] AdaGrad accumulator on every rank (checkpoint layout: the `embeddings/Adagrad` slot of
        tf_bundle).  Collective, like gather_embeddings()."""
        from ._lib import HoleError
        if getattr(self, "accum", None) is None:
            raise HoleError("the optimizer is not adagrad: there is no accumulator")
        self.check_barriers()
        return self._gather(self.accum)

    def load_embeddings(self, E):
        E = torch.as_tensor(E)
        mine = torch.cat([E[: self.R], E[self.begin:self.end]], dim=0)
        self.shard.zero_()
        self.shard[: mine.shape[0]].copy_(self.be.pad_rows(mine))
        return self.shards_ready()

    def shards_ready(self):
        """Collective: call after writing self.shard directly.  The peers' training kernels READ this
        shard over NVLink, so nobody may start a step before every rank's shard is in place."""
        torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        return self

    def check_barriers(self):
        """Raises if a peer ever failed to reach a step barrier (host synchronisation)."""
        self._since_check = 0
        if self.be.eng.shard_poll():
            raise RuntimeError("a peer did not reach a step barrier in time; the sharded tables are inconsistent")

    def gather_embeddings(self):
        self.check_barriers()
        return super().gather_embeddings()

    def rank(self, *a, **kw):
        self.check_barriers()
        return super().rank(*a, **kw)

    def score(self, triples):
        """sigma of this rank's triples [n,3] on the sharded table, read in place from the owners' shards over peer
        memory (score_on_shards).  Collective.  Two conditions keep the reads consistent:
          1. before the first read, torch.cuda.synchronize(), dist.barrier() and check_barriers(): every owner's
             apply of the last step has completed, on every rank, and no barrier timed out;
          2. the gathers are enqueued on this rank's current stream, ahead of its next hole_shard_steps call.  An
             owner's next apply waits for every rank's "delivered" flag of that step, which a rank raises only after
             its K1 / K3 of the step, so after these gathers: no row is overwritten under a reader."""
        torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.check_barriers()
        return score_on_shards(self.be.eng, [p[0] for p in self._peers], self.my_rank, self.R, self.rows_per, triples)

    def _as_slice(self, pos):
        pos = torch.as_tensor(pos)
        if pos.device != self.shard.device or pos.dtype != torch.int32 or not pos.is_contiguous():
            pos = pos.to(self.shard.device, non_blocking=True).to(torch.int32).contiguous()
        return pos

    def train_step(self, pos_local, seed, step, margin, lr, next_pos=None):
        """pos_local: this rank's [B,3] slice of the global batch (device int32 tensors are used as they
        are and must stay alive until the step has run).  next_pos: the slice of step + 1, if known --
        its corruption, routing and plan are then built on the side stream while this step runs."""
        eng = self.be.eng
        pos = self._as_slice(pos_local)
        keep = [pos]
        if getattr(self, "_prepared_key", None) != (pos.data_ptr(), pos.shape[0], int(seed), int(step)):
            eng.shard_prepare(pos, seed, step)              # nothing was built ahead for this step
        self._prepared_key = None
        if next_pos is not None:                            # enqueue before the step, so that it overlaps it
            nxt = self._as_slice(next_pos)
            keep.append(nxt)
            eng.shard_prepare(nxt, seed, step + 1)
            self._prepared_key = (nxt.data_ptr(), nxt.shape[0], int(seed), int(step) + 1)
        loss = eng.shard_step(pos, seed, step, margin, lr)
        self._keep = keep                                   # the side stream may still read them
        self._since_check += 1
        if self.check_every and self._since_check >= self.check_every:
            self.check_barriers()
        return loss

    def train_step_logloss(self, pos_local, seed, step, lr, l2, negative_ratio):
        """One --log_loss step (holE.py:194-196, 206-220, 296; hole_shard_step_logloss) of the global batch: the
        result of HoleEngine.train_step_logloss on the concatenated slices.  pos_local: this rank's [B,3] slice;
        negative_ratio <= the trainer's.  Returns (loss rows of my slice [(1+k), B] device, without the L2 term;
        my l2 part, a device scalar: half the sum of squares of the old rows I own, the relation rows counted on
        rank 0 -- summed over the ranks, the global l2_loss; zero when l2 == 0).  A hinge step prepared ahead with
        next_pos stays prepared."""
        pos = self._as_slice(pos_local)
        loss, l2_part = self.be.eng.shard_step_logloss(pos, seed, step, lr, l2, negative_ratio)
        self._keep_logloss = pos                            # read by the step's kernels
        self._since_check += 1
        if self.check_every and self._since_check >= self.check_every:
            self.check_barriers()
        return loss, l2_part

    def train_steps(self, triples_i32, batch_size, seed, first_step, margin, lrs):
        """n_steps consecutive steps on device-resident slices [n_steps*B, 3] without returning to the
        host (hole_shard_steps).  Returns this rank's per-step loss sums (device)."""
        sums = self.be.eng.shard_steps(triples_i32, batch_size, seed, first_step, margin, lrs)
        self._since_check += triples_i32.shape[0] // batch_size
        return sums

    def train_steps_host(self, triples_host, batch_size, seed, first_step, margin, lrs):
        """Same from pinned host triples; returns numpy loss sums (blocks)."""
        out = self.be.eng.shard_steps_host(triples_host, batch_size, seed, first_step, margin, lrs)
        self.check_barriers()
        return out


# --------------------------------------------------------------------------------------
# parity of the multi-GPU product path (tools/multi_gpu_check.py, tests/test_gpu_multi.py, bench.py)
# --------------------------------------------------------------------------------------
def parity_case(dist, rank, world, local, dim, Bl, steps, n_ent, seed, chunked, log=None):
    """Row-sharded training over the real peers + sharded ranking against a single-GPU engine run on
    rank 0 over the same global batches.  Returns (ok on every rank, result dict on rank 0)."""
    from . import data as D
    from .engine import HoleEngine
    kg = D.synthetic_kg(9, n_ent, Bl * world * steps, 5, dim, seed=seed, trained_scale=True, zipf_entities=True)
    off, ids = D.build_type_csr(kg.type_of)
    be = CudaBackend(kg.n_relations, kg.dim, Bl, local, kg.type_of, off, ids)
    tr = make_trainer(kg.n_relations, kg.n_entities, kg.dim, be, dist, log=log).load_embeddings(kg.E)
    mine = torch.from_numpy(kg.triples).view(steps, world, Bl, 3)[:, rank].contiguous().cuda()
    lrs = [0.1 / (1 + 0.01 * s) for s in range(steps)]
    if chunked and isinstance(tr, P2PRowShardedTrainer):
        tr.train_steps(mine.view(-1, 3), Bl, 3, 0, 0.2, lrs)
    else:
        for s in range(steps):
            tr.train_step(mine[s], 3, s, 0.2, lrs[s], next_pos=mine[s + 1] if s + 1 < steps else None)
    full = tr.gather_embeddings()
    q = torch.from_numpy(kg.triples[:1000])
    raw, filt = tr.rank(q, 0)
    res = {"trainer": type(tr).__name__, "world": world, "dim": dim, "batch_per_gpu": Bl, "steps": steps,
           "chunked_call": bool(chunked)}
    ok = True
    if rank == 0:
        e = HoleEngine(kg.n_rows, kg.dim, local).set_embeddings(kg.E).set_types(kg.type_of, off, ids)
        for s in range(steps):
            gb = kg.triples[s * Bl * world:(s + 1) * Bl * world]
            side, neg = e.corrupt_batch(gb, 3, s)
            e.train_step(gb, neg, side, 0.2, lrs[s])
        want = e.embeddings()
        diff = (full - want).abs().amax(dim=1)
        err = float(diff.max())
        bad = torch.nonzero(diff > 2e-6).flatten()
        if len(bad):                      # diagnostics: which rows, whose
            rows_per = row_partition(kg.n_entities, world)
            res["bad_rows"] = int(len(bad))
            res["bad_relation_rows"] = int((bad < kg.n_relations).sum())
            res["bad_rows_by_owner"] = [int(((bad >= kg.n_relations + o * rows_per) &
                                             (bad < kg.n_relations + (o + 1) * rows_per)).sum()) for o in range(world)]
            res["bad_first"] = [int(x) for x in bad[:8]]
        moved = float((want.cpu() - torch.from_numpy(kg.E)).abs().max())
        # ranking on the single-GPU table that equals the gathered sharded table up to ~1e-7
        e2 = HoleEngine(kg.n_rows, kg.dim, local).set_embeddings(full)
        r1, f1, _ = e2.rank(q, 0, kg.n_relations, kg.n_rows)
        same = float((r1 == raw).float().mean())
        res.update({"max_abs_err": err, "moved": moved, "rank_counts_equal": same,
                    "rank_counts_max_diff": int((r1 - raw).abs().max())})
        ok = err <= 2e-6 and moved > 1e-4 and same == 1.0
        res["ok"] = ok
        e.close()
        e2.close()
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.broadcast(flag, 0)
    tr.close()
    be.eng.close()
    return bool(flag.item()), res


# --------------------------------------------------------------------------------------
# bench.py --gpus N (N > 1)
# --------------------------------------------------------------------------------------
#: measured peer-copy bandwidth per direction on this pool's B200s (B200_PROFILING.md; nominal 900 GB/s)
NVLINK_PEAK = 770.0
NVLINK_PEAK_SRC = "measured peer copy, 770 GB/s per direction (B200_PROFILING.md; nominal NVLink 5: 900)"


def _nvlink_bytes_per_dir(B, world, dim_stride):
    """Per GPU and direction, one step: rows gathered from remote owners + deltas received as an owner
    (in), rows served + deltas sent (out): 2 * 3B * (G-1)/G rows of 4*stride bytes (SURVEY 8d, k = 4)."""
    return 2.0 * 3.0 * B * (world - 1) / world * 4.0 * dim_stride


def _timed_device(dist, fn):
    """Device time of fn() in ms, max over ranks; also the host time fn() took to enqueue."""
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    h0 = time.perf_counter()
    fn()
    host_ms = (time.perf_counter() - h0) * 1e3
    e1.record()
    torch.cuda.synchronize()
    dist.barrier()
    t = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()), host_ms


def _timed_wall(dist, fn):
    """Wall-clock ms of a blocking fn(), max over ranks."""
    torch.cuda.synchronize()
    dist.barrier()
    h0 = time.perf_counter()
    out = fn()
    t = torch.tensor([(time.perf_counter() - h0) * 1e3], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()), out


def bench_config4(args, dist, rank, world, local_rank, steps, warmup):
    """BASELINE.json configs[4]: HolE d=512, 20 M entities (41 GB fp32 table), row-sharded; every
    rank trains `--batch` triples per step.  The shards, type tables and triples are generated on
    the device (the table is never materialised on the host)."""
    from . import data as D
    cfg = D.CONFIGS["sharded_d512"]
    R, n_ent, dim, n_types = cfg["n_relations"], cfg["n_entities"], cfg["dim"], cfg["n_types"]
    Bl = args.batch
    rng = np.random.default_rng(cfg["seed"])
    p = np.full(n_types, (1.0 - cfg["dominant_type_frac"]) / (n_types - 1))
    p[0] = cfg["dominant_type_frac"]
    type_of = np.concatenate([np.zeros(R, np.int32), 1 + rng.choice(n_types, size=n_ent, p=p).astype(np.int32)])
    off, ids = D.build_type_csr(type_of)
    be = CudaBackend(R, dim, Bl, local_rank, type_of, off, ids)
    tr = P2PRowShardedTrainer(R, n_ent, dim, be, dist)
    gen = torch.Generator(device=be.device)
    gen.manual_seed(cfg["seed"] + 1)                       # relation replicas identical on every rank
    sd = D.xavier_stddev(R + n_ent, dim)
    tr.shard[:R].normal_(0.0, 1.0, generator=gen).clamp_(-2.0, 2.0).mul_(sd)
    gen.manual_seed(cfg["seed"] + 2 + rank)
    n_mine = tr.end - tr.begin
    tr.shard[R:R + n_mine].normal_(0.0, 1.0, generator=gen).clamp_(-2.0, 2.0).mul_(sd)
    tr.shards_ready()
    n = (steps + warmup) * Bl
    h = torch.randint(R, R + n_ent, (n,), generator=gen, device=be.device, dtype=torch.int32)
    t = torch.randint(R, R + n_ent, (n,), generator=gen, device=be.device, dtype=torch.int32)
    w = 1.0 / torch.arange(1, R + 1, device=be.device, dtype=torch.float64)
    r = torch.multinomial(w / w.sum(), n, replacement=True, generator=gen).to(torch.int32)
    tri = torch.stack([h, t, r], dim=1).contiguous()
    lrs = np.full(steps + warmup, 0.1, np.float32)
    tr.train_steps(tri[: warmup * Bl], Bl, 1, 0, 0.2, lrs[:warmup])
    ms, host_ms = _timed_device(dist, lambda: tr.train_steps(tri[warmup * Bl:], Bl, 1, warmup, 0.2, lrs[warmup:]))
    tr.check_barriers()
    value = steps * Bl * world / (ms * 1e-3)
    nv = _nvlink_bytes_per_dir(Bl, world, be.width) / (ms / steps * 1e-3) / 1e9
    out = {"workload": f"sharded_d512: BASELINE.json configs[4], HolE d=512, {n_ent:,} entities + {R} relations "
                       f"({(R + n_ent) * dim * 4 / 1e9:.1f} GB fp32 table) row-sharded over {world} GPUs, "
                       "uniform entities, Zipf relations, Xavier-scale rows generated on the device",
           "value": value, "unit": "triples/s", "ms_per_step": ms / steps, "batch_per_gpu": Bl, "steps": steps,
           "shard_gb_per_gpu": float(tr.shard.numel() * 4 / 1e9), "host_enqueue_us_per_step": host_ms / steps * 1e3,
           "roofline": {"bound": "nvlink", "achieved": nv, "peak": NVLINK_PEAK, "unit": "GB/s per direction per GPU",
                        "frac": nv / NVLINK_PEAK, "peak_source": NVLINK_PEAK_SRC,
                        "bytes_per_dir_per_step": _nvlink_bytes_per_dir(Bl, world, be.width)}}
    tr.close()
    del tr
    be.eng.close()
    torch.cuda.empty_cache()
    return out


def bench(args, dist, rank, world, local_rank):
    """Weak scaling: every rank trains `--batch` triples per step on the row-sharded BASELINE config 1
    table (value / e2e), then config 4 and the sharded ranking as sub-records.  Device time, max over
    ranks; rank 0 prints the JSON line."""
    import bench as B_
    from . import data as D
    from .engine import HOLE_SIDE_TAIL

    Bl, K, W = args.batch, args.steps, args.warmup
    kg = D.make_config(B_.WORKLOAD, n_triples=(K + W) * Bl * world)
    off, ids = D.build_type_csr(kg.type_of)
    be = CudaBackend(kg.n_relations, kg.dim, Bl, local_rank, kg.type_of, off, ids)
    tr = make_trainer(kg.n_relations, kg.n_entities, kg.dim, be, dist,
                      log=lambda m: print(m, file=sys.stderr) if rank == 0 else None).load_embeddings(kg.E)
    p2p = isinstance(tr, P2PRowShardedTrainer)
    # step s, rank r takes triples [(s*world + r)*Bl, +Bl)
    mine = torch.from_numpy(kg.triples).view(K + W, world, Bl, 3)[:, rank].contiguous()
    dev_tri = mine.cuda()
    host_tri = mine.pin_memory()
    lrs = B_.lr_schedule(5 * (K + W), 0, 30_000_000 // (Bl * world))

    # nvidia-smi's start-up (NVML initialisation) disturbs running GPU work for a few hundred
    # ms: start the clock sampler before the warm-up, not inside the timed region
    sampler = B_.ClockSampler(local_rank, period=0.25)
    if rank == 0 and os.environ.get("HOLE_NO_SAMPLER") != "1":
        sampler.start()
        time.sleep(1.0)
    B_.settle_clocks()

    def run_steps(k0, n, first_step):
        if p2p:
            return tr.train_steps(dev_tri[k0:k0 + n].view(-1, 3), Bl, 1, first_step, B_.MARGIN, lrs[first_step:])
        for s in range(n):
            tr.train_step(dev_tri[k0 + s], 1, first_step + s, B_.MARGIN, float(lrs[first_step + s]),
                          next_pos=dev_tri[k0 + s + 1] if s + 1 < n else None)

    run_steps(0, W, 0)
    be.eng.reset_launch_count()
    ms, host_ms = _timed_device(dist, lambda: run_steps(W, K, W))
    launches = be.eng.launch_count()
    if p2p:
        tr.check_barriers()
    value = K * Bl * world / (ms * 1e-3)

    # the same steps when every rank trains the triples whose HEAD it owns (a head-partitioned triple file):
    # one of the three entity rows of a triple is then local, a third of the NVLink traffic disappears
    head_local = None
    if p2p:
        loc = dev_tri.clone()
        n_mine = tr.end - tr.begin
        loc[:, :, 0] = tr.begin + (loc[:, :, 0] - kg.n_relations) % n_mine
        tr.train_steps(loc[:W].view(-1, 3), Bl, 1, 2 * (K + W), B_.MARGIN, lrs[2 * (K + W):])
        ms_hl, _ = _timed_device(dist, lambda: tr.train_steps(loc[W:].view(-1, 3), Bl, 1, 2 * (K + W) + W, B_.MARGIN,
                                                               lrs[2 * (K + W) + W:]))
        tr.check_barriers()
        head_local = {"workload": "same table and batch, each rank's triples have heads it owns (head-partitioned triple file)",
                      "value": K * Bl * world / (ms_hl * 1e-3), "unit": "triples/s", "ms_per_step": ms_hl / K}
        del loc

    # end to end: pinned host triples in, per-step loss sums out, inside the timed region
    if p2p:
        # warm-up with a call of the same shape (staging / pinned buffers are sized on first use)
        tr.train_steps_host(host_tri[W:].view(-1, 3), Bl, 1, K + W, B_.MARGIN, lrs[K + W:])
        ms_e2e, hs = _timed_wall(dist, lambda: tr.train_steps_host(host_tri[W:].view(-1, 3), Bl, 1, K + 2 * W,
                                                                   B_.MARGIN, lrs[K + 2 * W:]))
        mean_loss = float(hs[-1]) / Bl
    else:
        def e2e_pass():
            tot = 0.0
            for s in range(K):
                loss = tr.train_step(host_tri[W + s], 1, K + W + s, B_.MARGIN, float(lrs[K + W + s]))
                tot = float(loss.sum().item())
            return tot
        ms_e2e, last = _timed_wall(dist, e2e_pass)
        mean_loss = last / Bl
    e2e = K * Bl * world / (ms_e2e * 1e-3)
    clocks = sampler.stop() if rank == 0 else None
    phases = None
    if p2p:       # where a step's time goes: stream events at the phase boundaries (separate pass)
        be.eng.profile(True)
        run_steps(W, K, 3 * (K + W))
        ph, _ = be.eng.shard_profile_read()
        be.eng.profile(False)
        t = torch.tensor([ph[k] for k in ("post", "k1", "k3", "finish", "apply")], device="cuda", dtype=torch.float64)
        tmax, tmin = t.clone(), t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
        phases = {k: [round(float(tmin[i]) * 1e3, 1), round(float(tmax[i]) * 1e3, 1)]
                  for i, k in enumerate(("post", "k1", "k3", "finish", "apply"))}

    # sharded ranking: configs[3], 100k replicated queries x 1.2M candidates split over the ranks
    nq = int(os.environ.get("HOLE_BENCH_RANK_QUERIES", 100000))
    rng = np.random.default_rng(20170906)
    q = torch.from_numpy(kg.triples[rng.integers(0, len(kg.triples), size=nq)])
    tr.rank(q, HOLE_SIDE_TAIL)
    ms_rank, _ = _timed_device(dist, lambda: tr.rank(q, HOLE_SIDE_TAIL))
    stride = be.width
    if p2p:
        tr.close()
    del tr
    be.eng.close()
    torch.cuda.empty_cache()

    # parity of this very path on the real peers (small problem, after the timed regions)
    ok, par = parity_case(dist, rank, world, local_rank, 256, 2048, 4, 50000, 77, True)
    cfg4 = None
    if not getattr(args, "no_config4", False):
        try:
            cfg4 = bench_config4(args, dist, rank, world, local_rank, max(3, min(K, 20)), 3)
        except Exception as exc:          # reported beside the headline, never instead of it
            cfg4 = {"error": repr(exc)}
    if rank == 0:
        alg = (32 * kg.dim + 20)
        hbm_peak, src, _ = B_.peaks()
        nv = _nvlink_bytes_per_dir(Bl, world, stride) / (ms / K * 1e-3) / 1e9
        print(json.dumps({
            "metric": "HolE train triples/s", "value": value, "unit": "triples/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": B_.workload_desc(Bl), "batch": Bl, "global_batch": Bl * world,
                       "sharding": (f"table row-sharded over {world} GPUs (relations replicated); the training kernel "
                                    "gathers rows from the owners' shards and stages row deltas at the owners over "
                                    "NVLink peer memory; no NCCL call and no host synchronisation inside a step"
                                    if p2p else f"table row-sharded over {world} GPUs, NCCL all-to-all of rows and deltas"),
                       "margin": B_.MARGIN, "lr0": B_.LR0, "parallelism": f"rowshard{world}",
                       "l2": "table shard larger than L2; no flush",
                       "host_enqueue_us_per_step": host_ms / K * 1e3, "mean_loss_last_step": mean_loss,
                       "phase_us_min_max_over_ranks": phases},
            "e2e": {"value": e2e, "unit": "triples/s", "h2d_bytes_per_step": 12 * Bl * world, "d2h_bytes_per_step": 4 * world,
                    "call": "hole_shard_steps_host per rank (pinned host triples in, per-step loss sums out)"},
            "gpu_launches": int(launches), "clocks": clocks,
            "roofline": {"bound": "nvlink", "achieved": nv, "peak": NVLINK_PEAK, "unit": "GB/s per direction per GPU",
                         "frac": nv / NVLINK_PEAK, "traffic": None, "peak_source": NVLINK_PEAK_SRC,
                         "kernel": "hole_k1_kernel<.,.,2> (row gather + delta scatter over peer memory) + apply",
                         "bytes_per_dir_per_step": _nvlink_bytes_per_dir(Bl, world, stride),
                         "hbm_frac_per_gpu": value * alg / 1e9 / world / hbm_peak, "hbm_peak_source": src},
            "cpu_baseline": None,
            "parity": par,
            "head_local": head_local,
            "config4": cfg4,
            "ranking": {"workload": f"rank_diffbot_d256: {nq} queries x 1,200,000 candidates sharded over {world} GPUs (tail side)",
                        "ms": ms_rank, "scores_per_s": nq * 1.2e6 / (ms_rank * 1e-3)},
        }))
    dist.barrier()
    dist.destroy_process_group()
