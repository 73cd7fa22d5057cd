"""The row-sharded --log_loss step (hole_shard_step_logloss): every rank gathers its step's rows once into a local step
table, runs the k passes of the one-GPU step (K1 DM 3 + K3, accumulating into a local delta table) at the old table,
pushes the summed deltas to the owners, who decay their shard by the one-GPU L2 factor (global batch size) and add
the staged deltas in rank order.

Tolerances.  At world 1 the step is the one-GPU call bit for bit: the request list keeps the global row order (the
step-table row R + slot is monotone in the global row), so the plan, K1's order and K3's trees are the same, and both
apply x * scale + d.  At world > 1 a row's delta reaches the owner through two summation levels: each rank's K3 tree
over its own uses of the row (in its passes, no deeper than the global tree), then the owner's sum over the ranks
that list the row, at most world - 1 further fp32 adds.  Each add rounds by at most 2^-24 of the running sum of
|lr g|, so the cross-rank level adds lr * absg * (world - 1) * 2^-24 to an element's error, where absg is the sum of
|g| over every use of the row in every pass -- in test_gpu_update_paths._tree_tol's form,
lr * absg * (31 depth + 1) 2^-24, that is (world - 1) / 31 of a tree level.  The band of a step is DESIGN 7's one-step
band widened by it:
    tol = 2e-6 + 1e-5 |x| + lr * absg * (world - 1) * 2^-24.
  * Against the fp64 O.logloss_step (re-synchronised from the shards before every step): that band.
  * Against the one-GPU engine over chained steps: both take the same fp32 per-use gradients and differ only in how
    they sum them, each within its band of the fp64 step from the same state; the band after step s is the sum of
    the per-step bands of the steps that touched the element.  A row no step has touched is equal bit for bit (it is
    only scaled, by the same fp32 factor).
Relation replicas are bit-identical on every rank."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from graphembeddings_b200 import _lib
from graphembeddings_b200 import data as D
from oracle import hole_oracle as O
from oracle.philox import side_coin

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

LOSS_ATOL, ROW_ATOL, ROW_RTOL = 2e-6, 2e-6, 1e-5
DIMS = [2, 64, 66, 128, 130, 256, 258, 512, 514, 768]     # every K1 lane group, masked and full (as the AdaGrad tests)


@pytest.fixture(scope="module")
def eng_mod():
    from graphembeddings_b200 import build
    build.build()
    from graphembeddings_b200 import engine
    return engine


def _bits(x):
    return np.ascontiguousarray(x).view(np.uint32)


def _mb(B, k):
    return max(B, -(-(2 + k) * B // 3))


def _two_sided_seed(n, start=3):
    """A seed whose first n virtual steps take both corruption sides."""
    return next(s for s in range(start, start + 100) if len({side_coin(s, v) for v in range(n)}) == 2)


class _VirtualRanks:
    """`world` ranks of the row-sharded step on ONE GPU: one engine per rank, every "peer" buffer a local tensor,
    sized for log-loss steps of up to k negatives (max_batch = max(B, ceil((2+k)B/3)), as P2PRowShardedTrainer).
    A step runs compute on every rank, then apply on every rank, on one stream."""

    def __init__(self, eng_mod, kg, world, B, k):
        from graphembeddings_b200.sharded import row_partition
        self.eng_mod, self.kg = eng_mod, kg
        self.world, self.B, self.R, self.n_rows = world, B, kg.n_relations, kg.n_rows
        off, ids = D.build_type_csr(kg.type_of)
        self.rows_per = row_partition(kg.n_entities, world)
        self.mb = _mb(B, k)
        self.engs, self.bufs = [], []
        full = eng_mod.HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E)
        for r in range(world):
            e = eng_mod.HoleEngine(kg.n_relations + 3 * self.mb, kg.dim).set_types(kg.type_of, off, ids)
            e.set_relation_count(kg.n_relations)
            dev, w, cap = e.device, e.row_stride, 3 * self.mb
            shard = torch.zeros((self.R + self.rows_per, w), dtype=torch.float32, device=dev)
            b0, b1 = self._block(r)
            shard[: self.R] = full.table[: self.R]
            shard[self.R: self.R + (b1 - b0)] = full.table[b0:b1]
            self.bufs.append([shard,
                              torch.zeros((world, cap, w), dtype=torch.float32, device=dev),
                              torch.zeros((world, max(self.R, 1), w), dtype=torch.float32, device=dev),
                              torch.zeros((2, world, cap), dtype=torch.int32, device=dev),
                              torch.zeros((2, world, 2), dtype=torch.int32, device=dev),
                              torch.zeros((2, world), dtype=torch.int32, device=dev),
                              torch.zeros(1, dtype=torch.int32, device=dev)])
            self.engs.append(e)
        full.close()
        for r, e in enumerate(self.engs):
            pa = e.peer_array
            e.shard_init(world, r, self.R, kg.n_entities, self.rows_per, self.mb, self.bufs[r][0],
                         *[pa([self.bufs[j][i] for j in range(world)]) for i in range(6)], self.bufs[r][6], 5.0)

    def _block(self, r):
        b0 = self.R + r * self.rows_per
        return b0, max(b0, min(self.n_rows, b0 + self.rows_per))

    def slices(self, gb):
        t = torch.from_numpy(np.ascontiguousarray(gb)).to(self.engs[0].device)
        return [t[r * self.B:(r + 1) * self.B].contiguous() for r in range(self.world)]

    def logloss(self, gb, seed, step, lr, l2, k, want_l2_loss=True):
        """One log-loss step of the global batch gb: (loss [(1+k), world*B] host, l2 parts host, sides, neg [k, world*B])"""
        outs = [e.shard_step_logloss(sl, seed, step, lr, l2, k, phase="compute", want_corruption=True,
                                     want_l2_loss=want_l2_loss) for e, sl in zip(self.engs, self.slices(gb))]
        for e in self.engs:
            e.shard_step(None, seed, step, 0.0, lr, phase="apply")
        sides = outs[0][2]
        assert all(o[2] == sides for o in outs)
        loss = np.concatenate([o[0].cpu().numpy() for o in outs], axis=1)
        neg = np.concatenate([o[3].cpu().numpy() for o in outs], axis=1)
        return loss, np.array([float(o[1]) for o in outs]), sides, neg

    def table(self):
        for e in self.engs:
            assert not e.shard_poll()
        rel = self.bufs[0][0][: self.R]
        ents = []
        for r in range(self.world):
            assert torch.equal(self.bufs[r][0][: self.R], rel), f"relation replica of rank {r} differs"
            b0, b1 = self._block(r)
            ents.append(self.bufs[r][0][self.R: self.R + (b1 - b0)])
        tmp = self.eng_mod.HoleEngine(self.n_rows, self.kg.dim)
        tmp.table = torch.cat([rel] + ents).contiguous()
        out = tmp.embeddings().cpu().numpy()
        tmp.table = None
        tmp.close()
        return out

    def close(self):
        for e in self.engs:
            e.close()


def _single(eng_mod, kg):
    off, ids = D.build_type_csr(kg.type_of)
    e = eng_mod.HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E).set_types(kg.type_of, off, ids)
    e.set_relation_count(kg.n_relations)
    return e


def _abs_grads(E, pos, negs, sides):
    """Per element, the sum of |g| over every use of the row in every pass (the absg of the module docstring)."""
    Ew = E.astype(np.float64)
    acc = np.zeros_like(Ew)
    s_p = O.score(Ew, pos, np.float64)
    for col, dx in zip((0, 1, 2), O._side_grads(Ew, pos, O.sigmoid(s_p) - 1.0, np.float64)):
        np.add.at(acc, pos[:, col].astype(np.int64), np.abs(dx))
    for j, side in enumerate(sides):
        neg = O.corrupt_triples(pos, negs[j], side)
        s_n = O.score(Ew, neg, np.float64)
        for col, dx in zip((0, 1, 2), O._side_grads(Ew, neg, O.sigmoid(s_n), np.float64)):
            np.add.at(acc, neg[:, col].astype(np.int64), np.abs(dx))
    return acc


def _used(pos, negs):
    return np.unique(np.concatenate([pos.ravel(), np.asarray(negs).ravel()]).astype(np.int64))


def _check_fp64(tag, E0, E1, loss, l2_parts, pos, negs, sides, lr, l2, world):
    """One sharded step E0 -> E1 against the fp64 O.logloss_step from E0 (module docstring's band)."""
    E = E0.astype(np.float64)
    want_loss, want_l2 = O.logloss_step(E, pos, list(negs), sides, lr, l2, np.float64)
    assert np.abs(loss - want_loss).max() <= LOSS_ATOL, tag
    assert abs(l2_parts.sum() - want_l2) <= 1e-6 * want_l2, tag
    rows = _used(pos, negs)
    tol = ROW_ATOL + ROW_RTOL * np.abs(E[rows]) + lr * _abs_grads(E0, pos, negs, sides)[rows] * (world - 1) * 2.0**-24
    r = np.abs(E1[rows] - E[rows]) / tol
    assert (r <= 1.0).all(), (tag, float(r.max()))
    keep = np.ones(len(E0), bool)
    keep[rows] = False
    scale = np.float32(1.0) - np.float32(lr) * np.float32(1 + len(sides)) * np.float32(len(pos)) * np.float32(l2)
    want_keep = E0[keep] if l2 == 0.0 else (E0[keep] * scale).astype(np.float32)
    assert np.array_equal(_bits(E1[keep]), _bits(want_keep)), (tag, "an untouched row is not just scaled")
    return rows


def _run_checked(vr, kg, gbs, seed, lr, l2, k, first_step=0):
    """Log-loss steps on the global batches gbs, each checked against fp64 re-synchronised; returns (negs, sides)."""
    off, ids = D.build_type_csr(kg.type_of)
    out = []
    for s, gb in enumerate(gbs):
        step = first_step + s
        E0 = vr.table()
        loss, parts, sides, neg = vr.logloss(gb, seed, step, lr, l2, k)
        for j in range(k):
            side_o, neg_o = O.corrupt(gb, kg.type_of, off, ids, seed, step * k + j)
            assert side_o == sides[j] and np.array_equal(neg_o, neg[j]), (s, j)
        _check_fp64(f"step {step}", E0, vr.table(), loss, parts, gb, neg, sides, np.float32(lr), l2, vr.world)
        out.append((neg, sides))
    return out


# ---------------------------------------------------------------- world 1: the one-GPU call bit for bit
@pytest.mark.parametrize("l2", [0.0, 1e-3])
@pytest.mark.parametrize("k", [1, 2, 4])
def test_world1_is_the_single_gpu_step_bit_for_bit(eng_mod, k, l2):
    B, steps, dim = 300, 3, 150
    kg = D.synthetic_kg(7, 3000, steps * B, 5, dim, seed=20 + k, trained_scale=True, zipf_entities=True)
    seed = _two_sided_seed(steps * k)
    vr = _VirtualRanks(eng_mod, kg, 1, B, k)
    e = _single(eng_mod, kg)
    got_sides = set()
    for s in range(steps):
        gb = kg.triples[s * B:(s + 1) * B]
        loss, parts, sides, neg = vr.logloss(gb, seed, s, 0.05, l2, k)
        want_loss, want_l2, want_sides, want_neg = e.train_step_logloss(gb, seed, s, 0.05, l2, k, want_corruption=True,
                                                                        want_l2_loss=True)
        assert sides == want_sides and np.array_equal(neg, want_neg.cpu().numpy())
        assert np.array_equal(_bits(loss), _bits(want_loss.cpu().numpy())), s
        assert abs(parts[0] - float(want_l2)) <= 1e-6 * float(want_l2)
        assert np.array_equal(_bits(vr.table()), _bits(e.embeddings().cpu().numpy())), s
        got_sides |= set(sides)
    assert got_sides == {0, 1}
    assert np.abs(vr.table() - kg.E).max() > 1e-4
    vr.close()
    e.close()


# ---------------------------------------------------------------- worlds 2, 3, 8
@pytest.mark.parametrize("world,dim,B,k,l2", [(2, 256, 257, 2, 1e-3), (3, 150, 129, 1, 0.0), (3, 130, 100, 4, 1e-4),
                                              (8, 150, 65, 2, 1e-3)])
def test_parity_with_the_single_gpu_step(eng_mod, world, dim, B, k, l2):
    """Chained steps against HoleEngine.train_step_logloss on the concatenated batches: negatives, sides and the first
    step's loss rows bit for bit, tables within the summed per-step bands, rows no step touched bit for bit, the
    relation replicas identical; every step also against fp64 from the shards' own state."""
    steps, lr = 3, np.float32(0.05)
    kg = D.synthetic_kg(7, 2000, steps * world * B, 5, dim, seed=900 + world + k, trained_scale=True,
                        zipf_entities=True)
    seed = _two_sided_seed(steps * k)
    vr = _VirtualRanks(eng_mod, kg, world, B, k)
    e = _single(eng_mod, kg)
    band = np.zeros(kg.E.shape)
    touched = np.zeros(kg.n_rows, bool)
    for s in range(steps):
        gb = kg.triples[s * world * B:(s + 1) * world * B]
        E0 = vr.table()
        loss, parts, sides, neg = vr.logloss(gb, seed, s, lr, l2, k)
        want_loss, _, want_sides, want_neg = e.train_step_logloss(gb, seed, s, lr, l2, k, want_corruption=True)
        assert sides == want_sides and np.array_equal(neg, want_neg.cpu().numpy())
        if s == 0:
            assert np.array_equal(_bits(loss), _bits(want_loss.cpu().numpy()))
        else:
            assert np.abs(loss - want_loss.cpu().numpy()).max() <= LOSS_ATOL
        rows = _check_fp64(f"step {s}", E0, vr.table(), loss, parts, gb, neg, sides, lr, l2, world)
        Es = e.embeddings().cpu().numpy()
        absg = _abs_grads(E0, gb, neg, sides)[rows]
        band[rows] += ROW_ATOL + ROW_RTOL * np.abs(Es[rows]) + lr * absg * (world - 1) * 2.0**-24
        touched[rows] = True
        Eg = vr.table()
        assert (np.abs(Eg - Es) <= band).all(), (s, float((np.abs(Eg - Es) / np.maximum(band, 1e-300)).max()))
        assert np.array_equal(_bits(Eg[~touched]), _bits(Es[~touched])), s
    assert (~touched).any() and np.abs(Es - kg.E).max() > 1e-4
    vr.close()
    e.close()


@pytest.mark.parametrize("dim", DIMS)
def test_every_lane_group(eng_mod, dim):
    """The passes on the step table, the gather and the push at every K1 lane group, 2 or 3 ranks, ragged B."""
    world = 2 + DIMS.index(dim) % 2
    B = 61 + 2 * DIMS.index(dim)
    kg = D.synthetic_kg(7, 2000, 2 * world * B, 5, dim, seed=700 + dim, trained_scale=True, zipf_entities=True)
    vr = _VirtualRanks(eng_mod, kg, world, B, 2)
    _run_checked(vr, kg, [kg.triples[s * world * B:(s + 1) * world * B] for s in range(2)], dim, 0.1, 1e-4, 2)
    assert np.abs(vr.table() - kg.E).max() > 1e-4
    vr.close()


# ---------------------------------------------------------------- sharding edges
def test_trailing_ranks_that_own_no_rows(eng_mod):
    """10 entities over 8 ranks: ranks 5-7 own no rows (their shards hold relation rows only)."""
    world, B, k = 8, 6, 2
    kg = D.synthetic_kg(5, 10, 2 * world * B, 2, 64, seed=36, trained_scale=True, zipf_entities=True)
    vr = _VirtualRanks(eng_mod, kg, world, B, k)
    assert vr.rows_per * 5 == 10
    _run_checked(vr, kg, [kg.triples[s * world * B:(s + 1) * world * B] for s in range(2)], 5, 0.1, 1e-3, k)
    vr.close()


def test_one_row_listed_by_all_eight_ranks(eng_mod):
    world, B, k = 8, 40, 2
    kg = D.synthetic_kg(5, 800, 2 * world * B, 4, 64, seed=12, trained_scale=True, zipf_entities=True)
    hot = kg.n_relations + 333
    kg.triples[::B // 4, 0] = hot                   # four uses in every slice of both steps
    vr = _VirtualRanks(eng_mod, kg, world, B, k)
    gbs = [kg.triples[s * world * B:(s + 1) * world * B] for s in range(2)]
    _run_checked(vr, kg, gbs, 3, 0.1, 1e-3, k)
    assert all(all((gb[r * B:(r + 1) * B, 0] == hot).any() for r in range(world)) for gb in gbs)
    vr.close()


def test_rows_that_only_a_later_pass_uses_and_rows_in_two_roles(eng_mod):
    """k = 4: a corrupt entity that no earlier pass and no positive lists (its only use is in pass j > 0), and a row
    that is a positive entity in every pass and a corrupt entity in another."""
    world, B, k = 3, 120, 4
    kg = D.synthetic_kg(5, 900, world * B, 4, 130, seed=13, trained_scale=True, zipf_entities=True)
    vr = _VirtualRanks(eng_mod, kg, world, B, k)
    (neg, sides), = _run_checked(vr, kg, [kg.triples], 6, 0.1, 1e-3, k)
    ents = set(kg.triples[:, :2].ravel().tolist())
    late = set(neg[1:].ravel().tolist()) - set(neg[0].tolist()) - ents
    both = ents & set(neg.ravel().tolist())
    assert late and both
    vr.close()


@pytest.mark.parametrize("B,k", [(30, 4), (64, 1)])
def test_batch_at_the_staging_capacity(eng_mod, B, k):
    """(2 + k) B == 3 * max_batch: the request list may fill the staging slices and inboxes."""
    world = 2
    kg = D.synthetic_kg(5, 5000, world * B, 3, 64, seed=B + k, trained_scale=True)
    vr = _VirtualRanks(eng_mod, kg, world, B, k)
    assert (2 + k) * B == 3 * vr.mb
    _run_checked(vr, kg, [kg.triples], 7, 0.1, 1e-3, k)
    vr.close()


# ---------------------------------------------------------------- hinge and log-loss steps on one context
def test_mixed_sequence_with_a_hinge_step_prepared_ahead(eng_mod):
    """Hinge steps 0-1, each prepared one step ahead (hole_shard_prepare), hinge step 4 prepared, log-loss steps 2-3,
    then hinge steps 4 (prepared) and 5, against the one-GPU engine doing the same.  The log-loss steps leave the
    prepared step in place: its compute half launches fewer kernels than step 5's, which builds its own plan."""
    world, B, k, seed, lr, margin = 2, 150, 2, 4, np.float32(0.1), 0.2
    kg = D.synthetic_kg(6, 1500, 6 * world * B, 4, 128, seed=9, trained_scale=True, zipf_entities=True)
    vr = _VirtualRanks(eng_mod, kg, world, B, k)
    e = _single(eng_mod, kg)
    gbs = [kg.triples[s * world * B:(s + 1) * world * B] for s in range(6)]
    sl = [vr.slices(gb) for gb in gbs]               # kept alive: a prepared step is found by its triples' address
    band = np.zeros(kg.E.shape)

    def widen(gb, negs):
        Es = e.embeddings().cpu().numpy()
        rows = _used(gb, negs)
        band[rows] += ROW_ATOL + ROW_RTOL * np.abs(Es[rows])

    def prepare(s):
        for r, en in enumerate(vr.engs):
            en.shard_prepare(sl[s][r], seed, s)

    def hinge(s):
        torch.cuda.synchronize()
        n0 = vr.engs[0].launch_count()
        vr.engs[0].shard_step(sl[s][0], seed, s, margin, lr, phase="compute")
        launches = vr.engs[0].launch_count() - n0
        for r in range(1, world):
            vr.engs[r].shard_step(sl[s][r], seed, s, margin, lr, phase="compute")
        for en in vr.engs:
            en.shard_step(None, seed, s, margin, lr, phase="apply")
        side, neg = e.corrupt_batch(gbs[s], seed, s)
        e.train_step(gbs[s], neg, side, margin, lr)
        widen(gbs[s], neg.cpu().numpy())
        return launches

    prepare(0)
    prepare(1)
    hinge(0)
    hinge(1)
    prepare(4)
    for s in (2, 3):
        vr.logloss(gbs[s], seed, s, lr, 1e-3, k)
        _, _, _, neg = e.train_step_logloss(gbs[s], seed, s, lr, 1e-3, k, want_corruption=True)
        widen(gbs[s], neg.cpu().numpy())
    prepared = hinge(4)
    unprepared = hinge(5)
    assert prepared < unprepared, (prepared, unprepared)
    Eg, Es = vr.table(), e.embeddings().cpu().numpy()
    assert (np.abs(Eg - Es) <= band).all(), float((np.abs(Eg - Es) / np.maximum(band, 1e-300)).max())
    assert np.abs(Es - kg.E).max() > 1e-4
    vr.close()
    e.close()


# ---------------------------------------------------------------- refusals
def test_refusals_write_nothing_and_leave_the_context_usable(eng_mod):
    world, B = 2, 100
    kg = D.synthetic_kg(5, 600, 3 * world * B, 4, 64, seed=6, trained_scale=True, zipf_entities=True)
    off, ids = D.build_type_csr(kg.type_of)
    fresh = eng_mod.HoleEngine(kg.n_relations + 3 * B, kg.dim).set_types(kg.type_of, off, ids)
    pos = torch.from_numpy(kg.triples[:B]).cuda()
    with pytest.raises(_lib.HoleError, match="error -1"):         # before hole_shard_init
        fresh.shard_step_logloss(pos, 1, 0, 0.1, 0.0, 1)
    fresh.close()
    vr = _VirtualRanks(eng_mod, kg, world, B, 1)                   # max_batch = B: k = 1 fits, k = 2 does not
    gbs = [kg.triples[s * world * B:(s + 1) * world * B] for s in range(3)]
    _run_checked(vr, kg, gbs[:1], 2, 0.1, 1e-3, 1)
    e = vr.engs[0]
    snap = [b[0].clone() for b in vr.bufs]
    sl = vr.slices(gbs[1])[0]
    torch.cuda.synchronize()
    n0 = e.launch_count()
    for k in (2, 0, 65):                                           # over capacity, bad k
        with pytest.raises(_lib.HoleError, match="error -1"):
            e.shard_step_logloss(sl, 2, 1, 0.1, 1e-3, k)
    with pytest.raises(_lib.HoleError, match="error -1"):          # B = 0
        e.shard_step_logloss(sl[:0], 2, 1, 0.1, 1e-3, 1)
    acc = torch.full_like(vr.bufs[0][0], 0.1)
    e.shard_set_optimizer("adagrad", acc)
    with pytest.raises(_lib.HoleError, match="error -4"):          # AdaGrad has no log-loss step
        e.shard_step_logloss(sl, 2, 1, 0.1, 1e-3, 1)
    e.shard_set_optimizer("sgd", None)
    torch.cuda.synchronize()
    assert e.launch_count() == n0
    for t, b in zip(snap, vr.bufs):
        assert torch.equal(b[0], t)
    _run_checked(vr, kg, gbs[1:], 2, 0.1, 1e-3, 1, first_step=1)   # still training correctly
    vr.close()


# ---------------------------------------------------------------- the trainer at world 1
def test_world1_trainer_matches_the_single_gpu_engine(eng_mod):
    from graphembeddings_b200.sharded import CudaBackend, P2PRowShardedTrainer
    B, steps, dim, k = 256, 3, 150, 4
    kg = D.synthetic_kg(6, 2500, steps * B, 4, dim, seed=77, trained_scale=True, zipf_entities=True)
    off, ids = D.build_type_csr(kg.type_of)
    be = CudaBackend(kg.n_relations, dim, B, 0, kg.type_of, off, ids)
    tr = P2PRowShardedTrainer(kg.n_relations, kg.n_entities, dim, be, None, negative_ratio=k).load_embeddings(kg.E)
    assert tr.max_batch == 2 * B and be.eng.n_rows == kg.n_relations + 6 * B
    e = _single(eng_mod, kg)
    tri = torch.from_numpy(kg.triples).cuda()
    for s in range(steps):
        kk = 1 + s % k                                              # any k up to the trainer's
        loss, part = tr.train_step_logloss(tri[s * B:(s + 1) * B], 5, s, 0.05, 1e-3, kk)
        want, want_l2 = e.train_step_logloss(kg.triples[s * B:(s + 1) * B], 5, s, 0.05, 1e-3, kk)
        assert torch.equal(loss, want)
        assert abs(float(part) - float(want_l2)) <= 1e-6 * float(want_l2)
    E1, Es = tr.gather_embeddings().cpu().numpy(), e.embeddings().cpu().numpy()
    assert np.array_equal(_bits(E1), _bits(Es)) and np.abs(Es - kg.E).max() > 1e-4
    tr.close()
    be.eng.close()
    e.close()


# ---------------------------------------------------------------- real peers
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.parametrize("world", [2, 4, 8])
def test_real_peers_match_the_single_gpu_step(world):
    if not torch.cuda.is_available() or torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    from graphembeddings_b200 import build
    build.build()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           os.path.join(ROOT, "tools", "multi_gpu_logloss_check.py")]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    tail = (r.stdout + r.stderr)[-3000:]
    assert r.returncode == 0, tail
    assert "MULTI_GPU_LOGLOSS_CHECK OK" in r.stdout, tail
