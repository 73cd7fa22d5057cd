"""The row-sharded --log_loss step (hole_shard_step_logloss), restated in NumPy fp64 on top of oracle.hole_oracle,
and the Python surface around it.  No GPU needed.

A sharded log-loss step splits the global batch into `world` slices.  Rank k draws the k corrupt batches of its
slice with the Philox draws keyed on the global triple index k*B + i, takes every pass's gradient at the old table,
and sums its passes into one delta per row; the owner of a row adds the deltas of every listing rank in rank order
to its decayed row, E * (1 - lr (1+k) (world B) l2).  Each rank reports half the sum of squares of the old rows it
owns, the replicated relation rows on rank 0 only.  In exact arithmetic that is the one-GPU step on the
concatenated batch, so in fp64 it must equal O.logloss_step up to summation order."""
import ctypes as C
import os

import numpy as np
import pytest

from graphembeddings_b200 import _lib
from graphembeddings_b200 import data as D
from graphembeddings_b200.sharded import RowShardedTrainer, row_partition
from oracle import hole_oracle as O
from oracle import philox

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def slice_corruption(pos_slice, type_of, off, ids, seed, step, k, index_base):
    """Rank-local negatives of a slice: pass j is virtual step step*k + j, draws keyed on index_base + i."""
    sides, negs = [], []
    for j in range(k):
        v = step * k + j
        side = philox.side_coin(seed, v)
        ent = pos_slice[:, 0 if side else 1].astype(np.int64)
        ty = np.asarray(type_of)[ent].astype(np.int64)
        lo = off[ty]
        cnt = off[ty + 1] - lo
        draw = philox.entity_draw(seed, v, index_base + np.arange(len(pos_slice)), cnt)
        sides.append(side)
        negs.append(ids[lo + draw].astype(np.int32))
    return sides, np.stack(negs)


def sharded_logloss_step(E, pos, type_of, off, ids, seed, step, k, lr, l2, world, n_relations):
    """The sharded statement, in place on E: per-rank deltas summed over the rank's passes, the owners' rank-order
    sum on the decayed rows.  Returns (loss [(1+k), world*B] in global order, l2 parts [world], negs, sides)."""
    B = len(pos) // world
    rows_per = row_partition(len(E) - n_relations, world)
    E0 = E.copy()
    deltas, losses, negs, parts = [], [], [], []
    sides = None
    for r in range(world):
        sl = pos[r * B:(r + 1) * B]
        s_r, n_r = slice_corruption(sl, type_of, off, ids, seed, step, k, r * B)
        assert sides is None or s_r == sides                  # one side coin per pass, on every rank
        sides = s_r
        Er = E0.copy()
        loss_r, _ = O.logloss_step(Er, sl, list(n_r), s_r, lr, 0.0, np.float64)
        deltas.append(Er - E0)                                # the rank's passes, summed at the old table
        losses.append(loss_r)
        negs.append(n_r)
        b0 = n_relations + r * rows_per
        own = E0[b0:b0 + rows_per]
        parts.append(0.5 * np.sum(own ** 2) + (0.5 * np.sum(E0[:n_relations] ** 2) if r == 0 else 0.0))
    scale = 1.0 - lr * (1 + k) * (world * B) * l2
    E *= scale
    for d in deltas:                                          # rank order
        E += d
    return np.concatenate(losses, axis=1), np.array(parts), np.concatenate(negs, axis=1), sides


@pytest.mark.parametrize("l2", [0.0, 1e-3])
@pytest.mark.parametrize("k", [1, 3])
@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_sharded_statement_equals_the_global_batch_step(world, k, l2):
    B = 40
    kg = D.synthetic_kg(5, 400, 3 * world * B, 4, 20, seed=world + 10 * k, trained_scale=True, zipf_entities=True)
    off, ids = D.build_type_csr(kg.type_of)
    E = kg.E.astype(np.float64)
    Es = E.copy()
    crossing = 0
    for step in range(3):
        pos = kg.triples[step * world * B:(step + 1) * world * B]
        sides, negs = [], []
        for j in range(k):
            side, neg = O.corrupt(pos, kg.type_of, off, ids, 9, step * k + j)
            sides.append(side)
            negs.append(neg)
        want_l2 = 0.5 * np.sum(E ** 2)
        want, _ = O.logloss_step(E, pos, negs, sides, 0.05, l2, np.float64)
        got, parts, got_negs, got_sides = sharded_logloss_step(Es, pos, kg.type_of, off, ids, 9, step, k, 0.05, l2,
                                                               world, kg.n_relations)
        assert got_sides == sides and np.array_equal(got_negs, np.stack(negs))
        np.testing.assert_allclose(got, want, rtol=0, atol=1e-13)
        np.testing.assert_allclose(Es, E, rtol=0, atol=1e-13)
        np.testing.assert_allclose(parts.sum(), want_l2, rtol=1e-13, atol=0)
        listed = [set(np.concatenate([pos[r * B:(r + 1) * B, :2].ravel(), got_negs[:, r * B:(r + 1) * B].ravel()])
                      .tolist()) for r in range(world)]
        crossing += sum(1 for x in set().union(*listed) if sum(x in s for s in listed) > 1)
    if world > 1:
        assert crossing > 0                                   # Zipf entities: rows listed by several ranks
    assert np.abs(Es - kg.E).max() > 1e-3


def test_untouched_rows_are_only_scaled():
    """A row no pass of any rank uses: E <- E * scale (and E unchanged with l2 == 0)."""
    world, B, k = 3, 30, 2
    kg = D.synthetic_kg(4, 2000, world * B, 3, 16, seed=5, trained_scale=True)
    off, ids = D.build_type_csr(kg.type_of)
    for l2 in (0.0, 1e-3):
        E = kg.E.astype(np.float64)
        E0 = E.copy()
        _, _, negs, _ = sharded_logloss_step(E, kg.triples, kg.type_of, off, ids, 1, 0, k, 0.1, l2, world,
                                             kg.n_relations)
        used = np.zeros(len(E), bool)
        used[kg.triples.ravel()] = True
        used[negs.ravel()] = True
        assert (~used).sum() > 1000
        scale = 1.0 - 0.1 * (1 + k) * (world * B) * l2
        assert np.array_equal(E[~used], E0[~used] * scale)


def test_the_binding_declares_the_log_loss_step():
    assert _lib.ABI_VERSION == 7
    sig = (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_uint64, C.c_uint64, C.c_float, C.c_float,
                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p])
    assert _lib.SIGNATURES["hole_shard_step_logloss"] == sig
    assert _lib.SIGNATURES["hole_shard_step_logloss_compute"] == sig
    src = open(os.path.join(ROOT, "include", "hole_b200.h")).read()
    assert "HOLE_API int hole_shard_step_logloss(hole_ctx* ctx," in src
    assert "HOLE_API int hole_shard_step_logloss_compute(hole_ctx* ctx," in src


def test_the_all_to_all_trainer_refuses_log_loss():
    tr = RowShardedTrainer(3, 50, 16, backend=None)
    with pytest.raises(_lib.HoleError, match="P2PRowShardedTrainer"):
        tr.train_step_logloss(np.zeros((4, 3), np.int32), 1, 0, 0.1, 0.0, 1)
