"""The owner-side AdaGrad step of the row-sharded trainer (hole_shard_set_optimizer), restated in NumPy on top of
tests/adagrad_reference.py, and the Python surface around it.  No GPU needed.

A sharded AdaGrad step splits the global batch into `world` slices.  Rank k computes, at the shared table, the summed
gradient of every row its slice uses and stages it at the row's owner; the owner sums the staged rows of every rank
that lists the row in rank order, then applies one SparseApplyAdagrad update.  In exact arithmetic that is
TF's duplicate-index sum over the whole global batch, so in fp64 it must equal adagrad_reference.adagrad_step on the
concatenated batch up to summation order."""
import ctypes as C
import os

import numpy as np
import pytest

import adagrad_reference as R
from graphembeddings_b200 import _lib
from graphembeddings_b200 import data as D
from graphembeddings_b200.sharded import RowShardedTrainer
from oracle import hole_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def sharded_adagrad_step(E, A, pos, neg, side, margin, lr, world):
    """The owner-side statement, in place on E and A: per-slice summed gradients, summed over the slices in rank
    order, one update per touched row.  Returns (loss [world*B], the rows each slice lists)."""
    B = len(pos) // world
    total = np.zeros_like(E)
    touched = np.zeros(len(E), bool)
    losses, listed = [], []
    for k in range(world):
        sl = slice(k * B, (k + 1) * B)
        rows, g, loss = R.merged_gradient(E, pos[sl], neg[sl], side, margin, E.dtype.type)
        total[rows] += g                      # rank order: slice k is added after slices 0..k-1
        touched[rows] = True
        losses.append(loss)
        listed.append(set(rows.tolist()))
    rows = np.flatnonzero(touched)
    R.adagrad_apply(E, A, rows, total[rows], lr)
    return np.concatenate(losses), listed


@pytest.mark.parametrize("margin", [0.2, 0.0])           # 0.0: about half the hinges inactive
@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_owner_side_sum_equals_the_global_batch_step(world, margin):
    B = 48
    kg = D.synthetic_kg(5, 400, 3 * world * B, 4, 20, seed=world, trained_scale=True, zipf_entities=True)
    off, ids = D.build_type_csr(kg.type_of)
    E = kg.E.astype(np.float64)
    A = np.full_like(E, 0.1)
    Es, As = E.copy(), A.copy()
    crossing = 0
    for step in range(3):
        pos = kg.triples[step * world * B:(step + 1) * world * B]
        side, neg = O.corrupt(pos, kg.type_of, off, ids, 7, step)
        want = R.adagrad_step(E, A, pos, neg, side, margin, 0.3, np.float64)
        got, listed = sharded_adagrad_step(Es, As, pos, neg, side, margin, 0.3, world)
        np.testing.assert_allclose(got, want, rtol=0, atol=1e-13)
        np.testing.assert_allclose(Es, E, rtol=0, atol=1e-13)
        np.testing.assert_allclose(As, A, rtol=1e-13, atol=0)
        ents = [r for r in set().union(*listed) if r >= kg.n_relations]
        crossing += sum(1 for r in ents if sum(r in s for s in listed) > 1)
        if margin == 0.0:
            assert 0 < (want == 0).sum() < len(want)       # active and inactive hinges in one step
    if world > 1:
        assert crossing > 0                                # Zipf entities: rows listed by several ranks
    assert np.abs(Es - kg.E).max() > 1e-3


def test_a_row_whose_gradients_cancel_keeps_its_rows():
    """A row listed by two ranks whose gradients are exact opposites: g = 0, so the table and accumulator rows keep
    their values (A + 0 = A, x - lr 0 rsqrt(A) = x), as for an inactive hinge."""
    E = np.array([[1.0, -2.0], [0.5, 0.25]])
    A = np.full_like(E, 0.1)
    g = [np.array([[0.0, 0.0], [0.5, -1.0]]), np.array([[0.0, 0.0], [-0.5, 1.0]])]
    total = g[0] + g[1]
    E0, A0 = E.copy(), A.copy()
    R.adagrad_apply(E, A, np.array([0, 1]), total, 0.5)
    assert np.array_equal(E, E0) and np.array_equal(A, A0)


def test_the_binding_declares_hole_shard_set_optimizer():
    assert _lib.ABI_VERSION == 7
    assert _lib.SIGNATURES["hole_shard_set_optimizer"] == (C.c_int, [C.c_void_p, C.c_int, C.c_void_p])
    src = open(os.path.join(ROOT, "include", "hole_b200.h")).read()
    assert "HOLE_API int hole_shard_set_optimizer(hole_ctx* ctx, int optimizer, float* accum_shard);" in src
    assert "#define HOLE_ABI_VERSION 7" in src


def test_the_all_to_all_trainer_refuses_adagrad():
    tr = RowShardedTrainer(3, 50, 16, backend=None)
    assert tr.set_optimizer("sgd") is tr
    with pytest.raises(_lib.HoleError, match="P2PRowShardedTrainer"):
        tr.set_optimizer("adagrad")
    with pytest.raises(_lib.HoleError, match="P2PRowShardedTrainer"):
        tr.set_optimizer("adagrad", initial_accumulator=0.5)
