"""AdaGrad on the row-sharded step (hole_shard_set_optimizer): K1 / K3 stage each rank's summed gradient with
lr = -1, and hole_shard_adagrad_apply_kernel at the owner sums the staged rows of every listing rank in rank order,
then applies A += g^2; E -= lr g rsqrt(A) once.

Tolerances.  The fp32 gradient of a row reaches the update through two summation levels: each rank's K3 tree over
its own uses (tree_depth of the rank's use count, at most that of the global count), then the owner's sum over the
ranks that list the row, at most world - 1 further fp32 adds, each rounding by at most 2^-24 of the running sum of
|g|.  In adagrad_reference.tree_tolerance's form, where delta = absg (1e-6 + (31 depth + 1) 2^-24), those adds are
(world - 1) / 31 of a tree level:
    tolE, tolA = tree_tolerance(G, absg, depth + (world - 1) / 31, A0, lr, E_ref)
Its constant terms are the one-step band of DESIGN 7c (2e-6 + 1e-5 |x| on a row); nothing else is widened.
  * Against the fp64 reference (re-synchronised from the device's state before every step): that band per step;
    the plain 7c band (2e-6 + 1e-5 |x|, 1e-7 + 1e-5 |a|) in the default regime, as tests/test_gpu_adagrad.py.
  * Against the single-GPU engine over chained steps: both devices take the same fp32 per-use gradients and differ
    only in how they sum them, each within its band of the fp64 step from the same state; the band after step s is
    the sum of the per-step bands of the steps that touched the element (a difference carried in from an earlier
    step reaches the next step's gradient through the fp32 forward pass, which the constant terms cover).  SGD steps
    of a mixed sequence add the SGD one-step band 2e-6 + 1e-5 |x|.
Both accumulator regimes run: A0 >> g^2 (an SGD step at lr / sqrt(A0)) and A0 << g^2 (a step of ~lr sign(g)).
Rows and accumulator elements no step touches keep their bits; the relation rows of the table and of the
accumulator are bit-identical on every rank."""
import ctypes as C
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

import adagrad_reference as R
from graphembeddings_b200 import _lib
from graphembeddings_b200 import data as D
from oracle import hole_oracle as O
from oracle.philox import side_coin
from test_gpu_adagrad_paths import _row_depths, _row_sums

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

MARGIN, INIT, LOSS_ATOL = 0.2, 0.1, 2e-6
ROW_ATOL, ROW_RTOL, ACC_ATOL, ACC_RTOL = 2e-6, 1e-5, 1e-7, 1e-5
# (A0, lr): A0 >> g^2 (lr / sqrt(A0) = 0.1)  /  A0 << g^2 (steps of ~lr)
REGIMES = {"large": (100.0, 1.0), "small": (1e-6, 0.01)}
# first and last dim of every K1 lane group (GS 8 / 16 / 32 x V 1, 2, 3): masked and full
DIMS = [2, 64, 66, 128, 130, 256, 258, 512, 514, 768]


@pytest.fixture(scope="module")
def eng_mod():
    from graphembeddings_b200 import build
    build.build()
    from graphembeddings_b200 import engine
    return engine


def _f32(x):
    return float(np.float32(x))


def _bits(x):
    return np.ascontiguousarray(x).view(np.uint32)


def _two_sided_seed(steps, start=3):
    """The first Philox seed >= start whose side coins over `steps` steps take both sides."""
    return next(s for s in range(start, start + 100) if len({side_coin(s, k) for k in range(steps)}) == 2)


class _VirtualRanks:
    """`world` ranks of the row-sharded step on ONE GPU (as test_gpu_train._VirtualRanks): one engine per rank, every
    "peer" buffer a local tensor; a step runs compute on every rank, then apply on every rank, on one stream.  Also
    holds an AdaGrad accumulator shard per rank (set_optimizer).  E: start table (default kg.E)."""

    def __init__(self, eng_mod, kg, world, B, csr=None, E=None):
        from graphembeddings_b200.sharded import row_partition
        self.eng_mod, self.kg = eng_mod, kg
        self.world, self.B, self.R, self.n_rows = world, B, kg.n_relations, kg.n_rows
        off, ids = D.build_type_csr(kg.type_of) if csr is None else csr
        self.rows_per = row_partition(kg.n_entities, world)
        self.engs, self.bufs, self.accums = [], [], [None] * world
        full = eng_mod.HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E if E is None else E)
        for k in range(world):
            e = eng_mod.HoleEngine(kg.n_relations + 3 * B, kg.dim).set_types(kg.type_of, off, ids)
            e.set_relation_count(kg.n_relations)
            dev, w, cap = e.device, e.row_stride, 3 * B
            shard = torch.zeros((self.R + self.rows_per, w), dtype=torch.float32, device=dev)
            b0, b1 = self._block(k)
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
        for k, e in enumerate(self.engs):
            pa = e.peer_array
            e.shard_init(world, k, self.R, kg.n_entities, self.rows_per, B, self.bufs[k][0],
                         *[pa([self.bufs[j][i] for j in range(world)]) for i in range(6)], self.bufs[k][6], 5.0)

    def _block(self, k):
        b0 = self.R + k * self.rows_per
        return b0, max(b0, min(self.n_rows, b0 + self.rows_per))

    def set_optimizer(self, opt, init=INIT):
        """"adagrad": a fresh accumulator shard per rank, every element (pads, unused rows) = init; "sgd": none."""
        for k, e in enumerate(self.engs):
            if opt == "adagrad":
                self.accums[k] = torch.full_like(self.bufs[k][0], float(init))
                e.shard_set_optimizer("adagrad", self.accums[k])
            else:
                e.shard_set_optimizer("sgd", None)
                self.accums[k] = None
        return self

    def step(self, slices, seed, step, margin, lr):
        losses = [e.shard_step(slices[k], seed, step, margin, lr, phase="compute") for k, e in enumerate(self.engs)]
        for e in self.engs:
            e.shard_step(None, seed, step, margin, lr, phase="apply")
        return losses

    def _full(self, parts):
        """[N, dim] from every rank's [relations | block] rows; checks that the relation replicas are identical."""
        rel = parts[0][: self.R]
        ents = []
        for k in range(self.world):
            assert torch.equal(parts[k][: self.R], rel), f"relation replica of rank {k} differs"
            b0, b1 = self._block(k)
            ents.append(parts[k][self.R: self.R + (b1 - b0)])
        tmp = self.eng_mod.HoleEngine(self.n_rows, self.kg.dim)
        tmp.table = torch.cat([rel] + ents).contiguous()
        out = tmp.embeddings().cpu().numpy()
        tmp.table = None
        tmp.close()
        return out

    def table(self):
        for e in self.engs:
            assert not e.shard_poll()
        return self._full([b[0] for b in self.bufs])

    def accumulator(self):
        return self._full(self.accums)

    def state(self):
        return self.table(), self.accumulator()

    def close(self):
        for e in self.engs:
            e.close()


def _single(eng_mod, kg, csr=None, opt="adagrad", init=INIT):
    off, ids = D.build_type_csr(kg.type_of) if csr is None else csr
    e = eng_mod.HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E).set_types(kg.type_of, off, ids)
    e.set_relation_count(kg.n_relations)
    if opt == "adagrad":
        e.set_optimizer("adagrad", init)
    return e


def _slices(gb, world, dev):
    B = len(gb) // world
    t = torch.from_numpy(np.ascontiguousarray(gb)).to(dev)
    return [t[k * B:(k + 1) * B].contiguous() for k in range(world)]


def _ref(E0, A0, pos, neg, side, margin, lr, n_relations, world):
    """The fp64 AdaGrad step from (E0, A0) on the rows it uses, with the sharded band of each (module docstring)."""
    E64 = E0.astype(np.float64)
    slices, loss, _, _ = O.indexed_slices(E64, pos, neg, side, margin, np.float64)
    rows, G, absg = _row_sums([(i.astype(np.int64), g) for i, g in slices], len(E0))
    Er, Ar = E64[rows], A0[rows].astype(np.float64)
    R.adagrad_apply(Er, Ar, np.arange(len(rows)), G, lr)
    depth = _row_depths(pos, neg, len(E0), n_relations)[rows] + (world - 1) / 31
    tolE, tolA = R.tree_tolerance(G, absg, depth[:, None], A0[rows].astype(np.float64), lr, Er)
    return dict(loss=loss, rows=rows, E=Er, A=Ar, tolE=tolE, tolA=tolA)


def _check(tag, before, after, pos, neg, side, lr, kg, world, loss, flat=False):
    """One sharded step before -> after against the fp64 step from `before`: the sharded band (flat: DESIGN 7c's
    band), and untouched rows / accumulator elements bit for bit."""
    E0, A0 = before
    E1, A1 = after
    ref = _ref(E0, A0, pos, neg, side, MARGIN, lr, kg.n_relations, world)
    rows = ref["rows"]
    assert np.abs(loss - ref["loss"]).max() <= LOSS_ATOL, tag
    tolE, tolA = ref["tolE"], ref["tolA"]
    if flat:
        tolE, tolA = ROW_ATOL + ROW_RTOL * np.abs(ref["E"]), ACC_ATOL + ACC_RTOL * np.abs(ref["A"])
    for name, got, want, tol in (("E", E1[rows], ref["E"], tolE), ("A", A1[rows], ref["A"], tolA)):
        r = np.abs(got - want) / tol
        assert (r <= 1.0).all(), (tag, name, float(r.max()), int(rows[np.unravel_index(r.argmax(), r.shape)[0]]))
    keep = np.ones(len(E0), bool)
    keep[rows] = False
    assert np.array_equal(_bits(E1[keep]), _bits(E0[keep])), (tag, "an unused row changed")
    assert np.array_equal(_bits(A1[keep]), _bits(A0[keep])), (tag, "an unused accumulator row changed")
    return ref


def _run_checked(vr, kg, gbs, seed, lr, csr=None, flat=False, first_step=0):
    """Sharded steps on the global batches gbs, each checked against fp64 re-synchronised; returns the refs."""
    off, ids = D.build_type_csr(kg.type_of) if csr is None else csr
    refs = []
    for s, gb in enumerate(gbs):
        before = vr.state()
        losses = vr.step(_slices(gb, vr.world, vr.engs[0].device), seed, first_step + s, MARGIN, lr)
        side, neg = O.corrupt(gb, kg.type_of, off, ids, seed, first_step + s)
        loss = torch.cat(losses).cpu().numpy()
        refs.append(_check(f"step {s}", before, vr.state(), gb, neg, side, _f32(lr), kg, vr.world, loss, flat))
        refs[-1]["neg"], refs[-1]["side"] = neg, side
    return refs


# ---------------------------------------------------------------- parity with the single-GPU engine
def _parity(eng_mod, kg, world, B, seed, schedule, init, lr):
    """Chained sharded steps against the single-GPU engine on the concatenated global batches, with the optimizer
    schedule[s] at step s (a switch to AdaGrad starts both from fresh accumulators = init)."""
    vr = _VirtualRanks(eng_mod, kg, world, B)
    e = _single(eng_mod, kg, opt="sgd")
    N, dim = kg.n_rows, kg.dim
    bandE, bandA = np.zeros((N, dim)), np.zeros((N, dim))
    used = np.zeros(N, bool)
    opt, worst = "sgd", 0.0
    for s, want_opt in enumerate(schedule):
        if want_opt != opt:
            vr.set_optimizer(want_opt, init)
            e.set_optimizer(want_opt, init)
            bandA[:] = 0.0
            used[:] = False
            opt = want_opt
        gb = kg.triples[s * world * B:(s + 1) * world * B]
        E0 = e.embeddings().cpu().numpy()
        A0 = e.accumulator().cpu().numpy() if opt == "adagrad" else None
        losses = vr.step(_slices(gb, world, e.device), seed, s, MARGIN, lr)
        side, neg = e.corrupt_batch(gb, seed, s)
        want = e.train_step(gb, neg, side, MARGIN, lr).cpu().numpy().reshape(world, B)
        for k in range(world):
            assert np.abs(losses[k].cpu().numpy() - want[k]).max() <= LOSS_ATOL
        neg_h = neg.cpu().numpy()
        Es = e.embeddings().cpu().numpy()
        if opt == "adagrad":
            ref = _ref(E0, A0, gb, neg_h, side, MARGIN, _f32(lr), kg.n_relations, world)
            rows = ref["rows"]
            bandE[rows] += ref["tolE"]
            bandA[rows] += ref["tolA"]
        else:
            rows = np.unique(np.concatenate([gb.ravel(), neg_h]).astype(np.int64))
            bandE[rows] += ROW_ATOL + ROW_RTOL * np.abs(Es[rows])
        used[rows] = True
        Eg = vr.table()
        r = np.abs(Eg - Es) / np.maximum(bandE, 1e-300)
        assert (np.abs(Eg - Es) <= bandE).all(), (s, "E", float(r.max()))
        worst = max(worst, float(r.max()))
        if opt == "adagrad":
            Ag, As = vr.accumulator(), e.accumulator().cpu().numpy()
            assert (np.abs(Ag - As) <= bandA).all(), (s, "A", float((np.abs(Ag - As) / np.maximum(bandA, 1e-300)).max()))
            assert (Ag[~used] == np.float32(init)).all()                 # untouched: exactly the initial value
    moved = float(np.abs(Es - kg.E).max())
    vr.close()
    e.close()
    return worst, moved


@pytest.mark.parametrize("regime", list(REGIMES))
@pytest.mark.parametrize("world,dim,B", [(1, 150, 300), (2, 256, 257), (3, 150, 129), (4, 64, 200), (8, 150, 65)])
def test_parity_with_single_gpu_adagrad(eng_mod, world, dim, B, regime):
    """Three chained AdaGrad steps of `world` virtual ranks against HoleEngine.set_optimizer("adagrad") on the
    concatenated global batch: Zipf entities (rows listed by several ranks), ragged B, trained-scale rows, both
    corruption sides over the steps."""
    init, lr = REGIMES[regime]
    kg = D.synthetic_kg(7, 2000, 3 * world * B, 5, dim, seed=900 + world, trained_scale=True, zipf_entities=True)
    worst, moved = _parity(eng_mod, kg, world, B, _two_sided_seed(3), ["adagrad"] * 3, init, lr)
    print(f"world {world} {regime}: worst |sharded - single| / band = {worst:.2e}")
    assert moved > 1e-4


def test_mixed_optimizers_in_one_sequence_match_the_single_gpu_engine(eng_mod):
    kg = D.synthetic_kg(7, 2000, 5 * 2 * 150, 5, 128, seed=31, trained_scale=True, zipf_entities=True)
    _parity(eng_mod, kg, 2, 150, 5, ["sgd", "adagrad", "adagrad", "sgd", "adagrad"], 0.2, 0.1)


# ---------------------------------------------------------------- against the fp64 reference
@pytest.mark.parametrize("world,regime", [(2, "default"), (3, "default"), (8, "default"), (3, "large"),
                                          (3, "small")])
def test_steps_against_the_fp64_reference(eng_mod, world, regime):
    """Every step re-synchronised from the shards' state against adagrad_reference: DESIGN 7c's band in the default
    regime (A0 = 0.1), the sharded tree band in the two extreme ones."""
    B = 160
    init, lr = REGIMES.get(regime, (INIT, 0.2))
    kg = D.synthetic_kg(6, 1500, 4 * world * B, 4, 150, seed=40 + world, trained_scale=True, zipf_entities=True)
    vr = _VirtualRanks(eng_mod, kg, world, B).set_optimizer("adagrad", init)
    gbs = [kg.triples[s * world * B:(s + 1) * world * B] for s in range(4)]
    refs = _run_checked(vr, kg, gbs, _two_sided_seed(4, 17), lr, flat=regime == "default")
    assert {r["side"] for r in refs} == {0, 1}
    vr.close()


@pytest.mark.parametrize("dim", DIMS)
def test_every_lane_group(eng_mod, dim):
    """Every hole_shard_adagrad_apply_kernel<GS, V> instantiation (masked and full dims), 2 or 3 ranks, ragged B."""
    world = 2 + DIMS.index(dim) % 2
    B = 61 + 2 * DIMS.index(dim)
    kg = D.synthetic_kg(7, 2000, 3 * world * B, 5, dim, seed=700 + dim, trained_scale=True, zipf_entities=True)
    vr = _VirtualRanks(eng_mod, kg, world, B).set_optimizer("adagrad", INIT)
    gbs = [kg.triples[s * world * B:(s + 1) * world * B] for s in range(3)]
    _run_checked(vr, kg, gbs, dim, 0.3)
    assert np.abs(vr.table() - kg.E).max() > 1e-4
    vr.close()


# ---------------------------------------------------------------- edges
def test_one_hot_row_listed_by_all_eight_ranks(eng_mod):
    world, B = 8, 40
    kg = D.synthetic_kg(5, 800, 2 * world * B, 4, 64, seed=12, trained_scale=True, zipf_entities=True)
    hot = kg.n_relations + 333
    kg.triples[::B // 4, 0] = hot                   # four uses in every slice of both steps
    vr = _VirtualRanks(eng_mod, kg, world, B).set_optimizer("adagrad", INIT)
    gbs = [kg.triples[s * world * B:(s + 1) * world * B] for s in range(2)]
    refs = _run_checked(vr, kg, gbs, 3, 0.3)
    for gb in gbs:
        assert all((gb[k * B:(k + 1) * B, 0] == hot).any() for k in range(world))
    assert all(hot in r["rows"] for r in refs)
    vr.close()


def test_a_row_listed_only_by_a_higher_rank(eng_mod):
    """A row of rank 0's block that only rank 2's slice lists: the claim word's lowest set bit is 2."""
    world, B = 3, 100
    kg = D.synthetic_kg(5, 900, world * B, 4, 130, seed=13, trained_scale=True, zipf_entities=True)
    off, ids = D.build_type_csr(kg.type_of)
    from graphembeddings_b200.sharded import row_partition
    rows_per = row_partition(kg.n_entities, world)
    unused = np.setdiff1d(np.arange(kg.n_relations, kg.n_relations + rows_per), kg.triples[:, :2].ravel())
    for x in unused:
        gb = kg.triples.copy()
        gb[2 * B + 5, 1] = x
        _, neg = O.corrupt(gb, kg.type_of, off, ids, 4, 0)
        listed = [x in np.concatenate([gb[k * B:(k + 1) * B, :2].ravel(), neg[k * B:(k + 1) * B]]) for k in range(world)]
        if listed == [False, False, True]:
            break
    else:
        pytest.fail("no candidate row")
    kg.triples[:] = gb
    vr = _VirtualRanks(eng_mod, kg, world, B).set_optimizer("adagrad", INIT)
    ref = _run_checked(vr, kg, [gb], 4, 0.3)[0]
    assert x in ref["rows"]
    vr.close()


def test_trailing_ranks_that_own_no_rows(eng_mod):
    """20 entities over 16 ranks: ranks 10-15 own nothing, their accumulator shards hold relation rows only, and most
    slices list nothing of most owners."""
    world, B = 16, 3
    kg = D.synthetic_kg(7, 20, 3 * world * B, 3, 150, seed=36, trained_scale=True, zipf_entities=True)
    vr = _VirtualRanks(eng_mod, kg, world, B).set_optimizer("adagrad", INIT)
    assert vr.rows_per * 10 == 20
    gbs = [kg.triples[s * world * B:(s + 1) * world * B] for s in range(3)]
    _run_checked(vr, kg, gbs, 5, 0.3)
    for k in range(10, world):                      # the unused rows of an empty block keep the initial value
        assert torch.all(vr.accums[k][vr.R:] == INIT)
    vr.close()


def test_an_empty_call_changes_nothing(eng_mod):
    kg = D.synthetic_kg(5, 300, 4 * 64, 4, 64, seed=3, trained_scale=True)
    vr = _VirtualRanks(eng_mod, kg, 1, 64).set_optimizer("adagrad", INIT)
    e = vr.engs[0]
    tri = torch.from_numpy(kg.triples).to(e.device)
    e.shard_steps(tri[:2 * 64], 64, 1, 0, MARGIN, [0.2, 0.2])
    t0, a0 = vr.bufs[0][0].clone(), vr.accums[0].clone()
    empty = tri[:0]
    sums = e.shard_steps(empty, 64, 1, 2, MARGIN, [0.2])
    hs = e.shard_steps_host(np.zeros((0, 3), np.int32), 64, 1, 2, MARGIN, [0.2])
    torch.cuda.synchronize()
    assert sums.numel() == 0 and hs.size == 0
    assert torch.equal(vr.bufs[0][0], t0) and torch.equal(vr.accums[0], a0)
    vr.close()


def test_one_row_three_times_in_a_triple(eng_mod):
    """A type of one entity: (x, x, r) corrupted to x again uses row x three times in one triple."""
    rng = np.random.default_rng(5)
    Rn, P, dim, B, world = 4, 600, 130, 350, 2
    N = Rn + P + 1
    solo = N - 1
    type_of = np.array([0] * Rn + [1] * P + [2], np.int32)
    pos = np.stack([Rn + rng.integers(0, P, 2 * B), Rn + rng.integers(0, P, 2 * B), rng.integers(0, Rn, 2 * B)], 1)
    pos[::7, :2] = solo
    E = D.init_embeddings(N, dim, rng, trained_scale=True)
    kg = D.SyntheticKG(Rn, P + 1, dim, pos.astype(np.int32), type_of, E)
    vr = _VirtualRanks(eng_mod, kg, world, B).set_optimizer("adagrad", INIT)
    refs = _run_checked(vr, kg, [kg.triples, kg.triples], 8, 0.3)
    assert all((r["neg"][::7] == solo).all() for r in refs)
    vr.close()


# ---------------------------------------------------------------- multi-step entries
def test_multi_step_calls_equal_per_step_calls(eng_mod):
    """hole_shard_steps and hole_shard_steps_host under AdaGrad == hole_shard_step per step, bit for bit in the
    table and the accumulator, over 70 steps (SHARD_PREP_STEPS = 16 and SHARD_LOSS_CHUNK = 64 boundaries); two
    identical runs are bit-identical."""
    B, steps, dim = 50, 70, 66
    kg = D.synthetic_kg(7, 3000, steps * B, 5, dim, seed=62, trained_scale=True, zipf_entities=True)
    lrs = [0.3 / (1 + 0.02 * s) for s in range(steps)]
    runs = [_VirtualRanks(eng_mod, kg, 1, B).set_optimizer("adagrad", INIT) for _ in range(4)]
    tri = torch.from_numpy(kg.triples).to(runs[0].engs[0].device)
    sums = [runs[i].engs[0].shard_steps(tri, B, 3, 10, MARGIN, lrs).cpu().numpy() for i in (0, 1)]
    hs = runs[2].engs[0].shard_steps_host(kg.triples, B, 3, 10, MARGIN, lrs)
    want = []
    for s in range(steps):
        loss = runs[3].step([tri[s * B:(s + 1) * B]], 3, 10 + s, MARGIN, lrs[s])[0]
        want.append(float(loss.double().sum()))
    assert np.abs(sums[0] - np.array(want)).max() <= 1e-3
    assert np.array_equal(sums[0], sums[1]) and np.array_equal(hs, sums[0])
    ref = runs[3].state()
    for vr in runs[:3]:
        E, A = vr.state()
        assert np.array_equal(_bits(E), _bits(ref[0])) and np.array_equal(_bits(A), _bits(ref[1]))
    assert not np.array_equal(ref[1], np.full_like(ref[1], INIT))
    for vr in runs:
        vr.close()


# ---------------------------------------------------------------- switching and refusals
def test_sgd_adagrad_sgd_on_one_shard_context(eng_mod):
    """After switching back to SGD the steps are bit for bit those of a shard context that never used AdaGrad."""
    world, B = 2, 120
    kg = D.synthetic_kg(6, 1500, 6 * world * B, 4, 128, seed=9, trained_scale=True, zipf_entities=True)
    dev = torch.device("cuda", 0)
    gbs = [kg.triples[s * world * B:(s + 1) * world * B] for s in range(6)]
    a = _VirtualRanks(eng_mod, kg, world, B)
    for s, opt in enumerate(["sgd", "sgd", "adagrad", "adagrad", "sgd", "sgd"]):
        if s in (2, 4):
            a.set_optimizer(opt, 0.2)
        if s == 4:
            mid = a.table()
            b = _VirtualRanks(eng_mod, kg, world, B, E=mid)
        a.step(_slices(gbs[s], world, dev), 4, s, MARGIN, 0.1)
        if s >= 4:
            b.step(_slices(gbs[s], world, dev), 4, s, MARGIN, 0.1)
    assert np.array_equal(_bits(a.table()), _bits(b.table()))
    assert not np.array_equal(a.table(), mid)
    a.close()
    b.close()


def test_refusals_write_nothing_and_leave_the_context_usable(eng_mod):
    world, B = 2, 100
    kg = D.synthetic_kg(5, 600, 4 * world * B, 4, 64, seed=6, trained_scale=True, zipf_entities=True)
    fresh = eng_mod.HoleEngine(kg.n_rows, kg.dim)
    acc = torch.full((kg.n_rows, fresh.row_stride), INIT, device=fresh.device)
    for opt, a in (("adagrad", acc), ("sgd", None)):            # before hole_shard_init
        with pytest.raises(_lib.HoleError, match="error -1"):
            fresh.shard_set_optimizer(opt, a)
    fresh.close()
    vr = _VirtualRanks(eng_mod, kg, world, B).set_optimizer("adagrad", INIT)
    gbs = [kg.triples[s * world * B:(s + 1) * world * B] for s in range(2)]
    _run_checked(vr, kg, gbs[:1], 2, 0.3)
    e = vr.engs[0]
    snap = [(b[0].clone(), a.clone()) for b, a in zip(vr.bufs, vr.accums)]
    torch.cuda.synchronize()
    n0 = e.launch_count()
    ptr = C.c_void_p(vr.accums[0].data_ptr())
    for opt, p in ((_lib.HOLE_OPT_ADAGRAD, None), (_lib.HOLE_OPT_SGD, ptr), (2, ptr), (-1, None)):
        with pytest.raises(_lib.HoleError, match="error -1"):
            _lib.check(e.lib.hole_shard_set_optimizer(e._ctx, opt, p))
    with pytest.raises(_lib.HoleError, match="error -4"):       # the context's own optimizer stays SGD
        e.set_optimizer("adagrad")
    torch.cuda.synchronize()
    assert e.launch_count() == n0
    for (t, a), b, acc_k in zip(snap, vr.bufs, vr.accums):
        assert torch.equal(b[0], t) and torch.equal(acc_k, a)
    # still AdaGrad, and still training correctly
    _run_checked(vr, kg, gbs[1:], 2, 0.3, first_step=1)
    vr.close()


# ---------------------------------------------------------------- the trainer at world 1
def test_world1_trainer_matches_the_single_gpu_engine_and_round_trips_the_checkpoint_slot(eng_mod, tmp_path):
    from graphembeddings_b200 import hole, tf_bundle
    from graphembeddings_b200.sharded import CudaBackend, P2PRowShardedTrainer
    B, steps, dim = 256, 6, 150
    kg = D.synthetic_kg(6, 2500, steps * B, 4, dim, seed=77, trained_scale=True, zipf_entities=True)
    off, ids = D.build_type_csr(kg.type_of)
    A = np.random.default_rng(1).uniform(0.05, 1.0, size=kg.E.shape).astype(np.float32)
    lrs = [0.3 / (1 + 0.1 * s) for s in range(steps)]
    be = CudaBackend(kg.n_relations, dim, B, 0, kg.type_of, off, ids)
    tr = P2PRowShardedTrainer(kg.n_relations, kg.n_entities, dim, be, None).load_embeddings(kg.E)
    tr.set_optimizer("adagrad", 0.25).load_accumulator(A)
    assert np.array_equal(tr.gather_accumulator().cpu().numpy(), A)
    half, H = be.width // 2, dim // 2
    assert torch.all(tr.accum[:, H:half] == 0.25) and torch.all(tr.accum[:, half + H:] == 0.25)
    tri = torch.from_numpy(kg.triples).cuda()
    tr.train_steps(tri[:3 * B], B, 5, 0, MARGIN, lrs[:3])
    for s in range(3, steps):
        tr.train_step(tri[s * B:(s + 1) * B], 5, s, MARGIN, lrs[s])
    E1, A1 = tr.gather_embeddings().cpu().numpy(), tr.gather_accumulator().cpu().numpy()
    e = _single(eng_mod, kg, opt="adagrad", init=0.25).set_accumulator(A)
    e.train_steps(kg.triples, B, 5, 0, MARGIN, lrs)
    Es, As = e.embeddings().cpu().numpy(), e.accumulator().cpu().numpy()
    assert np.all(np.abs(E1 - Es) <= steps * (ROW_ATOL + ROW_RTOL * np.abs(Es)))
    assert np.all(np.abs(A1 - As) <= steps * (ACC_ATOL + ACC_RTOL * np.abs(As)))
    assert np.abs(Es - kg.E).max() > 1e-4 and not np.array_equal(A1, A)
    prefix = str(tmp_path / "model.ckpt")
    tf_bundle.save_bundle(prefix, {"embeddings": E1, hole.ADAGRAD_SLOT: A1})
    b = tf_bundle.load_bundle(prefix)
    assert np.array_equal(b[hole.ADAGRAD_SLOT], A1)
    tr.set_optimizer("adagrad", 0.25).load_accumulator(b[hole.ADAGRAD_SLOT])
    assert np.array_equal(tr.gather_accumulator().cpu().numpy(), A1)
    tr.set_optimizer("sgd")
    assert tr.accum is None
    with pytest.raises(_lib.HoleError, match="not adagrad"):
        tr.gather_accumulator()
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
def test_real_peers_match_single_gpu_adagrad(world):
    if not torch.cuda.is_available() or torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    from graphembeddings_b200 import build
    build.build()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           os.path.join(ROOT, "tools", "multi_gpu_adagrad_check.py")]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    tail = (r.stdout + r.stderr)[-3000:]
    assert r.returncode == 0, tail
    assert "MULTI_GPU_ADAGRAD_CHECK OK" in r.stdout, tail
