"""AdaGrad (hole_ctx_set_optimizer) through the combine tree at every depth and lane group, and through every
multi-step chunking path.

The AdaGrad step is K1 in DM 4 (a row used once) and hole_adagrad_apply_kernel<GS, V> (K3: the combine tree of a
row used more than once, whose root applies S += acc^2; E -= lr acc rsqrt(S) and stores S).  Every step below is
held, re-synchronised from the device's own table and accumulator before it, to the fp64 statement
(tests/adagrad_reference.py) within adagrad_reference.tree_tolerance: the band of the fp32 tree sum of each row's
per-use gradients at that row's tree depth, carried through the AdaGrad update.  A relation row's depth counts one
level more than its triple count gives: K1 first sums a relation's gradient over its run of up to T <= 32
triples (hole_k1.cuh) before K3 combines the runs.  Rows and accumulator elements the step does not use keep
their bits.  This file checks:
  1. one hot row at both sides of every depth edge (1 .. 32769 uses) under the three plan sorts, in both
     accumulator regimes (A0 >> g^2: SGD at lr / sqrt(A0); A0 << g^2: a step of ~lr sign(g)), and that dropping
     any one of its leaves would leave the tolerance;
  2. three- and four-level trees at every K1 lane group, for both optimizers (hole_apply_kernel and
     hole_adagrad_apply_kernel at all ten (GS, V, full) forms);
  3. the tree's counters over three consecutive four-level steps of one call;
  4. the multi-step calls (test_gpu_chunked's layouts, the adaptive plan sort, the large-B natural layouts, the
     relation-count hint) bit for bit against the per-step path, and at every chunk boundary against fp64;
  5. ragged and empty batches, three uses of one row in one triple, and optimizer switches inside a sequence.
The CPU tests at the top pin the tolerance on a simulated fp32 tree and keep the parametrizations covering every
lane-group form, depth edge, accumulator regime and chunk layout."""
import numpy as np
import pytest
import torch

import adagrad_reference as R
from graphembeddings_b200 import data as D
from oracle import hole_oracle as O
from test_gpu_chunked import SS_CAP, SUM_ATOL, VARIANTS, _lrs, _set_env, boundary_steps, chunk_sizes
from test_gpu_shapes import lane_group, regimes
from test_gpu_update_paths import (DIMS, HOLE_TREE_C, TREE_EDGES, _params, _tree_kg, _unpack, _uses,
                                   tree_depth)

LOSS_ATOL = 2e-6
MARGIN, HOT_MARGIN, LR, INIT = 0.2, 1.0, 0.1, 0.1      # HOT_MARGIN 1: every hinge of a hot-row batch is active
ACC_REGIMES = ["large", "small"]       # A0 = 1e3 max G^2 with lr = LR sqrt(A0)  /  A0 = 1e-6 with lr = LR
CAPS = np.array([HOLE_TREE_C**k for k in range(7)], np.int64)


def depth_of(counts):
    """tree_depth of every element of an array of use counts."""
    return np.searchsorted(CAPS, np.asarray(counts, np.int64), side="left")


# ---------------------------------------------------------------- A. the tolerance, on a simulated fp32 tree
def _fp32_tree_sum(g32):
    """The K3 tree on fp32 per-use gradients [n, D]: leaves are chunks of HOLE_TREE_C consecutive uses, every level
    sums up to HOLE_TREE_C nodes in order into a zeroed fp32 accumulator.  A single use is K1's row as it is."""
    x = g32
    while len(x) > 1:
        m = -(-len(x) // HOLE_TREE_C)
        pad = np.zeros((m * HOLE_TREE_C, x.shape[1]), np.float32)
        pad[:len(x)] = x
        pad = pad.reshape(m, HOLE_TREE_C, -1)
        acc = np.zeros((m, x.shape[1]), np.float32)
        for q in range(HOLE_TREE_C):
            acc = acc + pad[:, q]
        x = acc
    return x[0]


def _fp32_adagrad(x, A0, acc, lr):
    """The root's fp32 update: S = fma(acc, acc, A0); E = fma(-lr acc, rsqrt_rn(S), x)."""
    S = (A0.astype(np.float64) + acc.astype(np.float64)**2).astype(np.float32)
    r = (1.0 / np.sqrt(S.astype(np.float64))).astype(np.float32)
    E = ((-np.float32(lr) * acc).astype(np.float64) * r + x).astype(np.float32)
    return E, S


def _gradient_set(kind, n, D, rng):
    mag = rng.uniform(0.5, 1.5, (n, D))
    if kind == "random":
        return mag * rng.choice([-1.0, 1.0], (n, D))
    if kind == "same_sign":
        return mag
    h = n // 2                                  # "cancel": pairs +-g, plus one unpaired leaf when n is odd
    return np.concatenate([mag[:h], -mag[:h][rng.permutation(h)], mag[2 * h:]])


@pytest.mark.parametrize("regime", ACC_REGIMES)
@pytest.mark.parametrize("kind", ["random", "same_sign", "cancel"])
@pytest.mark.parametrize("n", [1, 32, 1024, 32768, 32769])
def test_tree_tolerance_on_a_simulated_fp32_tree(n, kind, regime):
    """The fp32 tree and update lie inside tree_tolerance of fp64, with every per-use gradient 0.9e-6 too large
    (the same sign for all: the worst case of the 1e-6 term); dropping or doubling any one leaf leaves it.  The
    accumulator shows every such leaf, except in the large-A0 regime with 32768 uses of one sign: there one leaf
    changes S by 2 G g ~ 2 A0 / (1e3 n), below S's own fp32 resolution, and the row shows it instead."""
    rng = np.random.default_rng(n + len(kind))
    Dm = 64
    g = _gradient_set(kind, n, Dm, rng)
    depth = tree_depth(n)
    G, absg = g.sum(0), np.abs(g).sum(0)
    x = rng.uniform(-1, 1, Dm).astype(np.float32)
    if regime == "large":
        A0 = np.float32(1e3 * max((G**2).max(), (g**2).max()))
        lr = np.float32(LR * np.sqrt(A0))
    else:
        A0, lr = np.float32(1e-6), np.float32(LR)
    A0v = np.full(Dm, A0, np.float32)
    E, S = _fp32_adagrad(x, A0v, _fp32_tree_sum((g * (1 + 9e-7)).astype(np.float32)), lr)
    A_ref = A0v.astype(np.float64) + G**2
    E_ref = x - float(lr) * G / np.sqrt(A_ref)
    tolE, tolA = R.tree_tolerance(G, absg, depth, A0v, float(lr), E_ref)
    assert (np.abs(E - E_ref) <= tolE).all(), float((np.abs(E - E_ref) / tolE).max())
    assert (np.abs(S - A_ref) <= tolA).all(), float((np.abs(S - A_ref) / tolA).max())
    for sgn in (-1.0, 1.0):                     # each leaf dropped / doubled
        Gp = G[None] + sgn * g
        if not (regime == "large" and kind == "same_sign" and depth >= 3):
            assert (np.abs(Gp**2 - G**2) / tolA).max(axis=1).min() > 1.0
        if regime == "large":
            Ep = x - float(lr) * Gp / np.sqrt(A0v + Gp**2)
            assert (np.abs(Ep - E_ref) / tolE).max(axis=1).min() > 1.0


# ---------------------------------------------------------------- coverage
def test_adagrad_path_coverage():
    """B.2 runs every (GS, V, full) form with both optimizers at three- and four-level trees; B.1 reaches both
    sides of every depth edge in both accumulator regimes; B.4 runs every chunk layout of test_gpu_chunked."""
    forms = {r[2] for r in regimes(lane_group) if r[2] is not None}
    assert len(forms) == 10
    lanes = {(lane_group(d), o) for d in _params(test_deep_trees_every_lane_group, "dim")
             for o in _params(test_deep_trees_every_lane_group, "optimizer")}
    assert lanes == {(f, o) for f in forms for o in ("sgd", "adagrad")}
    assert {tree_depth(n) for n in _params(test_deep_trees_every_lane_group, "n")} == {3, 4}
    assert [int(d) for d in depth_of(TREE_EDGES)] == [tree_depth(n) for n in TREE_EDGES]
    edges = _params(test_adagrad_tree_depth_edges, "n")
    for d in range(1, 5):
        assert max(n for n in range(1, 40000) if tree_depth(n) == d - 1) in edges
        assert min(n for n in range(1, 40000) if tree_depth(n) == d) in edges
    assert set(_params(test_adagrad_tree_depth_edges, "regime")) == set(ACC_REGIMES) == {"large", "small"}
    assert set(_params(test_tree_tolerance_on_a_simulated_fp32_tree, "regime")) == set(ACC_REGIMES)
    assert tree_depth(max(_params(test_adagrad_tree_counters_over_steps, "n"))) == 4
    got = _params(test_adagrad_ramped_chunks_and_host_path, "variant")
    assert sorted(map(repr, got)) == sorted(map(repr, VARIANTS))


# ---------------------------------------------------------------- GPU helpers
@pytest.fixture(scope="module")
def eng_mod():
    from graphembeddings_b200 import build
    build.build()
    from graphembeddings_b200 import engine
    return engine


def _engine(eng_mod, monkeypatch, kg, csr=None, A0=INIT, hint=None, env=None, optimizer="adagrad"):
    """A context created under exactly `env` (the switches are read by hole_ctx_create), AdaGrad with every
    accumulator element A0 unless optimizer == "sgd"."""
    _set_env(monkeypatch, env)
    off, ids = D.build_type_csr(kg.type_of) if csr is None else csr
    e = eng_mod.HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E).set_types(kg.type_of, off, ids)
    if hint is not None:
        e.set_relation_count(hint)
    _set_env(monkeypatch, None)
    if optimizer == "adagrad":
        e.set_optimizer("adagrad", A0)
    return e


def _state(e):
    return e.embeddings().cpu().numpy(), e.accumulator().cpu().numpy()


def _bits(x):
    return np.ascontiguousarray(x).view(np.uint32)


def _row_sums(slices, n_rows):
    """(rows, G, absg): every used row, its fp64 summed gradient and the sum of |g| over its per-use gradients."""
    dim = slices[0][1].shape[1]
    G, absg, used = np.zeros((n_rows, dim)), np.zeros((n_rows, dim)), np.zeros(n_rows, bool)
    for i, g in slices:
        o = np.argsort(i, kind="stable")
        u, start = np.unique(i[o], return_index=True)
        G[u] += np.add.reduceat(g[o], start, axis=0)
        absg[u] += np.add.reduceat(np.abs(g[o]), start, axis=0)
        used[u] = True
    rows = np.flatnonzero(used)
    return rows, G[rows], absg[rows]


def _row_depths(pos, neg, n_rows, n_relations):
    """Tree depth of every row: entity rows from their key count, relation rows one more than their triple count
    gives (K1 sums a relation over its run of up to T triples first)."""
    d = depth_of(_uses(pos, neg, n_rows))
    rel = np.bincount(pos[:, 2].astype(np.int64), minlength=n_rows)[:n_relations]
    d[:n_relations] = depth_of(rel) + (rel > 1)
    return d


def _ref(E0, A0, pos, neg, side, margin, lr, n_relations):
    """The fp64 AdaGrad step from (E0, A0) on the rows it uses, with the tree tolerance of each."""
    E64 = E0.astype(np.float64)
    slices, loss, _, _ = O.indexed_slices(E64, pos, neg, side, margin, np.float64)
    slices = [(i.astype(np.int64), g) for i, g in slices]
    rows, G, absg = _row_sums(slices, len(E0))
    Er, Ar = E64[rows], A0[rows].astype(np.float64)
    R.adagrad_apply(Er, Ar, np.arange(len(rows)), G, lr)
    depth = _row_depths(pos, neg, len(E0), n_relations)[rows]
    tolE, tolA = R.tree_tolerance(G, absg, depth[:, None], A0[rows].astype(np.float64), lr, Er)
    return dict(slices=slices, loss=loss, rows=rows, G=G, E=Er, A=Ar, tolE=tolE, tolA=tolA, depth=depth)


def _check(tag, before, after, pos, neg, side, margin, lr, n_relations, loss=None):
    """The device step before -> after (tables and accumulators in checkpoint layout) against the fp64 step."""
    E0, A0 = before
    E1, A1 = after
    ref = _ref(E0, A0, pos, neg, side, margin, lr, n_relations)
    rows = ref["rows"]
    if loss is not None:
        assert np.abs(loss - ref["loss"]).max() <= LOSS_ATOL, (tag, float(np.abs(loss - ref["loss"]).max()))
    for name, got, want, tol in (("E", E1[rows], ref["E"], ref["tolE"]), ("S", A1[rows], ref["A"], ref["tolA"])):
        r = np.abs(got - want) / tol
        assert (r <= 1.0).all(), (tag, name, float(r.max()), int(rows[np.unravel_index(r.argmax(), r.shape)[0]]))
    keep = np.ones(len(E0), bool)
    keep[rows] = False
    assert np.array_equal(_bits(E1[keep]), _bits(E0[keep])), (tag, "an unused row changed")
    assert np.array_equal(_bits(A1[keep]), _bits(A0[keep])), (tag, "an unused accumulator row changed")
    return ref


def _leaves_visible(ref, hot, n, A0, lr, on_rows):
    """Dropping any one of the hot row's n per-use gradients alone would leave the accumulator's tolerance (and,
    with on_rows, the row's): the tolerance cannot pass a lost or doubled leaf."""
    k = int(np.searchsorted(ref["rows"], hot))
    assert ref["rows"][k] == hot
    g = np.concatenate([g[i == hot] for i, g in ref["slices"]])
    assert len(g) == n
    G = ref["G"][k]
    Gp = G[None] - g
    assert (np.abs(Gp**2 - G**2) / ref["tolA"][k]).max(axis=1).min() > 1.0
    if on_rows:
        dE = lr * (G / np.sqrt(A0 + G**2) - Gp / np.sqrt(A0 + Gp**2))
        assert (np.abs(dE) / ref["tolE"][k]).max(axis=1).min() > 1.0


def _regime(regime, G):
    """(A0, lr) of an accumulator regime, both fp32-representable."""
    if regime == "large":
        A0 = np.float32(1e3 * (G**2).max())
        return float(A0), float(np.float32(LR * np.sqrt(A0)))
    return float(np.float32(1e-6)), float(np.float32(LR))


# ---------------------------------------------------------------- B.1 every depth edge
@pytest.mark.gpu
@pytest.mark.parametrize("regime", ACC_REGIMES)
@pytest.mark.parametrize("n", TREE_EDGES)
def test_adagrad_tree_depth_edges(eng_mod, monkeypatch, n, regime):
    """One hot entity row used exactly n times (test_gpu_update_paths._tree_kg), trained by one AdaGrad step
    under HOLE_SORT_SMALL 0, 1 and 2: bit-identical tables and accumulators; every used row, relation rows
    (~n/3 triples each) included, within the tree tolerance of fp64; the hot row's leaves each visible."""
    step = TREE_EDGES.index(n)
    seed = 40 + step
    kg, csr = _tree_kg(n, 1000 + n)
    hot = kg.n_rows - 1
    pos = kg.triples
    side, neg = O.corrupt(pos, kg.type_of, *csr, seed, step)
    assert (neg == hot).all() and _uses(pos, neg, kg.n_rows)[hot] == n
    slices, _, _, _ = O.indexed_slices(kg.E.astype(np.float64), pos, neg, side, HOT_MARGIN, np.float64)
    _, G, _ = _row_sums([(i.astype(np.int64), g) for i, g in slices], kg.n_rows)
    A0, lr = _regime(regime, G)
    outs = []
    for sort in ("0", "1", "2"):
        e = _engine(eng_mod, monkeypatch, kg, csr, A0=A0, env={"HOLE_SORT_SMALL": sort})
        before = _state(e)
        loss = e.train_step(pos, neg, side, HOT_MARGIN, lr).cpu().numpy()
        outs.append((e.table.clone(), e.accum.clone(), loss, _state(e)))
        e.close()
    for t, a, l, _ in outs[1:]:
        assert torch.equal(t, outs[0][0]) and torch.equal(a, outs[0][1]) and np.array_equal(l, outs[0][2])
    ref = _check(f"n={n} {regime}", before, outs[0][3], pos, neg, side, HOT_MARGIN, lr, kg.n_relations, outs[0][2])
    assert ref["depth"][ref["rows"] == hot][0] == tree_depth(n)
    _leaves_visible(ref, hot, n, A0, lr, on_rows=regime == "large")
    E1, A1 = outs[0][3]
    assert np.abs(E1[hot] - kg.E[hot]).max() > 1e-4 and (A1[hot] > np.float32(A0)).any()


# ---------------------------------------------------------------- B.2 deep trees at every lane group
def _hot_kg(n, dim, seed):
    """_tree_kg at any dim, with relation and pool rows of norms U(0.5, 1.5): the norm clip fires on about half."""
    rng = np.random.default_rng(seed)
    Rn, P = 3, 4096
    N = Rn + P + 1
    pos = np.stack([Rn + rng.integers(0, P, n), Rn + rng.integers(0, P, n), rng.integers(0, Rn, n)], 1)
    type_of = np.array([0] * Rn + [1] * P + [2], np.int32)
    E = rng.standard_normal((N, dim))
    E *= rng.uniform(0.5, 1.5, (N, 1)) / np.linalg.norm(E, axis=1, keepdims=True)
    E[-1] *= 0.05
    kg = D.SyntheticKG(Rn, P + 1, dim, pos.astype(np.int32), type_of, E.astype(np.float32))
    csr = (np.array([0, Rn, Rn + 1, Rn + 2], np.int64), np.array(list(range(Rn)) + [N - 1, N - 1], np.int32))
    return kg, csr


@pytest.mark.gpu
@pytest.mark.parametrize("optimizer", ["sgd", "adagrad"])
@pytest.mark.parametrize("n", [1025, 32769])
@pytest.mark.parametrize("dim", DIMS)
def test_deep_trees_every_lane_group(eng_mod, monkeypatch, dim, n, optimizer):
    """A hot row used n times (a three- or four-level tree) at the first and last dim of every lane group, so
    hole_apply_kernel / hole_adagrad_apply_kernel run at every (GS, V, full) form, at V 2 and 3 with NB = 4 row
    loads in flight and full level-1 nodes.  SGD against O.sgd_step within test_gpu_update_paths' tree band,
    AdaGrad against the fp64 step within tree_tolerance."""
    kg, csr = _hot_kg(n, dim, 2000 + dim + n)
    hot = kg.n_rows - 1
    norms = np.linalg.norm(kg.E[:-1], axis=1)
    assert (norms > 1).any() and (norms < 1).any()
    pos = kg.triples
    side, neg = O.corrupt(pos, kg.type_of, *csr, dim, 0)
    assert (neg == hot).all()
    lr = float(np.float32(LR))
    e = _engine(eng_mod, monkeypatch, kg, csr, A0=0.05, optimizer=optimizer)
    if optimizer == "adagrad":
        before = _state(e)
        loss = e.train_step(pos, neg, side, HOT_MARGIN, lr).cpu().numpy()
        ref = _check(f"dim={dim} n={n}", before, _state(e), pos, neg, side, HOT_MARGIN, lr, kg.n_relations, loss)
        _leaves_visible(ref, hot, n, 0.05, lr, on_rows=False)
    else:
        E0 = kg.E.astype(np.float64)
        loss = e.train_step(pos, neg, side, HOT_MARGIN, lr).cpu().numpy()
        got = e.embeddings().cpu().numpy()
        slices, l64, _, _ = O.indexed_slices(E0, pos, neg, side, HOT_MARGIN, np.float64)
        rows, G, absg = _row_sums([(i.astype(np.int64), g) for i, g in slices], kg.n_rows)
        want = E0[rows] - lr * G
        depth = _row_depths(pos, neg, kg.n_rows, kg.n_relations)[rows]
        tol = 2e-6 + 1e-5 * np.abs(want) + lr * absg * (1e-6 + (31 * depth[:, None] + 1) * 2.0**-24)
        assert np.abs(loss - l64).max() <= LOSS_ATOL
        r = np.abs(got[rows] - want) / tol
        assert (r <= 1).all(), float(r.max())
        g_hot = np.concatenate([g[i == hot] for i, g in slices])
        k = int(np.searchsorted(rows, hot))
        assert (lr * np.abs(g_hot) / tol[k]).max(axis=1).min() > 1.0
        keep = np.ones(kg.n_rows, bool)
        keep[rows] = False
        assert np.array_equal(_bits(got[keep]), _bits(kg.E[keep]))
    assert tree_depth(_uses(pos, neg, kg.n_rows)[hot]) == tree_depth(n)
    e.close()


# ---------------------------------------------------------------- B.3 counters over steps
@pytest.mark.gpu
@pytest.mark.parametrize("n", [32769])
def test_adagrad_tree_counters_over_steps(eng_mod, monkeypatch, n):
    """Three consecutive four-level AdaGrad steps in one train_steps call: the tree's ticket counters must reset
    themselves for the next step (a stale counter freezes the row, a stale S shows in the next step).  The call
    equals the per-step path bit for bit (table, accumulator, per-triple losses), and every per-step step is
    within the tree tolerance of the fp64 step re-run from the device's state before it."""
    steps, seed, first = 3, 12, 5
    kg, csr = _tree_kg(steps * n, 77)
    hot = kg.n_rows - 1
    lrs = np.array([eng_mod.inverse_time_decay(0.1, first + k, 2, 0.5) for k in range(steps)], np.float32)
    a = _engine(eng_mod, monkeypatch, kg, csr, A0=0.01)
    sums, loss_a = a.train_steps(torch.from_numpy(kg.triples).to(a.device), n, seed, first, HOT_MARGIN, lrs,
                                 want_loss=True)
    b = _engine(eng_mod, monkeypatch, kg, csr, A0=0.01)
    losses = []
    for k in range(steps):
        pos = kg.triples[k * n:(k + 1) * n]
        side, neg = b.corrupt_batch(pos, seed, first + k)
        neg = neg.cpu().numpy()
        before = _state(b)
        losses.append(b.train_step(pos, neg, side, HOT_MARGIN, lrs[k]))
        ref = _check(f"step {k}", before, _state(b), pos, neg, side, HOT_MARGIN, float(lrs[k]), kg.n_relations,
                     losses[-1].cpu().numpy())
        _leaves_visible(ref, hot, n, before[1][hot].astype(np.float64), float(lrs[k]), on_rows=False)
    assert torch.equal(a.table, b.table) and torch.equal(a.accum, b.accum)
    assert torch.equal(loss_a, torch.cat(losses))
    # a sum of 32769 losses near 1 is ~3.3e4, where one fp32 ulp is 2^-8: a relative band on top of SUM_ATOL
    want = loss_a.double().view(steps, n).sum(1).cpu().numpy()
    assert (np.abs(sums.cpu().numpy() - want) <= SUM_ATOL + 1e-6 * np.abs(want)).all()
    a.close(); b.close()


# ---------------------------------------------------------------- B.4 the chunking paths
def _per_step(e, tri, B, seed, first_step, lrs, n_relations, check_at=(), margin=MARGIN, sub_table=False):
    """The per-step AdaGrad path; at the steps in check_at the step is held to the fp64 step re-run from this
    engine's state (on the touched rows alone with sub_table).  Returns the per-triple losses."""
    n = len(tri) // B
    losses, check_at = [], set(check_at)
    for k in range(n):
        pos = tri[k * B:(k + 1) * B]
        side, neg = e.corrupt_batch(pos, seed, first_step + k)
        if k not in check_at:
            losses.append(e.train_step(pos, neg, side, margin, lrs[k]))
            continue
        pos_h, neg_h = pos.cpu().numpy() if isinstance(pos, torch.Tensor) else pos, neg.cpu().numpy()
        if sub_table:
            _check_touched(e, pos_h, neg_h, side, margin, float(lrs[k]), n_relations, losses)
            continue
        before = _state(e)
        losses.append(e.train_step(pos, neg, side, margin, lrs[k]))
        _check(f"step {first_step + k}", before, _state(e), pos_h, neg_h, side, margin, float(lrs[k]), n_relations,
               losses[-1].cpu().numpy())
    return torch.cat(losses)


def _check_touched(e, pos, neg, side, margin, lr, n_relations, losses):
    """One step checked on the rows it touches, re-indexed into a compact table (relations stay first); every
    other row and accumulator element keeps its bits."""
    rows = np.unique(np.concatenate([pos.ravel(), neg, np.arange(n_relations)]))
    assert (rows[:n_relations] == np.arange(n_relations)).all()
    rows_d = torch.from_numpy(rows).to(e.device)
    t0, a0 = e.table.clone(), e.accum.clone()
    before = (_unpack(t0[rows_d].cpu().numpy(), e.dim), _unpack(a0[rows_d].cpu().numpy(), e.dim))
    losses.append(e.train_step(pos, neg, side, margin, lr))
    after = (_unpack(e.table[rows_d].cpu().numpy(), e.dim), _unpack(e.accum[rows_d].cpu().numpy(), e.dim))
    sub = lambda x: np.searchsorted(rows, x).astype(np.int32)
    p = np.stack([sub(pos[:, 0]), sub(pos[:, 1]), pos[:, 2]], 1)
    _check("touched rows", before, after, p, sub(neg), side, margin, lr, n_relations, losses[-1].cpu().numpy())
    mask = torch.ones(e.n_rows, dtype=torch.bool, device=e.device)
    mask[rows_d] = False
    assert torch.equal(e.table[mask], t0[mask]) and torch.equal(e.accum[mask], a0[mask])


def _assert_same(tag, a, b, B, sums, ref_loss, loss=None):
    assert torch.equal(a.table, b.table), f"{tag}: table differs from the per-step path"
    assert torch.equal(a.accum, b.accum), f"{tag}: accumulator differs from the per-step path"
    if loss is not None:
        assert torch.equal(loss, ref_loss), f"{tag}: per-triple losses differ from the per-step path"
    s = sums.cpu().numpy() if isinstance(sums, torch.Tensor) else np.asarray(sums)
    err = np.abs(s - ref_loss.double().view(-1, B).sum(1).cpu().numpy())
    assert err.max() <= SUM_ATOL, (tag, int(err.argmax()), float(err.max()))


@pytest.mark.gpu
@pytest.mark.parametrize("variant", VARIANTS, ids=lambda v: f"{v[0]}-{v[1]}-{v[2]}")
def test_adagrad_ramped_chunks_and_host_path(eng_mod, monkeypatch, variant):
    """test_gpu_chunked's HOLE_PLAN_RAMP / HOLE_HOST_FIRST layouts of 40 steps at B = 1000 under AdaGrad: the
    device entry (with per-triple losses) and the host entry equal the per-step path bit for bit, and the
    per-step path is within the tree tolerance of fp64 on both sides of every chunk boundary."""
    entry, ramp, host_first, layout = variant
    B, n_steps, dim = 1000, 40, 150
    from_host = entry == "host"
    assert chunk_sizes(B, n_steps, ramp, host_first, from_host) == layout
    env = {}
    if ramp:
        env["HOLE_PLAN_RAMP"] = "%d,%d" % ramp
    if host_first:
        env["HOLE_HOST_FIRST"] = host_first
    kg = D.synthetic_kg(9, 20000, n_steps * B, 5, dim, seed=3 + len(layout), trained_scale=True, zipf_entities=True)
    seed, first_step = 77, 333
    lrs = _lrs(eng_mod, first_step, n_steps)
    a = _engine(eng_mod, monkeypatch, kg, env=env, hint=kg.n_relations)
    if from_host:
        sums, loss = a.train_steps_host(kg.triples, B, seed, first_step, MARGIN, lrs), None
    else:
        sums, loss = a.train_steps(kg.triples, B, seed, first_step, MARGIN, lrs, want_loss=True)
    b = _engine(eng_mod, monkeypatch, kg, hint=kg.n_relations)
    ref = _per_step(b, kg.triples, B, seed, first_step, lrs, kg.n_relations, boundary_steps(layout))
    _assert_same(f"{entry} {env}", a, b, B, sums, ref, loss)
    a.close(); b.close()


@pytest.mark.gpu
def test_adagrad_adaptive_plan_sort_switches_inside_a_call(eng_mod, monkeypatch):
    """test_gpu_chunked.test_adaptive_plan_sort_switches_inside_a_call under AdaGrad: the one-launch row sort
    and the radix chain alternate between the chunks of one call (steps [16, 28) have more than SS_CAP duplicated
    row uses); HOLE_SORT_SMALL 0, 1 and 2 give the per-step path's table, accumulator and losses bit for bit."""
    B, dim, n_rel, n_hub, n_spread = 4096, 64, 8, 40, 100000
    warm, n_steps, heavy = 8, 48, range(16, 28)
    layout = chunk_sizes(B, n_steps, (1, 2))
    assert chunk_sizes(B, warm, (1, 2)) == [1, 2, 4, 1] and layout == [1, 2, 4, 8, 16, 17]
    total = warm + n_steps
    rng = np.random.default_rng(12)
    type_of = np.concatenate([np.zeros(n_rel), np.ones(n_hub), np.full(n_spread, 2)]).astype(np.int32)
    hub0, spread0 = n_rel, n_rel + n_hub
    tri = np.empty((total * B, 3), np.int32)
    tri[:, 2] = rng.integers(0, n_rel, total * B)
    for k in range(total):
        lo, hi = (hub0, hub0 + n_hub) if k in heavy else (spread0, spread0 + n_spread)
        tri[k * B:(k + 1) * B, :2] = rng.integers(lo, hi, (B, 2))
    kg = D.SyntheticKG(n_rel, n_hub + n_spread, dim, tri, type_of,
                       D.init_embeddings(len(type_of), dim, rng, trained_scale=True))
    seed, first_step = 2024, 4000
    off, ids = D.build_type_csr(type_of)
    negs = [O.corrupt(tri[k * B:(k + 1) * B], type_of, off, ids, seed, first_step + k)[1] for k in range(total)]
    dups = []
    for k in range(total):
        _, cnt = np.unique(np.concatenate([tri[k * B:(k + 1) * B, 0], tri[k * B:(k + 1) * B, 1], negs[k]]),
                           return_counts=True)
        dups.append(int(cnt[cnt > 1].sum()))
    assert all(dups[k] > SS_CAP for k in heavy)
    assert all(dups[k] + B <= SS_CAP for k in range(total) if k not in heavy)
    lrs = _lrs(eng_mod, first_step, total)
    outs = []
    for mode in ("0", "1", "2"):
        e = _engine(eng_mod, monkeypatch, kg, env={"HOLE_PLAN_RAMP": "1,2", "HOLE_SORT_SMALL": mode})
        t = torch.from_numpy(tri).to(e.device)
        s0, l0 = e.train_steps(t[:warm * B], B, seed, first_step, MARGIN, lrs[:warm], want_loss=True)
        s1, l1 = e.train_steps(t[warm * B:], B, seed, first_step + warm, MARGIN, lrs[warm:], want_loss=True)
        outs.append((mode, e, torch.cat([s0, s1]), torch.cat([l0, l1])))
    b = _engine(eng_mod, monkeypatch, kg)
    check = sorted({0, warm - 1} | {warm + k for k in boundary_steps(layout)} | {15, 16, 27, 28})
    ref = _per_step(b, torch.from_numpy(tri).to(b.device), B, seed, first_step, lrs, n_rel, check)
    for mode, e, sums, loss in outs:
        _assert_same(f"HOLE_SORT_SMALL={mode}", e, b, B, sums, ref, loss)
        assert torch.equal(sums, outs[0][2])
        e.close()
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("B,dim,n_steps,n_ent,layout", [
    (16384, 64, 300, 50000, [128, 128, 44]),
    (32768, 256, 140, 200000, [64, 64, 12]),
])
def test_adagrad_natural_chunks_at_large_batches(eng_mod, monkeypatch, B, dim, n_steps, n_ent, layout):
    """hole_train_steps over three natural plan chunks at B = 16384 and 32768 (Zipf entities: rows used thousands
    of times a step) under AdaGrad: bit for bit the per-step path, loss sums within SUM_ATOL of the fp64 sums of
    its losses, and the boundary steps within the tree tolerance of fp64 on the touched rows."""
    assert chunk_sizes(B, n_steps) == layout
    kg = D.synthetic_kg(14, n_ent, n_steps * B, 6, dim, seed=B + dim, trained_scale=True, zipf_entities=True)
    seed, first_step = 0x5EED + B, 1000 + B
    lrs = _lrs(eng_mod, first_step, n_steps)
    a = _engine(eng_mod, monkeypatch, kg, hint=kg.n_relations)
    tri = torch.from_numpy(kg.triples).to(a.device)
    sums, loss = a.train_steps(tri, B, seed, first_step, MARGIN, lrs, want_loss=True)
    b = _engine(eng_mod, monkeypatch, kg, hint=kg.n_relations)
    ref = _per_step(b, tri, B, seed, first_step, lrs, kg.n_relations, boundary_steps(layout), sub_table=True)
    _assert_same(f"B={B}", a, b, B, sums, ref, loss)
    assert not torch.equal(a.accum, torch.full_like(a.accum, INIT))
    a.close(); b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("sort_small", ["0", "1"])
@pytest.mark.parametrize("hint", [None, 4, 200, 300])
def test_adagrad_relation_ids_and_the_hint(eng_mod, monkeypatch, hint, sort_small):
    """300 relations (ids above 255 in every batch) with no relation-count hint (the hint-less relation radix
    chain) and with hints of 4, 200 (relation ids above it) and 300, under HOLE_SORT_SMALL 0 and 1: one step
    within the tree tolerance of fp64 with relations above 255 trained, and a call of 12 steps in chunks
    1, 2, 4, 5 bit for bit the per-step path, which passes the boundary checks."""
    B, dim, n_rel, n_steps = 2000, 150, 300, 12
    layout = chunk_sizes(B, n_steps, (1, 2))
    assert layout == [1, 2, 4, 5]
    kg = D.synthetic_kg(n_rel, 4000, (n_steps + 1) * B, 5, dim, seed=hint or 1, trained_scale=True,
                        zipf_entities=True)
    kg.triples[::5, 2] = 256 + np.arange(len(kg.triples[::5])) % (n_rel - 256)
    assert hint is None or hint == n_rel or (kg.triples[:, 2] >= hint).any()
    env = {"HOLE_SORT_SMALL": sort_small}
    e = _engine(eng_mod, monkeypatch, kg, env=env, hint=hint)
    off, ids = D.build_type_csr(kg.type_of)
    pos = kg.triples[n_steps * B:]
    side, neg = O.corrupt(pos, kg.type_of, off, ids, 5, 9)
    before = _state(e)
    loss = e.train_step(pos, neg, side, MARGIN, 0.1).cpu().numpy()
    after = _state(e)
    _check(f"hint {hint}", before, after, pos, neg, side, MARGIN, float(np.float32(0.1)), n_rel, loss)
    assert (np.abs(after[0] - before[0]).max(axis=1) > 0)[256:n_rel].any()
    e.close()
    seed, first_step = 41, 7000
    lrs = _lrs(eng_mod, first_step, n_steps)
    tri = kg.triples[:n_steps * B]
    a = _engine(eng_mod, monkeypatch, kg, env=dict(env, HOLE_PLAN_RAMP="1,2"), hint=hint)
    sums, loss = a.train_steps(tri, B, seed, first_step, MARGIN, lrs, want_loss=True)
    b = _engine(eng_mod, monkeypatch, kg, env=env, hint=hint)
    ref = _per_step(b, tri, B, seed, first_step, lrs, n_rel, boundary_steps(layout))
    _assert_same(f"hint {hint}", a, b, B, sums, ref, loss)
    a.close(); b.close()


# ---------------------------------------------------------------- B.5 edges
@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 2, 31, 33, 513])
def test_adagrad_ragged_batches(eng_mod, monkeypatch, B):
    """Ragged batches (one triple, a partial lane group, one past a warp): two steps each within the tree
    tolerance of fp64, and a 3-step call equal to the per-step path bit for bit."""
    kg = D.synthetic_kg(5, 300, 8 * B, 4, 66, seed=B, trained_scale=True, zipf_entities=True)
    e = _engine(eng_mod, monkeypatch, kg, hint=kg.n_relations)
    lrs = _lrs(eng_mod, 3, 5)
    _per_step(e, kg.triples[:2 * B], B, 6, 3, lrs, kg.n_relations, check_at=(0, 1))
    a = _engine(eng_mod, monkeypatch, kg, hint=kg.n_relations)
    b = _engine(eng_mod, monkeypatch, kg, hint=kg.n_relations)
    sums, loss = a.train_steps(kg.triples[:3 * B], B, 6, 3, MARGIN, lrs, want_loss=True)
    ref = _per_step(b, kg.triples[:3 * B], B, 6, 3, lrs, kg.n_relations)
    _assert_same(f"B={B}", a, b, B, sums, ref, loss)
    e.close(); a.close(); b.close()


@pytest.mark.gpu
def test_adagrad_empty_batch_changes_nothing(eng_mod, monkeypatch):
    kg = D.synthetic_kg(5, 300, 1024, 4, 64, seed=3, trained_scale=True)
    e = _engine(eng_mod, monkeypatch, kg)
    e.train_steps(kg.triples, 512, 1, 0, MARGIN, [0.2, 0.2])
    t0, a0 = e.table.clone(), e.accum.clone()
    empty = np.zeros((0, 3), np.int32)
    loss = e.train_step(empty, np.zeros(0, np.int32), 0, MARGIN, 0.2)
    sums = e.train_steps(empty, 512, 1, 2, MARGIN, [0.2])
    hs = e.train_steps_host(empty, 512, 1, 2, MARGIN, [0.2])
    torch.cuda.synchronize()
    assert loss.numel() == 0 and sums.numel() == 0 and hs.size == 0
    assert torch.equal(e.table, t0) and torch.equal(e.accum, a0)
    e.close()


@pytest.mark.gpu
def test_adagrad_one_row_three_times_in_a_triple(eng_mod, monkeypatch):
    """A type of one entity: a triple (x, x, r) whose corruption is x again uses row x three times (head, tail,
    corrupt entity), and shares it between the positive and the negative triple."""
    rng = np.random.default_rng(5)
    Rn, P, dim, B = 4, 600, 130, 700
    N = Rn + P + 1
    solo = N - 1
    type_of = np.array([0] * Rn + [1] * P + [2], np.int32)
    pos = np.stack([Rn + rng.integers(0, P, B), Rn + rng.integers(0, P, B), rng.integers(0, Rn, B)], 1)
    pos[::7, :2] = solo
    E = D.init_embeddings(N, dim, rng, trained_scale=True)
    kg = D.SyntheticKG(Rn, P + 1, dim, pos.astype(np.int32), type_of, E)
    e = _engine(eng_mod, monkeypatch, kg, hint=Rn)
    off, ids = D.build_type_csr(type_of)
    for step in range(2):
        side, neg = O.corrupt(kg.triples, type_of, off, ids, 8, step)
        assert (neg[::7] == solo).all()
        before = _state(e)
        loss = e.train_step(kg.triples, neg, side, MARGIN, 0.3).cpu().numpy()
        _check(f"step {step}", before, _state(e), kg.triples, neg, side, MARGIN, float(np.float32(0.3)), Rn, loss)
    e.close()


@pytest.mark.gpu
def test_optimizer_switches_inside_a_sequence(eng_mod, monkeypatch):
    """SGD -> AdaGrad -> SGD on one context equals the same three phases each on a fresh context started from the
    previous phase's table, bit for bit: nothing of one optimizer (plans, counters, the sort decision) leaks into
    the next."""
    kg = D.synthetic_kg(6, 3000, 30 * 1024, 4, 128, seed=9, trained_scale=True, zipf_entities=True)
    B = 1024
    lrs = _lrs(eng_mod, 0, 30)
    phases = [("sgd", 0, 10), ("adagrad", 10, 20), ("sgd", 20, 30)]
    a = _engine(eng_mod, monkeypatch, kg, optimizer="sgd", hint=kg.n_relations)
    tables, accs = [], []
    for opt, k0, k1 in phases:
        if opt == "adagrad":
            a.set_optimizer("adagrad", 0.2)
        else:
            a.set_optimizer("sgd")
        a.train_steps(kg.triples[k0 * B:k1 * B], B, 4, k0, MARGIN, lrs[k0:k1])
        tables.append(a.table.clone())
        accs.append(a.accum.clone() if a.accum is not None else None)
    E = kg.E
    for (opt, k0, k1), t, acc in zip(phases, tables, accs):
        f = _engine(eng_mod, monkeypatch, D.SyntheticKG(kg.n_relations, kg.n_entities, kg.dim, kg.triples,
                                                        kg.type_of, E), optimizer="sgd", hint=kg.n_relations)
        if opt == "adagrad":
            f.set_optimizer("adagrad", 0.2)
        f.train_steps(kg.triples[k0 * B:k1 * B], B, 4, k0, MARGIN, lrs[k0:k1])
        assert torch.equal(f.table, t), opt
        if acc is not None:
            assert torch.equal(f.accum, acc)
        E = f.embeddings().cpu().numpy()
        f.close()
    assert not torch.equal(tables[0], tables[1]) and not torch.equal(tables[1], tables[2])
    a.close()
