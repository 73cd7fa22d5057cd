"""The delta-table and row-sharded training steps at every K1 lane group, and the gradient combine tree at
every depth.

K1 (csrc/hole_k1.cuh) has four update modes DM: 0 in place, 1 into a delta table (hole_train_step_ex), 2 the
row-sharded step (hole_shard_step: rows gathered from the owners' shards, deltas stored into the owners'
staging buffers), 3 a --log_loss pass (deltas accumulated over the passes).  Rows used more than once go
through K3 (hole_apply_kernel, csrc/hole_train.cu), a fan-in-32 combine tree whose root writes to the table,
the delta table, a peer's staging buffer or adds to the log-loss deltas.  This file checks:
  1. DM 1 at the first and last dim of every lane group, both sides, against the fp64 oracle; the row
     copies hole_gather_rows / hole_add_rows bit for bit;
  2. DM 2 with virtual ranks (test_gpu_train._VirtualRanks) at the same dims, both sides, against the
     single-GPU step and the fp64 oracle;
  3. the sharding edges: 16 ranks (HOLE_MAX_RANKS), ranks that own no rows, slices that request nothing
     from an owner, B < max_batch, and the refusal of 17 ranks;
  4. the combine tree on both sides of every depth edge (1, 32, 1024, 32768 uses) in every mode, with a
     tolerance derived from the fp64 per-use gradients, and its counters over consecutive steps.
The CPU test at the top keeps the parametrizations covering every lane-group form and every depth edge.
"""
import numpy as np
import pytest
import torch

from graphembeddings_b200 import data as D
from oracle import hole_oracle as O
from oracle.philox import side_coin
from test_gpu_shapes import lane_group, regimes, row_stride
from test_gpu_train import _VirtualRanks

HOLE_TREE_C = 32          # csrc/hole_common.cuh
HOLE_TREE_LEVELS = 6
HOLE_MAX_RANKS = 16
ROW_ATOL, ROW_RTOL, LOSS_ATOL = 2e-6, 1e-5, 2e-6
MARGIN, LR = 0.2, 0.1
SENTINEL = -1234.5

# first and last dim of every K1 lane-group regime (test_gpu_shapes.lane_group)
DIMS = [2, 64, 66, 128, 130, 256, 258, 512, 514, 768]
# both sides of every depth edge of the combine tree
TREE_EDGES = [1, 2, 32, 33, 1024, 1025, 32768, 32769]


def tree_depth(n):
    """Levels of the combine tree of hole_apply_kernel (csrc/hole_train.cu) for a row used n times in a step:
    0 = used once, K1 writes the row directly (gslot UNIQUE); otherwise the leaves are chunks of HOLE_TREE_C
    uses and each level combines up to HOLE_TREE_C nodes: 2-32 uses one level (the leaf is the root),
    33-1024 two, 1025-32768 three, 32769 and up four."""
    d, cap = 0, 1
    while n > cap:
        d += 1
        cap *= HOLE_TREE_C
    assert d <= HOLE_TREE_LEVELS
    return d


def dm2_seed(dim, steps=3):
    """The Philox seed of the DM 2 test at `dim`: the first seed >= dim whose side coins over the steps
    take both sides."""
    s = dim
    while len({side_coin(s, k) for k in range(steps)}) < 2:
        s += 1
    return s


def _params(test_fn, name):
    for m in getattr(test_fn, "pytestmark", []):
        if m.name == "parametrize" and m.args[0] == name:
            return [getattr(v, "values", (v,))[0] for v in m.args[1]]
    raise AssertionError(f"{test_fn.__name__} has no {name} parametrization")


def test_update_path_coverage():
    """DM 1 and DM 2 run every (GS, V, full) form of K1 on both sides; the tree tests reach both sides of
    every depth edge in every mode, and the counter test runs a four-level tree."""
    forms = {r[2] for r in regimes(lane_group) if r[2] is not None}
    assert len(forms) == 10
    dm1 = {(lane_group(d), s) for d in _params(test_delta_step_matches_oracle, "dim")
           for s in _params(test_delta_step_matches_oracle, "side")}
    assert dm1 == {(f, s) for f in forms for s in (0, 1)}
    assert {lane_group(d) for d in _params(test_gather_and_add_rows, "dim")} == forms
    dm2 = {(lane_group(d), side_coin(dm2_seed(d), k)) for d in _params(test_sharded_step_every_lane_group, "dim")
           for k in range(3)}
    assert dm2 == {(f, s) for f in forms for s in (0, 1)}
    assert [tree_depth(n) for n in TREE_EDGES] == [0, 1, 1, 2, 2, 3, 3, 4]
    edges = _params(test_combine_tree_depth_edges, "n")
    for d in range(1, 5):                       # the largest n of depth d-1 and the smallest of depth d
        assert max(n for n in range(1, 40000) if tree_depth(n) == d - 1) in edges
        assert min(n for n in range(1, 40000) if tree_depth(n) == d) in edges
    assert set(_params(test_combine_tree_depth_edges, "mode")) == {"dm0", "dm1", "dm2", "dm3"}
    assert tree_depth(max(_params(test_combine_tree_counters_over_steps, "n"))) == 4


# ---------------------------------------------------------------- GPU helpers
@pytest.fixture(scope="module")
def eng_mod():
    from graphembeddings_b200 import build
    build.build()
    from graphembeddings_b200 import engine
    return engine


def _engine(eng_mod, kg, csr=None):
    off, ids = D.build_type_csr(kg.type_of) if csr is None else csr
    return eng_mod.HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E).set_types(kg.type_of, off, ids), off, ids


def _unpack(tab, dim):
    """[N, row_stride] device layout -> [N, dim] ([Re | Im], each half padded to whole float4s)."""
    H, Hp = dim // 2, row_stride(dim) // 2
    return np.concatenate([tab[:, :H], tab[:, Hp:Hp + H]], axis=1)


def _band(got, want, rows):
    err, tol = np.abs(got[rows] - want[rows]), ROW_ATOL + ROW_RTOL * np.abs(want[rows])
    assert (err <= tol).all(), float((err - tol).max())


# ---------------------------------------------------------------- 1. DM 1 and the row copies
@pytest.mark.gpu
@pytest.mark.parametrize("dim", DIMS)
@pytest.mark.parametrize("side", [0, 1])
def test_delta_step_matches_oracle(eng_mod, dim, side):
    """hole_train_step_ex into a delta table filled with a sentinel: the table is bit-unchanged, every used
    row's delta is within the one-step band of (fp64 step - E0), every other row keeps the sentinel bits."""
    B = 600
    kg = D.synthetic_kg(7, 500, B, 5, dim, seed=300 + dim, trained_scale=True, zipf_entities=True)
    e, off, ids = _engine(eng_mod, kg)
    pos = kg.triples
    _, neg = O.corrupt(pos, kg.type_of, off, ids, 3, 0)
    pos_t, neg_t = torch.from_numpy(pos).to(e.device), torch.from_numpy(neg).to(e.device)
    before = e.table.clone()
    delta = torch.full_like(e.table, SENTINEL)
    loss = e.train_step_delta(pos_t, neg_t, side, MARGIN, LR, delta).cpu().numpy()
    assert torch.equal(e.table, before)
    E64 = kg.E.astype(np.float64)
    l64, _, _ = O.sgd_step(E64, pos, neg, side, MARGIN, LR, np.float64, "tf")
    assert np.abs(loss - l64).max() <= LOSS_ATOL
    used = np.unique(np.concatenate([pos.ravel(), neg]))
    d = _unpack(delta.cpu().numpy(), dim)
    want = E64 - kg.E.astype(np.float64)
    err, tol = np.abs(d[used] - want[used]), ROW_ATOL + ROW_RTOL * np.abs(E64[used])
    assert (err <= tol).all(), float((err - tol).max())
    assert np.abs(d[used]).max() > 1e-5
    unused = torch.ones(kg.n_rows, dtype=torch.bool, device=e.device)
    unused[torch.from_numpy(used).to(e.device).long()] = False
    sent = torch.tensor(SENTINEL, dtype=torch.float32).view(torch.int32).item()
    assert (delta[unused].view(torch.int32) == sent).all()
    e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("dim", DIMS)
def test_gather_and_add_rows(eng_mod, dim):
    """hole_gather_rows == torch indexing and hole_add_rows == the fp32 add, bit for bit, with an id offset
    and the last row of the table among the ids."""
    rng = np.random.default_rng(dim)
    N, off, K = 3000, 37, 500
    e = eng_mod.HoleEngine(N, dim).set_embeddings(D.init_embeddings(N, dim, rng, trained_scale=True))
    ids = rng.choice(N - off, size=K, replace=False)
    ids[rng.integers(0, K)] = N - 1 - off
    ids_t = torch.from_numpy(ids.astype(np.int64)).to(e.device)
    w = e.row_stride
    dst = torch.full((K, w), SENTINEL, dtype=torch.float32, device=e.device)
    e.gather_rows(e.table, ids_t, off, dst)
    assert torch.equal(dst, e.table[ids_t + off])
    rows = torch.from_numpy(rng.standard_normal((K, w)).astype(np.float32)).to(e.device)
    want = e.table.clone()
    want[ids_t + off] += rows
    e.add_rows(e.table, ids_t, off, rows)
    assert torch.equal(e.table, want)
    assert not torch.equal(dst, e.table[ids_t + off])
    e.close()


# ---------------------------------------------------------------- 2.-3. DM 2 with virtual ranks
def _run_sharded(eng_mod, kg, world, max_batch, Bs, seed, csr=None):
    """len(Bs) sharded steps of `world` virtual ranks (step s: slices of Bs[s] triples each) against the
    single-GPU engine on the concatenated global batch: loss <= 2e-6 per step, the first step within the
    one-step band of the fp64 oracle, the tables <= 2e-6 after the last step, relation replicas
    bit-identical and no flag time-out.  Returns the sides the steps took."""
    vr = _VirtualRanks(eng_mod, kg, world, max_batch, csr=csr)
    e, _, _ = _engine(eng_mod, kg, csr)
    dev = e.device
    sides, t0 = [], 0
    for s, B in enumerate(Bs):
        gb = kg.triples[t0:t0 + world * B]
        t0 += world * B
        tri = torch.from_numpy(gb).to(dev)
        losses = vr.step([tri[k * B:(k + 1) * B].contiguous() for k in range(world)], seed, s, MARGIN, LR)
        side, neg = e.corrupt_batch(gb, seed, s)
        assert side == side_coin(seed, s)
        sides.append(side)
        want = e.train_step(gb, neg, side, MARGIN, LR).cpu().numpy().reshape(world, B)
        for k in range(world):
            assert np.abs(losses[k].cpu().numpy() - want[k]).max() <= LOSS_ATOL
        if s == 0:
            E64 = kg.E.astype(np.float64)
            neg_h = neg.cpu().numpy()
            O.sgd_step(E64, gb, neg_h, side, MARGIN, LR, np.float64, "tf")
            _band(vr.table(), E64, np.unique(np.concatenate([gb.ravel(), neg_h])))
    assert t0 <= len(kg.triples)
    got = vr.table()
    ref = e.embeddings().cpu().numpy()
    assert np.abs(got - ref).max() <= 2e-6
    assert np.abs(ref - kg.E).max() > 1e-4
    e.close()
    for x in vr.engs:
        x.close()
    return sides


@pytest.mark.gpu
@pytest.mark.parametrize("dim", DIMS)
def test_sharded_step_every_lane_group(eng_mod, dim):
    """hole_shard_step at every lane group: 2 or 3 virtual ranks, ragged B, Zipf entities (rows requested by
    several ranks), three steps whose side coins take both sides."""
    world = 2 + DIMS.index(dim) % 2
    B = 61 + 2 * DIMS.index(dim)
    seed = dm2_seed(dim)
    kg = D.synthetic_kg(7, 2000, 3 * world * B, 5, dim, seed=700 + dim, trained_scale=True, zipf_entities=True)
    sides = _run_sharded(eng_mod, kg, world, B, [B] * 3, seed)
    assert sides == [side_coin(seed, s) for s in range(3)] and set(sides) == {0, 1}


EDGE_DIM = 150


def _owners(kg, rows_per, rows):
    return set(((np.asarray(rows) - kg.n_relations) // rows_per).tolist())


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["world16", "empty_owners", "small_batches"])
def test_sharding_edges(eng_mod, case):
    """world16: HOLE_MAX_RANKS ranks (bit 15 of the claim masks, 17 cut slots).  empty_owners: 20 entities
    over 16 ranks, ranks 10-15 own no rows and most slices request nothing from most owners.
    small_batches: steps with B < max_batch (staging stride 3 max_batch != 3B), B = 1 included, alternating
    with B = max_batch."""
    from graphembeddings_b200.sharded import row_partition
    world, n_ent, max_batch, Bs = {"world16": (16, 3000, 40, [40, 40, 23]),
                                   "empty_owners": (16, 20, 3, [3, 2, 3]),
                                   "small_batches": (3, 2000, 200, [200, 77, 200, 1])}[case]
    kg = D.synthetic_kg(7, n_ent, world * sum(Bs), 3, EDGE_DIM, seed=world + n_ent, trained_scale=True,
                        zipf_entities=True)
    rows_per = row_partition(n_ent, world)
    off, ids = D.build_type_csr(kg.type_of)
    if case == "empty_owners":
        assert rows_per * 10 == n_ent                         # ranks 10..15 own nothing
        t0, missing = 0, 0
        for s, B in enumerate(Bs):
            gb = kg.triples[t0:t0 + world * B]
            t0 += world * B
            _, neg = O.corrupt(gb, kg.type_of, off, ids, 5, s)
            for k in range(world):
                sl = slice(k * B, (k + 1) * B)
                asked = _owners(kg, rows_per, np.concatenate([gb[sl, 0], gb[sl, 1], neg[sl]]))
                missing += len(set(range(10)) - asked)
        assert missing > 0
    if case == "world16":
        top = _owners(kg, rows_per, kg.triples[:world * Bs[0], :2].ravel())
        assert world - 1 in top                                # the last rank owns rows the first step uses
    sides = _run_sharded(eng_mod, kg, world, max_batch, Bs, 5)
    assert sides == [side_coin(5, s) for s in range(len(Bs))]


@pytest.mark.gpu
def test_shard_init_refuses_17_ranks(eng_mod):
    """hole_shard_init with world = HOLE_MAX_RANKS + 1 raises HoleError and launches nothing; the same
    context then accepts HOLE_MAX_RANKS."""
    kg = D.synthetic_kg(3, 100, 10, 2, 8, seed=1)
    e, _, _ = _engine(eng_mod, kg)
    buf = torch.zeros(64, dtype=torch.float32, device=e.device)
    err = torch.zeros(1, dtype=torch.int32, device=e.device)

    def init(world):
        pa = e.peer_array([buf] * world)
        e.shard_init(world, 0, kg.n_relations, kg.n_entities, (kg.n_entities + world - 1) // world, 4, buf,
                     pa, pa, pa, pa, pa, pa, err, 1.0)

    torch.cuda.synchronize()
    n0 = e.launch_count()
    with pytest.raises(eng_mod.HoleError, match="world <= HOLE_MAX_RANKS"):
        init(HOLE_MAX_RANKS + 1)
    torch.cuda.synchronize()
    assert e.launch_count() == n0
    init(HOLE_MAX_RANKS)
    e.close()


# ---------------------------------------------------------------- 4. the combine tree
TREE_DIM, TREE_MARGIN, TREE_R, TREE_P = 8, 1.0, 3, 4096       # margin 1: every hinge is active


def _tree_kg(n_triples, seed):
    """TREE_R relations, TREE_P pool entities and one hot row (the last).  Heads and tails come from the
    pool; the type table sends every corruption to the hot row, so each triple uses it exactly once, as its
    corrupt entity (on either side)."""
    rng = np.random.default_rng(seed)
    R, P = TREE_R, TREE_P
    N = R + P + 1
    pos = np.stack([R + rng.integers(0, P, n_triples), R + rng.integers(0, P, n_triples),
                    rng.integers(0, R, n_triples)], 1).astype(np.int32)
    type_of = np.array([0] * R + [1] * P + [2], np.int32)
    E = rng.standard_normal((N, TREE_DIM))
    E *= rng.uniform(0.8, 0.95, (N, 1)) / np.linalg.norm(E, axis=1, keepdims=True)
    E[-1] *= 0.05
    kg = D.SyntheticKG(R, P + 1, TREE_DIM, pos, type_of, E.astype(np.float32))
    csr = (np.array([0, R, R + 1, R + 2], np.int64), np.array(list(range(R)) + [N - 1, N - 1], np.int32))
    return kg, csr


def _uses(pos, neg, n_rows):
    """Per-row key count of hole_plan_keys_kernel: head, tail and corrupt entity of every triple."""
    return np.bincount(np.concatenate([pos[:, 0], pos[:, 1], neg]).astype(np.int64), minlength=n_rows)


def _hinge_slices(E64, pos, neg, side):
    slices, loss, _, _ = O.indexed_slices(E64, pos, neg, side, TREE_MARGIN, np.float64)
    return [(i.astype(np.int64), g) for i, g in slices], loss


def _logloss_slices(E64, pos, negs, sides):
    out = []
    for tri, g in [(pos, O.sigmoid(O.score(E64, pos, np.float64)) - 1.0)] + [
            (O.corrupt_triples(pos, n, s), None) for n, s in zip(negs, sides)]:
        if g is None:
            g = O.sigmoid(O.score(E64, tri, np.float64))
        out += [(tri[:, c].astype(np.int64), dx) for c, dx in enumerate(O._side_grads(E64, tri, g, np.float64))]
    return out


def _tree_tol(want, slices, depth, lr):
    """2e-6 + 1e-5 |x| + lr * sum_i |g_i| * (1e-6 + (31 depth + 1) 2^-24) per element: the fp32 sums of the
    combine tree (31 adds per level) over the fp64 per-use gradients g_i."""
    absg = np.zeros_like(want)
    for i, g in slices:
        np.add.at(absg, i, np.abs(g))
    return ROW_ATOL + ROW_RTOL * np.abs(want) + lr * absg * (1e-6 + (31 * depth[:, None] + 1) * 2.0**-24)


def _check_tree(got, want, slices, counts, hot, n, lr, n_relations):
    """got vs want within the tree tolerance on the entity rows the step uses; the hot row has n uses in every
    group of counts (one per rank / per pass), and each of its per-use gradients alone exceeds the tolerance,
    so a dropped or doubled leaf cannot pass."""
    depth = np.max([[tree_depth(c) for c in cnt] for cnt in counts], axis=0)
    ent_rows = n_relations + np.flatnonzero(np.sum(counts, axis=0)[n_relations:])
    for cnt in counts:
        assert cnt[hot] == n
    assert depth[hot] == tree_depth(n)
    tol = _tree_tol(want, slices, depth, lr)
    g_hot = np.concatenate([g[i == hot] for i, g in slices])
    assert len(g_hot) == n * len(counts)
    assert (lr * np.abs(g_hot) / tol[hot]).max(axis=1).min() > 1.0
    err = np.abs(got[ent_rows] - want[ent_rows])
    assert (err <= tol[ent_rows]).all(), float((err - tol[ent_rows]).max())


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["dm0", "dm1", "dm2", "dm3"])
@pytest.mark.parametrize("n", TREE_EDGES)
def test_combine_tree_depth_edges(eng_mod, monkeypatch, mode, n):
    """One hot entity row used exactly n times in a step, in each update mode: dm0 train_step under the three
    plan sorts (HOLE_SORT_SMALL 0, 1, 2: bit-identical tables); dm1 train_step_delta twice on one context
    (bit-identical deltas, untouched table); dm2 two virtual ranks, the hot row owned by rank 1 and used n
    times by each rank's slice; dm3 train_step_logloss with k = 2 (n uses per pass).  The entity rows
    against the fp64 oracle within the derived tree tolerance; a second run is bit-identical."""
    step = TREE_EDGES.index(n)
    seed = 40 + step
    lr = LR
    world = 2 if mode == "dm2" else 1
    kg, csr = _tree_kg(world * n, 1000 + n)
    hot = kg.n_rows - 1
    E64 = kg.E.astype(np.float64)
    pos = kg.triples
    if mode in ("dm0", "dm1"):
        side, neg = O.corrupt(pos, kg.type_of, *csr, seed, step)
        slices, l64 = _hinge_slices(E64, pos, neg, side)
        want = E64.copy()
        O.sgd_step(want, pos, neg, side, TREE_MARGIN, lr, np.float64, "tf")
        counts = [_uses(pos, neg, kg.n_rows)]
        if mode == "dm0":
            tables = []
            for sort in ("0", "1", "2"):
                monkeypatch.setenv("HOLE_SORT_SMALL", sort)
                e, _, _ = _engine(eng_mod, kg, csr)
                monkeypatch.delenv("HOLE_SORT_SMALL")
                loss = e.train_step(pos, neg, side, TREE_MARGIN, lr).cpu().numpy()
                assert np.abs(loss - l64).max() <= LOSS_ATOL
                tables.append(e.table.clone())
                got = e.embeddings().cpu().numpy()
                e.close()
            assert torch.equal(tables[0], tables[1]) and torch.equal(tables[0], tables[2])
        else:
            e, _, _ = _engine(eng_mod, kg, csr)
            pos_t, neg_t = torch.from_numpy(pos).to(e.device), torch.from_numpy(neg).to(e.device)
            before = e.table.clone()
            deltas = []
            for _ in range(2):
                d = torch.full_like(e.table, SENTINEL)
                loss = e.train_step_delta(pos_t, neg_t, side, TREE_MARGIN, lr, d).cpu().numpy()
                assert np.abs(loss - l64).max() <= LOSS_ATOL
                deltas.append(d)
            assert torch.equal(deltas[0], deltas[1]) and torch.equal(e.table, before)
            d = _unpack(deltas[0].cpu().numpy(), TREE_DIM)
            assert (d[kg.n_relations:][counts[0][kg.n_relations:] == 0] == SENTINEL).all()   # unused entity rows
            got = kg.E.astype(np.float64) + d
            e.close()
    elif mode == "dm2":
        from graphembeddings_b200.sharded import row_partition
        rows_per = row_partition(kg.n_entities, 2)
        assert (hot - kg.n_relations) // rows_per == 1
        e, _, _ = _engine(eng_mod, kg, csr)
        side, neg = e.corrupt_batch(pos, seed, step)
        neg = neg.cpu().numpy()
        e.close()
        slices, l64 = _hinge_slices(E64, pos, neg, side)
        want = E64.copy()
        O.sgd_step(want, pos, neg, side, TREE_MARGIN, lr, np.float64, "tf")
        counts = [_uses(pos[k * n:(k + 1) * n], neg[k * n:(k + 1) * n], kg.n_rows) for k in range(2)]
        outs = []
        for _ in range(2):
            vr = _VirtualRanks(eng_mod, kg, 2, n, csr=csr)
            tri = torch.from_numpy(pos).to(vr.engs[0].device)
            losses = vr.step([tri[:n].contiguous(), tri[n:].contiguous()], seed, step, TREE_MARGIN, lr)
            loss = torch.cat(losses).cpu().numpy()
            assert np.abs(loss - l64).max() <= LOSS_ATOL
            outs.append(vr.table())
            for x in vr.engs:
                x.close()
        assert np.array_equal(outs[0], outs[1])
        got = outs[0]
    else:
        k = 2
        outs = []
        for _ in range(2):
            e, _, _ = _engine(eng_mod, kg, csr)
            loss, _, sides, negs = e.train_step_logloss(pos, seed, step, lr, 0.0, k, want_corruption=True)
            outs.append((loss.cpu().numpy(), e.embeddings().cpu().numpy()))
            negs = negs.cpu().numpy()
            assert not e._delta_ws.any()
            e.close()
        assert np.array_equal(outs[0][0], outs[1][0]) and np.array_equal(outs[0][1], outs[1][1])
        for j in range(k):
            assert (sides[j], negs[j].tolist()) == (side_coin(seed, step * k + j), [hot] * n)
        want = E64.copy()
        l64, _ = O.logloss_step(want, pos, list(negs), sides, lr, 0.0, np.float64)
        assert np.abs(outs[0][0] - l64).max() <= LOSS_ATOL
        slices = _logloss_slices(E64, pos, list(negs), sides)
        counts = [_uses(pos, negs[j], kg.n_rows) for j in range(k)]
        got = outs[0][1]
    _check_tree(got, want, slices, counts, hot, n, lr, kg.n_relations)
    assert np.abs(got[hot] - kg.E[hot]).max() > 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("n", [32769])
def test_combine_tree_counters_over_steps(eng_mod, n):
    """A four-level tree in three consecutive steps of one train_steps call: its ticket counters must reset
    themselves for the next step (a stale counter freezes the row).  The call equals the per-step path bit for
    bit, and every per-step step is within the tree tolerance of the fp64 oracle re-run from its table."""
    steps, seed, first = 3, 12, 5
    kg, csr = _tree_kg(steps * n, 77)
    hot = kg.n_rows - 1
    lrs = np.array([eng_mod.inverse_time_decay(0.1, first + k, 2, 0.5) for k in range(steps)], np.float32)
    a, _, _ = _engine(eng_mod, kg, csr)
    tri = torch.from_numpy(kg.triples).to(a.device)
    sums, loss_a = a.train_steps(tri, n, seed, first, TREE_MARGIN, lrs, want_loss=True)
    b, _, _ = _engine(eng_mod, kg, csr)
    losses = []
    for k in range(steps):
        pos = kg.triples[k * n:(k + 1) * n]
        side, neg = b.corrupt_batch(pos, seed, first + k)
        neg = neg.cpu().numpy()
        E64 = b.embeddings().cpu().numpy().astype(np.float64)
        losses.append(b.train_step(pos, neg, side, TREE_MARGIN, lrs[k]))
        slices, l64 = _hinge_slices(E64, pos, neg, side)
        want = E64.copy()
        O.sgd_step(want, pos, neg, side, TREE_MARGIN, float(lrs[k]), np.float64, "tf")
        assert np.abs(losses[-1].cpu().numpy() - l64).max() <= LOSS_ATOL
        _check_tree(b.embeddings().cpu().numpy(), want, slices, [_uses(pos, neg, kg.n_rows)], hot, n,
                    float(lrs[k]), kg.n_relations)
    assert torch.equal(a.table, b.table) and torch.equal(loss_a, torch.cat(losses))
    a.close(); b.close()
