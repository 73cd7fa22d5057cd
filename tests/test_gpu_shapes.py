"""The kernels on both sides of their embedding-dimension and table-size dispatch boundaries.

The host picks kernel templates, lane masks, ring depths and radix pass counts from the embedding dimension
and the table size.  The functions below restate those selections (each cites its source); the CPU test
pins them, and the GPU tests take their dims from them: the last dim of a regime and the first of the next.
Parity in each regime is checked by the existing tests, whose parametrizations carry these dims
(test_gpu_train, test_gpu_rank, test_gpu_topk, test_gpu_ccorr).  This file adds:
  * refusals: a dim a path does not build raises HoleError, launches nothing, writes no output or table,
    and leaves the context usable for what it does build;
  * the update plan at the row-key radix pass edges (255/256, 65,535/65,536, 2^24-1/2^24 rows): the three
    plan-sort strategies agree bit for bit, the step matches the fp64 oracle on the rows it uses and leaves
    every other row bit-unchanged; at 2^24 rows a multi-chunk train_steps call equals the per-step path;
  * the device loop at the first v2 and the last v3 lane-group dims, bit-equal to the per-step path;
  * the own-operands exact-count check of the archived ccorr mode at its widest query packers (NV 8, 12).
"""
import ctypes as C

import numpy as np
import pytest
import torch

from graphembeddings_b200 import data as D
from oracle import hole_oracle as O

SMEM = 227 * 1024                 # opt-in shared memory per block
EVEN_DIMS = range(2, 772, 2)      # 770 is the first dim the library refuses


# ---------------------------------------------------------------- dispatch mirror (host selection formulas)
def row_stride(dim):
    """hole_row_stride (csrc/hole_train.cu): [Re | Im], each half padded to whole float4s."""
    return 8 * ((dim // 2 + 3) // 4)


def lane_group(dim):
    """hole_ctx_create (csrc/hole_train.cu): lanes per row gs and float4s per lane and half v, from
    nvec = ceil(dim / 8); full = (nvec == GS * V) picks the unmasked template (hole_k1.cuh, hole_k1_launch).
    None: refused (v > 3)."""
    nvec = (dim // 2 + 3) // 4
    if nvec <= 8:
        gs, v = 8, 1
    elif nvec <= 16:
        gs, v = 16, 1
    else:
        gs, v = 32, (nvec + 31) // 32
    if v > 3:
        return None
    return gs, v, nvec == gs * v


def rank_stages(dim, parts):
    """rank_impl (csrc/hole_rank.cu): depth of the candidate k-block ring next to the resident query operand,
    min((227 KB - A - 2 KB) / 32 KB, MAX_STAGES = 4); parts = 1 (bf16) or 2 (bf16x3).  None: refused (< 2)."""
    num_kb = (dim + 63) // 64
    a_bytes = num_kb * parts * 128 * 64 * 2
    stages = min((SMEM - a_bytes - 2048) // (256 * 64 * 2), 4)
    return stages if stages >= 2 else None


def pq_iters(dim):
    """rank_impl (csrc/hole_rank.cu): PQ_ITERS of hole_rank_pack_query_kernel, ceil(row_stride / 256)."""
    return (row_stride(dim) // 2 + 127) // 128


def last_kb_mmas(dim):
    """rank_impl (csrc/hole_rank.cu): K = 16 slices of the last k-block that hold real columns."""
    num_kb = (dim + 63) // 64
    return (dim - (num_kb - 1) * 64 + 15) // 16


def cc_nv(dim):
    """cc_nv / HOLE_CC_DISPATCH (csrc/hole_train.cu) and the ccorr query packer (csrc/hole_rank.cu):
    (needed, instantiated) float4s per lane, needed = ceil(4 nvec / 32) rounded up to {1,2,3,4,6,8,12}."""
    need = (row_stride(dim) // 2 + 31) // 32
    return need, next(n for n in (1, 2, 3, 4, 6, 8, 12, need) if n >= need)


def row_passes(n_rows):
    """hole_ctx_create (csrc/hole_train.cu): smallest p with 2^(8p) - 1 >= n_rows (the absent key sorts
    last).  Also the relation-sort passes without a hole_ctx_set_relations hint."""
    p = 1
    while (1 << (8 * p)) - 1 < n_rows:
        p += 1
    return p


def route_passes(n_rows_global):
    """shard_route (csrc/hole_train.cu): byte passes covering n_rows_global - 1, at most 4."""
    p = 1
    while p < 4 and (n_rows_global - 1) >> (8 * p):
        p += 1
    return p


def regimes(fn):
    """[(first dim, last dim, value)] of the runs of fn over the even dims 2..770."""
    out = []
    for d in EVEN_DIMS:
        v = fn(d)
        if out and out[-1][2] == v:
            out[-1][1] = d
        else:
            out.append([d, d, v])
    return [tuple(r) for r in out]


def first_dim(pred):
    return next(d for d in EVEN_DIMS if pred(d))


def test_dispatch_mirror():
    """The regimes of every host selection, and the dims the GPU tests use at their edges."""
    assert regimes(lane_group) == [
        (2, 56, (8, 1, False)), (58, 64, (8, 1, True)),
        (66, 120, (16, 1, False)), (122, 128, (16, 1, True)),
        (130, 248, (32, 1, False)), (250, 256, (32, 1, True)),
        (258, 504, (32, 2, False)), (506, 512, (32, 2, True)),
        (514, 760, (32, 3, False)), (762, 768, (32, 3, True)),
        (770, 770, None)]
    assert regimes(lambda d: rank_stages(d, 1)) == [(2, 384, 4), (386, 512, 3), (514, 640, 2), (642, 770, None)]
    assert regimes(lambda d: rank_stages(d, 2)) == [(2, 192, 4), (194, 256, 3), (258, 320, 2), (322, 770, None)]
    assert regimes(pq_iters)[:3] == [(2, 256, 1), (258, 512, 2), (514, 768, 3)]
    assert regimes(cc_nv) == [
        (2, 64, (1, 1)), (66, 128, (2, 2)), (130, 192, (3, 3)), (194, 256, (4, 4)), (258, 320, (5, 6)),
        (322, 384, (6, 6)), (386, 448, (7, 8)), (450, 512, (8, 8)), (514, 576, (9, 12)), (578, 640, (10, 12)),
        (642, 704, (11, 12)), (706, 768, (12, 12)), (770, 770, (13, 13))]
    assert last_kb_mmas(514) == 1 and last_kb_mmas(640) == 4 and last_kb_mmas(2) == 1
    # the edges the refusal tests below use, found from the mirror
    assert first_dim(lambda d: lane_group(d) is None) == 770
    assert first_dim(lambda d: rank_stages(d, 1) is None) == 642
    assert first_dim(lambda d: rank_stages(d, 2) is None) == 322
    # table-size edges
    assert [row_passes(n) for n in (43, 255, 256, 65535, 65536, 2**24 - 1, 2**24)] == [1, 1, 2, 2, 3, 3, 4]
    assert [route_passes(n) for n in (1005, 256, 257, 2**24, 2**24 + 1, 3 * 2**24 + 5, 2**31)] == [2, 1, 2, 3, 4, 4, 4]
    assert row_stride(770) == 776 and row_stride(2) == 8


def _dims_of(test_fn):
    """The dims a test is parametrized with (first field of a "dim" or "dim,..." parametrization)."""
    for m in getattr(test_fn, "pytestmark", []):
        if m.name == "parametrize" and m.args[0].split(",")[0] == "dim":
            vals = [getattr(v, "values", v) for v in m.args[1]]
            return [v[0] if isinstance(v, tuple) else v for v in vals]
    raise AssertionError(f"{test_fn.__name__} has no dim parametrization")


def test_parity_tests_reach_every_regime():
    """The dims the parity tests of the other files run at cover every regime of the mirror."""
    import test_gpu_ccorr as CC
    import test_gpu_rank as RK
    import test_gpu_topk as TK
    import test_gpu_train as TR
    all_lane_groups = {r[2] for r in regimes(lane_group) if r[2] is not None}
    for fn in (TR.test_pack_unpack_roundtrip, TR.test_score_matches_oracle, TR.test_train_step_matches_oracle):
        assert {lane_group(d) for d in _dims_of(fn)} == all_lane_groups
    rank = _dims_of(RK.test_rank_counts_exact_vs_own_operands)
    assert {rank_stages(d, 1) for d in rank} == {4, 3, 2} and {pq_iters(d) for d in rank} == {1, 2, 3}
    assert 2 in rank and max(rank) == max(d for d in EVEN_DIMS if rank_stages(d, 1))
    x3 = _dims_of(RK.test_split_bf16_precision_matches_fp64_oracle)
    assert {rank_stages(d, 2) for d in x3} == {4, 3, 2} and max(x3) == max(d for d in EVEN_DIMS if rank_stages(d, 2))
    topk = _dims_of(TK.test_topk_matches_fp64_oracle)
    assert {2, 320, 640} <= set(topk) and {pq_iters(d) for d in topk} == {1, 2, 3}
    all_nv = {r[2][1] for r in regimes(cc_nv)} - {13}
    assert {cc_nv(d)[1] for d in _dims_of(CC.test_ccorr_score_matches_oracle)} == all_nv
    assert {cc_nv(d)[1] for d in _dims_of(CC.test_ccorr_train_steps_match_oracle)} == all_nv
    assert {cc_nv(d)[0] for d in _dims_of(CC.test_ccorr_score_matches_oracle)} >= {5, 8, 9, 12}   # rounded up and exact
    assert {cc_nv(d)[1] for d in _dims_of(CC.test_ccorr_ranking_matches_fp64_oracle)} >= {6}
    assert {cc_nv(d)[1] for d in _dims_of(test_ccorr_rank_counts_exact_vs_own_operands)} == {8, 12}
    assert {lane_group(d) for d in _dims_of(TR.test_logloss_step_matches_oracle)} == all_lane_groups


# ---------------------------------------------------------------- GPU helpers
@pytest.fixture(scope="module")
def eng_mod():
    from graphembeddings_b200 import build
    build.build()
    from graphembeddings_b200 import engine
    return engine


def _engine(eng_mod, kg, types=True):
    e = eng_mod.HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E)
    if types:
        off, ids = D.build_type_csr(kg.type_of)
        e.set_types(kg.type_of, off, ids)
    return e


def _check_one_step(e, kg, B, side, seed=3, lr=0.1, margin=0.2):
    """One hinge step on e against the fp64 oracle: sigma, loss, rows, and untouched rows bit-unchanged."""
    off, ids = D.build_type_csr(kg.type_of)
    pos = kg.triples[:B]
    _, neg = O.corrupt(pos, kg.type_of, off, ids, seed, 0)
    E0 = e.embeddings().cpu().numpy()
    loss, vp, vn = e.train_step(pos, neg, side, margin, lr, return_sigma=True)
    E64 = E0.astype(np.float64)
    l64, vp64, vn64 = O.sgd_step(E64, pos, neg, side, margin, lr, np.float64, "tf")
    assert np.abs(vp.cpu().numpy() - vp64).max() <= 1e-6 and np.abs(vn.cpu().numpy() - vn64).max() <= 1e-6
    assert np.abs(loss.cpu().numpy() - l64).max() <= 2e-6
    got = e.embeddings().cpu().numpy()
    err, tol = np.abs(got - E64), 2e-6 + 1e-5 * np.abs(E64)
    assert (err <= tol).all(), float((err - tol).max())
    untouched = np.setdiff1d(np.arange(kg.n_rows), np.concatenate([pos.ravel(), neg]))
    assert np.array_equal(got[untouched], E0[untouched])
    assert np.abs(got - E0).max() > 1e-5


# ---------------------------------------------------------------- 1. refusals
@pytest.mark.gpu
def test_dim_above_768_is_refused_at_context_creation(eng_mod):
    dim = first_dim(lambda d: lane_group(d) is None)
    with pytest.raises(eng_mod.HoleError, match=f"embedding_dim {dim}"):
        eng_mod.HoleEngine(100, dim)
    from graphembeddings_b200 import _lib
    assert _lib.load().hole_row_stride(dim) == row_stride(dim)
    e = eng_mod.HoleEngine(100, dim - 2)                 # the last built dim is accepted
    assert e.row_stride == row_stride(dim - 2)
    e.close()


def _rank_refusals(eng_mod, e, kg, precision):
    """rank, rank_prepare and topk at `precision` raise, launch nothing and write nothing."""
    b, en = kg.n_relations, kg.n_rows
    Q = len(kg.triples)
    table0 = e.table.clone()
    raw = torch.full((Q,), -7, dtype=torch.int32, device=e.device)
    filt = torch.full((Q,), -7, dtype=torch.int32, device=e.device)
    ts = torch.full((Q,), 1234.5, dtype=torch.float32, device=e.device)
    match = f"embedding_dim {kg.dim}"
    n0 = e.launch_count()
    with pytest.raises(eng_mod.HoleError, match=match):
        e.rank(kg.triples, 0, b, en, precision=precision, true_score=ts, raw_before=raw, filt_before=filt)
    with pytest.raises(eng_mod.HoleError, match=match):
        e.rank_prepare(b, en, precision=precision)
    k = 5
    ids = torch.full((Q, k), -7, dtype=torch.int32, device=e.device)
    sc = torch.full((Q, k), 1234.5, dtype=torch.float32, device=e.device)
    q = torch.from_numpy(kg.triples).to(e.device)
    from graphembeddings_b200 import _lib
    with pytest.raises(eng_mod.HoleError, match=match):       # hole_topk with sentinel output buffers
        _lib.check(e.lib.hole_topk(e._ctx, C.c_void_p(e.table.data_ptr()), b, en, C.c_void_p(q.data_ptr()), Q, 0,
                                   precision, k, None, None, C.c_void_p(ids.data_ptr()), C.c_void_p(sc.data_ptr()),
                                   C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    with pytest.raises(eng_mod.HoleError, match=match):
        e.topk(kg.triples, 0, b, en, k, precision=precision)
    torch.cuda.synchronize()
    assert e.launch_count() == n0
    assert (raw == -7).all() and (filt == -7).all() and (ts == 1234.5).all()
    assert (ids == -7).all() and (sc == 1234.5).all()
    assert torch.equal(e.table, table0)


@pytest.mark.gpu
def test_bf16x3_refusal_then_bf16_ranking_on_the_same_context(eng_mod):
    """First dim bf16x3 does not build (322): a clean refusal, then plain bf16 ranking at the same dim on
    the same context matches the exact count of its own operands."""
    from test_gpu_rank import _exact_from_operands
    dim = first_dim(lambda d: rank_stages(d, 2) is None)
    assert rank_stages(dim, 1) == 4
    kg = D.synthetic_kg(5, 1500, 300, 4, dim, seed=dim, trained_scale=True)
    e = _engine(eng_mod, kg, types=False)
    _rank_refusals(eng_mod, e, kg, eng_mod.HOLE_RANK_BF16X3)
    b, en = kg.n_relations, kg.n_rows
    raw, filt, ts = e.rank(kg.triples, 0, b, en)
    raw, filt, ts = raw.cpu().numpy(), filt.cpu().numpy(), ts.cpu().numpy()
    _exact_from_operands(e, kg, kg.triples, 0, b, en, raw, filt, ts)
    assert raw.max() > 100
    e.close()


@pytest.mark.gpu
def test_bf16_refusal_then_scoring_and_training_on_the_same_context(eng_mod):
    """First dim plain bf16 ranking does not build (642): a clean refusal at both precisions, then scoring
    and a hinge step at the same dim on the same context match the fp64 oracle."""
    dim = first_dim(lambda d: rank_stages(d, 1) is None)
    kg = D.synthetic_kg(7, 500, 1024, 5, dim, seed=dim, trained_scale=True, zipf_entities=True)
    e = _engine(eng_mod, kg)
    _rank_refusals(eng_mod, e, kg, eng_mod.HOLE_RANK_BF16)
    _rank_refusals(eng_mod, e, kg, eng_mod.HOLE_RANK_BF16X3)
    got = e.evaluate_triples(kg.triples).cpu().numpy()
    want = O.evaluate_triples(kg.E.astype(np.float64), kg.triples, np.float64)
    assert np.abs(got - want).max() <= 1e-6
    _check_one_step(e, kg, 1024, side=1)
    e.close()


# ---------------------------------------------------------------- 2. the device loop at the lane-group edges
@pytest.mark.gpu
@pytest.mark.parametrize("dim", [258, 768])
def test_device_loop_matches_per_step_at_lane_group_edges(eng_mod, monkeypatch, dim):
    """hole_train_steps in chunks 1, 2, 4, 1 (HOLE_PLAN_RAMP=1,2) equals the per-step path bit for bit at the
    first v2 lane-group dim (258, partial) and the last v3 dim (768, full), with the oracle re-run at the
    chunk boundaries."""
    from test_gpu_chunked import (MARGIN, _assert_matches_per_step, _engine as chunk_engine, _lrs, _per_step,
                                  boundary_steps, chunk_sizes)
    B, n_steps = 1000, 8
    layout = chunk_sizes(B, n_steps, (1, 2))
    assert layout == [1, 2, 4, 1]
    assert lane_group(dim) in [(32, 2, False), (32, 3, True)]
    kg = D.synthetic_kg(9, 4000, n_steps * B, 5, dim, seed=dim, trained_scale=True, zipf_entities=True)
    seed, first_step = 17, 250
    lrs = _lrs(eng_mod, first_step, n_steps)
    a = chunk_engine(eng_mod, monkeypatch, kg, {"HOLE_PLAN_RAMP": "1,2"})
    tri = torch.from_numpy(kg.triples).to(a.device)
    sums, loss = a.train_steps(tri, B, seed, first_step, MARGIN, lrs, want_loss=True)
    b = chunk_engine(eng_mod, monkeypatch, kg)
    ref = _per_step(b, tri, B, seed, first_step, lrs, check_at=boundary_steps(layout))
    _assert_matches_per_step(f"dim {dim}", a.table, b.table, sums, ref, B, loss)
    assert not torch.equal(a.embeddings().cpu(), torch.from_numpy(kg.E))
    a.close(); b.close()


# ---------------------------------------------------------------- 3. ccorr ranking at NV 8 and NV 12
@pytest.mark.gpu
@pytest.mark.parametrize("dim", [450, 514])
def test_ccorr_rank_counts_exact_vs_own_operands(eng_mod, dim):
    """The archived ccorr mode's query packer at NV 8 (450) and NV 12 (514), reachable only in plain bf16
    (bf16x3 stops at 320): counts exact against an fp64 contraction of the kernel's own operands."""
    from test_gpu_rank import _exact_from_operands
    assert cc_nv(dim)[1] in (8, 12) and rank_stages(dim, 1) is not None and rank_stages(dim, 2) is None
    kg = D.synthetic_kg(6, 2500, 300, 4, dim, seed=dim, trained_scale=True)
    e = _engine(eng_mod, kg, types=False).set_score_mode("ccorr_tanh")
    b, en = kg.n_relations, kg.n_rows
    for side in (0, 1):
        raw, filt, ts = e.rank(kg.triples, side, b, en)
        raw, filt, ts = raw.cpu().numpy(), filt.cpu().numpy(), ts.cpu().numpy()
        _exact_from_operands(e, kg, kg.triples, side, b, en, raw, filt, ts)
        assert raw.max() > 100
    e.close()


# ---------------------------------------------------------------- 4. table-size edges of the update plan
SIZE_EDGES = [255, 256, 65535, 65536, 2**24 - 1, 2**24]
N_REL, TOP = 4, 1000


def _device_table(n_rows, dim, seed):
    """A trained-scale table (row norms ~U(0.5, 1.5)) generated on the device."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn((n_rows, dim), generator=g, device="cuda")
    x *= (0.5 + torch.rand((n_rows, 1), generator=g, device="cuda")) / x.norm(dim=1, keepdim=True)
    return x


def _top_batch(n_rows, B, seed):
    """Triples over the top TOP rows (every entity row of a small table), with the largest id, unique and
    duplicated rows."""
    rng = np.random.default_rng(seed)
    lo = max(N_REL, n_rows - TOP)
    pos = np.stack([rng.integers(lo, n_rows, B), rng.integers(lo, n_rows, B), rng.integers(0, N_REL, B)], 1)
    neg = rng.integers(lo, n_rows, B)
    pos[0, 0] = pos[1, 1] = neg[2] = n_rows - 1
    _, cnt = np.unique(np.concatenate([pos[:, 0], pos[:, 1], neg]), return_counts=True)
    assert (cnt == 1).any() and (cnt > 1).any()
    return pos.astype(np.int32), neg.astype(np.int32)


@pytest.mark.gpu
@pytest.mark.parametrize("n_rows", SIZE_EDGES)
def test_update_plan_at_row_key_pass_edges(eng_mod, monkeypatch, n_rows):
    """One train_step on a table at each edge of the row-key radix pass count (1|2, 2|3, 3|4 passes), under
    HOLE_SORT_SMALL = 0 (radix chain), 1 (adaptive) and 2 (one-launch sort): the three tables are bit-identical;
    the rows the step uses are within the one-step band of the fp64 oracle (run on the sub-table of those rows,
    ids relabelled in order); every other row is bit-unchanged."""
    dim, B, margin, lr = 8, 512, 0.2, 0.1
    side = n_rows % 2
    E0 = _device_table(n_rows, dim, n_rows)
    pos, neg = _top_batch(n_rows, B, n_rows)
    tables, losses = [], []
    for mode in ("0", "1", "2"):
        monkeypatch.setenv("HOLE_SORT_SMALL", mode)
        e = eng_mod.HoleEngine(n_rows, dim)
        monkeypatch.delenv("HOLE_SORT_SMALL")
        e.set_embeddings(E0)
        losses.append(e.train_step(pos, neg, side, margin, lr).cpu().numpy())
        tables.append(e.table)
        e.table = None
        e.close()
    for t, l in zip(tables[1:], losses[1:]):
        assert torch.equal(t, tables[0]) and np.array_equal(l, losses[0])
    e = eng_mod.HoleEngine(n_rows, dim)
    e.table = tables[0]
    got = e.embeddings()
    e.table = None
    e.close()
    del tables
    used = np.unique(np.concatenate([pos.ravel(), neg]))
    used_t = torch.from_numpy(used.astype(np.int64)).to(got.device)
    E64 = E0[used_t].cpu().numpy().astype(np.float64)
    l64, _, _ = O.sgd_step(E64, np.searchsorted(used, pos).astype(np.int32), np.searchsorted(used, neg).astype(np.int32),
                           side, margin, lr, np.float64, "tf")
    assert np.abs(losses[0] - l64).max() <= 2e-6
    sub = got[used_t].cpu().numpy()
    err, tol = np.abs(sub - E64), 2e-6 + 1e-5 * np.abs(E64)
    assert (err <= tol).all(), float((err - tol).max())
    assert np.abs(sub - E0[used_t].cpu().numpy()).max() > 1e-5
    keep = torch.ones(n_rows, dtype=torch.bool, device=got.device)
    keep[used_t] = False
    assert torch.equal(got[keep], E0[keep])


@pytest.mark.gpu
@pytest.mark.parametrize("hint", [None, N_REL])
def test_chunked_steps_at_2_pow_24_rows(eng_mod, monkeypatch, hint):
    """2^24 rows (4 row-key passes): train_steps in chunks 1, 2, 1 (HOLE_PLAN_RAMP=1,2) equals the per-step path
    bit for bit, without a relation-count hint (a 4-pass relation radix chain) and with one.  Corrupt entities
    are drawn from the top TOP rows (their own type), so the high key bytes are set."""
    from test_gpu_chunked import MARGIN, _assert_matches_per_step, _lrs, _per_step, chunk_sizes
    n_rows, dim, B, n_steps = 2**24, 8, 2048, 4
    assert row_passes(n_rows) == 4
    layout = chunk_sizes(B, n_steps, (1, 2))
    assert layout == [1, 2, 1]
    E0 = _device_table(n_rows, dim, 24)
    tri = np.concatenate([_top_batch(n_rows, B, 100 + k)[0] for k in range(n_steps)])
    lo = n_rows - TOP                                        # types: 0 relations, 1 the top rows, 2 the rest
    type_of = np.full(n_rows, 2, np.int32)
    type_of[:N_REL] = 0
    type_of[lo:] = 1
    off = np.array([0, N_REL, N_REL + TOP, n_rows], np.int64)
    ids = np.concatenate([np.arange(N_REL), np.arange(lo, n_rows), np.arange(N_REL, lo)]).astype(np.int32)
    seed, first_step = 2**24 + 1, 77
    lrs = _lrs(eng_mod, first_step, n_steps)

    def make(env):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        e = eng_mod.HoleEngine(n_rows, dim)
        for k in env:
            monkeypatch.delenv(k)
        e.set_embeddings(E0).set_types(type_of, off, ids)
        if hint is not None:
            e.set_relation_count(hint)
        return e

    a = make({"HOLE_PLAN_RAMP": "1,2"})
    t = torch.from_numpy(tri).to(a.device)
    sums, loss = a.train_steps(t, B, seed, first_step, MARGIN, lrs, want_loss=True)
    b = make({})
    ref = _per_step(b, t, B, seed, first_step, lrs)
    _assert_matches_per_step(f"2^24 rows, hint {hint}", a.table, b.table, sums, ref, B, loss)
    _, neg = b.corrupt_batch(tri[:B], seed, first_step)
    assert int(neg.min()) >= lo and int(neg.max()) < n_rows
    assert not torch.equal(a.embeddings()[lo:], E0[lo:])
    a.close(); b.close()
