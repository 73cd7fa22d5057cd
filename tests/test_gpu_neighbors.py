"""Nearest neighbours (hole_neighbors through the C ABI and HoleEngine.neighbors) against the fp64 oracle, the
kernel's own operands, the other library paths and the CLI.

Standards (include/hole_b200.h, hole_neighbors):
  * the selection is exact on the contraction's own bf16 operands except within 2e-6 of the k-th similarity;
  * against the fp64 cosine of the fp32 table the id set is exact except within 3e-5 (bf16x3) / 4e-3 (bf16) of
    the k-th similarity; the returned similarities are within 2e-6 + 1e-5 |s| of the fp64 value of that id;
  * every row is sorted by (-similarity, id), holds neither the query's own row nor a filtered id, and is padded
    with (-1, -inf).
The tables are trained-scale (row norms vary), so cosine order differs from the clipped-dot order of the ranking
operands; test_selection_exact_vs_own_operands asserts that it does in its data.
"""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from graphembeddings_b200 import data as D
import neighbors_reference as N

pytestmark = pytest.mark.gpu

BAND_X3, BAND_BF16 = 3e-5, 4e-3


@pytest.fixture(scope="module")
def eng_mod():
    from graphembeddings_b200 import build
    build.build()
    from graphembeddings_b200 import engine
    return engine


def _setup(eng_mod, n_rel, n_ent, dim, seed, E=None):
    kg = D.synthetic_kg(n_rel, n_ent, 16, 4, dim, seed=seed, trained_scale=True)
    E = kg.E if E is None else E
    return kg, E, eng_mod.HoleEngine(kg.n_rows, kg.dim).set_embeddings(E)


def _np(*ts):
    return tuple(t.cpu().numpy() for t in ts)


def _random_filters(rng, qids, cand, n_max=40):
    fl = [np.sort(rng.choice(cand, size=int(rng.integers(0, n_max)), replace=False)).astype(np.int32) for _ in qids]
    foff = np.concatenate([[0], np.cumsum([len(f) for f in fl])]).astype(np.int64)
    return foff, np.concatenate(fl).astype(np.int32), [f.astype(np.int64) for f in fl]


def _check_rows(ids, sims, S, qids, cand, k, flists, band):
    """ids / sims [Q, k] from the device against fp64 similarities S [Q, len(cand)]."""
    want_ids, want_s = N.neighbors(S, qids, cand, k, flists)
    col = {int(c): j for j, c in enumerate(cand)}
    for q in range(len(S)):
        n = int((want_ids[q] >= 0).sum())
        assert np.all(ids[q, n:] == -1) and np.all(sims[q, n:] == -np.inf), q
        g = ids[q, :n].astype(np.int64)
        assert np.all(g >= 0) and len(set(g.tolist())) == n, q
        assert int(qids[q]) not in g, q
        gs = sims[q, :n].astype(np.float64)
        assert np.isfinite(gs).all(), q
        assert np.all((np.diff(gs) < 0) | ((np.diff(gs) == 0) & (np.diff(g) > 0))), q
        if flists is not None and len(flists[q]):
            assert not np.isin(g, flists[q]).any(), q
        if n == 0:
            continue
        sg = S[q, [col[int(x)] for x in g]]
        assert np.all(np.abs(gs - sg) <= 2e-6 + 1e-5 * np.abs(sg)), (q, np.abs(gs - sg).max())
        kth = want_s[q, n - 1]
        assert np.all(sg >= kth - band), q                              # nothing returned from beyond the band
        assert np.isin(want_ids[q, :n][want_s[q, :n] > kth + band], g).all(), q
    return want_ids, want_s


def test_selection_exact_vs_own_operands(eng_mod):
    """bf16: an fp64 contraction of the operands hole_neighbors packed selects the same ids (2e-6 band); the
    candidate operand is unit-normalised, and on this table that ranks differently from the clipped operand."""
    kg, E, e = _setup(eng_mod, 9, 3000, 150, seed=11)
    b, en = kg.n_relations, kg.n_rows
    rng = np.random.default_rng(1)
    qids = rng.choice(np.arange(b, en), size=300, replace=False)
    k = 20
    ids, _ = _np(*e.neighbors(qids, k, b, en, precision=eng_mod.HOLE_RANK_BF16))
    cand_op, qp = e.rank_debug_operands()
    cand_op, qp = cand_op.double().cpu().numpy()[: en - b], qp.double().cpu().numpy()[: len(qids)]
    assert np.abs(np.linalg.norm(cand_op, axis=1) - 1).max() < 1e-2          # normalised, not clipped
    S = -(qp @ cand_op.T)                                                    # the query operand is negated
    want_ids, want_s = N.neighbors(S, qids - b, np.arange(en - b), k)
    got = ids.astype(np.int64) - b
    for q in range(len(qids)):
        kth = want_s[q, k - 1]
        assert np.all(S[q, got[q]] >= kth - 2e-6), q
        assert np.isin(want_ids[q][want_s[q] > kth + 2e-6], got[q]).all(), q
        assert qids[q] - b not in got[q]
    # what a clipping packer would select: unit query . clip(E_j)
    E64 = E.astype(np.float64)
    nrm = np.linalg.norm(E64, axis=1)
    clipped = E64[b:en] * np.minimum(1.0, 1.0 / nrm[b:en])[:, None]
    Sc = (E64[qids] / nrm[qids, None]) @ clipped.T
    clip_ids, _ = N.neighbors(Sc, qids, np.arange(b, en), k)
    cos_ids, _ = N.neighbors(N.cosine(E, qids, np.arange(b, en)), qids, np.arange(b, en), k)
    differ = sum(set(a.tolist()) != set(c.tolist()) for a, c in zip(clip_ids, cos_ids))
    assert differ > len(qids) // 2, differ


@pytest.mark.parametrize("dim,bf16", [pytest.param(d, False, id=str(d)) for d in (2, 64, 150, 256, 320)] +
                         [pytest.param(640, True, id="640-bf16")])
def test_matches_fp64_oracle(eng_mod, dim, bf16):
    """Q = 300 (not a multiple of 128) over [b + 7, en - 100) (not a multiple of 256), queries inside and outside
    the range, k = 1, 10, 128 with and without a filter; and Q = 1."""
    kg, E, e = _setup(eng_mod, 9, 2600, dim, seed=100 + dim)
    b, en = kg.n_relations + 7, kg.n_rows - 100
    assert (en - b) % 256 != 0
    cand = np.arange(b, en)
    rng = np.random.default_rng(dim)
    qids = rng.choice(kg.n_rows, size=300, replace=False)
    assert ((qids < b) | (qids >= en)).any() and ((qids >= b) & (qids < en)).any()
    S = N.cosine(E, qids, cand)
    foff, fids, flists = _random_filters(rng, qids, cand)
    precision = eng_mod.HOLE_RANK_BF16 if bf16 else eng_mod.HOLE_RANK_BF16X3
    band = BAND_BF16 if bf16 else BAND_X3
    for k in (1, 10, 128):
        ids, sims = _np(*e.neighbors(qids, k, b, en, precision=precision))
        assert ids.shape == (300, k)
        _check_rows(ids, sims, S, qids, cand, k, None, band)
        ids, sims = _np(*e.neighbors(qids, k, b, en, foff, fids, precision=precision))
        _check_rows(ids, sims, S, qids, cand, k, flists, band)
    ids, sims = _np(*e.neighbors(qids[:1], 10, b, en, precision=precision))
    _check_rows(ids, sims, S[:1], qids[:1], cand, 10, None, band)


def test_zero_rows_as_query_and_candidate(eng_mod):
    kg = D.synthetic_kg(5, 2000, 16, 4, 64, seed=21, trained_scale=True)
    E = kg.E.copy()
    zeros = np.array([kg.n_relations + i for i in (0, 3, 250, 251, 1999)])
    E[zeros] = 0.0
    e = eng_mod.HoleEngine(kg.n_rows, kg.dim).set_embeddings(E)
    b, en = kg.n_relations, kg.n_rows
    cand = np.arange(b, en)
    qids = np.concatenate([zeros, np.arange(b + 10, b + 60)])
    S = N.cosine(E, qids, cand)
    for prec, band in ((eng_mod.HOLE_RANK_BF16X3, BAND_X3), (eng_mod.HOLE_RANK_BF16, BAND_BF16)):
        ids, sims = _np(*e.neighbors(qids, 128, b, en, precision=prec))
        _check_rows(ids, sims, S, qids, cand, 128, None, band)
        for q in range(len(zeros)):              # a zero query: every similarity is 0, so the id order
            want = [c for c in cand if c != zeros[q]][:128]
            assert ids[q].tolist() == want and np.all(sims[q] == 0)
        hit = np.isin(ids, zeros)
        assert np.all(sims[hit] == 0)            # a zero candidate has similarity 0 with every row
    # a range that is mostly zero rows: their similarity-0 ties in id order
    E2 = E.copy()
    E2[b + 300:b + 400] = 0.0
    e.set_embeddings(E2)
    e.rank_invalidate()
    q = np.array([b + 5])
    ids, sims = _np(*e.neighbors(q, 128, b + 290, b + 400))
    S2 = N.cosine(E2, q, np.arange(b + 290, b + 400))
    _check_rows(ids, sims, S2, q, np.arange(b + 290, b + 400), 128, None, BAND_X3)
    assert not np.isnan(sims).any()


def test_duplicated_rows_tie_in_id_order(eng_mod):
    """Twins (cos = 1) come first in ascending id order across tiles and work items; the row itself never."""
    kg = D.synthetic_kg(3, 60000, 16, 3, 64, seed=22, trained_scale=True)
    E = kg.E.copy()
    b = kg.n_relations
    groups = []
    for i in range(6):
        ids = [b + 1000 + 7 * i + o for o in (0, 1, 5, 130, 200, 256 * 11 + 3, 256 * 40, 256 * 100 + 129)]
        E[ids] = E[ids[0]] * np.float32(0.5 + i)     # identical rows
        groups.append(ids)
    e = eng_mod.HoleEngine(kg.n_rows, kg.dim).set_embeddings(E)
    for prec in (eng_mod.HOLE_RANK_BF16, eng_mod.HOLE_RANK_BF16X3):
        for g in groups:
            for src in (g[0], g[3]):
                ids, sims = _np(*e.neighbors([src], 12, b, kg.n_rows, precision=prec))
                twins = [x for x in g if x != src]
                assert ids[0, :len(twins)].tolist() == twins, (prec, src)
                assert np.all(sims[0, :len(twins)] == sims[0, 0]) and abs(sims[0, 0] - 1) < 1e-6
                assert src not in ids[0]


def test_relation_range_and_small_ranges(eng_mod):
    kg, E, e = _setup(eng_mod, 40, 1500, 150, seed=23)
    R = kg.n_relations
    rng = np.random.default_rng(3)
    qids = np.concatenate([np.arange(R), rng.choice(np.arange(R, kg.n_rows), size=30, replace=False)])
    cand = np.arange(R)
    S = N.cosine(E, qids, cand)
    ids, sims = _np(*e.neighbors(qids, 10, 0, R))
    _check_rows(ids, sims, S, qids, cand, 10, None, BAND_X3)
    ids, sims = _np(*e.neighbors(qids, 128, 0, R))              # k > R: relation queries get R - 1 rows
    _check_rows(ids, sims, S, qids, cand, 128, None, BAND_X3)
    assert np.all((ids[:R] >= 0).sum(1) == R - 1) and np.all((ids[R:] >= 0).sum(1) == R)
    b, en = R + 100, R + 106                                     # a range of 6 rows, k = 10
    q = np.array([R + 102, R + 500])
    ids, sims = _np(*e.neighbors(q, 10, b, en))
    _check_rows(ids, sims, N.cosine(E, q, np.arange(b, en)), q, np.arange(b, en), 10, None, BAND_X3)
    assert (ids[0] >= 0).sum() == 5 and (ids[1] >= 0).sum() == 6
    ids, sims = _np(*e.neighbors(q, 4, b, b))                    # empty range: all padding
    assert np.all(ids == -1) and np.all(sims == -np.inf)


def test_operand_cache_and_context(eng_mod):
    """prepare -> neighbors -> rank equals rank without the prepare; top-k and neighbours are unchanged by calls of
    the other kind on the same context; the ccorr_tanh score mode gives the same neighbours."""
    kg, E, e = _setup(eng_mod, 7, 3000, 150, seed=24)
    b, en = kg.n_relations, kg.n_rows
    tri = D.synthetic_kg(7, 3000, 260, 4, 8, seed=5, with_embeddings=False).triples
    qids = np.arange(b, b + 500)
    for prec in (eng_mod.HOLE_RANK_BF16, eng_mod.HOLE_RANK_BF16X3):
        e.rank_invalidate()
        r0 = e.rank(tri, 2, b, en, precision=prec)
        t0 = e.topk(tri, 0, b, en, 16, precision=prec)
        n0 = e.neighbors(qids, 16, b, en, precision=prec)
        e.rank_prepare(b, en, precision=prec)
        n1 = e.neighbors(qids, 16, b, en, precision=prec)          # never the prepared clipped operand
        r1 = e.rank(tri, 2, b, en, precision=prec)                 # never the normalised operand
        t1 = e.topk(tri, 0, b, en, 16, precision=prec)
        for x, y in zip(r0 + t0 + n0, r1 + t1 + n1):
            assert torch.equal(x, y), prec
    e.set_score_mode("ccorr_tanh")
    for prec in (eng_mod.HOLE_RANK_BF16, eng_mod.HOLE_RANK_BF16X3):
        n2 = e.neighbors(qids, 16, b, en, precision=prec)
        e.set_score_mode("complex")
        n3 = e.neighbors(qids, 16, b, en, precision=prec)
        e.set_score_mode("ccorr_tanh")
        assert torch.equal(n2[0], n3[0]) and torch.equal(n2[1], n3[1])


@pytest.mark.parametrize("precision", [0, 1])
def test_interleaved_with_topk_and_rank_over_many_chunks(eng_mod, precision):
    """Neighbours directly after hole_topk and hole_rank on the same context (each re-packs the shared candidate
    buffer and overwrites the shared query workspace), with Q = 1000 (not a multiple of 128) over 20,000 rows:
    8 query tiles and 9 candidate chunks per tile, so every query row merges 18 partial lists."""
    kg, E, e = _setup(eng_mod, 6, 20000, 64, seed=27)
    b, en = kg.n_relations, kg.n_rows
    rng = np.random.default_rng(8)
    qids = rng.choice(np.arange(b, en), size=1000, replace=False)
    tri = D.synthetic_kg(6, 20000, 1000, 4, 8, seed=9, with_embeddings=False).triples
    cand = np.arange(b, en)
    S = N.cosine(E, qids, cand)
    band = BAND_BF16 if precision == 0 else BAND_X3
    t0 = e.topk(tri, 0, b, en, 10, precision=precision)
    n0 = e.neighbors(qids, 10, b, en, precision=precision)           # right after hole_topk
    _check_rows(*_np(*n0), S, qids, cand, 10, None, band)
    r0 = e.rank(tri, 0, b, en, precision=precision)
    n1 = e.neighbors(qids, 10, b, en, precision=precision)           # right after hole_rank
    t1 = e.topk(tri, 0, b, en, 10, precision=precision)             # right after neighbours
    r1 = e.rank(tri, 0, b, en, precision=precision)
    for x, y in zip(n0 + t0 + r0, n1 + t1 + r1):
        assert torch.equal(x, y), precision


@pytest.mark.parametrize("dim,precision", [(642, 0), (322, 1)])
def test_refusals_leave_outputs_and_context_intact(eng_mod, dim, precision):
    kg, E, e = _setup(eng_mod, 3, 400, dim, seed=25)
    ids = torch.arange(3, 13, dtype=torch.int32, device="cuda")
    out = torch.full((10, 5), 12345, dtype=torch.int32, device="cuda")
    sim = torch.full((10, 5), 7.0, dtype=torch.float32, device="cuda")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    n0 = e.launch_count()
    rc = e.lib.hole_neighbors(e._ctx, C.c_void_p(e.table.data_ptr()), 3, kg.n_rows, C.c_void_p(ids.data_ptr()), 10,
                              precision, 5, None, None, C.c_void_p(out.data_ptr()), C.c_void_p(sim.data_ptr()), st)
    assert rc == -4
    torch.cuda.synchronize()
    assert torch.all(out == 12345) and torch.all(sim == 7.0)
    with pytest.raises(eng_mod.HoleError, match=f"embedding_dim {dim}"):
        e.neighbors(ids, 5, 3, kg.n_rows, precision=precision)
    assert e.launch_count() == n0
    # the context stays usable
    sig = e.evaluate_triples(kg.triples).cpu().numpy()
    assert np.isfinite(sig).all()
    if dim == 322:
        got, s = _np(*e.neighbors(ids, 5, 3, kg.n_rows, precision=eng_mod.HOLE_RANK_BF16))
        q = ids.cpu().numpy()
        _check_rows(got, s, N.cosine(E, q, np.arange(3, kg.n_rows)), q, np.arange(3, kg.n_rows), 5, None, BAND_BF16)


def test_argument_errors(eng_mod):
    kg, E, e = _setup(eng_mod, 3, 300, 64, seed=26)
    ids = torch.arange(3, 13, dtype=torch.int32, device="cuda")
    out = torch.empty((10, 129), dtype=torch.int32, device="cuda")
    sim = torch.empty((10, 129), dtype=torch.float32, device="cuda")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for k in (0, 129):
        rc = e.lib.hole_neighbors(e._ctx, C.c_void_p(e.table.data_ptr()), 3, 303, C.c_void_p(ids.data_ptr()), 10, 1,
                                  k, None, None, C.c_void_p(out.data_ptr()), C.c_void_p(sim.data_ptr()), st)
        assert rc == -1, k
        with pytest.raises(eng_mod.HoleError):
            e.neighbors(ids, k, 3, 303)
    for bad in ([-1], [5, kg.n_rows]):
        with pytest.raises(eng_mod.HoleError, match="must lie in"):
            e.neighbors(np.array(bad), 5, 3, 303)
    with pytest.raises(eng_mod.HoleError):                 # filter slice not ascending
        e.neighbors([10], 5, 3, 303, np.array([0, 2]), np.array([50, 40]))


# ---------------------------------------------------------------------------------------------- CLI
@pytest.fixture(scope="module")
def trained_dir(eng_mod, tmp_path_factory):
    from graphembeddings_b200 import hole
    from test_gpu_cli import _write_data_dir
    tmp = tmp_path_factory.mktemp("neighbors_cli")
    kg = D.synthetic_kg(8, 1500, 9000, 4, 64, seed=3, with_embeddings=False)
    d = tmp / "data"; d.mkdir()
    parts = _write_data_dir(str(d), kg, 600, 400)
    out = str(tmp / "run")
    args = ["--data_dir", str(d), "--output_dir", out, "--batch_size", "256", "--embedding_dim", "64",
            "--num_epochs", "2"]
    hole.main(args)
    return tmp, kg, parts, args, out


def test_cli_nearest_neighbors(eng_mod, trained_dir):
    from graphembeddings_b200 import hole, tf_bundle
    tmp, kg, parts, args, out = trained_dir
    path = os.path.join(out, "neighbors.tsv")
    logged = []
    cwd = os.getcwd()
    os.chdir(tmp)
    try:
        hole.infer_triples(hole.build_parser().parse_args(args + ["--infer", "--nearest_neighbors", "5"]),
                           log=lambda *a: logged.append(" ".join(map(str, a))))
    finally:
        os.chdir(cwd)
    rows = [line.rstrip("\n").split("\t") for line in open(path)]
    test = parts["test_positive_triples.txt"]
    ents, rels = np.unique(test[:, :2]), np.unique(test[:, 2])
    assert len(rows) == 5 * (len(ents) + len(rels))
    assert any(f"Wrote {len(rows)} nearest-neighbour lines" in m for m in logged)
    assert all(len(r) == 7 for r in rows)
    E = tf_bundle.load_bundle(os.path.join(out, "model.ckpt"))["embeddings"]
    e = eng_mod.HoleEngine(kg.n_rows, 64).set_embeddings(E)
    R = kg.n_relations
    for kind, qids, lo, hi in (("entity", ents, R, kg.n_rows), ("relation", rels, 0, R)):
        want_ids, want_s = _np(*e.neighbors(qids, 5, lo, hi))
        mine = {}
        for r in rows:
            if r[0] == kind:
                mine.setdefault(int(r[1]), []).append(r)
        assert sorted(mine) == qids.tolist()
        for i, q in enumerate(qids.tolist()):
            got = mine[q]
            assert [int(g[3]) for g in got] == [1, 2, 3, 4, 5]
            assert [int(g[2]) for g in got] == want_ids[i].tolist()
            sims = [float(g[4]) for g in got]
            assert np.all(np.diff(sims) <= 0)
            assert np.allclose(sims, want_s[i], rtol=0, atol=1e-7)
            assert all(g[5] == f"id{q} name{q}" and g[6] == f"id{g[2]} name{g[2]}" for g in got)
