"""Top-k link prediction (hole_topk through the C ABI and HoleEngine.topk) against the fp64 oracle, the
kernel's own operands, the other library paths and the CLI.

Standards (include/hole_b200.h, hole_topk):
  * the selection is exact on the contraction's own bf16 operands except within 2e-6 of the k-th score;
  * against the fp64 oracle on the fp32 table (split-bf16 operands) the id set is exact except within 3e-5
    of the k-th score; the returned fp32 scores are within 2e-6 + 1e-5 |s| of the fp64 score of that id;
  * every row is sorted by (score, id) and padded with (-1, +inf).
"""
import os

import numpy as np
import pytest
import torch

from graphembeddings_b200 import data as D
from oracle import hole_ccorr as OC
from oracle import hole_oracle as O
import topk_reference as T

pytestmark = pytest.mark.gpu

BAND_X3 = 3e-5


@pytest.fixture(scope="module")
def eng_mod():
    from graphembeddings_b200 import build
    build.build()
    from graphembeddings_b200 import engine
    return engine


def _setup(eng_mod, n_rel, n_ent, n_q, dim, seed):
    kg = D.synthetic_kg(n_rel, n_ent, n_q, 4, dim, seed=seed, trained_scale=True)
    return kg, eng_mod.HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E)


def _filter_lists(foff, fids):
    if foff is None:
        return None
    return [fids[foff[q]:foff[q + 1]].astype(np.int64) for q in range(len(foff) - 1)]


def _check_rows(ids, scores, S, cand, k, flists, band, score_tol=True):
    """ids / scores [R, k] from the device against fp64 scores S [R, len(cand)] of candidates cand."""
    want_ids, want_s = T.topk(S, cand, k, flists)
    col = {int(c): j for j, c in enumerate(cand)}
    for q in range(len(S)):
        n = int((want_ids[q] >= 0).sum())
        got = ids[q]
        assert np.all(got[n:] == -1) and np.all(np.isinf(scores[q, n:])), q
        g = got[:n].astype(np.int64)
        assert np.all(g >= 0) and len(set(g.tolist())) == n, q
        # sorted by (score, id)
        gs = scores[q, :n].astype(np.float64)
        assert np.all((np.diff(gs) > 0) | ((np.diff(gs) == 0) & (np.diff(g) > 0))), q
        if flists is not None and len(flists[q]):
            assert not np.isin(g, flists[q]).any(), q
        if n == 0:
            continue
        sg = S[q, [col[int(x)] for x in g]]
        if score_tol:
            assert np.all(np.abs(gs - sg) <= 2e-6 + 1e-5 * np.abs(sg)), (q, np.abs(gs - sg).max())
        kth = want_s[q, n - 1]
        assert np.all(sg <= kth + band), q                              # nothing returned from beyond the band
        sure = want_ids[q, :n][want_s[q, :n] < kth - band]
        assert np.isin(sure, g).all(), q                                # everything clearly inside is returned
    return want_ids, want_s


def _oracle_scores(E64, queries, side, cand):
    if side == 2:
        return np.concatenate([O.all_scores(E64, queries, "tail", cand, np.float64),
                               O.all_scores(E64, queries, "head", cand, np.float64)])
    return O.all_scores(E64, queries, "tail" if side == 0 else "head", cand, np.float64)


def _filters(kg, queries, side, seed):
    known = D.synthetic_kg(kg.n_relations, kg.n_entities, 20000, 4, 8, seed=seed, with_embeddings=False).triples
    if side == 2:
        ft = D.build_filter_csr(queries, known, "tail")
        fh = D.build_filter_csr(queries, known, "head")
        return np.concatenate([ft[0], fh[0][1:] + ft[0][-1]]), np.concatenate([ft[1], fh[1]])
    return D.build_filter_csr(queries, known, "tail" if side == 0 else "head")


@pytest.mark.parametrize("side", [0, 1])
def test_selection_exact_vs_own_operands(eng_mod, side):
    """bf16 operands: an fp64 contraction of the operands hole_topk packed selects the same ids (2e-6 band)."""
    kg, e = _setup(eng_mod, 9, 3000, 300, 150, seed=70 + side)
    b, en = kg.n_relations, kg.n_rows
    foff, fids = _filters(kg, kg.triples, side, 95)
    k = 20
    ids, sc = e.topk(kg.triples, side, b, en, k, foff, fids, precision=eng_mod.HOLE_RANK_BF16)
    cand_op, qp = e.rank_debug_operands()
    S = qp.double().cpu().numpy()[: len(kg.triples)] @ cand_op.double().cpu().numpy()[: en - b].T
    local = [f.astype(np.int64) - b for f in _filter_lists(foff, fids)]
    got = ids.cpu().numpy().astype(np.int64) - b
    got[ids.cpu().numpy() < 0] = -1
    want_ids, want_s = T.topk(S, np.arange(en - b), k, local)
    for q in range(len(S)):
        g = got[q][got[q] >= 0]
        kth = want_s[q, k - 1]
        assert np.all(S[q, g] <= kth + 2e-6)
        assert np.isin(want_ids[q][want_s[q] < kth - 2e-6], g).all()


@pytest.mark.parametrize("dim,bf16", [pytest.param(d, False, id=str(d)) for d in (64, 150, 256, 2, 320)] +
                         [pytest.param(640, True, id="640-bf16")])
@pytest.mark.parametrize("side", [0, 1, 2])
def test_topk_matches_fp64_oracle(eng_mod, dim, bf16, side):
    """Split-bf16: Q = 300 (not a multiple of 128) over [b + 7, en - 100) (not a multiple of 256), filtered,
    k = 1, 10, 128; and Q = 1.  Dims 2 and 320 are the smallest and the largest bf16x3 builds; 640, the largest
    plain bf16 build (3 query-packer iterations, 2-stage ring), runs in bf16: there the id set is exact outside
    the bf16 score bound 4e-3 |q| |e| of the k-th score (|e| <= 1 after the clip), and the returned scores, which
    the merge kernel recomputes in fp32, keep the fp32 tolerance."""
    kg, e = _setup(eng_mod, 9, 2600, 300, dim, seed=80 + dim + side)
    b, en = kg.n_relations + 7, kg.n_rows - 100
    assert (en - b) % 256 != 0
    cand = np.arange(b, en)
    E64 = kg.E.astype(np.float64)
    S = _oracle_scores(E64, kg.triples, side, cand)
    foff, fids = _filters(kg, kg.triples, side, 94)
    precision = eng_mod.HOLE_RANK_BF16 if bf16 else eng_mod.HOLE_RANK_BF16X3
    band = BAND_X3
    if bf16:
        sides = ("tail", "head") if side == 2 else (("tail",) if side == 0 else ("head",))
        qn = max(np.linalg.norm(O.query_vectors(E64, kg.triples, s, np.float64), axis=1).max() for s in sides)
        band = 4e-3 * qn
    for k in (1, 10, 128):
        ids, sc = e.topk(kg.triples, side, b, en, k, foff, fids, precision=precision)
        assert ids.shape == (S.shape[0], k)
        _check_rows(ids.cpu().numpy(), sc.cpu().numpy(), S, cand, k, _filter_lists(foff, fids), band)
    ids, sc = e.topk(kg.triples[:1], side, b, en, 10, precision=precision)
    S1 = _oracle_scores(E64, kg.triples[:1], side, cand)
    _check_rows(ids.cpu().numpy(), sc.cpu().numpy(), S1, cand, 10, None, band)


def test_k_larger_than_the_candidates_pads(eng_mod):
    kg, e = _setup(eng_mod, 5, 800, 40, 64, seed=3)
    b, en = kg.n_relations + 100, kg.n_relations + 150
    cand = np.arange(b, en)
    S = _oracle_scores(kg.E.astype(np.float64), kg.triples, 0, cand)
    ids, sc = e.topk(kg.triples, 0, b, en, 100)
    ids, sc = ids.cpu().numpy(), sc.cpu().numpy()
    assert np.all(ids[:, 50:] == -1) and np.all(np.isinf(sc[:, 50:])) and np.all(ids[:, :50] >= b)
    _check_rows(ids, sc, S, cand, 100, None, BAND_X3)
    ids, sc = e.topk(kg.triples, 0, b, b, 5)                 # empty range: all padding
    assert torch.all(ids == -1) and torch.all(torch.isinf(sc))


def test_many_chunks(eng_mod):
    """Q <= 3 over 400 k candidates: hundreds of work items, each with two partial lists, merged."""
    kg, e = _setup(eng_mod, 4, 400_000, 3, 64, seed=12)
    b, en = kg.n_relations, kg.n_rows
    cand = np.arange(b, en)
    S = _oracle_scores(kg.E.astype(np.float64), kg.triples, 0, cand)
    rng = np.random.default_rng(1)
    fl = [np.sort(rng.choice(cand, size=5000, replace=False)).astype(np.int32) for _ in range(3)]
    foff = np.concatenate([[0], np.cumsum([len(f) for f in fl])]).astype(np.int64)
    fids = np.concatenate(fl)
    for k in (10, 128):
        ids, sc = e.topk(kg.triples, 0, b, en, k, foff, fids)
        _check_rows(ids.cpu().numpy(), sc.cpu().numpy(), S, cand, k, _filter_lists(foff, fids), BAND_X3)


def test_exact_ties_go_to_the_smaller_id(eng_mod):
    """Duplicated candidate rows score bit-identically: copies inside one tile, across the two column halves
    of a tile and across work items must come out in ascending id order."""
    n_rel, n_ent, dim = 3, 60000, 64
    kg = D.synthetic_kg(n_rel, n_ent, 4, 3, dim, seed=21, trained_scale=True)
    E = kg.E.copy()
    qv = O.query_vectors(E.astype(np.float64), kg.triples, "tail", np.float64)
    offs = [0, 1, 5, 130, 200, 256 * 11 + 3, 256 * 40, 256 * 100 + 129]
    groups = []
    for i in range(len(kg.triples)):
        base = n_rel + 1000 + 7 * i          # groups interleave but never collide
        row = (-qv[i] / np.linalg.norm(qv[i]) * 0.9).astype(np.float32)
        ids = [base + o for o in offs]
        E[ids] = row
        groups.append(ids)
    e = eng_mod.HoleEngine(kg.n_rows, dim).set_embeddings(E)
    b, en = n_rel, kg.n_rows
    for prec in (eng_mod.HOLE_RANK_BF16, eng_mod.HOLE_RANK_BF16X3):
        ids, sc = e.topk(kg.triples, 0, b, en, 12, precision=prec)
        ids, sc = ids.cpu().numpy(), sc.cpu().numpy()
        for i, g in enumerate(groups):
            assert ids[i, :len(g)].tolist() == sorted(g), (prec, i)
            assert np.all(sc[i, :len(g)] == sc[i, 0])


def test_filter_excludes_and_pads(eng_mod):
    kg, e = _setup(eng_mod, 5, 1200, 50, 64, seed=33)
    b, en = kg.n_relations, kg.n_relations + 300
    cand = np.arange(b, en)
    rng = np.random.default_rng(2)
    keep = [np.sort(rng.choice(cand, size=4, replace=False)) for _ in range(len(kg.triples))]
    fl = [np.setdiff1d(cand, kp).astype(np.int32) for kp in keep]    # all but 4 candidates filtered
    foff = np.concatenate([[0], np.cumsum([len(f) for f in fl])]).astype(np.int64)
    ids, sc = e.topk(kg.triples, 0, b, en, 10, foff, np.concatenate(fl))
    ids, sc = ids.cpu().numpy(), sc.cpu().numpy()
    for q in range(len(kg.triples)):
        assert sorted(ids[q, :4].tolist()) == keep[q].tolist()
        assert np.all(ids[q, 4:] == -1) and np.all(np.isinf(sc[q, 4:]))
    # with and without a filter: the filtered list is the unfiltered one with the filtered ids removed
    kg, e = _setup(eng_mod, 5, 3000, 100, 150, seed=34)
    b, en = kg.n_relations, kg.n_rows
    foff, fids = _filters(kg, kg.triples, 0, 93)
    fl = _filter_lists(foff, fids)
    idf, scf = e.topk(kg.triples, 0, b, en, 10, foff, fids)
    idn, scn = e.topk(kg.triples, 0, b, en, 128)
    idf, scf, idn, scn = idf.cpu().numpy(), scf.cpu().numpy(), idn.cpu().numpy(), scn.cpu().numpy()
    for q in range(len(kg.triples)):
        keep_n = ~np.isin(idn[q], fl[q])
        want, want_s = idn[q][keep_n][:10], scn[q][keep_n][:10]
        assert len(want) == 10
        same = idf[q] == want
        assert np.all(same | (np.abs(scf[q] - want_s) <= 2 * BAND_X3)), q
        assert np.array_equal(scf[q][same], want_s[same])


def test_consistent_with_score_and_rank(eng_mod):
    """The returned score is hole_score's triple score; hole_rank with a prediction as the true candidate
    (same filter) puts it at the prediction's position."""
    kg, e = _setup(eng_mod, 7, 2500, 200, 150, seed=41)
    b, en = kg.n_relations, kg.n_rows
    foff, fids = _filters(kg, kg.triples, 0, 92)
    k = 8
    ids, sc = e.topk(kg.triples, 0, b, en, k, foff, fids)
    ids, sc = ids.cpu().numpy(), sc.cpu().numpy().astype(np.float64)
    Q = len(kg.triples)
    tri = np.repeat(kg.triples, k, axis=0)
    tri[:, 1] = ids.reshape(-1)
    sig = e.evaluate_triples(tri).cpu().numpy().astype(np.float64)
    assert np.abs(sig - 1.0 / (1.0 + np.exp(-sc.reshape(-1)))).max() <= 1e-6
    # rank each prediction: filtered count before it == its position
    foff_k = np.concatenate([[0], np.cumsum(np.repeat(np.diff(foff), k))]).astype(np.int64)
    fids_k = np.concatenate([fids[foff[q]:foff[q + 1]] for q in range(Q) for _ in range(k)]).astype(np.int32)
    _, filt, _ = e.rank(tri, 0, b, en, foff_k, fids_k, precision=eng_mod.HOLE_RANK_BF16X3)
    filt = filt.cpu().numpy().reshape(Q, k)
    S = _oracle_scores(kg.E.astype(np.float64), kg.triples, 0, np.arange(b, en))
    checked = 0
    for q in range(Q):
        s = np.sort(S[q][~np.isin(np.arange(b, en), fids[foff[q]:foff[q + 1]])])[: k + 1]
        if np.min(np.diff(s)) > 2 * BAND_X3:           # no near-tie around the top k
            assert filt[q].tolist() == list(range(k)), q
            checked += 1
    assert checked > Q // 4


def test_prepared_cache_and_determinism(eng_mod):
    kg, e = _setup(eng_mod, 7, 3000, 260, 150, seed=43)
    b, en = kg.n_relations, kg.n_rows
    foff, fids = _filters(kg, kg.triples, 2, 91)
    for prec in (eng_mod.HOLE_RANK_BF16, eng_mod.HOLE_RANK_BF16X3):
        e.rank_invalidate()
        i0, s0 = e.topk(kg.triples, 2, b, en, 16, foff, fids, precision=prec)
        i1, s1 = e.topk(kg.triples, 2, b, en, 16, foff, fids, precision=prec)
        e.rank_prepare(b, en, precision=prec)
        i2, s2 = e.topk(kg.triples, 2, b, en, 16, foff, fids, precision=prec)
        assert torch.equal(i0, i1) and torch.equal(s0, s1)
        assert torch.equal(i0, i2) and torch.equal(s0, s2)
    e.rank_invalidate()


@pytest.mark.parametrize("side", [0, 1])
def test_ccorr_tanh_mode(eng_mod, side):
    kg, e = _setup(eng_mod, 6, 1500, 120, 64, seed=47 + side)
    e.set_score_mode("ccorr_tanh")
    b, en = kg.n_relations, kg.n_rows
    cand = np.arange(b, en)
    S = OC.all_scores(kg.E.astype(np.float64), kg.triples, "tail" if side == 0 else "head", cand, np.float64)
    foff, fids = _filters(kg, kg.triples, side, 90)
    ids, sc = e.topk(kg.triples, side, b, en, 10, foff, fids)
    ids, sc = ids.cpu().numpy(), sc.cpu().numpy()
    _check_rows(ids, sc, S, cand, 10, _filter_lists(foff, fids), BAND_X3)
    tri = np.repeat(kg.triples, 10, axis=0)
    tri[:, 1 if side == 0 else 0] = ids.reshape(-1)
    th = e.evaluate_triples(tri).cpu().numpy().astype(np.float64)
    assert np.abs(th - np.tanh(sc.reshape(-1).astype(np.float64))).max() <= 1e-6


def test_error_codes(eng_mod):
    import ctypes as C
    kg, e = _setup(eng_mod, 3, 300, 10, 64, seed=1)
    for k in (0, 129):
        with pytest.raises(eng_mod.HoleError):
            e.topk(kg.triples, 0, 3, 303, k)
    q = torch.as_tensor(kg.triples).cuda()
    out = torch.empty((10, 5), dtype=torch.int32, device="cuda")
    sco = torch.empty((10, 5), dtype=torch.float32, device="cuda")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for a, b in ((None, sco), (out, None)):
        rc = e.lib.hole_topk(e._ctx, C.c_void_p(e.table.data_ptr()), 3, 303, C.c_void_p(q.data_ptr()), 10, 0, 1, 5,
                             None, None, None if a is None else C.c_void_p(a.data_ptr()),
                             None if b is None else C.c_void_p(b.data_ptr()), st)
        assert rc == -1
    with pytest.raises(eng_mod.HoleError):                 # filter slice not ascending
        e.topk(kg.triples[:1], 0, 3, 303, 5, np.array([0, 2]), np.array([50, 40]))


# ---------------------------------------------------------------------------------------------- CLI
def _write_data_dir(d, kg, n_valid, n_test):
    with open(os.path.join(d, "entity_metadata.tsv"), "w") as f:
        f.write("Index\tId\tName\tType\n")
        for i in range(kg.n_rows):
            f.write(f"{i}\tid{i}\tname{i}\t{'RELATION' if i < kg.n_relations else 'T%d' % kg.type_of[i]}\n")
    with open(os.path.join(d, "relation_ids.txt"), "w") as f:
        for r in range(kg.n_relations):
            f.write(f"rel{r}\t{r}\n")
    n = len(kg.triples)
    parts = {"triples.txt": kg.triples[: n - n_valid - n_test],
             "triples-valid.txt": kg.triples[n - n_valid - n_test: n - n_test],
             "test_positive_triples.txt": kg.triples[n - n_test:]}
    for name, tr in parts.items():
        np.savetxt(os.path.join(d, name), tr, fmt="%d", delimiter="\t")
    return parts


@pytest.fixture(scope="module")
def trained_dir(eng_mod, tmp_path_factory):
    from graphembeddings_b200 import hole
    tmp = tmp_path_factory.mktemp("topk_cli")
    kg = D.synthetic_kg(8, 1500, 9000, 4, 64, seed=3, with_embeddings=False)
    d = tmp / "data"; d.mkdir()
    parts = _write_data_dir(str(d), kg, 600, 400)
    out = str(tmp / "run")
    args = ["--data_dir", str(d), "--output_dir", out, "--batch_size", "256", "--embedding_dim", "64",
            "--num_epochs", "2"]
    hole.main(args)
    return tmp, kg, parts, args, out


def test_cli_predict_top_k(trained_dir):
    from graphembeddings_b200 import hole, tf_bundle
    tmp, kg, parts, args, out = trained_dir
    pred = os.path.join(out, "predictions.tsv")
    cwd = os.getcwd()
    os.chdir(tmp)
    try:
        hole.infer_triples(hole.build_parser().parse_args(args + ["--infer"]), log=lambda *a: None)
        assert not os.path.exists(pred)
        hole.infer_triples(hole.build_parser().parse_args(args + ["--infer", "--predict_top_k", "3"]),
                           log=lambda *a: None)
    finally:
        os.chdir(cwd)
    rows = [line.rstrip("\n").split("\t") for line in open(pred)]
    E64 = tf_bundle.load_bundle(os.path.join(out, "model.ckpt"))["embeddings"].astype(np.float64)
    test = parts["test_positive_triples.txt"]
    known = np.concatenate([parts["triples.txt"], parts["triples-valid.txt"]])
    test_set = set(map(tuple, test.tolist()))
    cand = np.arange(kg.n_relations, kg.n_rows)
    n_lines = 0
    for side, kc in (("tail", 0), ("head", 1)):
        pairs = np.unique(test[:, [kc, 2]], axis=0)
        q = np.zeros((len(pairs), 3), dtype=np.int32)
        q[:, kc], q[:, 2] = pairs[:, 0], pairs[:, 1]
        S = O.all_scores(E64, q, side, cand, np.float64)
        foff, fids = D.build_filter_csr(q, known, side)
        want_ids, want_s = T.topk(S, cand, 3, _filter_lists(foff, fids))
        mine = {}
        for r_ in rows:
            if r_[0] == side:
                h, t, r, pos = int(r_[1]), int(r_[2]), int(r_[3]), int(r_[4])
                mine.setdefault((h if side == "tail" else t, r), []).append((pos, h, t, float(r_[5]), float(r_[6]),
                                                                            r_[7]))
        assert len(mine) == len(pairs)
        for i, (a, r) in enumerate(pairs.tolist()):
            got = sorted(mine[(a, r)])
            assert [g[0] for g in got] == [1, 2, 3]
            gid = [g[2] if side == "tail" else g[1] for g in got]
            for (pos, h, t, s, v, it), c, ws in zip(got, gid, want_s[i]):
                assert abs(s - S[i, c - kg.n_relations]) <= 2e-6 + 1e-5 * abs(s)
                assert abs(v - 1.0 / (1.0 + np.exp(-s))) <= 1e-6
                assert it == str((h, t, r) in test_set)
            kth = want_s[i, 2]
            assert np.all(S[i, np.array(gid) - kg.n_relations] <= kth + BAND_X3)
            assert np.isin(want_ids[i][want_s[i] < kth - BAND_X3], gid).all()
            n_lines += 3
    assert n_lines == len(rows)
