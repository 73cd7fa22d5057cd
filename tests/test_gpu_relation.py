"""Relation prediction (HOLE_SIDE_RELATION through hole_rank / hole_rank_ex / hole_topk, HoleEngine and the CLI)
against the kernel's own operands, the fp64 statement of tests/relation_reference.py and the other library paths.

Standards (tests/test_gpu_rank.py, tests/test_gpu_topk.py):
  * counts are exact against an fp64 contraction of the kernel's own bf16 operands outside +-2e-6 of the threshold;
  * split-bf16 counts are exact against the fp64 oracle outside +-3e-5 of the threshold, MRR within 1e-4;
  * top-k: the id set is exact outside 3e-5 of the k-th score, scores within 2e-6 + 1e-5 |s|, rows sorted by
    (score, id), filtered, padded with (-1, +inf).
"""
import math
import os

import numpy as np
import pytest
import torch

from graphembeddings_b200 import data as D
from oracle import hole_oracle as O
import relation_reference as RR
from test_gpu_shapes import cc_nv, pq_iters, rank_stages
from test_gpu_topk import _check_rows, _filter_lists

pytestmark = pytest.mark.gpu

REL = 3                              # HOLE_SIDE_RELATION
BAND_X3 = 3e-5
OWN_DIMS = [2, 150, 258, 640]        # plain bf16: query-packer iterations 1, 1, 2, 3
CCORR_DIMS = [2, 128, 150, 256, 320, 450, 640]     # ccorr query-packer NV 1, 2, 3, 4, 6, 8, 12


@pytest.fixture(scope="module")
def eng_mod():
    from graphembeddings_b200 import build
    build.build()
    from graphembeddings_b200 import engine
    return engine


def _setup(eng_mod, n_rel, n_ent, n_q, dim, seed, rel_range=None):
    """Synthetic table and queries; rel_range = (lo, hi) moves every query's relation into [lo, hi)."""
    kg = D.synthetic_kg(n_rel, n_ent, n_q, 4, dim, seed=seed, trained_scale=True)
    if rel_range is not None:
        kg.triples[:, 2] = np.random.default_rng(seed).integers(*rel_range, size=len(kg.triples))
    return kg, eng_mod.HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E)


def _known(kg, seed):
    """Known triples sharing the queries' (h, t) pairs (several relations each, duplicates, some the query's own),
    plus unrelated ones."""
    rng = np.random.default_rng(seed)
    q = kg.triples
    sel = q[rng.random(len(q)) < 0.6]
    parts = [np.stack([sel[:, 0], sel[:, 1], rng.integers(0, kg.n_relations, len(sel))], 1) for _ in range(3)]
    parts.append(sel[: len(sel) // 4])
    parts.append(D.synthetic_kg(kg.n_relations, kg.n_entities, 5000, 4, 8, seed=seed, with_embeddings=False).triples)
    return np.concatenate(parts).astype(np.int32)


def _own_operand_check(e, queries, b, en, raw, filt, ts, foff=None, fids=None, eps=2e-6):
    """Counts against an fp64 contraction of the operands the last call packed (test_gpu_rank's standard)."""
    cand, qp = e.rank_debug_operands()
    S = qp.double().cpu().numpy()[: len(queries)] @ cand.double().cpu().numpy()[: en - b].T
    tj = queries[:, 2].astype(np.int64) - b
    thr = S[np.arange(len(queries)), tj]
    assert np.abs(ts - thr).max() < eps
    ids = np.arange(S.shape[1])
    lo = (S < thr[:, None] - eps).sum(1)
    hi = (S <= thr[:, None] + eps).sum(1) - 1
    exact = ((S < thr[:, None]) | ((S == thr[:, None]) & (ids[None, :] < tj[:, None]))).sum(1)
    assert np.all(raw >= lo) and np.all(raw <= hi)
    assert np.all((raw == exact) | (hi > lo))
    if foff is not None:
        for q in range(len(queries)):
            f = fids[foff[q]:foff[q + 1]].astype(np.int64) - b
            f = f[(f >= 0) & (f < S.shape[1])]
            before = (S[q, f] < thr[q]) | ((S[q, f] == thr[q]) & (f < tj[q]))
            sure = int((S[q, f] < thr[q] - eps).sum())
            maybe = int((S[q, f] <= thr[q] + eps).sum())
            assert raw[q] - maybe <= filt[q] <= raw[q] - sure
            if hi[q] == lo[q]:
                assert filt[q] == raw[q] - int(before.sum())
    return S


def _oracle_check(S, cand, queries, raw, filt, ts, foff, fids, band=BAND_X3, true_tol=True):
    """Split-bf16 counts against fp64 scores S [Q, len(cand)]: exact outside the band, MRR within 1e-4."""
    tj = queries[:, 2].astype(np.int64) - cand[0]
    thr = S[np.arange(len(queries)), tj]
    if true_tol:
        assert np.abs(ts - thr).max() < band
    lo = (S < thr[:, None] - band).sum(1)
    hi = (S <= thr[:, None] + band).sum(1) - 1
    oraw, ofilt = O.rank_counts(S, cand, queries[:, 2], _filter_lists(foff, fids))
    assert np.all(raw >= lo) and np.all(raw <= hi)
    assert np.all((raw == oraw) | (hi > lo))
    assert np.all((filt == ofilt) | (hi > lo))
    assert np.all(filt <= raw) and np.all(filt >= 0)
    got, want = O.score_mrr(raw + 1, filt + 1), O.score_mrr(oraw + 1, ofilt + 1)
    for key in ("raw_mrr", "filtered_mrr"):
        assert abs(got[key] - want[key]) <= 1e-4, (key, got, want)


def _np(*ts):
    return [t.cpu().numpy() for t in ts]


# ---------------------------------------------------------------------------------------------- counts
def test_dims_reach_every_query_packer():
    assert {pq_iters(d) for d in OWN_DIMS} == {1, 2, 3} and max(OWN_DIMS) == 640 and rank_stages(640, 1) == 2
    assert {cc_nv(d)[1] for d in CCORR_DIMS} == {1, 2, 3, 4, 6, 8, 12}
    assert all(rank_stages(d, 1) for d in CCORR_DIMS) and rank_stages(320, 2) == 2


@pytest.mark.parametrize("dim", OWN_DIMS)
def test_counts_exact_vs_own_operands(eng_mod, dim):
    kg, e = _setup(eng_mod, 300, 2000, 700, dim, seed=dim)
    foff, fids = D.build_filter_csr(kg.triples, _known(kg, dim), "relation")
    assert (np.diff(foff) > 0).mean() > 0.4
    raw, filt, ts = _np(*e.rank(kg.triples, REL, 0, kg.n_relations, foff, fids))
    _own_operand_check(e, kg.triples, 0, kg.n_relations, raw, filt, ts, foff, fids)
    assert raw.max() > 100 and (filt < raw).any()
    e.close()


@pytest.mark.parametrize("n_rel,rng_,dim", [(14, (0, 14), 150), (300, (0, 300), 150), (300, (7, 290), 64),
                                            (300, (0, 300), 320)])
def test_split_bf16_counts_match_fp64_oracle(eng_mod, n_rel, rng_, dim):
    """Relation counts 14 (one padded tile) and 300, a range not starting at row 0; Q = 300 and Q = 1; dim 320 is
    the largest bf16x3 build."""
    b, en = rng_
    kg, e = _setup(eng_mod, n_rel, 2000, 300, dim, seed=n_rel + b + dim, rel_range=rng_)
    cand = np.arange(b, en)
    foff, fids = D.build_filter_csr(kg.triples, _known(kg, 5), "relation")
    S = RR.all_scores(kg.E.astype(np.float64), kg.triples, cand)
    raw, filt, ts = _np(*e.rank(kg.triples, REL, b, en, foff, fids, precision=eng_mod.HOLE_RANK_BF16X3))
    _oracle_check(S, cand, kg.triples, raw, filt, ts, foff, fids)
    raw1, filt1, ts1 = _np(*e.rank(kg.triples[:1], REL, b, en, foff[:2], fids[: foff[1]],
                                   precision=eng_mod.HOLE_RANK_BF16X3))
    _oracle_check(S[:1], cand, kg.triples[:1], raw1, filt1, ts1, foff[:2], fids[: foff[1]])
    assert raw1[0] == raw[0] and filt1[0] == filt[0]
    e.close()


def test_exact_ties_go_to_the_smaller_relation_id(eng_mod):
    kg, _ = _setup(eng_mod, 40, 1500, 200, 64, seed=9)
    E = kg.E.copy()
    E[[3, 17, 29]] = E[8]                                   # four relations with bit-identical scores
    e = eng_mod.HoleEngine(kg.n_rows, kg.dim).set_embeddings(E)
    kg.triples[:, 2] = np.array([3, 8, 17, 29, 5])[np.arange(len(kg.triples)) % 5]
    for prec in (eng_mod.HOLE_RANK_BF16, eng_mod.HOLE_RANK_BF16X3):
        raw, filt, ts = _np(*e.rank(kg.triples, REL, 0, 40, precision=prec))
        if prec == eng_mod.HOLE_RANK_BF16:
            S = _own_operand_check(e, kg.triples, 0, 40, raw, filt, ts)
            for q in range(len(kg.triples)):
                r = int(kg.triples[q, 2])
                if r in (3, 8, 17, 29):                     # the tied smaller ids rank before r, the larger after
                    i = (3, 8, 17, 29).index(r)
                    strict = int((S[q] < S[q, r] - 2e-6).sum())
                    loose = int((S[q] <= S[q, r] + 2e-6).sum()) - 1
                    assert strict + i <= raw[q] <= loose - (3 - i), (q, r)
        ids, sc = _np(*e.topk(kg.triples, REL, 0, 40, 40, precision=prec))
        for q in range(len(kg.triples)):
            pos = [int(np.flatnonzero(ids[q] == r)[0]) for r in (3, 8, 17, 29)]
            assert pos == list(range(pos[0], pos[0] + 4)), (prec, q, pos)
            assert np.all(sc[q, pos] == sc[q, pos[0]])
    e.close()


# ---------------------------------------------------------------------------------------------- top-k
@pytest.mark.parametrize("n_rel", [14, 300])
def test_topk_matches_fp64_oracle(eng_mod, n_rel):
    kg, e = _setup(eng_mod, n_rel, 2000, 300, 150, seed=30 + n_rel)
    cand = np.arange(n_rel)
    E64 = kg.E.astype(np.float64)
    S = RR.all_scores(E64, kg.triples, cand)
    foff, fids = D.build_filter_csr(kg.triples, _known(kg, 6), "relation")
    for k in (1, 10, 128):
        ids, sc = _np(*e.topk(kg.triples, REL, 0, n_rel, k, foff, fids))
        assert ids.shape == (len(kg.triples), k)
        _check_rows(ids, sc, S, cand, k, _filter_lists(foff, fids), BAND_X3)
        if k > n_rel:
            assert np.all(ids[:, n_rel:] == -1) and np.all(np.isinf(sc[:, n_rel:]))
    ids, sc = _np(*e.topk(kg.triples[:1], REL, 0, n_rel, 10))
    _check_rows(ids, sc, S[:1], cand, 10, None, BAND_X3)
    e.close()


# ---------------------------------------------------------------------------------------------- dims
@pytest.mark.parametrize("dim", [2, 258, 320])
def test_split_bf16_topk_and_counts_across_packer_iterations(eng_mod, dim):
    kg, e = _setup(eng_mod, 60, 1500, 300, dim, seed=200 + dim)
    cand = np.arange(60)
    S = RR.all_scores(kg.E.astype(np.float64), kg.triples, cand)
    foff, fids = D.build_filter_csr(kg.triples, _known(kg, 7), "relation")
    raw, filt, ts = _np(*e.rank(kg.triples, REL, 0, 60, foff, fids, precision=eng_mod.HOLE_RANK_BF16X3))
    _oracle_check(S, cand, kg.triples, raw, filt, ts, foff, fids)
    ids, sc = _np(*e.topk(kg.triples, REL, 0, 60, 10, foff, fids))
    _check_rows(ids, sc, S, cand, 10, _filter_lists(foff, fids), BAND_X3)
    e.close()


@pytest.mark.parametrize("dim,precision", [(642, 0), (322, 1)])
def test_refusals_for_the_relation_side(eng_mod, dim, precision):
    """First dims the ranking kernel does not build: HoleError, no kernel launched, outputs untouched; the same
    context then ranks relations at the other precision (322) or scores (642)."""
    kg, e = _setup(eng_mod, 20, 500, 100, dim, seed=dim)
    Q, R = len(kg.triples), kg.n_relations
    raw = torch.full((Q,), -7, dtype=torch.int32, device=e.device)
    filt = torch.full((Q,), -7, dtype=torch.int32, device=e.device)
    ts = torch.full((Q,), 1234.5, dtype=torch.float32, device=e.device)
    table0 = e.table.clone()
    n0 = e.launch_count()
    with pytest.raises(eng_mod.HoleError, match=f"embedding_dim {dim}"):
        e.rank(kg.triples, REL, 0, R, precision=precision, true_score=ts, raw_before=raw, filt_before=filt)
    with pytest.raises(eng_mod.HoleError, match=f"embedding_dim {dim}"):
        e.topk(kg.triples, REL, 0, R, 5, precision=precision)
    torch.cuda.synchronize()
    assert e.launch_count() == n0
    assert (raw == -7).all() and (filt == -7).all() and (ts == 1234.5).all() and torch.equal(e.table, table0)
    if precision == 1:
        raw, filt, ts = _np(*e.rank(kg.triples, REL, 0, R))
        _own_operand_check(e, kg.triples, 0, R, raw, filt, ts)
    else:
        got = e.evaluate_triples(kg.triples).cpu().numpy()
        assert np.abs(got - O.evaluate_triples(kg.E.astype(np.float64), kg.triples, np.float64)).max() <= 1e-6
    e.close()


# ---------------------------------------------------------------------------------------------- ccorr_tanh
@pytest.mark.parametrize("dim", CCORR_DIMS)
def test_ccorr_tanh_mode(eng_mod, dim):
    """Every ccorr query-packer NV: counts exact on the kernel's own operands (bf16); up to dim 320 also split-bf16
    counts and top-k against the definition of the archived score."""
    n_rel = 50
    kg, e = _setup(eng_mod, n_rel, 800, 120, dim, seed=300 + dim)
    e.set_score_mode("ccorr_tanh")
    foff, fids = D.build_filter_csr(kg.triples, _known(kg, 8), "relation")
    raw, filt, ts = _np(*e.rank(kg.triples, REL, 0, n_rel, foff, fids))
    _own_operand_check(e, kg.triples, 0, n_rel, raw, filt, ts, foff, fids)
    assert raw.max() > 10
    if rank_stages(dim, 2) is None:
        e.close()
        return
    cand = np.arange(n_rel)
    S = RR.ccorr_all_scores(kg.E.astype(np.float64), kg.triples, cand)
    raw, filt, ts = _np(*e.rank(kg.triples, REL, 0, n_rel, foff, fids, precision=eng_mod.HOLE_RANK_BF16X3))
    _oracle_check(S, cand, kg.triples, raw, filt, ts, foff, fids)
    ids, sc = _np(*e.topk(kg.triples, REL, 0, n_rel, 10, foff, fids))
    # the fp32 query vector is an O(H) correlation sum: its score is held to the band, not to the fp32 bound
    _check_rows(ids, sc, S, cand, 10, _filter_lists(foff, fids), BAND_X3, score_tol=False)
    sel = np.take_along_axis(S, ids.astype(np.int64), axis=1)
    assert np.abs(sc - sel).max() <= BAND_X3
    tri = np.repeat(kg.triples, 10, axis=0)
    tri[:, 2] = ids.reshape(-1)
    th = e.evaluate_triples(tri).cpu().numpy().astype(np.float64)
    assert np.abs(th - np.tanh(sc.reshape(-1).astype(np.float64))).max() <= BAND_X3
    e.close()


# ---------------------------------------------------------------------------------------------- consistency
def test_top1_is_consistent_with_score_and_rank(eng_mod):
    kg, e = _setup(eng_mod, 200, 2500, 400, 150, seed=41)
    ids, sc = _np(*e.topk(kg.triples, REL, 0, 200, 1))
    q = kg.triples.copy()
    q[:, 2] = ids[:, 0]
    sig = e.evaluate_triples(q).cpu().numpy().astype(np.float64)
    logit = np.log(sig) - np.log1p(-sig)
    s = sc[:, 0].astype(np.float64)
    assert np.all(np.abs(logit - s) <= 2e-6 + 1e-5 * np.abs(s))
    raw, _, _ = _np(*e.rank(q, REL, 0, 200, precision=eng_mod.HOLE_RANK_BF16X3))
    S = np.sort(RR.all_scores(kg.E.astype(np.float64), kg.triples, np.arange(200)), axis=1)
    clear = S[:, 1] - S[:, 0] > 2 * BAND_X3
    assert clear.mean() > 0.5 and np.all(raw[clear] == 0)
    e.close()


def test_rank_ex_with_a_query_table_equals_rank(eng_mod):
    kg, e = _setup(eng_mod, 100, 2000, 300, 150, seed=43)
    Q, R = len(kg.triples), kg.n_relations
    foff, fids = D.build_filter_csr(kg.triples, _known(kg, 9), "relation")
    raw, filt, ts = e.rank(kg.triples, REL, 0, R, foff, fids)
    # the h and t rows from a separate table [h rows | t rows]; the relation column indexes the main table
    rows = torch.as_tensor(np.concatenate([kg.triples[:, 0], kg.triples[:, 1]]).astype(np.int64), device=e.device)
    qtab = e.table.index_select(0, rows).contiguous()
    ql = torch.as_tensor(np.stack([np.arange(Q), Q + np.arange(Q), kg.triples[:, 2]], 1).astype(np.int32),
                         device=e.device)
    raw2 = torch.zeros(Q, dtype=torch.int32, device=e.device)
    filt2 = torch.zeros_like(raw2)
    ts2 = torch.zeros(Q, dtype=torch.float32, device=e.device)
    fo = torch.as_tensor(foff, device=e.device)
    fi = torch.as_tensor(fids, device=e.device)
    e.rank_ex(ql, REL, 0, R, query_table=qtab, filter_off=fo, filter_ids=fi, true_score=ts2, raw_before=raw2,
              filt_before=filt2)
    assert torch.equal(raw, raw2) and torch.equal(filt, filt2) and torch.equal(ts, ts2)
    e.close()


def test_relation_call_between_prepared_entity_calls(eng_mod):
    kg, e = _setup(eng_mod, 30, 3000, 300, 150, seed=47)
    R, N = kg.n_relations, kg.n_rows
    tail0 = e.rank(kg.triples, 0, R, N)
    rel0 = e.rank(kg.triples, REL, 0, R)
    top0 = e.topk(kg.triples, REL, 0, R, 5)
    e.rank_prepare(R, N)
    tail1 = e.rank(kg.triples, 0, R, N)
    rel1 = e.rank(kg.triples, REL, 0, R)                   # drops the prepared entity operand
    top1 = e.topk(kg.triples, REL, 0, R, 5)
    tail2 = e.rank(kg.triples, 0, R, N)                    # re-packs
    for a, b in zip(tail0 + tail0, tail1 + tail2):
        assert torch.equal(a, b)
    for a, b in zip(rel0, rel1):
        assert torch.equal(a, b)
    assert torch.equal(top0[0], top1[0]) and torch.equal(top0[1], top1[1])
    e.close()


def test_sharded_rank_refuses_relation_and_both(eng_mod):
    from graphembeddings_b200.sharded import CudaBackend, RowShardedTrainer
    kg, e = _setup(eng_mod, 6, 1000, 50, 64, seed=51)
    e.close()
    tr = RowShardedTrainer(kg.n_relations, kg.n_entities, kg.dim, CudaBackend(kg.n_relations, kg.dim, 64, 0),
                           None).load_embeddings(kg.E)
    for side in (eng_mod.HOLE_SIDE_RELATION, eng_mod.HOLE_SIDE_BOTH):
        with pytest.raises(eng_mod.HoleError, match="gather_embeddings"):
            tr.rank(torch.from_numpy(kg.triples), side)
    raw, _ = tr.rank(torch.from_numpy(kg.triples), eng_mod.HOLE_SIDE_TAIL)
    assert raw.shape == (len(kg.triples),)


# ---------------------------------------------------------------------------------------------- full size
def test_full_size_fb15k_queries_against_fp64_on_the_gpu(eng_mod, golden_dir):
    """The 59,071 real FB15k test queries x 1,345 relations at d = 150 on a table the engine fitted to test + valid,
    filtered against valid: split-bf16 counts against an fp64 contraction done with torch on the GPU."""
    z = np.load(os.path.join(golden_dir, "fb15k_test_valid_triples.npz"))
    test, valid = z["test"], z["valid"]
    R_, N, dim = 1345, 16296, 150
    kg = D.make_config("fb15k_d150", n_triples=1000, zipf_entities=True)
    off, ids = D.build_type_csr(kg.type_of)
    e = eng_mod.HoleEngine(N, dim).set_embeddings(kg.E).set_types(kg.type_of, off, ids).set_relation_count(R_)
    fit = np.concatenate([test, valid]).astype(np.int32)
    rng = np.random.default_rng(0)
    for epoch in range(20):
        perm = rng.permutation(len(fit))[: (len(fit) // 2048) * 2048]
        e.train_steps(fit[perm], 2048, 1, epoch * 100, 0.2, [0.5] * (len(perm) // 2048))
    foff, fids = D.build_filter_csr(test, valid, "relation")
    raw, filt, ts = e.rank(test, REL, 0, R_, foff, fids, precision=eng_mod.HOLE_RANK_BF16X3)
    # fp64 on the GPU: clipped rows, q = [a e + b f ; a f - b e], S = q . clip(E_r)
    E = e.embeddings().double()
    E = E * torch.clamp(E.norm(dim=1, keepdim=True).reciprocal(), max=1.0)
    H = dim // 2
    tq = torch.as_tensor(test.astype(np.int64), device=e.device)
    h, t = E[tq[:, 0]], E[tq[:, 1]]
    a, b, c, d = h[:, :H], h[:, H:], t[:, :H], t[:, H:]
    S = torch.cat([a * c + b * d, a * d - b * c], 1) @ E[:R_].T
    tj = tq[:, 2]
    thr = S.gather(1, tj[:, None])
    cand = torch.arange(R_, device=e.device)
    before = (S < thr) | ((S == thr) & (cand[None] < tj[:, None]))
    oraw = before.sum(1)
    qi = torch.repeat_interleave(torch.arange(len(test), device=e.device), torch.as_tensor(np.diff(foff), device=e.device))
    hit = torch.zeros(len(test), dtype=torch.int64, device=e.device)
    hit.index_add_(0, qi, before[qi, torch.as_tensor(fids.astype(np.int64), device=e.device)].long())
    ofilt = oraw - hit
    lo = (S < thr - BAND_X3).sum(1)
    hi = (S <= thr + BAND_X3).sum(1) - 1
    raw, filt = raw.long(), filt.long()
    assert float((ts.double() - thr[:, 0]).abs().max()) < BAND_X3
    assert bool(((raw >= lo) & (raw <= hi)).all())
    assert bool(((raw == oraw) | (hi > lo)).all()) and bool(((filt == ofilt) | (hi > lo)).all())
    got = O.score_mrr(*_np(raw + 1, filt + 1))
    want = O.score_mrr(*_np(oraw + 1, ofilt + 1))
    for key in ("raw_mrr", "filtered_mrr"):
        assert abs(got[key] - want[key]) <= 1e-4, (key, got, want)
    assert float(oraw.double().mean()) < 0.45 * R_           # fitted: better than a random table's R / 2
    assert len(fids) > 0 and int(hit.sum()) > 0
    e.close()


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


def _infer(hole, tmp, args):
    logged = []
    cwd = os.getcwd()
    os.chdir(tmp)
    try:
        m = hole.infer_triples(hole.build_parser().parse_args(args), log=lambda *a: logged.append(" ".join(map(str, a))))
    finally:
        os.chdir(cwd)
    return m, logged


def _lines(path, side):
    return [r.rstrip("\n").split("\t") for r in open(path) if r.startswith(side + "\t")]


def test_cli_relation_prediction(eng_mod, tmp_path):
    from graphembeddings_b200 import hole, tf_bundle
    kg = D.synthetic_kg(8, 1500, 9000, 4, 64, seed=3, with_embeddings=False)
    d = tmp_path / "data"; d.mkdir()
    parts = _write_data_dir(str(d), kg, 600, 400)
    out = str(tmp_path / "run")
    args = ["--data_dir", str(d), "--output_dir", out, "--batch_size", "256", "--embedding_dim", "64",
            "--num_epochs", "2"]
    hole.main(args)
    pred = os.path.join(out, "predictions.tsv")
    base, _ = _infer(hole, tmp_path, args + ["--infer", "--predict_top_k", "5"])
    assert "relation" not in base and not _lines(pred, "relation") and _lines(pred, "tail")
    n_results = sum(1 for _ in open(tmp_path / "inference_results.tsv"))
    m, logged = _infer(hole, tmp_path, args + ["--infer", "--relation_prediction", "--predict_top_k", "5"])
    assert sum(1 for _ in open(tmp_path / "inference_results.tsv")) == 2 * n_results    # entity sides only
    assert {k: v for k, v in m.items() if k != "relation"} == base
    # logged metrics against the fp64 oracle's ranks
    E64 = tf_bundle.load_bundle(os.path.join(out, "model.ckpt"))["embeddings"].astype(np.float64)
    test = np.unique(parts["test_positive_triples.txt"], axis=0)
    known = np.concatenate([parts["triples.txt"], parts["triples-valid.txt"]])
    test = test[~D.rows_in(test, known)]
    R = kg.n_relations
    foff, fids = D.build_filter_csr(test, known, "relation")
    S = RR.all_scores(E64, test, np.arange(R))
    oraw, ofilt = O.rank_counts(S, np.arange(R), test[:, 2], _filter_lists(foff, fids))
    want = O.score_mrr(oraw + 1, ofilt + 1)
    for key, v in want.items():
        assert abs(m["relation"][key] - v) <= 1e-4, (key, m["relation"], want)
    assert any("Relation prediction" in line for line in logged)
    assert sum("Filtered MRR" in line for line in logged) == 2
    # the relation lines of predictions.tsv are HoleEngine.topk's
    rows = _lines(pred, "relation")
    pairs = np.unique(parts["test_positive_triples.txt"][:, :2], axis=0)
    q = np.zeros((len(pairs), 3), np.int32)
    q[:, :2] = pairs
    qf, qi = D.build_filter_csr(q, known, "relation")
    e = eng_mod.HoleEngine(kg.n_rows, 64).set_embeddings(E64.astype(np.float32))
    ids, sc = _np(*e.topk(q, REL, 0, R, 5, qf, qi))
    test_set = set(map(tuple, parts["test_positive_triples.txt"].tolist()))
    want_rows = []
    for i, (h, t) in enumerate(pairs.tolist()):
        for pos in range(5):
            if ids[i, pos] < 0:
                break
            r = int(ids[i, pos])
            s = np.float64(sc[i, pos])
            want_rows.append(["relation", str(h), str(t), str(r), str(pos + 1), "{:.9g}".format(s),
                              "{:.6f}".format(1.0 / (1.0 + np.exp(-s))), str((h, t, r) in test_set)])
    assert rows == want_rows and len(rows) > len(pairs)
    # the archived score variant: the value column is tanh
    m2, _ = _infer(hole, tmp_path, args + ["--infer", "--relation_prediction", "--predict_top_k", "3",
                                          "--score_variant", "ccorr_tanh"])
    assert 0 < m2["relation"]["filtered_mrr"] <= 1
    rows = _lines(pred, "relation")
    assert rows and all(abs(float(r_[6]) - math.tanh(float(r_[5]))) <= 1e-6 for r_ in rows)
    e.close()
