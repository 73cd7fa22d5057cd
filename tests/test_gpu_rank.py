"""Parity of the tensor-core ranking path (hole_rank through the C ABI).

Standards (north_star / SURVEY 8c):
  * the tcgen05 contraction + rank-count epilogue are checked EXACTLY against an fp64
    contraction of the kernel's own bf16 operands: counts must agree except for candidates
    whose score lies within 2e-6 of the threshold (fp32 accumulation noise);
  * the bf16 operands agree with the oracle's clipped rows / query vectors to 1 bf16 ulp
    (|d| <= 2^-8 |x|);
  * scores agree with the fp32 oracle within the bf16 bound 4e-3 * |q| |e|; filtered MRR and
    Hits@k within 1e-2 absolute on random embeddings (near-ties dominate there) and 1e-3 on
    a structured table.
"""
import numpy as np
import pytest
import torch

from graphembeddings_b200 import data as D
from oracle import hole_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng_mod():
    from graphembeddings_b200 import build
    build.build()
    from graphembeddings_b200 import engine
    return engine


def _setup(eng_mod, n_rel, n_ent, n_q, dim, seed, trained=True):
    kg = D.synthetic_kg(n_rel, n_ent, n_q, 4, dim, seed=seed, trained_scale=trained)
    e = eng_mod.HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E)
    return kg, e


def _exact_from_operands(e, kg, queries, side, ent_begin, ent_end, raw, filt, tscore, foff=None, fids=None,
                         eps=2e-6):
    cand, qp = e.rank_debug_operands()
    C = cand.double().cpu().numpy()[: ent_end - ent_begin]
    Qm = qp.double().cpu().numpy()[: len(queries)]
    S = Qm @ C.T
    col = 1 if side == 0 else 0
    tj = queries[:, col].astype(np.int64) - ent_begin
    thr = S[np.arange(len(queries)), tj]
    assert np.abs(tscore - thr).max() < eps
    ids = np.arange(S.shape[1])
    lo = ((S < thr[:, None] - eps) | ((np.abs(S - thr[:, None]) <= eps) & False)).sum(1)
    hi = (S <= thr[:, None] + eps).sum(1) - 1      # minus the true candidate itself
    exact = ((S < thr[:, None]) | ((S == thr[:, None]) & (ids[None, :] < tj[:, None]))).sum(1)
    assert np.all(raw >= lo) and np.all(raw <= hi)
    assert np.all((raw == exact) | (hi > lo))            # outside a near-tie the count is exact
    if foff is not None:
        for q in range(len(queries)):
            f = fids[foff[q]:foff[q + 1]].astype(np.int64) - ent_begin
            f = f[(f >= 0) & (f < S.shape[1])]
            sure = int((S[q, f] < thr[q] - eps).sum())
            maybe = int((S[q, f] <= thr[q] + eps).sum())
            assert raw[q] - maybe <= filt[q] <= raw[q] - sure
    return S, thr


@pytest.mark.parametrize("dim", [64, 150, 256, 512, 2, 514, 640])     # 514, 640: 2-stage ring, 3 query-packer iterations
@pytest.mark.parametrize("side", [0, 1])
def test_rank_counts_exact_vs_own_operands(eng_mod, dim, side):
    kg, e = _setup(eng_mod, 11, 3000, 700, dim, seed=dim + side)
    b, en = kg.n_relations, kg.n_rows
    known = D.synthetic_kg(11, 3000, 20000, 4, 8, seed=99, with_embeddings=False).triples
    foff, fids = D.build_filter_csr(kg.triples, known, "tail" if side == 0 else "head")
    raw, filt, ts = e.rank(kg.triples, side, b, en, foff, fids)
    raw, filt, ts = raw.cpu().numpy(), filt.cpu().numpy(), ts.cpu().numpy()
    _exact_from_operands(e, kg, kg.triples, side, b, en, raw, filt, ts, foff, fids)
    assert np.all(filt <= raw) and np.all(filt >= 0)
    assert raw.max() > 100


def test_operands_match_oracle_to_one_bf16_ulp(eng_mod):
    kg, e = _setup(eng_mod, 7, 1000, 300, 150, seed=3)
    for side, name in ((0, "tail"), (1, "head")):
        e.rank(kg.triples, side, kg.n_relations, kg.n_rows)
        cand, qp = e.rank_debug_operands()
        Y, _, _ = O.clip_rows(kg.E[kg.n_relations:].astype(np.float64))
        got = cand.float().cpu().numpy()[: kg.n_entities, : kg.dim]
        assert np.abs(got - Y).max() <= 2.0 ** -8 * np.abs(Y).max()
        assert np.all(np.abs(got - Y) <= 2.0 ** -8 * np.abs(Y) + 1e-12)
        assert np.all(cand.float().cpu().numpy()[:, kg.dim:] == 0)
        qv = O.query_vectors(kg.E.astype(np.float64), kg.triples, name, np.float64)
        gq = qp.float().cpu().numpy()[: len(kg.triples), : kg.dim]
        assert np.all(np.abs(gq - qv) <= 2.0 ** -8 * np.abs(qv) + 1e-9)


def test_scores_within_bf16_bound_and_metrics_close(eng_mod):
    kg, e = _setup(eng_mod, 9, 5000, 1000, 256, seed=11)
    b, en = kg.n_relations, kg.n_rows
    cand_ids = np.arange(b, en)
    raw, filt, ts = e.rank(kg.triples, 0, b, en)
    S = O.all_scores(kg.E, kg.triples, "tail", cand_ids, np.float32)
    tj = kg.triples[:, 1] - b
    thr = S[np.arange(len(tj)), tj]
    qn = np.linalg.norm(O.query_vectors(kg.E, kg.triples, "tail"), axis=1)
    assert np.all(np.abs(ts.cpu().numpy() - thr) <= 4e-3 * qn * 1.0)
    oraw, _ = O.rank_counts(S, cand_ids, kg.triples[:, 1])
    m_gpu = O.score_mrr(raw.cpu().numpy() + 1, raw.cpu().numpy() + 1)
    m_ref = O.score_mrr(oraw + 1, oraw + 1)
    assert abs(m_gpu["filtered_mrr"] - m_ref["filtered_mrr"]) < 1e-2
    assert abs(m_gpu["hits10"] - m_ref["hits10"]) < 1.0
    # mean rank moves by at most a few places out of 5000
    assert abs(m_gpu["raw_mean_pos"] - m_ref["raw_mean_pos"]) < 5.0


def test_structured_table_metrics_match_oracle(eng_mod):
    """A table where the true tail really is the best candidate for most queries: build t so
    that conj-related score is strongly negative (lower is better)."""
    rng = np.random.default_rng(5)
    n_rel, n_ent, dim, Qn = 5, 4000, 128, 600
    kg = D.synthetic_kg(n_rel, n_ent, Qn, 3, dim, seed=5, trained_scale=True)
    E = kg.E.astype(np.float64)
    # make each query's true tail = -(h*r) direction + noise  => most negative score
    qv = O.query_vectors(E, kg.triples, "tail", np.float64)
    # distinct tails per query
    tails = n_rel + rng.permutation(n_ent)[:Qn]
    kg.triples[:, 1] = tails
    E[tails] = -qv / np.linalg.norm(qv, axis=1, keepdims=True) * 0.9 + 0.02 * rng.standard_normal(qv.shape)
    kg.E = E.astype(np.float32)
    e = eng_mod.HoleEngine(kg.n_rows, dim).set_embeddings(kg.E)
    raw, filt, ts = e.rank(kg.triples, 0, n_rel, kg.n_rows)
    S = O.all_scores(kg.E, kg.triples, "tail", np.arange(n_rel, kg.n_rows), np.float32)
    oraw, _ = O.rank_counts(S, np.arange(n_rel, kg.n_rows), kg.triples[:, 1])
    m_gpu = O.score_mrr(raw.cpu().numpy() + 1, raw.cpu().numpy() + 1)
    m_ref = O.score_mrr(oraw + 1, oraw + 1)
    assert m_ref["hits1"] > 60.0
    assert abs(m_gpu["filtered_mrr"] - m_ref["filtered_mrr"]) < 1e-3
    assert abs(m_gpu["hits1"] - m_ref["hits1"]) < 0.5
    assert abs(m_gpu["hits10"] - m_ref["hits10"]) < 0.5


def test_candidate_shards_accumulate_like_one_call(eng_mod):
    """Ranking over [b, m) then [m, e) with combined true scores equals one call over [b, e):
    the multi-GPU protocol (candidate shards, counts summed)."""
    kg, e = _setup(eng_mod, 6, 2500, 400, 150, seed=21)
    b, en = kg.n_relations, kg.n_rows
    mid = b + 1111
    raw1, filt1, ts1 = e.rank(kg.triples, 0, b, en)
    ts = torch.zeros(len(kg.triples), dtype=torch.float32, device="cuda")
    raw = torch.zeros(len(kg.triples), dtype=torch.int32, device="cuda")
    filt = torch.zeros(len(kg.triples), dtype=torch.int32, device="cuda")
    # phase 1: every shard writes the true scores it owns
    scratch_r = torch.zeros_like(raw); scratch_f = torch.zeros_like(filt)
    e.rank(kg.triples, 0, b, mid, true_score=ts, compute_true=True, raw_before=scratch_r, filt_before=scratch_f)
    e.rank(kg.triples, 0, mid, en, true_score=ts, compute_true=True, raw_before=scratch_r, filt_before=scratch_f)
    # phase 2: count against the combined thresholds
    e.rank(kg.triples, 0, b, mid, true_score=ts, compute_true=False, raw_before=raw, filt_before=filt)
    e.rank(kg.triples, 0, mid, en, true_score=ts, compute_true=False, raw_before=raw, filt_before=filt)
    assert torch.equal(ts, ts1)
    assert torch.equal(raw, raw1)


def test_ragged_sizes_and_ties(eng_mod):
    """Q and N not multiples of the tile sizes; duplicated candidate rows give exact ties that
    must be broken by the smaller candidate id (holE.py:434 tuple order)."""
    kg, e0 = _setup(eng_mod, 3, 777, 130, 64, seed=8)
    E = kg.E.copy()
    t = kg.triples[:, 1]
    dup_lo = np.clip(t - 1, kg.n_relations, None)
    dup_hi = np.clip(t + 1, None, kg.n_rows - 1)
    # make the neighbours exact copies of the true tail where that does not clash
    free = np.ones(kg.n_rows, bool); free[t] = False
    n_lo = n_hi = 0
    want_extra = np.zeros(len(t), np.int64)
    for i in range(len(t)):
        if free[dup_lo[i]] and dup_lo[i] != t[i]:
            E[dup_lo[i]] = E[t[i]]; free[dup_lo[i]] = False; want_extra[i] += 1; n_lo += 1
        if free[dup_hi[i]] and dup_hi[i] != t[i]:
            E[dup_hi[i]] = E[t[i]]; free[dup_hi[i]] = False; n_hi += 1
    assert n_lo > 20 and n_hi > 20
    e = eng_mod.HoleEngine(kg.n_rows, 64).set_embeddings(E)
    raw, _, ts = e.rank(kg.triples, 0, kg.n_relations, kg.n_rows)
    cand, qp = e.rank_debug_operands()
    S = qp.double().cpu().numpy()[: len(t)] @ cand.double().cpu().numpy()[: kg.n_entities].T
    tj = t - kg.n_relations
    thr = S[np.arange(len(t)), tj]
    ids = np.arange(S.shape[1])
    exact = ((S < thr[:, None]) | ((S == thr[:, None]) & (ids[None] < tj[:, None]))).sum(1)
    raw = raw.cpu().numpy()
    # exact ties (identical rows) are resolved exactly; only fp32-noise near-ties may move a count, and
    # then only inside the band
    strict = (S < thr[:, None] - 2e-6).sum(1)
    loose = (S <= thr[:, None] + 2e-6).sum(1) - 1
    assert np.all(raw >= strict + want_extra) and np.all(raw <= loose)
    assert np.all((raw == exact) | (loose > strict + want_extra))


def test_empty_queries_and_errors(eng_mod):
    kg, e = _setup(eng_mod, 3, 300, 10, 64, seed=1)
    r, f, t = e.rank(np.zeros((0, 3), np.int32), 0, 3, 303)
    assert r.numel() == 0
    with pytest.raises(eng_mod.HoleError):
        e.rank(kg.triples, 0, 3, 99999)          # range outside the table
    with pytest.raises(eng_mod.HoleError):
        e.rank(kg.triples, 0, 3, 303, precision=7)           # unknown precision


def test_sharded_rank_single_rank_matches_engine(eng_mod):
    from graphembeddings_b200.sharded import CudaBackend, RowShardedTrainer
    kg, e = _setup(eng_mod, 6, 2500, 300, 150, seed=33)
    known = D.synthetic_kg(6, 2500, 8000, 4, 8, seed=98, with_embeddings=False).triples
    foff, fids = D.build_filter_csr(kg.triples, known, "tail")
    raw1, filt1, _ = e.rank(kg.triples, 0, kg.n_relations, kg.n_rows, foff, fids)
    be = CudaBackend(kg.n_relations, kg.dim, 64, 0)
    tr = RowShardedTrainer(kg.n_relations, kg.n_entities, kg.dim, be, None).load_embeddings(kg.E)
    raw2, filt2 = tr.rank(torch.from_numpy(kg.triples), 0, foff, fids)
    assert torch.equal(raw1, raw2) and torch.equal(filt1, filt2)


def test_both_sides_in_one_pass_equals_two_calls(eng_mod):
    kg, e = _setup(eng_mod, 6, 2500, 300, 150, seed=35)
    known = D.synthetic_kg(6, 2500, 8000, 4, 8, seed=97, with_embeddings=False).triples
    ft = D.build_filter_csr(kg.triples, known, "tail")
    fh = D.build_filter_csr(kg.triples, known, "head")
    rt, flt, tst = e.rank(kg.triples, 0, kg.n_relations, kg.n_rows, *ft)
    rh, flh, tsh = e.rank(kg.triples, 1, kg.n_relations, kg.n_rows, *fh)
    fo = np.concatenate([ft[0], fh[0][1:] + ft[0][-1]])
    fi = np.concatenate([ft[1], fh[1]])
    rb, flb, tsb = e.rank(kg.triples, eng_mod.HOLE_SIDE_BOTH, kg.n_relations, kg.n_rows, fo, fi)
    Q = len(kg.triples)
    assert torch.equal(rb[:Q], rt) and torch.equal(rb[Q:], rh)
    assert torch.equal(flb[:Q], flt) and torch.equal(flb[Q:], flh)
    assert torch.equal(tsb[:Q], tst) and torch.equal(tsb[Q:], tsh)


def test_full_size_config3_sample_against_fp64_contraction(eng_mod):
    """BASELINE config 3 shape (1,200,000 candidates, d=256): rank 2,048 queries and check a
    sample of them exactly against an fp64 contraction of the kernel's own bf16 operands
    (done on the GPU with torch), plus size-independent invariants for all of them."""
    kg = D.make_config("rank_diffbot_d256", n_triples=2048, trained_scale=True)
    e = eng_mod.HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E)
    b, en = kg.n_relations, kg.n_rows
    raw, filt, ts = e.rank(kg.triples, 0, b, en)
    N = kg.n_entities
    assert int(raw.min()) >= 0 and int(raw.max()) <= N - 1
    assert torch.equal(raw, filt)                       # no filter given
    cand, qp = e.rank_debug_operands()
    idx = torch.arange(0, 2048, 32, device="cuda")      # 64 sampled queries
    S = qp[idx].double() @ cand[:N].double().T           # [64, 1.2M] fp64
    tj = torch.as_tensor(kg.triples[idx.cpu().numpy(), 1] - b, device="cuda").long()
    thr = S[torch.arange(len(idx)), tj]
    assert float((ts[idx].double() - thr).abs().max()) < 2e-6
    eps = 2e-6
    lo = (S < (thr - eps)[:, None]).sum(1)
    hi = (S <= (thr + eps)[:, None]).sum(1) - 1
    r = raw[idx].long()
    assert bool(((r >= lo) & (r <= hi)).all())
    ids = torch.arange(N, device="cuda")
    exact = ((S < thr[:, None]) | ((S == thr[:, None]) & (ids[None, :] < tj[:, None]))).sum(1)
    assert bool(((r == exact) | (hi > lo)).all())       # a count differs only where a near-tie exists
    # candidate-shard invariance at full size: two halves accumulate to the same counts
    raw2 = torch.zeros_like(raw); f2 = torch.zeros_like(raw)
    mid = b + 600_123
    e.rank(kg.triples, 0, b, mid, true_score=ts.clone(), compute_true=False, raw_before=raw2, filt_before=f2)
    e.rank(kg.triples, 0, mid, en, true_score=ts.clone(), compute_true=False, raw_before=raw2, filt_before=f2)
    assert torch.equal(raw2, raw)


@pytest.mark.parametrize("dim", [64, 150, 256, 258, 320])     # 258, 320: the 2-stage ring at bf16x3
@pytest.mark.parametrize("side", [0, 1])
def test_split_bf16_precision_matches_fp64_oracle(eng_mod, dim, side):
    """HOLE_RANK_BF16X3 (hi.hi + lo.hi + hi.lo on the tensor cores): ranks agree with the fp64
    oracle on the fp32 table except for candidates within 3e-5 of the threshold -- two orders of
    magnitude tighter than plain bf16 operands."""
    kg, e = _setup(eng_mod, 9, 3000, 500, dim, seed=50 + dim + side)
    b, en = kg.n_relations, kg.n_rows
    name, col = ("tail", 1) if side == 0 else ("head", 0)
    S = O.all_scores(kg.E.astype(np.float64), kg.triples, name, np.arange(b, en), np.float64)
    tj = kg.triples[:, col].astype(np.int64) - b
    thr = S[np.arange(len(tj)), tj]
    known = D.synthetic_kg(9, 3000, 20000, 4, 8, seed=96, with_embeddings=False).triples
    foff, fids = D.build_filter_csr(kg.triples, known, name)
    raw, filt, ts = e.rank(kg.triples, side, b, en, foff, fids, precision=eng_mod.HOLE_RANK_BF16X3)
    raw, filt, ts = raw.cpu().numpy(), filt.cpu().numpy(), ts.cpu().numpy()
    eps = 3e-5
    assert np.abs(ts - thr).max() < eps
    lo = (S < thr[:, None] - eps).sum(1)
    hi = (S <= thr[:, None] + eps).sum(1) - 1
    assert np.all(raw >= lo) and np.all(raw <= hi)
    exact = (S < thr[:, None]).sum(1)
    frac_x3 = np.mean(raw == exact)
    raw_bf, _, _ = e.rank(kg.triples, side, b, en)
    frac_bf = np.mean(raw_bf.cpu().numpy() == exact)
    assert np.all((raw == exact) | (hi > lo))            # exact wherever no candidate sits inside the band
    assert frac_x3 >= frac_bf
    assert np.all(filt <= raw) and np.all(filt >= 0)
