"""The archived FFT / tanh score variant as a score mode of the engine (SURVEY.md section 8f item 4),
through the C ABI, against oracle/hole_ccorr.py (fp64 yardstick; fp32 tolerances written below)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng_mod():
    from graphembeddings_b200 import engine
    return engine


def _table(n, dim, seed, scale=1.0):
    rng = np.random.default_rng(seed)
    E = rng.standard_normal((n, dim))
    E *= (scale * rng.uniform(0.5, 1.5, size=(n, 1))) / np.linalg.norm(E, axis=1, keepdims=True)
    return E.astype(np.float32)


def _triples(rng, n_rel, n, B):
    return np.stack([rng.integers(n_rel, n, B), rng.integers(n_rel, n, B), rng.integers(0, n_rel, B)],
                    axis=1).astype(np.int32)


@pytest.mark.parametrize("dim", [8, 64, 150, 256, 384, 66, 128, 290, 450, 514, 768])   # NV 1, 2, 3, 4, 6, 8, 12
def test_ccorr_score_matches_oracle(eng_mod, dim):
    from oracle import hole_ccorr as oc
    n, B = 300, 257
    E = _table(n, dim, 100 + dim)
    rng = np.random.default_rng(dim)
    tri = _triples(rng, 6, n, B)
    e = eng_mod.HoleEngine(n, dim).set_embeddings(E).set_score_mode("ccorr_tanh")
    got = e.evaluate_triples(tri).cpu().numpy()
    want = np.tanh(oc.raw_score(E.astype(np.float64), tri, np.float64))
    assert np.abs(got - want).max() <= 2e-6          # |s| <= 1 by the clip; fp32 accumulation over H^2 terms
    e.close()


@pytest.mark.parametrize("dim,side,margin", [(8, 0, 1.0), (8, 1, 0.2), (150, 0, 1.0), (150, 1, 1.0), (256, 0, 0.2),
                                             (256, 1, 1.0), (384, 1, 1.0), (66, 0, 1.0), (290, 1, 1.0),
                                             (450, 0, 0.2), (768, 1, 1.0)])
def test_ccorr_train_steps_match_oracle(eng_mod, dim, side, margin):
    """Chained steps with duplicate rows (few entities, fewer relations), clipped and unclipped rows."""
    from oracle import hole_ccorr as oc
    n, n_rel, B, steps, lr = 120, 4, 96, 3, 0.1
    E = _table(n, dim, 7 + dim + side)
    rng = np.random.default_rng(11 * dim + side)
    e = eng_mod.HoleEngine(n, dim).set_embeddings(E).set_score_mode("ccorr_tanh")
    e.set_relation_count(n_rel)
    ref = E.astype(np.float64)
    for s in range(steps):
        pos = _triples(rng, n_rel, n, B)
        neg = rng.integers(n_rel, n, B).astype(np.int32)
        neg[:5] = pos[:5, 0 if side else 1]                      # corrupt entity equal to the original one
        loss, vp, vn = e.train_step(pos, neg, side, margin, lr, return_sigma=True)
        wl, wvp, wvn = oc.sgd_step(ref, pos, neg, side, margin, lr, dtype=np.float64)
        assert np.abs(vp.cpu().numpy() - wvp).max() <= 3e-6
        assert np.abs(vn.cpu().numpy() - wvn).max() <= 3e-6
        # rows whose hinge sits within rounding of the kink may differ by a whole gradient: none here
        assert np.abs(wvp - wvn + margin).min() > 1e-4
        assert np.abs(loss.cpu().numpy() - wl).max() <= 5e-6
        got = e.embeddings().cpu().numpy().astype(np.float64)
        err = np.abs(got - ref)
        assert (err <= 3e-6 + 1e-5 * np.abs(ref)).all(), float(err.max())
    assert np.abs(ref - E).max() > 1e-3                           # the steps moved the table
    e.close()


def test_ccorr_train_steps_device_loop_matches_single_steps(eng_mod):
    """hole_train_steps (device corruption, chunked plan) in the archived mode equals the same steps taken
    one by one with the corruption it reports."""
    from graphembeddings_b200 import data as D
    dim, B, steps = 64, 256, 5
    kg = D.make_config("fb15k_d150", n_triples=B * steps, dim=dim, trained_scale=True)
    off, ids = D.build_type_csr(kg.type_of)
    a = eng_mod.HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E).set_types(kg.type_of, off, ids).set_score_mode("ccorr_tanh")
    a.set_relation_count(kg.n_relations)
    tri = torch.from_numpy(kg.triples).cuda()
    sums = a.train_steps(tri, B, 3, 0, 1.0, [0.1] * steps)
    b = eng_mod.HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E).set_types(kg.type_of, off, ids).set_score_mode("ccorr_tanh")
    b.set_relation_count(kg.n_relations)
    tot = []
    for s in range(steps):
        pos = kg.triples[s * B:(s + 1) * B]
        side, neg = b.corrupt_batch(pos, 3, s)
        tot.append(float(b.train_step(pos, neg, side, 1.0, 0.1).sum()))
    np.testing.assert_allclose(sums.cpu().numpy(), np.array(tot), rtol=1e-5)
    assert torch.equal(a.embeddings(), b.embeddings())
    a.close(); b.close()


@pytest.mark.parametrize("dim", [64, 150, 256, 290, 320])
@pytest.mark.parametrize("side", [0, 1])
def test_ccorr_ranking_matches_fp64_oracle(eng_mod, dim, side):
    """All-candidate ranking in the archived mode (the score is linear in the candidate entity, so the same
    tensor-core contraction runs on another query vector): split-bf16 ranks agree with the fp64 oracle's
    scores, computed from the definition, except for candidates within 3e-5 of the threshold."""
    from oracle import hole_ccorr as oc
    n_rel, n, Q = 6, 1500, 160
    E = _table(n, dim, 300 + dim + side)
    rng = np.random.default_rng(dim + side)
    q = _triples(rng, n_rel, n, Q)
    e = eng_mod.HoleEngine(n, dim).set_embeddings(E).set_score_mode("ccorr_tanh")
    name, col = ("tail", 1) if side == 0 else ("head", 0)
    S = oc.all_scores(E.astype(np.float64), q, name, np.arange(n_rel, n), np.float64)
    tj = q[:, col].astype(np.int64) - n_rel
    thr = S[np.arange(Q), tj]
    raw, filt, ts = e.rank(q, side, n_rel, n, precision=eng_mod.HOLE_RANK_BF16X3)
    raw, ts = raw.cpu().numpy(), ts.cpu().numpy()
    eps = 3e-5
    assert np.abs(ts - thr).max() < eps
    lo = (S < thr[:, None] - eps).sum(1)
    hi = (S <= thr[:, None] + eps).sum(1) - 1
    assert np.all(raw >= lo) and np.all(raw <= hi)
    exact = (S < thr[:, None]).sum(1)
    assert np.all((raw == exact) | (hi > lo))      # exact wherever no candidate sits in the near-tie band
    # plain bf16 operands: scores within the bf16 bound
    raw_bf, _, ts_bf = e.rank(q, side, n_rel, n)
    assert np.abs(ts_bf.cpu().numpy() - thr).max() < 4e-3
    e.close()


def test_ccorr_mode_refuses_what_it_does_not_build(eng_mod):
    from graphembeddings_b200 import data as D
    kg = D.synthetic_kg(4, 60, 64, 3, 16, seed=1)
    off, ids = D.build_type_csr(kg.type_of)
    e = eng_mod.HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E).set_types(kg.type_of, off, ids).set_score_mode("ccorr_tanh")
    with pytest.raises(eng_mod.HoleError):
        e.train_step_logloss(kg.triples, 1, 0, 0.1)
    e.set_score_mode("complex")
    e.train_step_logloss(kg.triples, 1, 0, 0.1)
    e.close()
