"""CPU checks of the type-constrained contract statement (tests/typed_reference.py): against a brute-force
per-query loop, and, with one type covering every entity, against the all-entity count and
topk_reference.topk."""
import numpy as np
import pytest

import topk_reference
import typed_reference as R
from graphembeddings_b200 import data as D


def _case(seed, n_rows=300, n_types=9, Q=80, ties=True):
    rng = np.random.default_rng(seed)
    type_of = rng.integers(0, n_types, size=n_rows)
    type_of[:n_types] = np.arange(n_types)
    off, ids = D.build_type_csr(type_of, n_types)
    scores = rng.normal(size=(Q, n_rows))
    if ties:
        scores = np.round(scores, 1)               # many exact ties
    true = rng.integers(0, n_rows, size=Q)
    filters = [sorted(set(rng.integers(0, n_rows, size=int(rng.integers(0, 12))).tolist()) | (
        {int(true[q])} if rng.random() < 0.3 else set())) for q in range(Q)]
    return type_of, off, ids, scores, true, filters


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_counts_match_brute_force(seed):
    type_of, off, ids, scores, true, filters = _case(seed)
    raw, filt = R.rank_counts(scores, true, type_of[true], off, ids, filters)
    for q in range(len(true)):
        t, tau = int(true[q]), int(type_of[true[q]])
        r = f = 0
        for j in range(len(type_of)):
            if type_of[j] != tau:
                continue
            if scores[q, j] < scores[q, t] or (scores[q, j] == scores[q, t] and j < t):
                r += 1
                f += 0 if j in filters[q] else 1
        assert raw[q] == r and filt[q] == f


@pytest.mark.parametrize("seed", [0, 1])
def test_topk_matches_brute_force(seed):
    type_of, off, ids, scores, true, filters = _case(seed)
    taus = np.random.default_rng(seed + 10).integers(0, 9, size=len(true))
    got_i, got_s = R.topk(scores, taus, off, ids, 12, filters)
    for q, tau in enumerate(taus):
        cand = [j for j in range(len(type_of)) if type_of[j] == tau and j not in filters[q]]
        cand.sort(key=lambda j: (scores[q, j], j))
        want = cand[:12] + [-1] * (12 - len(cand[:12]))
        assert got_i[q].tolist() == want
        n = min(12, len(cand))
        assert np.array_equal(got_s[q, :n], scores[q, want[:n]]) and np.isinf(got_s[q, n:]).all()


def test_one_type_reduces_to_all_entities():
    _, _, _, scores, true, filters = _case(3)
    n_rows = scores.shape[1]
    type_of = np.zeros(n_rows, dtype=np.int64)
    off, ids = D.build_type_csr(type_of, 1)
    raw, filt = R.rank_counts(scores, true, type_of[true], off, ids, filters)
    st = scores[np.arange(len(true)), true]
    j = np.arange(n_rows)
    before = (scores < st[:, None]) | ((scores == st[:, None]) & (j[None, :] < true[:, None]))
    assert np.array_equal(raw, before.sum(1))
    want_f = [int(before[q].sum()) - len(set(filters[q]) & set(np.flatnonzero(before[q]).tolist()))
              for q in range(len(true))]
    assert np.array_equal(filt, want_f)
    got = R.topk(scores, type_of[true], off, ids, 9, filters)
    want = topk_reference.topk(scores, np.arange(n_rows), 9, filters)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
