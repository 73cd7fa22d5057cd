"""The nearest-neighbour contract (tests/neighbors_reference.py, what hole_neighbors computes) against scipy's cosine
distance, and on hand-made cases."""
import numpy as np
import pytest
from scipy.spatial.distance import cdist

import neighbors_reference as N


def _table(seed, n=300, dim=24):
    """Random rows of varied norm, with zero rows and duplicated rows."""
    rng = np.random.default_rng(seed)
    E = rng.normal(size=(n, dim)) * rng.uniform(0.05, 3.0, size=(n, 1))
    E[[3, 40, 41, 200]] = 0.0
    E[[17, 90, 250]] = E[5]
    E[[61, 62]] = E[60]
    return E.astype(np.float32)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_cosine_matches_scipy_and_zero_rows_are_zero(seed):
    E = _table(seed)
    qids = np.arange(len(E))
    cand = np.arange(20, len(E) - 10)
    S = N.cosine(E, qids, cand)
    zero = ~np.any(E != 0, axis=1)
    nz_q, nz_c = ~zero[qids], ~zero[cand]
    want = 1.0 - cdist(E[qids][nz_q].astype(np.float64), E[cand][nz_c].astype(np.float64), "cosine")
    assert np.abs(S[np.ix_(nz_q, nz_c)] - want).max() < 1e-12
    assert np.all(S[zero[qids]] == 0) and np.all(S[:, zero[cand]] == 0)
    assert np.isfinite(S).all()


@pytest.mark.parametrize("k", [1, 7, 50])
def test_selection_matches_a_scipy_argsort(k):
    E = _table(5)
    rng = np.random.default_rng(9)
    qids = rng.choice(len(E), size=40, replace=False)
    cand = np.arange(10, 280)
    flists = [np.sort(rng.choice(cand, size=rng.integers(0, 30), replace=False)) for _ in qids]
    ids, sims = N.neighbors(N.cosine(E, qids, cand), qids, cand, k, flists)
    E64 = E.astype(np.float64)
    for q, qi in enumerate(qids):
        ok = (cand != qi) & ~np.isin(cand, flists[q])
        c = cand[ok]
        if not np.any(E[qi]):
            want = c[:k]                                  # all similarities 0: id order
        else:
            s = np.zeros(len(c))
            nz = np.any(E[c] != 0, axis=1)
            s[nz] = 1.0 - cdist(E64[qi][None], E64[c[nz]], "cosine")[0]
            want = c[np.lexsort((c, -np.round(s, 12)))[:k]]
        assert ids[q, :len(want)].tolist() == want.tolist()
        assert np.all(np.diff(sims[q, :len(want)]) <= 0)


def test_self_is_excluded_and_twins_are_returned_in_id_order():
    E = _table(3)
    cand = np.arange(len(E))
    ids, sims = N.neighbors(N.cosine(E, [5, 60], cand), [5, 60], cand, 4)
    assert ids[0, :3].tolist() == [17, 90, 250] and np.allclose(sims[0, :3], 1.0)
    assert 5 not in ids[0]
    assert ids[1, :2].tolist() == [61, 62] and 60 not in ids[1]


def test_query_outside_the_range_excludes_nothing():
    E = _table(4)
    cand = np.arange(100, 200)
    ids, _ = N.neighbors(N.cosine(E, [5], cand), [5], cand, len(cand))
    assert sorted(ids[0].tolist()) == cand.tolist()
    ids, _ = N.neighbors(N.cosine(E, [150], cand), [150], cand, len(cand))
    assert 150 not in ids[0] and ids[0, -1] == -1


def test_exact_ties_go_to_the_smaller_id():
    E = np.zeros((8, 4), np.float32)
    E[0] = [1, 0, 0, 0]
    E[[6, 2, 4]] = [2, 0, 0, 0]                          # cos = 1 at three norms
    E[[1, 7]] = [0, 1, 0, 0]                             # cos = 0, as the zero rows 3 and 5
    ids, sims = N.neighbors(N.cosine(E, [0], np.arange(8)), [0], np.arange(8), 7)
    assert ids[0].tolist() == [2, 4, 6, 1, 3, 5, 7]
    assert sims[0].tolist() == [1, 1, 1, 0, 0, 0, 0]


def test_filter_slices_and_padding():
    E = _table(6)
    cand = np.arange(50, 60)
    qids = [55, 0]
    flists = [np.array([50, 51, 52, 53]), np.array([57])]
    ids, sims = N.neighbors(N.cosine(E, qids, cand), qids, cand, 8, flists)
    assert sorted(ids[0, :5].tolist()) == [54, 56, 57, 58, 59]       # 10 - 4 filtered - itself
    assert np.all(ids[0, 5:] == -1) and np.all(sims[0, 5:] == -np.inf)
    assert 57 not in ids[1] and np.all(ids[1] >= 0)
    ids, sims = N.neighbors(N.cosine(E, qids, cand[:0]), qids, cand[:0], 3)
    assert np.all(ids == -1) and np.all(sims == -np.inf)
