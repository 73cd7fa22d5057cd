"""fp64 NumPy statement of the nearest-neighbour contract (include/hole_b200.h, hole_neighbors), shared by
tests/test_neighbors_oracle.py (held to scipy's cosine distance) and tests/test_gpu_neighbors.py (held against
the device).  TEST INFRASTRUCTURE ONLY."""
import numpy as np


def cosine(E, query_ids, cand_ids):
    """S[q, j] = cos(E[query_ids[q]], E[cand_ids[j]]) over the whole row in float64; 0 when either row is zero."""
    E = np.asarray(E, dtype=np.float64)
    n = np.linalg.norm(E, axis=1)
    U = np.divide(E, n[:, None], out=np.zeros_like(E), where=n[:, None] > 0)
    return U[np.asarray(query_ids, dtype=np.int64)] @ U[np.asarray(cand_ids, dtype=np.int64)].T


def neighbors(S, query_ids, cand_ids, k, filter_lists=None):
    """Row q: the k candidates with the highest S[q], by descending similarity, ties to the smaller id, never the
    query's own row, skipping filter_lists[q].  Returns (ids int64[Q, k], sims float64[Q, k]); rows with fewer
    than k candidates left are padded with id -1 and similarity -inf."""
    S = np.asarray(S, dtype=np.float64)
    cand_ids = np.asarray(cand_ids, dtype=np.int64)
    Q = S.shape[0]
    ids = np.full((Q, k), -1, dtype=np.int64)
    vals = np.full((Q, k), -np.inf, dtype=np.float64)
    for q in range(Q):
        keep = cand_ids != int(query_ids[q])
        if filter_lists is not None:
            keep &= ~np.isin(cand_ids, np.asarray(list(filter_lists[q]), dtype=np.int64))
        c, s = cand_ids[keep], S[q, keep]
        order = np.lexsort((c, -s))[:k]
        ids[q, :len(order)] = c[order]
        vals[q, :len(order)] = s[order]
    return ids, vals
