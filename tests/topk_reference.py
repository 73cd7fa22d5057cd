"""fp64 NumPy statement of the top-k prediction contract (include/hole_b200.h, hole_topk), shared by
tests/test_topk_oracle.py (held to the reference's own heap pops) and tests/test_gpu_topk.py (held against the
device).  TEST INFRASTRUCTURE ONLY."""
import numpy as np


def topk(scores, cand_ids, k, filter_lists=None):
    """The first k pops of the reference heap (holE.py:427-472, cut at max_triples) for every query row,
    skipping in-sample candidates: ascending by (score, candidate id) (holE.py:231, 434, 446-453), in float64.

    scores[q, j] is candidate cand_ids[j] for query q; filter_lists[q] = ids to skip (train/valid-true).
    Returns (ids int64[Q, k], scores float64[Q, k]); rows with fewer than k candidates left are padded with
    id -1 and score +inf."""
    scores = np.asarray(scores, dtype=np.float64)
    cand_ids = np.asarray(cand_ids, dtype=np.int64)
    Q = scores.shape[0]
    ids = np.full((Q, k), -1, dtype=np.int64)
    vals = np.full((Q, k), np.inf, dtype=np.float64)
    for q in range(Q):
        keep = np.ones(len(cand_ids), dtype=bool)
        if filter_lists is not None:
            keep &= ~np.isin(cand_ids, np.asarray(list(filter_lists[q]), dtype=np.int64))
        c, s = cand_ids[keep], scores[q, keep]
        order = np.lexsort((c, s))[:k]
        ids[q, :len(order)] = c[order]
        vals[q, :len(order)] = s[order]
    return ids, vals
