"""fp64 NumPy statement of the type-constrained ranking and top-k contract (include/hole_b200.h, hole_rank_typed /
hole_topk_typed), reusing topk_reference for the selection.  TEST INFRASTRUCTURE ONLY."""
import numpy as np

import topk_reference


def rank_counts(scores, true_ids, query_types, csr_off, csr_ids, filter_lists=None):
    """scores[q, e]: the score of entity row e for query q (all rows); true_ids[q]: the true row; query_types[q]:
    its type.  Returns (raw int64[Q], filt int64[Q]):
        raw[q]  = #{j of type tau_q : (s_j, j) < (s_true, true)}
        filt[q] = raw[q] - #{f in filter[q] of type tau_q : (s_f, f) < (s_true, true)}   (repeated ids once)."""
    scores = np.asarray(scores, dtype=np.float64)
    Q = scores.shape[0]
    raw = np.zeros(Q, dtype=np.int64)
    filt = np.zeros(Q, dtype=np.int64)
    for q in range(Q):
        tau, t = int(query_types[q]), int(true_ids[q])
        cand = np.asarray(csr_ids[csr_off[tau]:csr_off[tau + 1]], dtype=np.int64)
        s, st = scores[q, cand], scores[q, t]
        before = (s < st) | ((s == st) & (cand < t))
        raw[q] = int(before.sum())
        f = np.unique(np.asarray(filter_lists[q] if filter_lists is not None else [], dtype=np.int64))
        filt[q] = raw[q] - int(np.isin(cand[before], f).sum())
    return raw, filt


def topk(scores, query_types, csr_off, csr_ids, k, filter_lists=None):
    """The first k candidates of each query's type by ascending (score, id), skipping its filter list; padded with
    (-1, +inf).  Returns (ids int64[Q, k], scores float64[Q, k])."""
    scores = np.asarray(scores, dtype=np.float64)
    Q = scores.shape[0]
    ids = np.full((Q, k), -1, dtype=np.int64)
    out = np.full((Q, k), np.inf)
    for q in range(Q):
        tau = int(query_types[q])
        cand = np.asarray(csr_ids[csr_off[tau]:csr_off[tau + 1]], dtype=np.int64)
        fl = None if filter_lists is None else [filter_lists[q]]
        i, s = topk_reference.topk(scores[q:q + 1, cand], cand, k, fl)
        ids[q], out[q] = i[0], s[0]
    return ids, out
