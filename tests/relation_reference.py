"""fp64 NumPy statement of relation prediction (include/hole_b200.h, HOLE_SIDE_RELATION): the scores of every
relation row for (h, ?, t), shared by tests/test_relation_oracle.py and tests/test_gpu_relation.py.
TEST INFRASTRUCTURE ONLY.  Built on the oracle package, which it leaves unchanged; O.rank_counts and
topk_reference.topk are side-agnostic and apply to these scores as they are."""
import numpy as np

from oracle import hole_ccorr as OC
from oracle import hole_oracle as O


def query_vectors(E, queries, dtype=np.float64):
    """Complex score: q = [a e + b f ; a f - b e] = [Re w ; -Im w] with w = clip(h) o conj(clip(t)), so that
    score(h, r, t) = clip(E_r) . q (ds/dy_r of SURVEY App. A.3)."""
    queries = np.asarray(queries)
    a, b = O.get_embedding(E, queries[:, 0], dtype)
    e, f = O.get_embedding(E, queries[:, 1], dtype)
    return np.concatenate([a * e + b * f, a * f - b * e], axis=1)


def ccorr_query_vectors(E, queries, dtype=np.float64):
    """Archived score: q = [Re c + Im c ; Re c - Im c] with c = ccorr(clip(h), clip(t)), c_k = sum_j conj(h_j) t_{j+k},
    so that s(h, r, t) = Re sum_k (1 - i) r_k c_k = clip(E_r) . q."""
    queries = np.asarray(queries)
    H = E.shape[1] // 2
    h, t = (O.clip_rows(E[queries[:, col].astype(np.int64)].astype(dtype, copy=False))[0] for col in (0, 1))
    c = OC.ccorr_fft(h[:, :H] + 1j * h[:, H:], t[:, :H] + 1j * t[:, H:])
    return np.concatenate([c.real + c.imag, c.real - c.imag], axis=1).astype(dtype)


def all_scores(E, queries, cand_ids, dtype=np.float64):
    """Complex score of every relation candidate for every query, [Q, C] (GEMM form)."""
    y, _, _ = O.clip_rows(E[np.asarray(cand_ids, dtype=np.int64)].astype(dtype, copy=False))
    return query_vectors(E, queries, dtype) @ y.T


def ccorr_all_scores(E, queries, cand_ids, dtype=np.float64):
    """Archived raw score s of every relation candidate, [Q, C], straight from the definition (OC.raw_score on the
    expanded triples (h, t, candidate)), not through the query vector."""
    queries = np.asarray(queries)
    cand_ids = np.asarray(cand_ids)
    out = np.empty((len(queries), len(cand_ids)), dtype=dtype)
    for i, (h, t, _) in enumerate(queries.tolist()):
        tri = np.empty((len(cand_ids), 3), dtype=np.int64)
        tri[:, 0], tri[:, 1], tri[:, 2] = h, t, cand_ids
        out[i] = OC.raw_score(E, tri, dtype)
    return out
