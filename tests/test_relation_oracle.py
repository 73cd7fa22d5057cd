"""Relation prediction on the CPU: the query vectors of tests/relation_reference.py against the score definitions,
the "relation" filter CSR, and the --relation_prediction flag."""
import numpy as np
import pytest

from graphembeddings_b200 import data as D
from oracle import hole_ccorr as OC
from oracle import hole_oracle as O
import relation_reference as RR


def _table(scale):
    """fp64 table whose rows have norms scale * U(0.5, 1.5): some rows are clipped, some are not."""
    rng = np.random.default_rng(7)
    E = rng.standard_normal((60, 22))
    E *= scale * rng.uniform(0.5, 1.5, size=(60, 1)) / np.linalg.norm(E, axis=1, keepdims=True)
    queries = np.stack([rng.integers(10, 60, 40), rng.integers(10, 60, 40), rng.integers(0, 10, 40)], 1)
    return E, queries


@pytest.mark.parametrize("scale", [0.5, 1.0, 2.0])
@pytest.mark.parametrize("mode", ["complex", "ccorr_tanh"])
def test_query_vector_times_relation_row_is_the_score(mode, scale):
    E, q = _table(scale)
    _, _, clipped = O.clip_rows(E)
    if scale == 1.0:
        assert clipped.any() and not clipped.all()
    y, _, _ = O.clip_rows(E[q[:, 2]])
    if mode == "complex":
        got = np.sum(RR.query_vectors(E, q) * y, axis=1)
        want = O.score(E, q, np.float64)
    else:
        got = np.sum(RR.ccorr_query_vectors(E, q) * y, axis=1)
        want = OC.raw_score(E, q, np.float64, direct=True)
    assert np.abs(got - want).max() <= 1e-12
    # the all-candidate forms: column r of row q is the score of (h, r, t)
    cand = np.arange(10)
    S = RR.all_scores(E, q, cand) if mode == "complex" else RR.ccorr_all_scores(E, q, cand)
    assert np.abs(S[np.arange(len(q)), q[:, 2]] - want).max() <= 1e-12


def test_filter_csr_relation_side():
    known = np.array([[5, 6, 3], [5, 6, 1], [5, 6, 3],      # duplicate (5, 6, 3)
                      [6, 5, 2],                            # the reversed pair is another key
                      [7, 8, 0], [5, 6, 2], [7, 8, 4], [7, 9, 1]], dtype=np.int32)
    queries = np.array([[7, 8, 1], [5, 6, 0], [9, 9, 9], [6, 5, 0], [5, 6, 3]], dtype=np.int32)
    off, ids = D.build_filter_csr(queries, known, "relation")
    assert off.dtype == np.int64 and ids.dtype == np.int32
    got = [ids[off[i]:off[i + 1]].tolist() for i in range(len(queries))]
    assert got == [[0, 4], [1, 2, 3], [], [2], [1, 2, 3]]
    # the order of the known triples does not matter
    perm = np.random.default_rng(0).permutation(len(known))
    off2, ids2 = D.build_filter_csr(queries, known[perm], "relation")
    assert np.array_equal(off, off2) and np.array_equal(ids, ids2)


def test_relation_prediction_flag():
    from graphembeddings_b200 import hole
    base = ["--data_dir", "d", "--output_dir", "o"]
    assert hole.build_parser().parse_args(base + ["--infer"]).relation_prediction is False
    f = hole.build_parser().parse_args(base + ["--infer", "--relation_prediction", "--predict_top_k", "5"])
    assert f.relation_prediction is True and f.predict_top_k == 5
