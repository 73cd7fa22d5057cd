"""The top-k contract (tests/topk_reference.py, what hole_topk computes) against the reference's own heap order, on the
reference-executed cases of tests/golden/ranking_ref.json (holE.py:427-472, quantised values with exact ties)."""
import heapq
import json
import os

import numpy as np
import pytest

import topk_reference as T


def _cases(golden_dir):
    with open(os.path.join(golden_dir, "ranking_ref.json")) as f:
        return json.load(f)["cases"]


def _case_arrays(c):
    triples = np.array(c["triples"], dtype=np.int64)
    vals = np.array(c["values"], dtype=np.float32)
    true_t = {int(h): {int(r): set(ts) for r, ts in rr.items()} for h, rr in c["true_triples"].items()}
    test_t = {int(h): {int(r): set(ts) for r, ts in rr.items()} for h, rr in c["test_triples"].items()}
    # one head per case: the heap's tuple order (value, (h, t, r)) is (value, composite (t, r))
    comp = triples[:, 1] * 1000 + triples[:, 2]
    in_sample = [int(x) for x, (h, t, r) in zip(comp, triples.tolist()) if t in true_t.get(h, {}).get(r, ())]
    return triples, vals, comp, in_sample, test_t


def _heap_pops(vals, triples, in_sample_comp):
    heap = [(float(v), tuple(int(x) for x in tr)) for v, tr in zip(vals, triples)]
    heapq.heapify(heap)
    pops = []
    while heap:
        _, (h, t, r) = heapq.heappop(heap)
        if t * 1000 + r not in in_sample_comp:
            pops.append(t * 1000 + r)
    return pops


@pytest.mark.parametrize("k", [1, 3, 10, 200])
def test_topk_is_the_first_k_new_pops_of_the_reference_heap(golden_dir, k):
    for c in _cases(golden_dir):
        triples, vals, comp, in_sample, _ = _case_arrays(c)
        pops = _heap_pops(vals, triples, set(in_sample))
        ids, s = T.topk(vals[None, :].astype(np.float64), comp, k, [in_sample])
        n = min(k, len(pops))
        assert ids[0, :n].tolist() == pops[:n]
        assert np.all(ids[0, n:] == -1) and np.all(np.isinf(s[0, n:]))
        assert np.all(np.diff(s[0, :n]) >= 0)


@pytest.mark.parametrize("k", [1, 5, 20])
def test_reference_filtered_positions_land_in_the_oracle_top_k(golden_dir, k):
    """Every test triple the reference reports at filtered position p <= k is the oracle's p-th prediction."""
    checked = 0
    for c in _cases(golden_dir):
        triples, vals, comp, in_sample, test_t = _case_arrays(c)
        ids, _ = T.topk(vals[None, :].astype(np.float64), comp, k, [in_sample])
        # the reference records the test triples in pop order: ascending (value, t, r)
        items = sorted((float(v), t, r) for v, (h, t, r) in zip(vals, triples.tolist())
                       if t in test_t.get(h, {}).get(r, ()) and t * 1000 + r not in in_sample)
        assert len(items) == len(c["filtered_positions"])
        for (_, t, r), p in zip(items, c["filtered_positions"]):
            if p <= k:
                assert ids[0, p - 1] == t * 1000 + r
                checked += 1
    assert checked > 0
