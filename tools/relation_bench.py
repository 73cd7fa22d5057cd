"""Relation prediction (HOLE_SIDE_RELATION) timed against the tail-side entity call on the same queries.

    python tools/relation_bench.py [--reps 20] [--out FILE]

Prints one JSON line.  Workloads:
  fb15k:   the real 59,071 FB15k test queries (tests/golden/fb15k_test_valid_triples.npz) x 1,345 relations, d=150,
           filtered against the FB15k valid triples (the synthetic trained-scale table of rank_fb15k_d150);
  diffbot: 100,000 queries x 14 relations, d=256, unfiltered (rank_diffbot_d256).
Per workload and operand precision (bf16, bf16x3): milliseconds per call of hole_rank and hole_topk (k = 10) on the
relation side and, for scale, on the tail side over all entities (14,951 / 1,200,000 candidates).  Median of
--reps, CUDA events, the four calls alternating after warm-up; the operand cache holds one candidate range, so
every call re-packs its candidate operand, as an evaluation that alternates sides does.  Also the split of each
relation call between the packers, the contraction and the top-k merge (torch.profiler, a separate pass).
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

from graphembeddings_b200 import data as D  # noqa: E402
from graphembeddings_b200._lib import check  # noqa: E402
from graphembeddings_b200.engine import (HOLE_RANK_BF16, HOLE_RANK_BF16X3, HOLE_SIDE_RELATION,  # noqa: E402
                                         HOLE_SIDE_TAIL, HoleEngine, _ptr, _stream)
from topk_bench import _gpu_info, _kernel_split, _time  # noqa: E402

K = 10


def _calls(e, q, R, N, filters, precision):
    """name -> zero-argument call; outputs preallocated, no host synchronisation inside."""
    Q = q.shape[0]
    (rfo, rfi), (tfo, tfi) = filters
    out = {}
    for side, name, b, en, fo, fi in ((HOLE_SIDE_RELATION, "relation", 0, R, rfo, rfi),
                                      (HOLE_SIDE_TAIL, "tail", R, N, tfo, tfi)):
        raw = torch.zeros(Q, dtype=torch.int32, device="cuda")
        filt, ts = torch.zeros_like(raw), torch.zeros(Q, dtype=torch.float32, device="cuda")
        ids = torch.empty((Q, K), dtype=torch.int32, device="cuda")
        sc = torch.empty((Q, K), dtype=torch.float32, device="cuda")

        def rank(side=side, b=b, en=en, fo=fo, fi=fi, raw=raw, filt=filt, ts=ts):
            e.rank_ex(q, side, b, en, filter_off=fo, filter_ids=fi, precision=precision, true_score=ts,
                      raw_before=raw, filt_before=filt)

        def topk(side=side, b=b, en=en, fo=fo, fi=fi, ids=ids, sc=sc):
            check(e.lib.hole_topk(e._ctx, _ptr(e.table), b, en, _ptr(q), Q, side, precision, K, _ptr(fo), _ptr(fi),
                                  _ptr(ids), _ptr(sc), _stream()))

        out[f"{name}_rank"], out[f"{name}_topk{K}"] = rank, topk
    return out


def bench(label, e, queries, R, N, filters, reps):
    q = torch.as_tensor(queries, dtype=torch.int32).cuda().contiguous()
    dev = [tuple(None if x is None else torch.as_tensor(x).cuda() for x in f) for f in filters]
    res = {"workload": label, "queries": int(q.shape[0]), "relations": R, "entities": N - R, "dim": e.dim,
           "filtered": filters[0][0] is not None}
    for pname, prec in (("bf16", HOLE_RANK_BF16), ("bf16x3", HOLE_RANK_BF16X3)):
        calls = _calls(e, q, R, N, dev, prec)
        for _ in range(3):
            for fn in calls.values():
                fn()
        torch.cuda.synchronize()
        times = {k: [] for k in calls}
        for _ in range(reps):
            for k, fn in calls.items():
                times[k].append(_time(fn))
        r = {k: {"ms": float(np.median(v)), "ms_min": float(np.min(v))} for k, v in times.items()}
        for k in ("relation_rank", f"relation_topk{K}"):
            r[k]["kernels_ms"] = _kernel_split(calls[k])
        r["relation_rank_over_tail_rank"] = r["relation_rank"]["ms"] / r["tail_rank"]["ms"]
        r[f"relation_topk{K}_over_tail_topk{K}"] = r[f"relation_topk{K}"]["ms"] / r[f"tail_topk{K}"]["ms"]
        r["relation_flop"] = 2.0 * e.dim * q.shape[0] * R
        res[pname] = r
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "relation_bench needs a GPU"
    out = {"gpu": _gpu_info(), "k": K}
    kg = D.make_config("rank_fb15k_d150", trained_scale=True)
    npz = np.load(os.path.join(ROOT, "tests", "golden", "fb15k_test_valid_triples.npz"))
    test, valid = npz["test"], npz["valid"]
    filters = (D.build_filter_csr(test, valid, "relation"), D.build_filter_csr(test, valid, "tail"))
    e = HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E)
    out["fb15k"] = bench("FB15k test queries x 1,345 relations, d=150, filtered against valid", e, test,
                         kg.n_relations, kg.n_rows, filters, a.reps)
    e.close()
    del e
    torch.cuda.empty_cache()
    kg = D.make_config("rank_diffbot_d256", trained_scale=True)
    e = HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E)
    out["diffbot"] = bench("100,000 queries x 14 relations, d=256, unfiltered", e, kg.triples, kg.n_relations,
                           kg.n_rows, ((None, None), (None, None)), a.reps)
    e.close()
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
