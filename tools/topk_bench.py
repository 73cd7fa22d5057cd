"""Top-k link prediction (hole_topk) against the counting ranking call (hole_rank) on the same queries.

    python tools/topk_bench.py [--reps 10] [--out FILE]

Prints one JSON line.  Workloads:
  config 2: the real 59,071 FB15k test queries (tests/golden/fb15k_test_valid_triples.npz), both sides in one call,
            14,951 candidates, d=150, filtered against the FB15k valid triples (the synthetic trained-scale table
            of BASELINE config rank_fb15k_d150);
  config 3: 100,000 queries x 1,200,000 candidates, d=256, tail side, unfiltered (rank_diffbot_d256).
Each runs at k = 10 and 100 with bf16 operands; the candidate operand is packed once (hole_rank_prepare), as an
evaluation over a static table does.  Per k: milliseconds per call (median of --reps, CUDA events, top-k and
counting calls alternating after warm-up), candidate scores/s, the ratio to the counting call, the split of
the top-k call between the contraction and the merge kernel (torch.profiler, a separate pass), and an output
check of 16 sampled queries against an fp64 top-k of the same table (bf16 band 4e-3 |q|).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from graphembeddings_b200 import data as D  # noqa: E402
from graphembeddings_b200._lib import check  # noqa: E402
from graphembeddings_b200.engine import (HOLE_RANK_BF16, HOLE_SIDE_BOTH, HOLE_SIDE_TAIL,  # noqa: E402
                                         HoleEngine)
from oracle import hole_oracle as O  # noqa: E402


def _gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name()


def _p(t):
    return C.c_void_p(0) if t is None else C.c_void_p(t.data_ptr())


class Workload:
    def __init__(self, eng, queries, side, b, en, foff=None, fids=None):
        self.e, self.side, self.b, self.en = eng, side, b, en
        self.q = torch.as_tensor(queries, dtype=torch.int32).cuda().contiguous()
        self.nq = self.q.shape[0]
        self.rows = self.nq * (2 if side == HOLE_SIDE_BOTH else 1)
        self.foff = None if foff is None else torch.as_tensor(foff, dtype=torch.int64).cuda()
        self.fids = None if fids is None else torch.as_tensor(fids, dtype=torch.int32).cuda()
        self.raw = torch.zeros(self.rows, dtype=torch.int32, device="cuda")
        self.filt = torch.zeros_like(self.raw)
        self.ts = torch.zeros(self.rows, dtype=torch.float32, device="cuda")
        self.stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def rank(self):
        check(self.e.lib.hole_rank(self.e._ctx, _p(self.e.table), self.b, self.en, _p(self.q), self.nq, self.side,
                                   HOLE_RANK_BF16, _p(self.foff), _p(self.fids), _p(self.ts), 1, _p(self.raw),
                                   _p(self.filt), self.stream))

    def topk(self, k, ids, scores):
        check(self.e.lib.hole_topk(self.e._ctx, _p(self.e.table), self.b, self.en, _p(self.q), self.nq, self.side,
                                   HOLE_RANK_BF16, k, _p(self.foff), _p(self.fids), _p(ids), _p(scores),
                                   self.stream))


def _time(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def _kernel_split(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {"contraction_ms": 0.0, "merge_ms": 0.0, "packing_ms": 0.0}
    for ev in prof.key_averages():
        t = ev.device_time_total / 1e3 if hasattr(ev, "device_time_total") else ev.cuda_time_total / 1e3
        if "hole_topk_merge" in ev.key:
            out["merge_ms"] += t
        elif "hole_rank_kernel" in ev.key:
            out["contraction_ms"] += t
        elif "hole_rank_pack" in ev.key:
            out["packing_ms"] += t
    return out


def _check(w, E, ids, scores, k, sample, filters):
    """Sampled rows against an fp64 top-k (torch on the GPU) of the same table: id sets equal outside the bf16
    band 4e-3 |q| around the k-th score, returned scores within that band of the fp64 score."""
    names = ("tail", "head")
    Ed = torch.as_tensor(E[w.b:w.en], device="cuda").double()
    Ed = Ed * torch.clamp(1.0 / Ed.norm(dim=1, keepdim=True), max=1.0)
    ok, worst = 0, 0.0
    for row in sample:
        src, sd = (row, 0) if row < w.nq else (row - w.nq, 1)
        if w.side != HOLE_SIDE_BOTH:
            sd = 0 if w.side == HOLE_SIDE_TAIL else 1
        qv = O.query_vectors(E.astype(np.float64), w.q[src:src + 1].cpu().numpy(), names[sd], np.float64)[0]
        s = Ed @ torch.as_tensor(qv, device="cuda")
        if filters is not None:
            fl = filters[1][filters[0][row]:filters[0][row + 1]].astype(np.int64) - w.b
            fl = fl[(fl >= 0) & (fl < w.en - w.b)]
            s[torch.as_tensor(fl, device="cuda")] = float("inf")
        want = torch.topk(s, k, largest=False).values
        kth = float(want[-1])
        band = 4e-3 * float(np.linalg.norm(qv))
        g = ids[row].long() - w.b
        sg = s[g]
        inside = bool((sg <= kth + band).all())
        sure = (s < kth - band).nonzero().flatten()
        covered = bool(torch.isin(sure, g).all())
        worst = max(worst, float((scores[row].double() - sg).abs().max()))
        ok += int(inside and covered and bool(torch.isfinite(sg).all()))
    return {"sampled_rows": len(sample), "rows_within_band": ok, "max_abs_score_err_vs_fp64": worst}


def bench(name, w, E, ks, reps, filters=None):
    res = {"workload": name, "queries_rows": w.rows, "candidates": w.en - w.b, "dim": int(E.shape[1])}
    w.e.rank_prepare(w.b, w.en, HOLE_RANK_BF16)
    rng = np.random.default_rng(5)
    sample = np.sort(rng.choice(w.rows, size=16, replace=False))
    for k in ks:
        ids = torch.empty((w.rows, k), dtype=torch.int32, device="cuda")
        sc = torch.empty((w.rows, k), dtype=torch.float32, device="cuda")
        for _ in range(2):
            w.rank()
            w.topk(k, ids, sc)
        torch.cuda.synchronize()
        t_rank, t_topk = [], []
        for _ in range(reps):
            t_rank.append(_time(w.rank))
            t_topk.append(_time(lambda: w.topk(k, ids, sc)))
        mr, mt = float(np.median(t_rank)), float(np.median(t_topk))
        n_scores = float(w.rows) * (w.en - w.b)
        res[f"k{k}"] = {"topk_ms": mt, "rank_ms": mr, "ratio_to_rank": mt / mr,
                        "topk_scores_per_s": n_scores / (mt * 1e-3), "rank_scores_per_s": n_scores / (mr * 1e-3),
                        "topk_ms_all": t_topk, "rank_ms_all": t_rank,
                        "topk_kernels": _kernel_split(lambda: w.topk(k, ids, sc)),
                        "check": _check(w, E, ids, sc, k, sample, filters)}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    ap.add_argument("--skip-config3", action="store_true")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "topk_bench needs a GPU"
    out = {"gpu": _gpu_info(), "precision": "bf16 operands, fp32 accumulate; fp32 rescore"}
    # config 2
    kg = D.make_config("rank_fb15k_d150", trained_scale=True)
    npz = np.load(os.path.join(ROOT, "tests", "golden", "fb15k_test_valid_triples.npz"))
    test, valid = npz["test"], npz["valid"]
    ft, fh = D.build_filter_csr(test, valid, "tail"), D.build_filter_csr(test, valid, "head")
    fo = np.concatenate([ft[0], fh[0][1:] + ft[0][-1]])
    fi = np.concatenate([ft[1], fh[1]])
    e = HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E)
    w = Workload(e, test, HOLE_SIDE_BOTH, kg.n_relations, kg.n_rows, fo, fi)
    out["config2"] = bench("FB15k test queries, both sides, 14,951 candidates, d=150, filtered", w, kg.E, (10, 100),
                           a.reps, (fo, fi))
    e.close()
    del w, e
    torch.cuda.empty_cache()
    if not a.skip_config3:
        kg = D.make_config("rank_diffbot_d256", trained_scale=True)
        e = HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E)
        w = Workload(e, kg.triples, HOLE_SIDE_TAIL, kg.n_relations, kg.n_rows)
        out["config3"] = bench("100,000 queries x 1,200,000 candidates, d=256, tail side", w, kg.E, (10, 100),
                               max(3, a.reps // 2))
        e.close()
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
