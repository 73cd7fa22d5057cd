"""Nearest neighbours (hole_neighbors) on the ranking contraction, next to top-k link prediction (hole_topk).

    python tools/neighbors_bench.py [--reps 10] [--out FILE]

Prints one JSON line.  Workloads, all at k = 10:
  fb15k:      all 14,951 entity rows against themselves, d=150 (the trained-scale table of BASELINE config
              rank_fb15k_d150), bf16 and bf16x3;
  config3:    100,000 entity queries x 1,200,000 entity rows, d=256 (rank_diffbot_d256), bf16, alternating in the
              same process with hole_topk on the tail side (same Q, same k; neither call keeps a prepared operand,
              since each drops the other's, so both re-pack their candidates);
  all_pairs:  the k-NN graph of all 1,200,000 entity rows of that table in one bf16 call: 1.44e12 similarities.
Per workload: milliseconds per call (median of --reps after warm-up, CUDA events), similarities/s, FLOP/s at
2*D per similarity on the true D and its share of the sustained bf16 tensor figure (MEASURED_PEAKS.json through
rank_bench; null without it), the contraction / merge / packing split (torch.profiler, a separate pass), and a
check of 16 sampled query rows against an fp64 cosine top-k of the same table (id set outside the precision's
band, similarity error).  The GPU's name and power limit are read in the same run.
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
from graphembeddings_b200.engine import HOLE_RANK_BF16, HOLE_RANK_BF16X3, HOLE_SIDE_TAIL, HoleEngine  # noqa: E402
from graphembeddings_b200.rank_bench import _tensor_peak_sustained  # noqa: E402

K = 10
BANDS = {HOLE_RANK_BF16: 4e-3, HOLE_RANK_BF16X3: 3e-5}
NAMES = {HOLE_RANK_BF16: "bf16", HOLE_RANK_BF16X3: "bf16x3"}


def _gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name()


def _p(t):
    return C.c_void_p(t.data_ptr())


class Calls:
    """Library calls on preallocated device tensors (the engine's argument checks and allocations stay out of the
    timed window)."""

    def __init__(self, e, b, en, Q):
        self.e, self.b, self.en = e, b, en
        self.ids = torch.empty((Q, K), dtype=torch.int32, device="cuda")
        self.vals = torch.empty((Q, K), dtype=torch.float32, device="cuda")
        self.tk_ids, self.tk_scores = torch.empty_like(self.ids), torch.empty_like(self.vals)
        self.st = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def neighbors(self, q, precision):
        check(self.e.lib.hole_neighbors(self.e._ctx, _p(self.e.table), self.b, self.en, _p(q), q.shape[0], precision,
                                        K, None, None, _p(self.ids), _p(self.vals), self.st))

    def topk(self, tq, precision):
        check(self.e.lib.hole_topk(self.e._ctx, _p(self.e.table), self.b, self.en, _p(tq), tq.shape[0],
                                   HOLE_SIDE_TAIL, precision, K, None, None, _p(self.tk_ids), _p(self.tk_scores), self.st))


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
        elif "_pack_" in ev.key:
            out["packing_ms"] += t
    return out


def _check(E, qids, b, en, ids, sims, rows, band):
    """Sampled rows against an fp64 cosine top-k of the same table (torch on the GPU)."""
    Ed = torch.as_tensor(E[b:en], device="cuda").double()
    n = Ed.norm(dim=1, keepdim=True)
    U = torch.where(n > 0, Ed / n, torch.zeros_like(Ed))
    ok, worst = 0, 0.0
    for row in rows:
        qi = int(qids[row])
        qv = torch.as_tensor(E[qi], device="cuda").double()
        qv = qv / qv.norm() if float(qv.norm()) > 0 else qv
        s = U @ qv
        if b <= qi < en:
            s[qi - b] = -float("inf")                              # the row itself is never returned
        kth = float(torch.topk(s, K).values[-1])
        g = ids[row].long() - b
        sg = s[g]
        inside = bool((sg >= kth - band).all())
        covered = bool(torch.isin((s > kth + band).nonzero().flatten(), g).all())
        worst = max(worst, float((sims[row].double() - sg).abs().max()))
        ok += int(inside and covered and bool(torch.isfinite(sg).all()))
    return {"sampled_rows": len(rows), "rows_within_band": ok, "max_abs_sim_err_vs_fp64": worst}


def _rates(ms, Q, Nc, dim):
    sims = float(Q) * Nc
    flops = sims * 2 * dim
    peak = _tensor_peak_sustained()
    return {"similarities_per_s": sims / (ms * 1e-3), "tflops": flops / (ms * 1e-3) / 1e12,
            "frac_of_sustained_bf16_peak": (flops / (ms * 1e-3) / 1e12 / peak) if peak else None}


def bench_neighbors(e, E, qids, b, en, precision, reps, name):
    q = torch.as_tensor(qids, dtype=torch.int32, device="cuda")
    c = Calls(e, b, en, len(qids))

    def call():
        c.neighbors(q, precision)
    for _ in range(2):
        call()
    torch.cuda.synchronize()
    t = [_time(call) for _ in range(reps)]
    ms = float(np.median(t))
    ids, sims = c.ids, c.vals
    rows = np.sort(np.random.default_rng(5).choice(len(qids), size=16, replace=False))
    res = {"workload": name, "precision": NAMES[precision], "queries": len(qids), "candidates": en - b,
           "dim": int(E.shape[1]), "k": K, "ms": ms, "ms_all": t, **_rates(ms, len(qids), en - b, E.shape[1]),
           "kernels": _kernel_split(call), "check": _check(E, qids, b, en, ids, sims, rows, BANDS[precision])}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "neighbors_bench needs a GPU"
    out = {"gpu": _gpu_info(), "k": K, "sustained_bf16_tflops": _tensor_peak_sustained(),
           "note": "selection at the operand precision, similarities rescored in fp32"}
    # fb15k: all entity rows against themselves
    kg = D.make_config("rank_fb15k_d150", trained_scale=True)
    e = HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E)
    b, en = kg.n_relations, kg.n_rows
    ents = np.arange(b, en)
    out["fb15k"] = [bench_neighbors(e, kg.E, ents, b, en, p, a.reps, "all 14,951 FB15k entity rows x themselves, d=150")
                    for p in (HOLE_RANK_BF16, HOLE_RANK_BF16X3)]
    e.close()
    del e
    # config 3 shape: neighbours and tail-side top-k alternating
    kg = D.make_config("rank_diffbot_d256", trained_scale=True)
    e = HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E)
    b, en = kg.n_relations, kg.n_rows
    qids = torch.as_tensor(np.random.default_rng(7).choice(np.arange(b, en), size=100_000, replace=False),
                           dtype=torch.int32, device="cuda")
    tq = torch.as_tensor(kg.triples, dtype=torch.int32, device="cuda")
    c = Calls(e, b, en, len(qids))
    nb_call, tk_call = (lambda: c.neighbors(qids, HOLE_RANK_BF16)), (lambda: c.topk(tq, HOLE_RANK_BF16))
    for _ in range(2):
        nb_call()
        tk_call()
    torch.cuda.synchronize()
    reps3 = max(3, a.reps // 2)
    tn, tt = [], []
    for _ in range(reps3):
        tn.append(_time(nb_call))
        tt.append(_time(tk_call))
    mn, mt = float(np.median(tn)), float(np.median(tt))
    nb_call()
    ids, sims = c.ids, c.vals
    rows = np.sort(np.random.default_rng(5).choice(len(qids), size=16, replace=False))
    out["config3"] = {"workload": "100,000 entity queries x 1,200,000 rows, d=256, bf16", "k": K,
                      "neighbors_ms": mn, "topk_tail_ms": mt, "ratio_to_topk": mn / mt,
                      "neighbors_ms_all": tn, "topk_ms_all": tt, **_rates(mn, len(qids), en - b, kg.dim),
                      "neighbors_kernels": _kernel_split(nb_call), "topk_kernels": _kernel_split(tk_call),
                      "check": _check(kg.E, qids.cpu().numpy(), b, en, ids, sims, rows, BANDS[HOLE_RANK_BF16])}
    del ids, sims, c
    # all-pairs k-NN graph of the 1.2 M entity rows in one call
    out["all_pairs"] = bench_neighbors(e, kg.E, np.arange(b, en), b, en, HOLE_RANK_BF16, max(3, a.reps // 3),
                                       "k-NN graph of all 1,200,000 entity rows, d=256, one call")
    e.close()
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
