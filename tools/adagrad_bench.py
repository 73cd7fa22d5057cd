"""SGD against AdaGrad training steps on config 1 (bench.py's workload: 1,200,014 x 256 table, B = 32768), in one
process, alternating the two optimizers: one hole_train_steps call of 20 steps and one of 200 steps each, repeated,
then K1 / K3 times per step from the library's event hook (hole_profile_enable) in a separate pass.

The HBM roofline counts the algorithmic bytes of a triple's four rows: SGD reads and writes 4 table rows
(32 D + 20 B with the triple and the corrupt id), AdaGrad also 4 accumulator rows (64 D + 20 B; 16,404 B at
D = 256).  The card's name and power limit are read in the same run.

    python tools/adagrad_bench.py [--reps 3] [--out profiles/r06_adagrad_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from graphembeddings_b200.engine import HoleEngine  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--batch", type=int, default=32768)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    B, W, calls = args.batch, args.warmup, (20, 200)
    kg, off, ids = bench.make_workload((W + max(calls)) * B)
    dev_tri = torch.from_numpy(kg.triples).cuda()
    batch_count = kg.triples.shape[0] // B
    peak, peak_src, _ = bench.peaks()
    engines = {}
    for opt in ("sgd", "adagrad"):
        e = HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E).set_types(kg.type_of, off, ids)
        e.set_relation_count(kg.n_relations)
        e.set_optimizer(opt)
        bench.warm_up(e, dev_tri, B, W, 0, batch_count)
        engines[opt] = e
    bytes_per_triple = {"sgd": 32 * kg.dim + 20, "adagrad": 64 * kg.dim + 20}
    runs = {(opt, K): [] for opt in engines for K in calls}
    for _ in range(args.reps):
        for K in calls:
            for opt, e in engines.items():      # alternating, same process, same data
                v, ms = bench.timed_train(e, dev_tri, B, K, 0, batch_count, first_step=W)
                runs[(opt, K)].append(ms)
    prof = {}
    for opt, e in engines.items():
        torch.cuda.synchronize()
        e.profile(True)
        e.train_steps(dev_tri[W * B:(W + 20) * B], B, 1, W, bench.MARGIN, bench.lr_schedule(20, W, batch_count))
        k1, k3, n = e.profile_read()
        e.profile(False)
        prof[opt] = {"k1_us": k1 / n * 1e3, "k3_us": k3 / n * 1e3, "steps": n}
    rec = {"card": card(), "peak_hbm_gbs": peak, "peak_source": peak_src, "batch": B, "dim": kg.dim,
           "n_rows": kg.n_rows, "workload": bench.workload_desc(B), "bytes_per_triple": bytes_per_triple,
           "timing": "CUDA events around one hole_train_steps call", "results": {}}
    for (opt, K), ms in runs.items():
        med = float(np.median(ms))
        tps = B / (med * 1e-3)
        rec["results"][f"{opt}_{K}"] = {
            "ms_per_step_median": med, "ms_per_step_all": ms, "triples_per_s": tps,
            "roofline_triples_per_s": peak * 1e9 / bytes_per_triple[opt],
            "frac_of_hbm_roofline": tps * bytes_per_triple[opt] / (peak * 1e9)}
    rec["kernels"] = prof
    for K in calls:
        rec["results"][f"adagrad_over_sgd_{K}"] = (rec["results"][f"adagrad_{K}"]["ms_per_step_median"] /
                                                   rec["results"][f"sgd_{K}"]["ms_per_step_median"])
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
