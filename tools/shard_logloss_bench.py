"""The row-sharded --log_loss step (P2PRowShardedTrainer.train_step_logloss = hole_shard_step_logloss) against the
one-GPU step (HoleEngine.train_step_logloss = hole_train_step_logloss) at N = 1: config 1's table (1,200,014 x 256,
bench.py's workload), B = 32768 triples per step, the workloads (k, l2) of DESIGN 7's table.  Both live in one
process and are timed alternately, --reps times each, with CUDA events around `--steps` consecutive one-step calls
(after --warmup steps of each workload).  Then, in a separate pass, the hole_shard_profile_read phase split of the
sharded step [corruption + route + post, gather, plan wait + k passes, push + finish, apply].  The card's name, power
limit and max SM clock are read in the same run.  Prints one JSON line (and writes it to --out).  N > 1 needs peers:
not measured here.

    python tools/shard_logloss_bench.py [--reps 3] [--out profiles/r08_shard_logloss_bench_n1.json]
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
from graphembeddings_b200.sharded import CudaBackend, P2PRowShardedTrainer  # noqa: E402

WORKLOADS = ((1, 0.0), (2, 0.0), (4, 0.0), (1, 1e-9))
PHASES = ("route_post", "gather", "passes", "push_finish", "apply")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name()


def timed(fn, steps):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(steps):
        fn(s)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--batch", type=int, default=32768)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    B, S, W = args.batch, args.steps, args.warmup
    n_steps = W + S
    kg, off, ids = bench.make_workload(n_steps * B)
    tri = torch.from_numpy(kg.triples).cuda()
    kmax = max(k for k, _ in WORKLOADS)
    be = CudaBackend(kg.n_relations, kg.dim, B, 0, kg.type_of, off, ids)
    tr = P2PRowShardedTrainer(kg.n_relations, kg.n_entities, kg.dim, be, None, negative_ratio=kmax).load_embeddings(kg.E)
    e = HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E).set_types(kg.type_of, off, ids)
    e.set_relation_count(kg.n_relations)
    batch = [tri[s * B:(s + 1) * B] for s in range(n_steps)]
    lr = 0.1

    def sharded(k, l2, s0):
        return lambda s: tr.train_step_logloss(batch[s0 + s], 1, s0 + s, lr, l2, k)

    def single(k, l2, s0):
        return lambda s: e.train_step_logloss(batch[s0 + s], 1, s0 + s, lr, l2, k)

    for k, l2 in WORKLOADS:
        timed(sharded(k, l2, 0), W)
        timed(single(k, l2, 0), W)
    runs = {(name, k, l2): [] for name in ("sharded", "single") for k, l2 in WORKLOADS}
    for _ in range(args.reps):
        for k, l2 in WORKLOADS:
            runs[("sharded", k, l2)].append(timed(sharded(k, l2, W), S))
            runs[("single", k, l2)].append(timed(single(k, l2, W), S))
    phases = {}
    eng = be.eng
    for k, l2 in WORKLOADS:
        torch.cuda.synchronize()
        eng.profile(True)
        for s in range(S):
            sharded(k, l2, W)(s)
        ph, n = eng.shard_profile_read()
        eng.profile(False)
        phases[f"k{k}_l2_{l2:g}"] = {name: round(ph[key] * 1e3, 1) for name, key in
                                     zip(PHASES, ("post", "k1", "k3", "finish", "apply"))}
    tr.check_barriers()
    rec = {"card": card(), "n_gpus": 1, "batch": B, "dim": kg.dim, "n_rows": kg.n_rows,
           "workload": bench.workload_desc(B), "steps_per_timing": S, "reps": args.reps,
           "timing": "CUDA events around --steps consecutive one-step calls, sharded and one-GPU alternating",
           "phase_us_per_step": phases, "phases": "sharded step: [corruption + route + post, gather (incl. its "
           "flag wait), the k passes (incl. the wait for their plan, built beside post and gather), push + finish, "
           "claim + decay + apply]", "results": {},
           "n_gt_1": "not measured (needs peers)"}
    for k, l2 in WORKLOADS:
        tag = f"k{k}_l2_{l2:g}"
        r = {}
        for name in ("sharded", "single"):
            us = runs[(name, k, l2)]
            r[name] = {"us_per_step_median": float(np.median(us)), "us_per_step_all": [round(u, 1) for u in us]}
        r["sharded_over_single"] = r["sharded"]["us_per_step_median"] / r["single"]["us_per_step_median"]
        rec["results"][tag] = r
    tr.close()
    be.eng.close()
    e.close()
    line = json.dumps(rec)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
