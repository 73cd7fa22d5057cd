"""SGD against AdaGrad on the row-sharded NVLink trainer (P2PRowShardedTrainer, hole_shard_steps), run under torchrun:
config 1's table (1,200,014 x 256, bench.py's workload) row-sharded over the ranks, B = 32768 triples per GPU and
step.  Two trainers (one SGD, one AdaGrad) live in one process and are timed alternately, `--reps` times each, with
CUDA events around one hole_shard_steps call of 20 and of 200 steps (max over ranks).  Then, in a separate pass, the
hole_shard_profile_read phase split [post, K1, K3, finish, apply] per step (min and max over ranks).  The card's
name and power limit are read in the same run.  Rank 0 prints one JSON line (and writes it to --out).

    python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tools/shard_adagrad_bench.py \
        [--reps 3] [--out profiles/r07_shard_adagrad_bench_nN.json]
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
import torch.distributed as dist  # noqa: E402

import bench  # noqa: E402
from graphembeddings_b200.sharded import CudaBackend, P2PRowShardedTrainer, _timed_device  # noqa: E402

PHASES = ("post", "k1", "k3", "finish", "apply")


def card(local):
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", str(local)], capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name(local)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--batch", type=int, default=32768)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    Bl, W, calls = args.batch, args.warmup, (20, 200)
    n_steps = W + max(calls)
    kg, off, ids = bench.make_workload(n_steps * Bl * world)
    mine = torch.from_numpy(kg.triples).view(n_steps, world, Bl, 3)[:, rank].contiguous().cuda()
    lrs = bench.lr_schedule(n_steps, 0, kg.triples.shape[0] // (Bl * world))
    trainers = {}
    for opt in ("sgd", "adagrad"):
        be = CudaBackend(kg.n_relations, kg.dim, Bl, local, kg.type_of, off, ids)
        tr = P2PRowShardedTrainer(kg.n_relations, kg.n_entities, kg.dim, be, dist).load_embeddings(kg.E)
        tr.set_optimizer(opt)
        tr.train_steps(mine[:W].view(-1, 3), Bl, 1, 0, bench.MARGIN, lrs[:W])
        trainers[opt] = tr
    runs = {(opt, K): [] for opt in trainers for K in calls}
    for _ in range(args.reps):
        for K in calls:
            for opt, tr in trainers.items():          # alternating, same process, same data
                ms, _ = _timed_device(dist, lambda: tr.train_steps(mine[W:W + K].view(-1, 3), Bl, 1, W, bench.MARGIN,
                                                                   lrs[W:W + K]))
                runs[(opt, K)].append(ms / K)
    phases = {}
    for opt, tr in trainers.items():
        tr.check_barriers()
        eng = tr.be.eng
        torch.cuda.synchronize()
        eng.profile(True)
        tr.train_steps(mine[W:W + 20].view(-1, 3), Bl, 1, W, bench.MARGIN, lrs[W:W + 20])
        ph, n = eng.shard_profile_read()
        eng.profile(False)
        t = torch.tensor([ph[k] for k in PHASES], device="cuda", dtype=torch.float64)
        tmax, tmin = t.clone(), t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
        phases[opt] = {k: [round(float(tmin[i]) * 1e3, 1), round(float(tmax[i]) * 1e3, 1)] for i, k in enumerate(PHASES)}
    for tr in trainers.values():
        tr.check_barriers()
        tr.close()
        tr.be.eng.close()
    if rank == 0:
        rec = {"card": card(local), "n_gpus": world, "batch_per_gpu": Bl, "global_batch": Bl * world, "dim": kg.dim,
               "n_rows": kg.n_rows, "workload": bench.workload_desc(Bl),
               "timing": "CUDA events around one hole_shard_steps call, max over ranks", "reps": args.reps,
               "phase_us_min_max_over_ranks": phases, "results": {}}
        for (opt, K), ms in runs.items():
            med = float(np.median(ms))
            rec["results"][f"{opt}_{K}"] = {"us_per_step_median": med * 1e3, "us_per_step_all": [m * 1e3 for m in ms],
                                            "triples_per_s": Bl * world / (med * 1e-3)}
        for K in calls:
            rec["results"][f"adagrad_over_sgd_{K}"] = (rec["results"][f"adagrad_{K}"]["us_per_step_median"] /
                                                       rec["results"][f"sgd_{K}"]["us_per_step_median"])
        line = json.dumps(rec)
        print(line, flush=True)
        if args.out:
            os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
            with open(args.out, "w") as f:
                f.write(line + "\n")
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
