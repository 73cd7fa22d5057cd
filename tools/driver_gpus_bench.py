"""Times hole.py's training loop on config 1 (BASELINE.json configs[1]: 1.2 M entities, d = 256, 30 M triples):
hole.run_training_sharded on N GPUs and, at N = 1, the one-GPU hole.run_training on the same data, alternately.
Validation is off (an empty validation file) and every run trains two epochs; the timed window is the driver's
loop over the second one (its shuffle, the rank's share of the batches and the training calls, batch_count - 1 steps),
from the "Training epoch 2" log line to the "Done training" one, with a device synchronise at both ends.  The first
epoch warms the engines up (workspaces sized on first use); start-up (table initialisation, the triples' upload) and
the final checkpoint lie outside the window.  Prints one JSON line (rank 0).

    python tools/driver_gpus_bench.py [--batch 32768] [--repeats 3]
    python -m torch.distributed.run --nproc-per-node N tools/driver_gpus_bench.py --gpus N
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from graphembeddings_b200 import data as D
from graphembeddings_b200 import hole


def _card(local_rank):
    q = subprocess.run(["nvidia-smi", "-i", str(local_rank), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return {"name": torch.cuda.get_device_name(local_rank), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


class _LoopTimer:
    """A driver log that synchronises the device and reads the clock at the loop's first and last lines."""

    def __init__(self):
        self.t0 = self.t1 = None

    def __call__(self, *a):
        msg = " ".join(str(x) for x in a)
        if msg.startswith("Training epoch 2") or msg.startswith("Done training"):
            torch.cuda.synchronize()
            t = time.perf_counter()
            if msg.startswith("Training epoch 2"):
                self.t0 = t
            else:
                self.t1 = t

    @property
    def seconds(self):
        return self.t1 - self.t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--batch", type=int, default=32768, help="global batch (--batch_size)")
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank, local_rank = int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}; launch with torch.distributed.run")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    kg = D.make_config("diffbot_d256", with_embeddings=False)
    data = hole.HolEData()
    data.entity_count, data.relation_count = kg.n_rows, kg.n_relations
    data.id_to_type = dict(enumerate(kg.type_of.tolist()))
    data.triples, data.triple_count = kg.triples, len(kg.triples)
    data.validation_triples = np.zeros((0, 3), np.int32)
    steps = data.triple_count // args.batch - 1       # the steps of one epoch (holE.py:340)

    def run(sharded):
        tmp = tempfile.mkdtemp(prefix="driver_bench_") if rank == 0 else None
        if dist is not None:
            box = [tmp]
            dist.broadcast_object_list(box, src=0)
            tmp = box[0]
        out = os.path.join(tmp, "run")              # made by the driver (rank 0)
        flags = hole.build_parser().parse_args(["--data_dir", "-", "--output_dir", out, "--batch_size",
                                                str(args.batch), "--embedding_dim", str(kg.dim), "--num_epochs", "2",
                                                "--gpus", str(world)])
        timer = _LoopTimer()
        if sharded:
            hole.run_training_sharded(data, flags, dist, rank, world, local_rank, seed=1, log=timer)
        else:
            eng, _ = hole.run_training(data, flags, seed=1, log=timer)
            eng.close()
        if rank == 0:
            shutil.rmtree(tmp, ignore_errors=True)
            return steps * args.batch / timer.seconds
        return None

    paths = ("sharded", "single") if world == 1 else ("sharded",)
    rates = {p: [] for p in paths}
    for _ in range(args.repeats):
        for p in paths:
            rates[p].append(run(p == "sharded"))
            torch.cuda.empty_cache()
    if rank == 0:
        res = {"metric": "hole.py driver training loop, global triples/s", "n_gpus": world, "card": _card(local_rank),
               "workload": f"config 1 (diffbot_d256): {kg.n_entities:,} entities + {kg.n_relations} relations, d={kg.dim}, "
                           f"{data.triple_count:,} triples, global batch {args.batch}, the second epoch's {steps} steps, validation off",
               "repeats": args.repeats,
               "sharded_triples_per_s": {"median": float(np.median(rates["sharded"])), "all": rates["sharded"]}}
        if "single" in rates:
            res["single_gpu_driver_triples_per_s"] = {"median": float(np.median(rates["single"])), "all": rates["single"]}
            res["sharded_over_single"] = res["sharded_triples_per_s"]["median"] / res["single_gpu_driver_triples_per_s"]["median"]
        print(json.dumps(res), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
