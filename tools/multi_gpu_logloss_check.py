"""torchrun check on N GPUs (real CUDA-IPC peers over NVLink) of the --log_loss step on the row-sharded trainer
(P2PRowShardedTrainer.train_step_logloss = hole_shard_step_logloss): trains on the real peers, gathers the table and
compares it on rank 0 with a single-GPU HoleEngine.train_step_logloss run over the same global batches, together
with every step's loss rows and the sum of the ranks' L2 parts.  Band after s steps: s times the one-step band of
DESIGN 7 (2e-6 + 1e-5 |x|).  Prints one JSON line per case and MULTI_GPU_LOGLOSS_CHECK OK on rank 0; exits non-zero
on a mismatch.

    python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tools/multi_gpu_logloss_check.py
"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist

from graphembeddings_b200 import data as D
from graphembeddings_b200.engine import HoleEngine
from graphembeddings_b200.sharded import CudaBackend, P2PRowShardedTrainer


def run_case(rank, world, local, dim, Bl, steps, n_ent, seed, k, l2):
    kg = D.synthetic_kg(9, n_ent, Bl * world * steps, 5, dim, seed=seed, trained_scale=True, zipf_entities=True)
    off, ids = D.build_type_csr(kg.type_of)
    be = CudaBackend(kg.n_relations, kg.dim, Bl, local, kg.type_of, off, ids)
    tr = P2PRowShardedTrainer(kg.n_relations, kg.n_entities, kg.dim, be, dist, negative_ratio=k).load_embeddings(kg.E)
    mine = torch.from_numpy(kg.triples).view(steps, world, Bl, 3)[:, rank].contiguous().cuda()
    lrs = [0.05 / (1 + 0.01 * s) for s in range(steps)]
    losses, parts = [], []
    for s in range(steps):
        loss, part = tr.train_step_logloss(mine[s], 3, s, lrs[s], l2, k)
        everyone = [torch.empty_like(loss) for _ in range(world)]
        dist.all_gather(everyone, loss)
        losses.append(torch.cat(everyone, dim=1))
        dist.all_reduce(part)
        parts.append(float(part))
    E = tr.gather_embeddings()
    res = {"trainer": type(tr).__name__, "world": world, "dim": dim, "batch_per_gpu": Bl, "steps": steps,
           "negative_ratio": k, "l2": l2}
    ok = True
    if rank == 0:
        e = HoleEngine(kg.n_rows, kg.dim, local).set_embeddings(kg.E).set_types(kg.type_of, off, ids)
        e.set_relation_count(kg.n_relations)
        loss_err, l2_err = 0.0, 0.0
        for s in range(steps):
            gb = kg.triples[s * Bl * world:(s + 1) * Bl * world]
            want, want_l2 = e.train_step_logloss(gb, 3, s, lrs[s], l2, k)
            loss_err = max(loss_err, float((losses[s] - want).abs().max()))
            if l2 != 0.0:
                l2_err = max(l2_err, abs(parts[s] - float(want_l2)) / float(want_l2))
        Ew = e.embeddings()
        rE = ((E - Ew).abs() / (steps * (2e-6 + 1e-5 * Ew.abs()))).max().item()
        moved = float((Ew.cpu() - torch.from_numpy(kg.E)).abs().max())
        res.update({"max_abs_err_table": float((E - Ew).abs().max()), "err_over_band_table": rE,
                    "max_abs_err_loss": loss_err, "max_rel_err_l2": l2_err, "moved": moved})
        ok = rE <= 1.0 and loss_err <= steps * 2e-6 and l2_err <= 1e-5 and moved > 1e-4
        res["ok"] = ok
        e.close()
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.broadcast(flag, 0)
    tr.close()
    be.eng.close()
    if rank == 0:
        print("MULTI_GPU_LOGLOSS_CHECK " + json.dumps(res), flush=True)
    return bool(flag.item())


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ok = True
    for dim, Bl, steps, n_ent, seed, k, l2 in [(256, 2048, 4, 50000, 77, 1, 1e-6),
                                                (150, 777, 3, 3000, 78, 4, 0.0),
                                                (64, 300, 3, 500, 79, 2, 1e-4)]:
        ok &= run_case(rank, world, local, dim, Bl, steps, n_ent, seed, k, l2)
    if rank == 0:
        print("MULTI_GPU_LOGLOSS_CHECK", "OK" if ok else "FAILED", flush=True)
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
