"""torchrun check on N GPUs (real CUDA-IPC peers over NVLink) of AdaGrad on the row-sharded trainer
(P2PRowShardedTrainer.set_optimizer("adagrad") = hole_shard_set_optimizer): trains on the real peers, gathers the
table and the accumulator, and compares them on rank 0 with a single-GPU AdaGrad HoleEngine run over the same
global batches.  Band after k steps: k times the one-step band of DESIGN 7c (2e-6 + 1e-5 |x| on a row, 1e-7 + 1e-5 |a|
on the accumulator).  Prints one JSON line per case and MULTI_GPU_ADAGRAD_CHECK OK on rank 0; exits non-zero on a
mismatch.

    python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tools/multi_gpu_adagrad_check.py
"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist

from graphembeddings_b200 import data as D
from graphembeddings_b200.engine import HoleEngine
from graphembeddings_b200.sharded import CudaBackend, P2PRowShardedTrainer, make_trainer

MARGIN = 0.2


def run_case(rank, world, local, dim, Bl, steps, n_ent, seed, chunked, init):
    kg = D.synthetic_kg(9, n_ent, Bl * world * steps, 5, dim, seed=seed, trained_scale=True, zipf_entities=True)
    off, ids = D.build_type_csr(kg.type_of)
    be = CudaBackend(kg.n_relations, kg.dim, Bl, local, kg.type_of, off, ids)
    tr = make_trainer(kg.n_relations, kg.n_entities, kg.dim, be, dist, log=print).load_embeddings(kg.E)
    assert isinstance(tr, P2PRowShardedTrainer), type(tr).__name__
    tr.set_optimizer("adagrad", init)
    mine = torch.from_numpy(kg.triples).view(steps, world, Bl, 3)[:, rank].contiguous().cuda()
    lrs = [0.3 / (1 + 0.01 * s) for s in range(steps)]
    if chunked:
        tr.train_steps(mine.view(-1, 3), Bl, 3, 0, MARGIN, lrs)
    else:
        for s in range(steps):
            tr.train_step(mine[s], 3, s, MARGIN, lrs[s], next_pos=mine[s + 1] if s + 1 < steps else None)
    E, A = tr.gather_embeddings(), tr.gather_accumulator()
    res = {"trainer": type(tr).__name__, "world": world, "dim": dim, "batch_per_gpu": Bl, "steps": steps,
           "chunked_call": bool(chunked), "initial_accumulator": init}
    ok = True
    if rank == 0:
        e = HoleEngine(kg.n_rows, kg.dim, local).set_embeddings(kg.E).set_types(kg.type_of, off, ids)
        e.set_relation_count(kg.n_relations)
        e.set_optimizer("adagrad", init)
        for s in range(steps):
            gb = kg.triples[s * Bl * world:(s + 1) * Bl * world]
            side, neg = e.corrupt_batch(gb, 3, s)
            e.train_step(gb, neg, side, MARGIN, lrs[s])
        Ew, Aw = e.embeddings(), e.accumulator()
        rE = ((E - Ew).abs() / (steps * (2e-6 + 1e-5 * Ew.abs()))).max().item()
        rA = ((A - Aw).abs() / (steps * (1e-7 + 1e-5 * Aw.abs()))).max().item()
        moved = float((Ew.cpu() - torch.from_numpy(kg.E)).abs().max())
        grown = float((Aw - init).max())
        res.update({"max_abs_err_table": float((E - Ew).abs().max()), "max_abs_err_accumulator": float((A - Aw).abs().max()),
                    "err_over_band_table": rE, "err_over_band_accumulator": rA, "moved": moved,
                    "accumulator_growth": grown})
        ok = rE <= 1.0 and rA <= 1.0 and moved > 1e-4 and grown > 0
        res["ok"] = ok
        e.close()
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.broadcast(flag, 0)
    tr.close()
    be.eng.close()
    if rank == 0:
        print("MULTI_GPU_ADAGRAD_CHECK " + json.dumps(res), flush=True)
    return bool(flag.item())


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ok = True
    for dim, Bl, steps, n_ent, seed, chunked, init in [(256, 2048, 4, 50000, 77, False, 0.1),
                                                        (150, 777, 5, 3000, 78, True, 0.1),
                                                        (64, 300, 3, 500, 79, True, 1e-3)]:
        ok &= run_case(rank, world, local, dim, Bl, steps, n_ent, seed, chunked, init)
    if rank == 0:
        print("MULTI_GPU_ADAGRAD_CHECK", "OK" if ok else "FAILED", flush=True)
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
