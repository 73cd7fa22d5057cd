"""Type-constrained ranking and top-k (hole_rank_typed / hole_topk_typed) against the all-entity calls (hole_rank /
hole_topk) on the same queries.

    python tools/typed_bench.py [--reps 10] [--out FILE]

Prints one JSON line.  Workloads:
  rank_fb15k_d150: the 59,071 FB15k test queries (tests/golden/fb15k_test_valid_triples.npz) over the synthetic
                   trained-scale table of that BASELINE config, whose 815 entity types follow the FB15k type
                   histogram; tail and head side separately, filtered against the valid triples; bf16 and bf16x3;
                   rank and top-10;
  rank_diffbot_d256: 100,000 queries x 1,200,000 entities, d=256, 12 types (one of 99 % of the rows), tail, bf16,
                   unfiltered, rank.
Per case: milliseconds per call (median of --reps, CUDA events, typed and all-entity calls alternating after
warm-up), their ratio beside the ratio of (128-query x 256-candidate) tile pairs computed from the shapes, and the
typed call's kernel split (plan / packing / contraction / merge; torch.profiler, a separate pass).  The
all-entity calls re-pack their candidate operand every call, as the typed calls do.  The GPU name and power limit
are read in the same run.
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
from graphembeddings_b200.engine import HOLE_RANK_BF16, HOLE_RANK_BF16X3, HoleEngine  # noqa: E402

TAIL, HEAD = 0, 1


def _gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name()


def _p(t):
    return C.c_void_p(0) if t is None else C.c_void_p(t.data_ptr())


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
    out = {"plan_ms": 0.0, "packing_ms": 0.0, "contraction_ms": 0.0, "merge_ms": 0.0}
    for ev in prof.key_averages():
        t = ev.device_time_total / 1e3 if hasattr(ev, "device_time_total") else ev.cuda_time_total / 1e3
        if "hole_typed_" in ev.key:
            out["plan_ms"] += t
        elif "hole_topk_merge" in ev.key:
            out["merge_ms"] += t
        elif "hole_rank_kernel" in ev.key:
            out["contraction_ms"] += t
        elif "hole_rank_pack" in ev.key or "gather_true" in ev.key:
            out["packing_ms"] += t
    return out


def tile_pairs(taus, type_counts, n_candidates):
    """(typed, all-entity) tile pairs of 128 queries x 256 candidates, from shapes; the all-entity call ranks
    n_candidates rows (the entity range, without the relation rows)."""
    nq = np.bincount(taus, minlength=len(type_counts))
    typed = int(np.sum(-(-nq // 128) * -(-type_counts // 256) * (nq > 0)))
    return typed, int(-(-len(taus) // 128) * -(-n_candidates // 256))


def case(e, q, side, prec, b, en, foff, fids, k, reps):
    dev = e.device
    Q = q.shape[0]
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    n_types = e.csr_off.shape[0] - 1
    tcol = 1 if side == TAIL else 0
    taus = e.type_of[q[:, tcol].long()].contiguous()
    # the all-entity call with the same known-triple filter (a different question: it ranks against every entity)
    raw, filt = torch.zeros(Q, dtype=torch.int32, device=dev), torch.zeros(Q, dtype=torch.int32, device=dev)
    ts = torch.zeros(Q, dtype=torch.float32, device=dev)
    if k:
        ids = torch.empty((Q, k), dtype=torch.int32, device=dev)
        sc = torch.empty((Q, k), dtype=torch.float32, device=dev)
        typed = lambda: check(e.lib.hole_topk_typed(e._ctx, _p(e.table), _p(q), _p(taus), Q, side, prec, k,
                                                    _p(e.csr_off), _p(e.csr_ids), n_types, _p(foff), _p(fids),
                                                    _p(ids), _p(sc), s))
        untyped = lambda: check(e.lib.hole_topk(e._ctx, _p(e.table), b, en, _p(q), Q, side, prec, k, _p(foff),
                                                _p(fids), _p(ids), _p(sc), s))
    else:
        typed = lambda: check(e.lib.hole_rank_typed(e._ctx, _p(e.table), _p(q), Q, side, prec, _p(e.type_of),
                                                    _p(e.csr_off), _p(e.csr_ids), n_types, _p(foff), _p(fids),
                                                    _p(ts), _p(raw), _p(filt), s))

        def untyped():
            raw.zero_(); filt.zero_()
            check(e.lib.hole_rank(e._ctx, _p(e.table), b, en, _p(q), Q, side, prec, _p(foff), _p(fids), _p(ts), 1,
                                  _p(raw), _p(filt), s))
    for _ in range(2):
        typed(); untyped()
    torch.cuda.synchronize()
    tt, tu = [], []
    for _ in range(reps):
        tt.append(_time(typed))
        tu.append(_time(untyped))
    mt, mu = float(np.median(tt)), float(np.median(tu))
    counts = (e.csr_off[1:] - e.csr_off[:-1]).cpu().numpy()
    pt, pu = tile_pairs(taus.cpu().numpy(), counts, en - b)
    return {"side": "tail" if side == TAIL else "head", "precision": "bf16x3" if prec == HOLE_RANK_BF16X3 else "bf16",
            "call": f"top-{k}" if k else "rank", "queries": Q, "typed_ms": mt, "all_entity_ms": mu,
            "measured_ratio": mt / mu, "tile_pairs_typed": pt, "tile_pairs_all_entity": pu,
            "tile_pair_ratio_from_shapes": pt / pu, "typed_ms_all": tt, "all_entity_ms_all": tu,
            "typed_kernels": _kernel_split(typed)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "typed_bench needs a GPU"
    out = {"gpu": _gpu_info(), "cases": []}
    kg = D.make_config("rank_fb15k_d150", trained_scale=True)
    npz = np.load(os.path.join(ROOT, "tests", "golden", "fb15k_test_valid_triples.npz"))
    test, valid = npz["test"], npz["valid"]
    e = HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E).set_types(kg.type_of, *D.build_type_csr(kg.type_of))
    q = torch.as_tensor(test, dtype=torch.int32).cuda().contiguous()
    for side, name in ((TAIL, "tail"), (HEAD, "head")):
        fo, fi = D.build_filter_csr(test, valid, name)
        fo, fi = torch.as_tensor(fo).cuda(), torch.as_tensor(fi, dtype=torch.int32).cuda()
        for prec in (HOLE_RANK_BF16, HOLE_RANK_BF16X3):
            for k in (0, 10):
                r = case(e, q, side, prec, kg.n_relations, kg.n_rows, fo, fi, k, a.reps)
                r["workload"] = "rank_fb15k_d150"
                out["cases"].append(r)
    e.close()
    torch.cuda.empty_cache()
    kg = D.make_config("rank_diffbot_d256", trained_scale=True)
    e = HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E).set_types(kg.type_of, *D.build_type_csr(kg.type_of))
    q = torch.as_tensor(kg.triples, dtype=torch.int32).cuda().contiguous()
    r = case(e, q, TAIL, HOLE_RANK_BF16, kg.n_relations, kg.n_rows, None, None, 0, max(3, a.reps // 2))
    r["workload"] = "rank_diffbot_d256"
    out["cases"].append(r)
    e.close()
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
