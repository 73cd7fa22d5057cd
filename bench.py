#!/usr/bin/env python
"""bench.py -- HolE training throughput on B200 (BASELINE.json metric), one JSON line.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--batch B] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of B synthetic triples: Philox
type-safe corruption, fused gather/clip/score/sigmoid/hinge forward+backward, deterministic
sparse SGD update.  Workload at N=1: BASELINE.json configs[1] (HolE d=256, 1,200,014-row
shared table, 12 types with one holding 99 %, Zipf relations) -- the table (1.2 GB) is far
larger than L2, so no flush is needed between steps.

  value    whole-job triples/s with the triples already resident in HBM
  e2e      same metric through the C-ABI host-buffer call (hole_train_steps_host): the
           step's triples are copied from pinned host memory and the step's loss is read
           back inside the timed region
  roofline algorithmic bytes (32*D + 20 per triple, SURVEY.md 8d) / summed duration of the
           step's two hot kernels, measured with CUDA events in a second pass
  cpu_baseline  oracle/hole_ref.c (C/OpenMP port of the reference arithmetic) on a bounded
           sample of the same workload, on this box's host cores

`--impl reference` times that CPU port alone (TensorFlow 1.2, which holE.py needs, cannot be
installed offline; see DESIGN.md).

`--dump-outputs DIR` (N = 1) writes what the timed call left to its caller, so that two builds can be
compared output for output on identical seeded inputs: loss_sums.npy (the per-step loss sums it
returned) and embeddings.npy (table rows after its last step, float32, at the row ids in
embedding_rows.npy; see dump_rows).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOAD = "diffbot_d256"


def workload_desc(batch):
    """The same string in both arms and at every N (the driver compares config.workload)."""
    return ("diffbot_d256: BASELINE.json configs[1], HolE d=256, 1,200,014-row shared table (14 relations + "
            "1.2M typed entities, 12 types, one holding 99 %), Zipf relations, type-safe Philox corruption, "
            f"B={batch} triples per step per GPU")


MARGIN, LR0 = 0.2, 0.1
#: dram__bytes_read.sum + dram__bytes_write.sum per step (K1 + K3) from the `ncu --set full`
#: captures under profiles/ for (batch, dim); other configurations report null
NCU_TRAFFIC = {(32768, 256): 158.4e6}   # profiles/r02_k1_raw.csv (98.5 + 45.5 MB) + r01_k3_raw.csv (14.4 MB)


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)", p
    return 6650.0, "fallback (B200_PROFILING.md)", {}


class ClockSampler:
    """SM clocks / throttle reasons during the timed region, polled every 100 ms through NVML
    in a background thread (an `nvidia-smi -lms` child process takes driver locks often enough
    to slow a launch-heavy multi-GPU step; NVML calls from this process are far lighter).
    Falls back to nvidia-smi when pynvml is unavailable."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0, period=0.1):
        self.index, self.period = index, period
        self.proc, self.lines, self.samples, self.reason_bits = None, [], [], 0
        self.max_clock, self.thread, self.stop_flag, self.nvml = None, None, False, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_clock = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
            self.thread = threading.Thread(target=self._poll_nvml, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _poll_nvml(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                self.samples.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
                self.reason_bits |= int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
            except Exception:
                try:
                    self.reason_bits |= int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
                except Exception:
                    pass
            time.sleep(self.period)

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.thread.join(timeout=2)
            bits = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
                    "sw_power_cap": 0x4}
            reasons = sorted(k for k, v in bits.items() if self.reason_bits & v)
            return {"sm_mhz": float(np.median(self.samples)) if self.samples else None,
                    "sm_max_mhz": self.max_clock, "samples": len(self.samples), "reasons": reasons,
                    "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        self.thread.join(timeout=2)
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            c = [x.strip() for x in l.split(",")]
            if len(c) < 7:
                continue
            try:
                sm.append(float(c[0])); mx = float(c[1])
            except ValueError:
                continue
            for n, v in zip(names, c[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx,
                "samples": len(sm), "reasons": sorted(reasons), "source": "nvidia-smi"}


def settle_clocks(seconds=0.25):
    """Keep the GPU busy with device fills for a moment: after the clock sampler's start-up pause the SM
    and memory clocks have dropped to idle, and W = 3-5 warm-up steps (0.3 ms) are too short to raise them
    again.  Not a step; nothing of the workload runs here."""
    import torch
    buf = torch.empty(64 << 20, dtype=torch.float32, device="cuda")
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        for _ in range(8):
            buf.fill_(1.0)
        torch.cuda.synchronize()
    del buf


def make_workload(n_triples, with_embeddings=True):
    from graphembeddings_b200 import data as D
    kg = D.make_config(WORKLOAD, n_triples=n_triples, with_embeddings=with_embeddings)
    off, ids = D.build_type_csr(kg.type_of)
    return kg, off, ids


def lr_schedule(n_steps, first_step, batch_count):
    f = np.float32
    return np.array([f(LR0) / (f(1.0) + f(0.5) * (f(s) / f(32 * batch_count)))
                     for s in range(first_step, first_step + n_steps)], dtype=np.float32)


DUMP_SAMPLE = 16384      # rows per sampled set: at most 2 * 16384 + relations rows of d=256 floats (~34 MB)


def dump_rows(kg, last_batch):
    """Row ids whose final values --dump-outputs writes: every relation row, a seeded sample of the entity
    rows the last step's triples use, and a seeded sample of all entity rows.  The table itself (1.2 GB) is
    too large to write whole."""
    rng = np.random.default_rng(20170904)
    used = np.unique(last_batch[:, :2])
    ents = np.arange(kg.n_relations, kg.n_rows)
    return np.unique(np.concatenate([np.arange(kg.n_relations),
                                     rng.choice(used, min(DUMP_SAMPLE, len(used)), replace=False),
                                     rng.choice(ents, min(DUMP_SAMPLE, len(ents)), replace=False)]))


def write_dump(out_dir, loss_sums, rows, table_rows):
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss_sums.npy"), loss_sums)
    np.save(os.path.join(out_dir, "embedding_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "embeddings.npy"), np.ascontiguousarray(table_rows, dtype=np.float32))


def cpu_port_throughput(kg, off, ids, B, min_seconds, max_steps, warmup=1):
    """Time oracle/hole_ref.c train steps (corruption drawn by the NumPy Philox oracle
    outside the timed region); cycles over the generated batches until `min_seconds` of CPU
    work are done.  Returns (triples/s, cores, steps, seconds)."""
    from oracle import hole_oracle as O
    from oracle import hole_ref as R
    E = np.ascontiguousarray(kg.E, np.float32).copy()
    sc = R.TrainScratch(B, kg.dim)
    n_avail = min(kg.triples.shape[0] // B, 32)
    negs = [O.corrupt(kg.triples[s * B:(s + 1) * B], kg.type_of, off, ids, 1, s) for s in range(n_avail)]
    for s in range(min(warmup, n_avail)):
        R.train_step(E, kg.triples[s * B:(s + 1) * B], negs[s][1], negs[s][0], MARGIN, LR0, sc)
    done, t0 = 0, time.perf_counter()
    while done < max_steps:
        s = done % n_avail
        R.train_step(E, kg.triples[s * B:(s + 1) * B], negs[s][1], negs[s][0], MARGIN, LR0, sc)
        done += 1
        if time.perf_counter() - t0 >= min_seconds:
            break
    dt = time.perf_counter() - t0
    return done * B / dt, R.threads(), done, dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    B, K, W = args.batch, args.steps, args.warmup
    kg, off, ids = make_workload((K + W) * B)
    from oracle import hole_oracle as O
    from oracle import hole_ref as R
    # all the host threads this process may use (torchrun exports OMP_NUM_THREADS=1 to its workers;
    # the other ranks have exited, the cores are free)
    R.set_threads(int(os.environ.get("HOLE_REF_THREADS", len(os.sched_getaffinity(0)))))
    E = np.ascontiguousarray(kg.E, np.float32)
    sc = R.TrainScratch(B, kg.dim)
    negs = [O.corrupt(kg.triples[s * B:(s + 1) * B], kg.type_of, off, ids, 1, s) for s in range(K + W)]
    for s in range(W):
        R.train_step(E, kg.triples[s * B:(s + 1) * B], negs[s][1], negs[s][0], MARGIN, LR0, sc)
    sums = np.empty(K, np.float64)
    t0 = time.perf_counter()
    for s in range(W, W + K):
        sums[s - W], _ = R.train_step(E, kg.triples[s * B:(s + 1) * B], negs[s][1], negs[s][0], MARGIN, LR0, sc)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        rows = dump_rows(kg, kg.triples[(W + K - 1) * B:(W + K) * B])
        write_dump(args.dump_outputs, sums, rows, E[rows])
    v = K * B / dt
    sample = f"{K} steps of B={B} triples of the {WORKLOAD} workload (corruption ids precomputed)"
    print(json.dumps({
        "impl": "reference", "metric": "HolE train triples/s", "value": v, "unit": "triples/s",
        "n_gpus": args.gpus, "steps": K, "warmup": W, "ms_per_step": dt / K * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": workload_desc(B),
                   "batch": B, "note": "CPU port of holE.py arithmetic (TensorFlow 1.2 not installable)"},
        "cpu_baseline": {"value": v, "unit": "triples/s", "cores": R.threads(), "kind": "port",
                         "sample": sample},
        "e2e": {"value": v, "unit": "triples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def timed_train(eng, dev_tri, B, K, W, batch_count, first_step=0):
    """(triples/s, ms per step) of one hole_train_steps call of K steps after W warm-up steps."""
    import torch
    warm_up(eng, dev_tri, B, W, first_step, batch_count)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tri, lrs = dev_tri[W * B:(W + K) * B], lr_schedule(K, first_step + W, batch_count)
    ev0.record()
    eng.train_steps(tri, B, 1, first_step + W, MARGIN, lrs)
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    return K * B / (ms * 1e-3), ms / K


def warm_up(eng, dev_tri, B, W, first_step, batch_count):
    """The W untimed warm-up steps, issued as TWO calls (W - 2 and 2 steps).  One-time costs of a context do
    not all fall into its first call: the first call's update plan reports how many duplicated uses a step
    has, and the second call is the first to run the one-launch sort (tools/first_call_probe.py: ~140 us, once
    per context; every later call is at the steady state the timed call is meant to measure)."""
    if W <= 0:
        return
    a = W - 2 if W >= 3 else max(W - 1, 1)
    for k0, n in ((0, a), (a, W - a)):
        if n > 0:
            eng.train_steps(dev_tri[k0 * B:(k0 + n) * B], B, 1, first_step + k0, MARGIN,
                            lr_schedule(n, first_step + k0, batch_count))


def coverage_records(args, eng1, kg1, dev_tri1, peak):
    """The other shapes north_star names, measured beside the headline with the same timer (one
    hole_train_steps call of K steps, CUDA events): BASELINE configs[0] (FB15k shape, d=150 -- the 9.8 MB
    table is L2-resident, so its "fraction of the HBM roofline" is an algorithmic-bytes rate that can
    exceed 1), the script's default B=512 (launch-latency bound), and the trained-scale / Zipf-entity
    variants of configs[1] (clip backward and deep combine trees inside the timed region)."""
    import torch
    from graphembeddings_b200 import data as D
    from graphembeddings_b200.engine import HoleEngine
    K, W = args.steps, args.warmup
    out = {}

    def record(name, eng, kg, tri, B, note, long_call=0):
        v, ms = timed_train(eng, tri, B, K, W, max(16, kg.triples.shape[0] // B), first_step=1000)
        out[name] = {"workload": note, "batch": B, "value": v, "unit": "triples/s", "ms_per_step": ms, "steps": K,
                     "frac_of_hbm_roofline": v * (32 * kg.dim + 20) / 1e9 / peak}
        if long_call:
            # the same batch size in ONE call of long_call steps (what the training loop issues between two
            # validation points): the first chunk's update plan, which nothing can hide, is paid once per call
            n = min(long_call, tri.shape[0] // B - W)
            v2, ms2 = timed_train(eng, tri, B, n, W, max(16, kg.triples.shape[0] // B), first_step=3000)
            out[name].update({"long_call": {"steps": n, "value": v2, "ms_per_step": ms2}})

    # configs[1] at the drop-in default batch size (holE.py:602)
    record("diffbot_d256_B512", eng1, kg1, dev_tri1, 512,
           "configs[1] table, B=512 (holE.py's default batch size): launch-latency bound", long_call=10 * K)
    for tag, kw, note in (("trained_scale", dict(trained_scale=True), "row norms ~U(0.5,1.5): every clip-backward branch runs"),
                          ("zipf_entities", dict(zipf_entities=True), "Zipf(1) entities: hot rows with thousands of uses per step")):
        kg = D.make_config(WORKLOAD, n_triples=(K + W) * args.batch, **kw)
        off, ids = D.build_type_csr(kg.type_of)
        eng = HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E).set_types(kg.type_of, off, ids)
        eng.set_relation_count(kg.n_relations)
        record("diffbot_d256_" + tag, eng, kg, torch.from_numpy(kg.triples).cuda(), args.batch,
               f"configs[1] shape, B={args.batch}, {note}")
        if tag == "trained_scale":
            # SURVEY section 8f item 4: the archived FFT / tanh score variant (direct O(H^2) correlations on CUDA
            # cores: compute-bound, ~4 * 4 * H^2 FMAs per triple, not an HBM-roofline kernel)
            eng.set_score_mode("ccorr_tanh")
            v, ms = timed_train(eng, torch.from_numpy(kg.triples).cuda(), args.batch, min(K, 10), min(W, 3),
                                max(16, kg.triples.shape[0] // args.batch), first_step=2000)
            H = kg.dim // 2
            out["diffbot_d256_ccorr_tanh"] = {
                "workload": f"configs[1] shape, B={args.batch}, archived score variant tanh(sum r*ccorr(h,t)) "
                            "(holE-20170724/graph.pbtxt:6221-6521), margin as the headline",
                "batch": args.batch, "value": v, "unit": "triples/s", "ms_per_step": ms, "steps": min(K, 10),
                "fp32_tflops": v * (4 * 8 * H * H) / 1e12, "bound": "fp32 FMA (CUDA cores)"}
            eng.set_score_mode("complex")
        eng.close()
        del eng, kg
    for tag, kw in (("uniform", {}), ("zipf", dict(zipf_entities=True))):
        kg = D.make_config("fb15k_d150", n_triples=max((K + W) * args.batch, 483142), **kw)
        off, ids = D.build_type_csr(kg.type_of)
        eng = HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E).set_types(kg.type_of, off, ids)
        eng.set_relation_count(kg.n_relations)
        tri = torch.from_numpy(kg.triples).cuda()
        record(f"fb15k_d150_{tag}_B{args.batch}", eng, kg, tri, args.batch,
               f"BASELINE.json configs[0]: FB15k shape (16,296 x 150 table, L2-resident), {tag} entities, B={args.batch}")
        if tag == "uniform":
            record("fb15k_d150_uniform_B512", eng, kg, tri, 512,
                   "BASELINE.json configs[0]: FB15k shape, B=512 (holE.py's default batch size)", long_call=10 * K)
        eng.close()
    return out


def config4_single_gpu(args, peak):
    """BASELINE.json configs[4] (20 M entities x d=512 = 41 GB) on ONE GPU: the N=1 point of that config's
    scaling curve (the sharded runs report it at N > 1).  Table generated on the device."""
    import torch
    from graphembeddings_b200 import data as D
    from graphembeddings_b200.engine import HoleEngine
    cfg = D.CONFIGS["sharded_d512"]
    R, n_ent, dim, n_types = cfg["n_relations"], cfg["n_entities"], cfg["dim"], cfg["n_types"]
    B, K, W = args.batch, min(args.steps, 20), 3
    rng = np.random.default_rng(cfg["seed"])
    p = np.full(n_types, (1.0 - cfg["dominant_type_frac"]) / (n_types - 1))
    p[0] = cfg["dominant_type_frac"]
    type_of = np.concatenate([np.zeros(R, np.int32), 1 + rng.choice(n_types, size=n_ent, p=p).astype(np.int32)])
    off, ids = D.build_type_csr(type_of)
    eng = HoleEngine(R + n_ent, dim).set_types(type_of, off, ids)
    eng.set_relation_count(R)
    gen = torch.Generator(device=eng.device)
    gen.manual_seed(cfg["seed"] + 1)
    eng.table = torch.empty((R + n_ent, eng.row_stride), dtype=torch.float32, device=eng.device)
    eng.table.normal_(0.0, 1.0, generator=gen).clamp_(-2.0, 2.0).mul_(D.xavier_stddev(R + n_ent, dim))
    n = (K + W) * B
    h = torch.randint(R, R + n_ent, (n,), generator=gen, device=eng.device, dtype=torch.int32)
    t = torch.randint(R, R + n_ent, (n,), generator=gen, device=eng.device, dtype=torch.int32)
    w = 1.0 / torch.arange(1, R + 1, device=eng.device, dtype=torch.float64)
    r = torch.multinomial(w / w.sum(), n, replacement=True, generator=gen).to(torch.int32)
    tri = torch.stack([h, t, r], dim=1).contiguous()
    v, ms = timed_train(eng, tri, B, K, W, 500_000_000 // B)
    out = {"workload": f"sharded_d512: BASELINE.json configs[4], HolE d=512, {n_ent:,} entities + {R} relations "
                       "(41.0 GB fp32 table) on one GPU, uniform entities, Zipf relations",
           "value": v, "unit": "triples/s", "ms_per_step": ms, "batch": B, "steps": K,
           "frac_of_hbm_roofline": v * (32 * dim + 20) / 1e9 / peak}
    eng.close()
    del eng
    torch.cuda.empty_cache()
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist
    from graphembeddings_b200.engine import HoleEngine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}; launch with torch.distributed.run")
    torch.cuda.set_device(local_rank)
    if world > 1:
        if args.dump_outputs:
            raise SystemExit("--dump-outputs writes the single-GPU timed call's outputs; use --gpus 1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        from graphembeddings_b200 import sharded
        return sharded.bench(args, dist, rank, world, local_rank)

    B, K, W = args.batch, args.steps, args.warmup
    t_gen = time.time()
    kg, off, ids = make_workload((K + W) * B)
    eng = HoleEngine(kg.n_rows, kg.dim, local_rank).set_embeddings(kg.E).set_types(kg.type_of, off, ids)
    eng.set_relation_count(kg.n_relations)
    batch_count = 30_000_000 // B      # the named config has 30 M triples per epoch
    dev_tri = torch.from_numpy(kg.triples).cuda()
    host_tri = torch.from_numpy(kg.triples).pin_memory()
    t_gen = time.time() - t_gen

    def barrier():
        torch.cuda.synchronize()

    # ---- device-resident throughput ("value")
    # (nvidia-smi's start-up disturbs running GPU work for a few hundred ms: the clock sampler
    # starts before the warm-up, not inside the timed region)
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(1.0)
    settle_clocks()
    warm_up(eng, dev_tri, B, W, 0, batch_count)
    barrier()
    eng.reset_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    timed_tri, timed_lrs = dev_tri[W * B:(W + K) * B], lr_schedule(K, W, batch_count)   # (host prep: not part of a step)
    ev0.record()
    sums = eng.train_steps(timed_tri, B, 1, W, MARGIN, timed_lrs)
    ev1.record()
    barrier()
    launches = eng.launch_count()
    ms = ev0.elapsed_time(ev1)
    value = K * B / (ms * 1e-3)
    mean_loss = float(sums.mean().item()) / B
    if args.dump_outputs:
        # before the e2e and roofline passes below train the same table further
        rows = dump_rows(kg, kg.triples[(W + K - 1) * B:(W + K) * B])
        table_rows = eng.embeddings()[torch.from_numpy(rows).to(eng.device)].cpu().numpy()
        write_dump(args.dump_outputs, sums.cpu().numpy(), rows, table_rows)

    # ---- end to end from pinned host triples ("e2e")
    # (warm-up with a call of the timed call's shape: staging and pinned buffers are sized on first use)
    eng.train_steps_host(host_tri[W * B:(W + K) * B], B, 1, W + K, MARGIN, lr_schedule(K, W + K, batch_count))
    barrier()
    e2e_tri, e2e_lrs = host_tri[W * B:(W + K) * B], lr_schedule(K, 2 * W + K, batch_count)
    t0 = time.perf_counter()
    hs = eng.train_steps_host(e2e_tri, B, 1, 2 * W + K, MARGIN, e2e_lrs)
    e2e_s = time.perf_counter() - t0
    e2e = K * B / e2e_s
    assert np.isfinite(hs).all()

    # ---- roofline: CUDA events around the two hot kernels of every step (separate pass)
    eng.profile(True)
    eng.train_steps(dev_tri[W * B:(W + K) * B], B, 1, 3 * W + 2 * K, MARGIN, lr_schedule(K, W, batch_count))
    k1_ms, k3_ms, n_prof = eng.profile_read()
    eng.profile(False)
    clocks = sampler.stop()      # sampled across the value, e2e and roofline passes
    peak, peak_src, _ = peaks()
    alg_bytes = (32 * kg.dim + 20) * B
    kern_s = (k1_ms + k3_ms) * 1e-3 / max(n_prof, 1)
    achieved = alg_bytes / kern_s / 1e9

    # ---- CPU baseline on a bounded sample
    cpu_v, cores, cpu_steps, cpu_dt = cpu_port_throughput(kg, off, ids, B, args.cpu_seconds, 100000)

    out = {
        "metric": "HolE train triples/s", "value": value, "unit": "triples/s", "n_gpus": 1,
        "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {
            "workload": workload_desc(B),
            "batch": B, "margin": MARGIN, "lr0": LR0, "triples_generated": int(kg.triples.shape[0]),
            "epoch_triples": 30_000_000, "l2": "table (1.2 GB) larger than L2; no flush",
            "clock_settle": "0.25 s of device fills after the clock sampler's start-up pause, before the warm-up steps",
            "warmup_calls": "the W warm-up steps are two calls (W-2 and 2 steps): the second training call of a context "
                            "still carries one-time costs (tools/first_call_probe.py)",
            "mean_loss_last_pass": mean_loss, "gen_seconds": round(t_gen, 1)},
        "e2e": {"value": e2e, "unit": "triples/s", "h2d_bytes_per_step": 12 * B,
                "d2h_bytes_per_step": 4, "call": "hole_train_steps_host (pinned host triples in, loss sums out)"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": NCU_TRAFFIC.get((B, kg.dim)), "peak_source": peak_src,
                     "kernel": "hole_k1_kernel + hole_apply_kernel (one step)",
                     "k1_us": k1_ms * 1e3 / max(n_prof, 1), "k3_us": k3_ms * 1e3 / max(n_prof, 1),
                     "algorithmic_bytes_per_launch": alg_bytes,
                     "whole_step_frac": value * (32 * kg.dim + 20) / 1e9 / peak},
        "cpu_baseline": {"value": cpu_v, "unit": "triples/s", "cores": cores, "kind": "port",
                         "sample": f"{cpu_steps} steps of B={B} ({cpu_dt:.1f} s) of the same workload, "
                                   "oracle/hole_ref.c (C/OpenMP)"},
    }
    if not args.no_coverage:
        try:
            out["coverage"] = coverage_records(args, eng, kg, dev_tri, peak)
        except Exception as exc:      # reported beside the headline, never instead of it
            out["coverage"] = {"error": repr(exc)}
    ranking = None
    if not args.no_ranking:
        try:
            from graphembeddings_b200 import rank_bench
            ranking = rank_bench.run(eng, kg, quick=False)
        except Exception as exc:  # ranking is reported beside the headline, never instead of it
            ranking = {"error": repr(exc)}
    if ranking is not None:
        out["ranking"] = ranking
    if not args.no_config4:
        eng.close()
        del eng, dev_tri
        torch.cuda.empty_cache()
        try:
            out["config4"] = config4_single_gpu(args, peak)
        except Exception as exc:
            out["config4"] = {"error": repr(exc)}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=32768)
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--no-ranking", action="store_true")
    ap.add_argument("--no-config4", action="store_true", help="skip the 20M-entity d=512 sub-record")
    ap.add_argument("--no-coverage", action="store_true", help="N = 1: skip the configs[0] / B=512 / variant sub-records")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="N = 1: write the timed call's loss sums and a fixed sample of its final table rows as .npy")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
