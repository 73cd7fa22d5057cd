"""The --gpus N driver (hole.run_training_sharded) and its validation on the shards (sharded.score_on_shards).

Tolerances.  score_on_shards reads the rows it scores bit for bit (hole_gather_rows) and scores them with hole_score,
so sigma is bit-identical to hole_score on the gathered table; the corruption of a slice at index_base o_k is
hole_corrupt's over the whole file, exactly.  A sharded run and a one-GPU run of the driver differ only in how the
steps sum a row's gradients, so their tables differ within the one-step band of DESIGN 7c (2e-6 + 1e-5 |x| on a row,
1e-7 + 1e-5 |a| on the accumulator) times the number of steps, as in test_gpu_shard_adagrad.py's world-1 trainer test;
across ranks the owner's sum adds at most world - 1 fp32 adds, (world - 1) / 31 of a tree level (DESIGN 7c), which
widens the band by that factor.  valid_loss_mean is a mean of hinges of sigma, 1/4-Lipschitz in a score that moves by
at most 3 sqrt(dim) times the largest element difference of its three (clipped) rows, so two runs' means agree
within 1.5 sqrt(dim) times the table band.  The widened band of the torchrun CLI test (2, 4 and 8 GPUs) is derived, not
yet checked against runs on real peers."""
import os
import shutil
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from graphembeddings_b200 import data as D
from test_gpu_cli import _write_data_dir
from test_gpu_shard_adagrad import _VirtualRanks

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROW_ATOL, ROW_RTOL, ACC_ATOL, ACC_RTOL = 2e-6, 1e-5, 1e-7, 1e-5


@pytest.fixture(scope="module")
def eng_mod():
    from graphembeddings_b200 import build
    build.build()
    from graphembeddings_b200 import engine
    return engine


# ---------------------------------------------------------------- score_on_shards on virtual ranks
def _whole(eng_mod, vr):
    e = eng_mod.HoleEngine(vr.n_rows, vr.kg.dim).set_embeddings(vr.table())
    off, ids = D.build_type_csr(vr.kg.type_of)
    return e.set_types(vr.kg.type_of, off, ids)


def _check_validation_on_shards(eng_mod, vr, valid, seed, step):
    """Every virtual rank corrupts and scores its slice of `valid` as evaluate_batch_sharded does; the ranks' results
    in rank order are evaluate_batch's on the gathered table, bit for bit."""
    from graphembeddings_b200 import hole
    from graphembeddings_b200.sharded import score_on_shards
    dev = vr.engs[0].device
    whole = _whole(eng_mod, vr)
    v = torch.from_numpy(np.ascontiguousarray(valid)).to(dev)
    side_w, neg_w = whole.corrupt_batch(v, seed, step)
    loss_w, vp_w, vn_w = hole.evaluate_batch(whole, v, seed, step, 0.2)
    o = hole.valid_split(len(valid), vr.world)
    shards = [b[0] for b in vr.bufs]
    negs, vps, vns = [], [], []
    for k, e in enumerate(vr.engs):
        part = v[o[k]:o[k + 1]]
        side, neg = e.corrupt_batch(part, seed, step, o[k])
        assert side == side_w
        corrupt = part.clone()
        corrupt[:, 0 if side else 1] = neg
        s = score_on_shards(e, shards, k, vr.R, vr.rows_per, torch.cat([part, corrupt]))
        negs.append(neg)
        vps.append(s[:len(part)])
        vns.append(s[len(part):])
    assert torch.equal(torch.cat(negs), neg_w)
    vp, vn = torch.cat(vps), torch.cat(vns)
    assert torch.equal(vp, vp_w) and torch.equal(vn, vn_w)
    assert torch.equal(torch.clamp(vp - vn + 0.2, min=0.0), loss_w)
    whole.close()


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_score_on_shards_is_hole_score_on_the_gathered_table(eng_mod, world):
    """Rows owned by every rank, relation rows as heads and tails, a file shorter than the ranks (empty slices), and
    the table after a few sharded steps."""
    B = 64
    kg = D.synthetic_kg(7, 900, 3 * world * B + 500, 4, 150, seed=60 + world, trained_scale=True, zipf_entities=True)
    vr = _VirtualRanks(eng_mod, kg, world, B)
    valid = kg.triples[3 * world * B:].copy()
    valid[:7, 0] = np.arange(7)               # relation rows (replicated) as heads and tails
    valid[7:12, 1] = np.arange(5)
    owners = (valid[:, :2].astype(np.int64) - kg.n_relations) // vr.rows_per
    assert set(np.unique(owners[owners >= 0])) == set(range(world))
    _check_validation_on_shards(eng_mod, vr, valid, 11, 0)
    _check_validation_on_shards(eng_mod, vr, valid[:world - 1], 11, 1)         # every slice <= 1 row, one empty
    _check_validation_on_shards(eng_mod, vr, valid[:0], 11, 2)
    dev = vr.engs[0].device
    for s in range(3):
        gb = torch.from_numpy(kg.triples[s * world * B:(s + 1) * world * B]).to(dev)
        vr.step([gb[k * B:(k + 1) * B].contiguous() for k in range(world)], 5, s, 0.2, 0.3)
    assert np.abs(vr.table() - kg.E).max() > 1e-4
    _check_validation_on_shards(eng_mod, vr, valid, 11, 3)
    vr.close()


def test_score_on_shards_with_trailing_ranks_that_own_no_rows(eng_mod):
    """10 entities over 8 ranks: rows_per = 2, ranks 5-7 own nothing."""
    world, B = 8, 4
    kg = D.synthetic_kg(3, 10, 2 * world * B + 40, 3, 66, seed=8, trained_scale=True)
    vr = _VirtualRanks(eng_mod, kg, world, B)
    assert vr.rows_per == 2
    _check_validation_on_shards(eng_mod, vr, kg.triples[2 * world * B:], 4, 0)
    dev = vr.engs[0].device
    gb = torch.from_numpy(kg.triples[:world * B]).to(dev)
    vr.step([gb[k * B:(k + 1) * B].contiguous() for k in range(world)], 4, 0, 0.2, 0.3)
    _check_validation_on_shards(eng_mod, vr, kg.triples[2 * world * B:], 4, 1)
    vr.close()


def test_all_to_all_trainer_scores_bit_for_bit(eng_mod):
    """RowShardedTrainer.score (rows routed with _route / _a2a into the side table) is hole_score on the whole table:
    relation rows as heads and tails, an empty call, and the table after a few all-to-all steps."""
    from graphembeddings_b200.sharded import CudaBackend, RowShardedTrainer
    B = 64
    kg = D.synthetic_kg(7, 900, 3 * B + 500, 4, 150, seed=21, trained_scale=True, zipf_entities=True)
    off, ids = D.build_type_csr(kg.type_of)
    be = CudaBackend(kg.n_relations, kg.dim, B, 0, kg.type_of, off, ids)
    tr = RowShardedTrainer(kg.n_relations, kg.n_entities, kg.dim, be).load_embeddings(kg.E)
    t = kg.triples.copy()
    t[:7, 0] = np.arange(7)
    t[7:12, 1] = np.arange(5)
    tt = torch.from_numpy(t).to(be.device)
    for s in range(4):
        if s:
            tr.train_step(tt[(s - 1) * B:s * B], 3, s, 0.2, 0.3)
        whole = eng_mod.HoleEngine(kg.n_rows, kg.dim).set_embeddings(tr.gather_embeddings())
        assert torch.equal(tr.score(tt), whole.evaluate_triples(tt)), s
        whole.close()
    assert np.abs(tr.gather_embeddings().cpu().numpy() - kg.E).max() > 1e-4
    assert tr.score(tt[:0]).numel() == 0
    be.eng.close()


def test_world1_all_to_all_driver_matches_the_one_gpu_driver(eng_mod, tmp_path, monkeypatch):
    """HOLE_SHARDED_NCCL=1 (and a machine without peer memory): the driver on the all-to-all RowShardedTrainer, one
    train_step per step and validation through RowShardedTrainer.score, against the one-GPU driver with SGD."""
    from graphembeddings_b200 import hole, sharded
    calls = {"score": 0, "train_step": 0}
    for name in calls:
        orig = getattr(sharded.RowShardedTrainer, name)

        def counted(self, *a, _orig=orig, _name=name, **kw):
            calls[_name] += 1
            return _orig(self, *a, **kw)
        monkeypatch.setattr(sharded.RowShardedTrainer, name, counted)
    monkeypatch.setenv("HOLE_SHARDED_NCCL", "1")
    kg = D.synthetic_kg(8, 1500, 20000, 4, 64, seed=3, with_embeddings=False)
    d = tmp_path / "data"; d.mkdir()
    _write_data_dir(str(d), kg, 600, 400)
    one, shd = str(tmp_path / "one"), str(tmp_path / "shd")
    common = ["--data_dir", str(d), "--batch_size", "256", "--embedding_dim", "64", "--num_epochs", "1",
              "--learning_rate", "0.5"]
    hole.main(common + ["--output_dir", one])
    step = _sharded_world1(common + ["--output_dir", shd])
    assert step == (20000 - 1000) // 256 - 1
    assert calls["train_step"] == step and calls["score"] == 2 * len(_rows(shd)), calls
    assert _events(shd)[0] == 1
    _compare_runs(one, shd, step, 64, False)


# ---------------------------------------------------------------- the driver at world 1 against the one-GPU driver
def _rows(out):
    return [dict(kv.split("=") for kv in line.strip().split("\t")) for line in open(os.path.join(out, "summaries.tsv"))]


def _events(out):
    """(number of events files, the (step, tags) of every summary record over all of them, sorted).  The writer names
    its file by the second it was created and appends to it, so a run resumed in the same second as the run its
    directory was copied from writes into the copied file: compare the records, not the number of files."""
    from graphembeddings_b200 import tf_events
    ev = [f for f in os.listdir(out) if f.startswith("events.out.tfevents.")]
    recs = [e for f in ev for e in tf_events.read_events(os.path.join(out, f)) if e["file_version"] is None]
    return len(ev), sorted((e["step"], tuple(sorted(list(e["scalars"]) + list(e["histograms"])))) for e in recs)


def _tags(out):
    return {t for _, tags in _events(out)[1] for t in tags}


def _ckpt(out):
    from graphembeddings_b200 import hole, tf_bundle
    return tf_bundle.load_bundle(os.path.join(out, "model.ckpt")), hole


def _pockets(rows, tol):
    """The steps of the pocket saves, and whether any decision lay within tol of the running best."""
    best, steps, close = 2.0, [], False
    for r in rows:
        v = float(r["valid_loss_mean"])
        close |= abs(v - best) <= tol
        if v < best:
            best = v
            steps.append(int(r["step"]))
    return steps, close


def _compare_runs(a, b, steps, dim, adagrad, widen=1.0):
    """Run directories a and b of the same training: checkpoints, summaries.tsv and events."""
    (ca, hole), (cb, _) = _ckpt(a), _ckpt(b)
    ra, rb = _rows(a), _rows(b)
    assert [r["step"] for r in ra] == [r["step"] for r in rb]
    tol_vlm = 1.5 * np.sqrt(dim) * steps * widen * (ROW_ATOL + ROW_RTOL * 1.5)
    va, vb = (np.array([float(r["valid_loss_mean"]) for r in rs]) for rs in (ra, rb))
    assert np.abs(va - vb).max() <= tol_vlm, (np.abs(va - vb).max(), tol_vlm)
    assert _events(a)[1] == _events(b)[1]
    pa, close_a = _pockets(ra, 2 * tol_vlm)
    pb, close_b = _pockets(rb, 2 * tol_vlm)
    if not (close_a or close_b):
        assert pa == pb
        assert int(ca["batch/Variable"]) == int(cb["batch/Variable"])
    if int(ca["batch/Variable"]) == int(cb["batch/Variable"]):
        Ea, Eb = ca["embeddings"], cb["embeddings"]
        assert np.all(np.abs(Ea - Eb) <= steps * widen * (ROW_ATOL + ROW_RTOL * np.abs(Ea))), np.abs(Ea - Eb).max()
        assert (hole.ADAGRAD_SLOT in ca) == (hole.ADAGRAD_SLOT in cb) == adagrad
        if adagrad:
            Aa, Ab = ca[hole.ADAGRAD_SLOT], cb[hole.ADAGRAD_SLOT]
            assert np.all(np.abs(Aa - Ab) <= steps * widen * (ACC_ATOL + ACC_RTOL * np.abs(Aa)))
    return ca, cb


def _sharded_world1(args):
    from graphembeddings_b200 import hole
    flags = hole.build_parser().parse_args(args)
    return hole.run_training_sharded(hole.init_data(flags), flags, None, 0, 1, 0, seed=flags.seed,
                                     max_steps=flags.max_steps, log=lambda *a: None)


@pytest.mark.parametrize("optimizer", ["sgd", "adagrad"])
def test_world1_driver_matches_the_one_gpu_driver(eng_mod, tmp_path, optimizer):
    from graphembeddings_b200 import hole, tf_bundle
    kg = D.synthetic_kg(8, 1500, 20000, 4, 64, seed=3, with_embeddings=False)
    d = tmp_path / "data"; d.mkdir()
    _write_data_dir(str(d), kg, 600, 400)
    one, shd = str(tmp_path / "one"), str(tmp_path / "shd")
    common = ["--data_dir", str(d), "--batch_size", "256", "--embedding_dim", "64", "--num_epochs", "2",
              "--optimizer", optimizer, "--learning_rate", "0.5" if optimizer == "sgd" else "0.1"]
    hole.main(common + ["--output_dir", one])
    step = _sharded_world1(common + ["--output_dir", shd])
    batch_count = (20000 - 1000) // 256
    assert step == 2 * (batch_count - 1)
    for name in ("model.ckpt.index", "checkpoint", "projector_config.pbtxt", "summaries.tsv"):
        assert os.path.exists(os.path.join(shd, name)), name
    assert _events(shd)[0] == 1 and "batch/eval/summaries/max" in _tags(shd)
    _compare_runs(one, shd, step, 64, optimizer == "adagrad")
    # refuses to clobber an existing output_dir, as the one-GPU driver does
    with pytest.raises(Exception, match="already exists"):
        _sharded_world1(common + ["--output_dir", shd])
    # resume either run's checkpoint on the other path: the same continued training
    for src, tag in ((one, "one_to"), (shd, "shd_to")):
        a, b = str(tmp_path / f"{tag}_one"), str(tmp_path / f"{tag}_shd")
        shutil.copytree(src, a)
        shutil.copytree(src, b)
        step0 = int(tf_bundle.load_bundle(os.path.join(src, "model.ckpt"))["batch/Variable"])
        more = common + ["--resume_checkpoint", "--max_steps", "9"]
        hole.main(more + ["--output_dir", a])
        _sharded_world1(more + ["--output_dir", b])
        ca, cb = _compare_runs(a, b, step + 9, 64, optimizer == "adagrad")
        assert int(cb["batch/Variable"]) > step0
    # --infer reads the sharded run's checkpoint unchanged
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        m = hole.infer_triples(hole.build_parser().parse_args(common + ["--output_dir", shd, "--infer"]),
                               log=lambda *a: None)
    finally:
        os.chdir(cwd)
    assert 0 < m["filtered_mrr"] <= 1


def test_world1_driver_refuses_a_checkpoint_without_the_adagrad_slot(eng_mod, tmp_path):
    from graphembeddings_b200 import hole
    kg = D.synthetic_kg(8, 600, 6000, 4, 64, seed=4, with_embeddings=False)
    d = tmp_path / "data"; d.mkdir()
    _write_data_dir(str(d), kg, 300, 200)
    out = str(tmp_path / "run")
    common = ["--data_dir", str(d), "--output_dir", out, "--batch_size", "128", "--embedding_dim", "64"]
    _sharded_world1(common + ["--num_epochs", "1"])
    with pytest.raises(SystemExit, match="no embeddings/Adagrad slot"):
        _sharded_world1(common + ["--resume_checkpoint", "--optimizer", "adagrad", "--max_steps", "3"])


# ---------------------------------------------------------------- several GPUs: torchrun the CLI
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _torchrun(world, args):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()), "-m", "graphembeddings_b200.hole"]
    r = subprocess.run(cmd + args + ["--gpus", str(world)], cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, (r.stdout + r.stderr)[-3000:]
    return r.stdout


@pytest.mark.parametrize("world", [2, 4, 8])
def test_torchrun_cli_matches_the_one_gpu_cli(tmp_path, world):
    if not torch.cuda.is_available() or torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    from graphembeddings_b200 import build, hole
    build.build()
    kg = D.synthetic_kg(8, 3000, 40000, 4, 64, seed=5, with_embeddings=False)
    d = tmp_path / "data"; d.mkdir()
    _write_data_dir(str(d), kg, 1000, 400)
    widen = 1.0 + (world - 1) / 31
    for optimizer in ("sgd", "adagrad"):
        one, many = str(tmp_path / f"one_{optimizer}"), str(tmp_path / f"many_{optimizer}")
        common = ["--data_dir", str(d), "--batch_size", "512", "--embedding_dim", "64", "--num_epochs", "2",
                  "--optimizer", optimizer]
        hole.main(common + ["--output_dir", one])
        out = _torchrun(world, common + ["--output_dir", many])
        assert "triples/s" in out
        assert _events(many)[0] == 1              # rank 0 alone writes the events
        steps = 2 * ((40000 - 1400) // 512 - 1)
        _compare_runs(one, many, steps, 64, optimizer == "adagrad", widen)
        # resumed: 9 more steps from the one-GPU checkpoint on both paths
        a, b = one + "_r", many + "_r"
        shutil.copytree(one, a)
        shutil.copytree(one, b)
        more = common + ["--resume_checkpoint", "--max_steps", "9"]
        hole.main(more + ["--output_dir", a])
        _torchrun(world, more + ["--output_dir", b])
        _compare_runs(a, b, steps + 9, 64, optimizer == "adagrad", widen)
