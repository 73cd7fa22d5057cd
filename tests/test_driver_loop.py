"""hole.py's training loop on the CPU.  run_training, and run_training_sharded at world 1 on both row-sharded trainers,
run with fakes in place of every call that touches a device, so that the loop itself is under test: the schedule of
steps, learning rates, triples, validation points, corruptions, pocket checkpoints and outputs.  The fake engine and
the fake trainers share one toy model (a score and an update of a CPU table), so both drivers compute the same
numbers, and the one-GPU records are checked against the holE.py schedule restated here."""
import math
import os

import numpy as np
import pytest
import torch

from graphembeddings_b200 import hole, sharded, tf_events
from graphembeddings_b200.engine import inverse_time_decay

R, N, DIM, B = 4, 40, 8, 8
BATCH_COUNT = 50                  # valid_every = 3: stretches of 2, 3, ..., 3 and 2 steps an epoch
_write_checkpoint = hole.write_checkpoint


# ---------------------------------------------------------------- the toy model and its fakes
def _toy_score(table, t):
    """Row by row in Python: a vectorised CPU sigmoid rounds a batch's tail differently from its body."""
    x = (20.0 * ((table[t[:, 0].long()] + table[t[:, 2].long()]) * table[t[:, 1].long()]).double().sum(1)).tolist()
    return torch.tensor([1.0 / (1.0 + math.exp(-v)) for v in x], dtype=torch.float32)


def _toy_train(table, triples, batch_size, first_step, lrs):
    t = torch.as_tensor(triples).long()
    for k, lr in enumerate(lrs):
        s = t[k * batch_size:(k + 1) * batch_size]
        table.index_add_(0, s[:, 0], (0.5 if (first_step + k) % 3 else -1.0) * float(lr) * table[s[:, 1]])


def _toy_corrupt(t, seed, step, index_base):
    t = torch.as_tensor(t).long()
    i = torch.arange(t.shape[0]) + index_base
    return int(step % 2), (R + (7 * t[:, 0] + 3 * t[:, 1] + 5 * i + seed + 11 * step) % (N - R)).to(torch.int32)


def _new_record():
    return {"init": [], "train": [], "corrupt": [], "ckpt": [], "logloss": [], "score_mode": None, "closed": []}


class _FakeEngine:
    """HoleEngine's surface that the drivers use, on a CPU table."""

    def __init__(self, rec, E=None):
        self.rec, self.device, self.accum = rec, torch.device("cpu"), None
        self.table = None if E is None else torch.as_tensor(E, dtype=torch.float32).clone()
        if E is not None:
            rec["init"].append(self.table.clone())

    def set_score_mode(self, mode):
        self.rec["score_mode"] = mode
        return self

    def corrupt_batch(self, t, seed, step, index_base=0):
        self.rec["corrupt"].append((int(step), int(index_base), torch.as_tensor(t).tolist()))
        return _toy_corrupt(t, seed, step, index_base)

    def evaluate_triples(self, t):
        return _toy_score(self.table, t)

    def train_steps(self, triples, batch_size, seed, first_step, margin, lrs):
        n = triples.shape[0] // batch_size
        self.rec["train"].append((int(first_step), n, [float(x) for x in lrs], triples.tolist()))
        _toy_train(self.table, triples, batch_size, first_step, lrs)
        return torch.zeros(n)

    def train_step_logloss(self, triples, seed, step, lr, l2, negative_ratio):
        self.rec["train"].append((int(step), 1, [float(lr)], triples.tolist()))
        self.rec["logloss"].append((seed, l2, negative_ratio))
        _toy_train(self.table, triples, triples.shape[0], step, [lr])
        return torch.zeros((1 + negative_ratio, triples.shape[0])), torch.zeros(())

    def embeddings(self):
        return self.table.clone()

    def close(self):
        self.rec["closed"].append("engine")


class _FakeBackend:
    def __init__(self, rec):
        self.eng, self.device = _FakeEngine(rec), torch.device("cpu")


class _FakeTrainer:
    """The row-sharded trainers' device methods on the toy model (placed before the real class in the bases)."""

    def load_embeddings(self, E):
        self.table = torch.as_tensor(E, dtype=torch.float32).clone()
        self.rec["init"].append(self.table.clone())
        return self

    def gather_embeddings(self):
        return self.table.clone()

    def score(self, triples):
        return _toy_score(self.table, triples)

    def check_barriers(self):
        pass

    def close(self):
        self.rec["closed"].append(type(self).__name__)


class _FakeAllToAll(_FakeTrainer, sharded.RowShardedTrainer):
    def train_step(self, pos_local, seed, step, margin, lr, next_pos=None):
        self.rec["train"].append((int(step), 1, [float(lr)], pos_local.tolist()))
        _toy_train(self.table, pos_local, pos_local.shape[0], step, [lr])
        return torch.zeros(pos_local.shape[0])


class _FakeP2P(_FakeTrainer, sharded.P2PRowShardedTrainer):
    def __init__(self, *a):
        sharded.RowShardedTrainer.__init__(self, *a)        # no peer buffers

    def train_steps(self, triples_i32, batch_size, seed, first_step, margin, lrs):
        return _FakeEngine.train_steps(self, triples_i32, batch_size, seed, first_step, margin, lrs)


@pytest.fixture(autouse=True)
def _no_device(monkeypatch):
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **kw: None)
    monkeypatch.delenv("HOLE_SHARDED_NCCL", raising=False)


# ---------------------------------------------------------------- runs
def _data(n_valid):
    rng = np.random.default_rng(5)

    def triples(n):
        return np.stack([rng.integers(R, N, n), rng.integers(R, N, n), rng.integers(0, R, n)], 1).astype(np.int32)
    d = hole.HolEData()
    d.entity_count, d.relation_count = N, R
    d.id_to_type = {i: 0 if i < R else 1 + i % 3 for i in range(N)}
    d.triples = triples(BATCH_COUNT * B + 3)
    d.triple_count = d.triples.shape[0]
    d.validation_triples = triples(n_valid)
    return d


def _flags(out, args):
    return hole.build_parser().parse_args(["--data_dir", "-", "--output_dir", out, "--batch_size", str(B),
                                           "--embedding_dim", str(DIM), "--num_epochs", "2", "--seed", "3",
                                           "--learning_rate", "0.5", "--learning_decay_steps", "0.5"] + args)


def _record_checkpoints(monkeypatch, rec):
    def recorded(output_dir, E, global_step, A=None):
        rec["ckpt"].append(int(global_step))
        _write_checkpoint(output_dir, E, global_step, A)
    monkeypatch.setattr(hole, "write_checkpoint", recorded)


def _run_one_gpu(monkeypatch, out, data, args):
    rec, log = _new_record(), []
    monkeypatch.setattr(hole, "make_engine", lambda n, r, dim, E, id_to_type=None, device=0: _FakeEngine(rec, E))
    _record_checkpoints(monkeypatch, rec)
    flags = _flags(out, args)
    eng, step = hole.run_training(data, flags, seed=flags.seed, max_steps=flags.max_steps,
                                  log=lambda *a: log.append(" ".join(str(x) for x in a)))
    assert isinstance(eng, _FakeEngine)
    return rec, log, step, flags


def _run_sharded(monkeypatch, out, data, args, trainer):
    rec, log = _new_record(), []
    monkeypatch.setattr(sharded, "CudaBackend", lambda *a: _FakeBackend(rec))

    def make_trainer(n_relations, n_entities, dim, backend, dist, log=None):
        tr = trainer(n_relations, n_entities, dim, backend, dist)
        tr.rec = rec
        return tr
    monkeypatch.setattr(sharded, "make_trainer", make_trainer)
    _record_checkpoints(monkeypatch, rec)
    flags = _flags(out, args)
    step = hole.run_training_sharded(data, flags, None, 0, 1, 0, seed=flags.seed, max_steps=flags.max_steps,
                                     log=lambda *a: log.append(" ".join(str(x) for x in a)))
    return rec, log, step


def _resume_from(out, step):
    """A checkpoint at `step` in `out`, as a run that stopped there leaves it; returns its table."""
    E = np.random.default_rng(9).standard_normal((N, DIM)).astype(np.float32) * 0.3
    os.makedirs(out)
    hole.write_checkpoint(out, torch.from_numpy(E), step)
    return E


# ---------------------------------------------------------------- the schedule, restated
def _expected(data, flags, first_step):
    """holE.py's loop: every step's (global step, lr, triples), every validation point's (global step, lr, validation
    triples, next training batch), and the first step of every stretch between validation points."""
    bc = data.triple_count // flags.batch_size
    ve = max(1, bc // 16)
    decay_steps = flags.learning_decay_steps * bc
    gen = torch.Generator().manual_seed(flags.seed)
    vrng = np.random.default_rng(flags.seed + 1)
    valid = data.validation_triples
    steps, points, starts = [], [], []
    g = first_step
    for _ in range(flags.num_epochs):
        perm = torch.randperm(data.triple_count, generator=gen).numpy()
        for batch in range(1, bc):
            if flags.max_steps is not None and g - first_step >= flags.max_steps:
                return steps, points, starts
            lr = float(inverse_time_decay(flags.learning_rate, g, decay_steps, flags.learning_decay_rate))
            tb = data.triples[perm[(batch - 1) * flags.batch_size:batch * flags.batch_size]].tolist()
            if batch % ve == 0 and len(valid):
                vb = valid[vrng.integers(0, len(valid), size=flags.batch_size)] if flags.valid_sample else valid
                points.append((g, lr, vb.tolist(), tb))
            if batch == 1 or batch % ve == 0:
                starts.append(g)
            steps.append((g, lr, tb))
            g += 1
    return steps, points, starts


def _per_step(train):
    return [(first + k, lrs[k], t[k * B:(k + 1) * B]) for first, n, lrs, t in train for k in range(n)]


def _rows(out):
    with open(os.path.join(out, "summaries.tsv")) as f:
        return [dict(kv.split("=") for kv in line.rstrip("\n").split("\t")) for line in f]


def _check_one_gpu_run(rec, log, step, flags, data, out, first_step=0, resumed=False):
    steps, points, starts = _expected(data, flags, first_step)
    assert step == first_step + len(steps)
    assert _per_step(rec["train"]) == steps
    if not flags.log_loss:            # one multi-step call per stretch
        assert [c[0] for c in rec["train"]] == starts
    rows = _rows(out)
    assert [(int(r["step"]), float(r["learning_rate"])) for r in rows] == [p[:2] for p in points]
    if flags.log_loss:
        k = flags.negative_ratio
        want = [(g * k + j, 0, vb) for g, _, vb, _ in points for j in range(k)]
        assert all("pos_mean" not in r for r in rows)
    else:
        want = [c for g, _, vb, tb in points for c in ((g, 0, vb), (g, 0, tb))]
        assert all("pos_mean" in r and "neg_mean" in r for r in rows)
    assert rec["corrupt"] == want
    best, saves = 2.0, []
    for r in rows:                    # pocket: holE.py:357-360
        if float(r["valid_loss_mean"]) < best:
            best = float(r["valid_loss_mean"])
            saves.append(int(r["step"]))
    if not saves and not resumed:     # never validated: the final save
        saves = [step]
    assert rec["ckpt"] == saves
    if saves:
        assert hole.load_checkpoint(out)[1] == saves[-1]
    lines = [m for m in log if m.startswith(("Training epoch", "Done training", "Trained"))]
    assert lines[-2] == ("Done training -- step limit reached" if flags.max_steps is not None
                         else "Done training -- epoch limit reached")
    assert lines[-1].startswith(f"Trained {len(steps)} steps in ")
    assert "Training epoch 1..." in lines
    return rows


CASES = {
    "sgd": ([], 30, None),
    "max_steps": (["--max_steps", "7"], 30, None),
    "resume": (["--resume_checkpoint", "--max_steps", "10"], 30, 37),
    "valid_sample": (["--valid_sample"], 30, None),
    "empty_valid": ([], 0, None),
}


# ---------------------------------------------------------------- tests
@pytest.mark.parametrize("case", list(CASES))
def test_one_gpu_loop_follows_the_holE_schedule(monkeypatch, tmp_path, case):
    args, n_valid, resume_step = CASES[case]
    data, out = _data(n_valid), str(tmp_path / "run")
    E0 = _resume_from(out, resume_step) if resume_step is not None else None
    rec, log, step, flags = _run_one_gpu(monkeypatch, out, data, args)
    rows = _check_one_gpu_run(rec, log, step, flags, data, out, resume_step or 0, resume_step is not None)
    if E0 is not None:
        assert torch.equal(rec["init"][0], torch.from_numpy(E0))      # trained on from the checkpoint's table
    if case == "sgd":
        assert step == 2 * (BATCH_COUNT - 1) and "Training epoch 2..." in log
        assert len(rec["ckpt"]) > 2                          # the pocket saved more than once
    if case == "max_steps":
        assert [c[1] for c in rec["train"]] == [2, 3, 2]     # the last stretch cut short
    if case == "empty_valid":
        assert rows == [] and rec["corrupt"] == [] and rec["ckpt"] == [step]


def test_one_gpu_log_loss_and_ccorr_tanh(monkeypatch, tmp_path):
    data = _data(30)
    out = str(tmp_path / "log_loss")
    rec, log, step, flags = _run_one_gpu(monkeypatch, out, data, ["--log_loss", "--negative_ratio", "2",
                                                                  "--l2_regularization", "0.01", "--max_steps", "20"])
    _check_one_gpu_run(rec, log, step, flags, data, out)
    assert rec["logloss"] == [(3, 0.01, 2)] * 20 and rec["score_mode"] is None
    out = str(tmp_path / "ccorr")
    rec, log, step, flags = _run_one_gpu(monkeypatch, out, data, ["--score_variant", "ccorr_tanh", "--max_steps", "20"])
    _check_one_gpu_run(rec, log, step, flags, data, out)
    assert rec["score_mode"] == "ccorr_tanh"


def test_ccorr_tanh_with_log_loss_is_refused_before_any_output(monkeypatch, tmp_path):
    def touched(*a, **kw):
        raise AssertionError("made the engine before refusing")
    monkeypatch.setattr(hole, "make_engine", touched)
    out = str(tmp_path / "run")
    with pytest.raises(SystemExit, match="ccorr_tanh has no --log_loss branch"):
        hole.run_training(_data(30), _flags(out, ["--score_variant", "ccorr_tanh", "--log_loss"]))
    assert not os.path.exists(out)


def _events(out):
    recs = []
    for f in sorted(os.listdir(out)):
        if f.startswith("events.out.tfevents."):
            recs += [(e["step"], e["file_version"], e["scalars"],
                      {t: {k: np.asarray(v).tolist() for k, v in h.items()} for t, h in e["histograms"].items()})
                     for e in tf_events.read_events(os.path.join(out, f))]          # all but wall_time
    return recs


def _checkpoint_files(out):
    names = sorted(f for f in os.listdir(out) if f.startswith("model.ckpt"))
    return {f: open(os.path.join(out, f), "rb").read() for f in names}


@pytest.mark.parametrize("trainer", [_FakeAllToAll, _FakeP2P], ids=["all_to_all", "p2p"])
@pytest.mark.parametrize("case", list(CASES))
def test_world1_sharded_loop_is_the_one_gpu_loop(monkeypatch, tmp_path, case, trainer):
    args, n_valid, resume_step = CASES[case]
    data = _data(n_valid)
    one, shd = str(tmp_path / "one"), str(tmp_path / "shd")
    if resume_step is not None:
        _resume_from(one, resume_step)
        _resume_from(shd, resume_step)
    rec1, log1, step1, _ = _run_one_gpu(monkeypatch, one, data, args)
    rec, log, step = _run_sharded(monkeypatch, shd, data, args, trainer)
    assert step == step1
    if trainer is _FakeP2P:           # the same multi-step calls
        assert rec["train"] == rec1["train"]
    else:                             # one train_step per step
        assert _per_step(rec["train"]) == _per_step(rec1["train"]) and {c[1] for c in rec["train"]} == {1}
    for key in ("corrupt", "ckpt"):
        assert rec[key] == rec1[key], key
    assert len(rec["init"]) == 1 and torch.equal(rec["init"][0], rec1["init"][0])
    with open(os.path.join(one, "summaries.tsv")) as a, open(os.path.join(shd, "summaries.tsv")) as b:
        assert a.read() == b.read()
    assert _events(shd) == _events(one)
    assert _checkpoint_files(shd) == _checkpoint_files(one)
    assert log[1:-1] == log1[1:-1]    # all but the header and the closing "Trained ..." line
    assert rec["closed"][-1] == "engine"
    if trainer is _FakeP2P:
        assert rec["closed"] == [trainer.__name__, "engine"]


def test_sharded_refuses_an_existing_output_dir_before_making_the_trainer(monkeypatch, tmp_path):
    out = str(tmp_path / "run")
    os.makedirs(out)

    def touched(*a, **kw):
        raise AssertionError("made the trainer before refusing")
    monkeypatch.setattr(sharded, "CudaBackend", touched)
    with pytest.raises(Exception, match="already exists"):
        hole.run_training_sharded(_data(30), _flags(out, []), None, 0, 1, 0)
    monkeypatch.setattr(hole, "make_engine", touched)
    with pytest.raises(Exception, match="already exists"):
        hole.run_training(_data(30), _flags(out, []))
