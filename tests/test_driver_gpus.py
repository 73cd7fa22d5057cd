"""The --gpus N driver's host logic: its refusals come before any CUDA work, the ranks' shares of every global batch
make up the one-GPU batch in order, and the validation split covers the file exactly."""
import numpy as np
import pytest
import torch

from graphembeddings_b200 import hole

BASE = ["--data_dir", "/nonexistent/data", "--output_dir", "/nonexistent/out", "--batch_size", "512"]


@pytest.fixture
def no_cuda(monkeypatch):
    """Any step past the refusals fails the test: CUDA, the process group and the data loader."""
    def touched(*a, **kw):
        raise AssertionError("reached CUDA / process-group / data work before refusing")
    monkeypatch.setattr(torch.cuda, "set_device", touched)
    monkeypatch.setattr(torch.distributed, "init_process_group", touched)
    monkeypatch.setattr(hole, "init_data", touched)
    monkeypatch.setattr(hole, "infer_triples", touched)
    monkeypatch.setattr(hole, "run_training", touched)
    monkeypatch.delenv("HOLE_SHARDED_NCCL", raising=False)


@pytest.mark.parametrize("world,extra,match", [
    (4, ["--gpus", "4", "--batch_size", "510"], r"multiple of --gpus 4: use --batch_size 508 or 512"),
    (2, ["--gpus", "2", "--log_loss"], r"--log_loss has no row-sharded step.*--gpus 1"),
    (2, ["--gpus", "2", "--score_variant", "ccorr_tanh"], r"ccorr_tanh has no row-sharded step.*--gpus 1"),
    (8, ["--gpus", "8", "--infer"], r"--infer runs on one GPU.*--gpus 1"),
    (1, ["--gpus", "2"], r"--gpus 2 but WORLD_SIZE=1.*torch.distributed.run --nproc-per-node 2"),
    (4, ["--gpus", "2"], r"--gpus 2 but WORLD_SIZE=4"),
    (2, [], r"--gpus 1 but WORLD_SIZE=2"),
    (2, ["--gpus", "0"], r"--gpus must be >= 1"),
])
def test_refusals_come_before_any_cuda_work(no_cuda, monkeypatch, world, extra, match):
    monkeypatch.setenv("WORLD_SIZE", str(world))
    with pytest.raises(SystemExit, match=match):
        hole.main(BASE + extra)


def test_adagrad_without_peer_memory_is_refused_before_any_cuda_work(no_cuda, monkeypatch):
    for k, v in (("WORLD_SIZE", "2"), ("RANK", "0"), ("LOCAL_RANK", "0"), ("HOLE_SHARDED_NCCL", "1")):
        monkeypatch.setenv(k, v)
    with pytest.raises(SystemExit, match=r"adagrad on several GPUs needs the NVLink peer-memory trainer.*HOLE_SHARDED_NCCL"):
        hole.main(BASE + ["--gpus", "2", "--optimizer", "adagrad"])
    monkeypatch.delenv("HOLE_SHARDED_NCCL")
    with pytest.raises(AssertionError, match="before refusing"):     # accepted: goes on to the launch
        hole.main(BASE + ["--gpus", "2", "--optimizer", "adagrad"])


def test_one_gpu_keeps_the_single_gpu_path(no_cuda, monkeypatch):
    """--gpus 1 without torch.distributed.run is today's driver: no check of its own, no process group."""
    monkeypatch.delenv("WORLD_SIZE", raising=False)
    seen = []
    monkeypatch.setattr(hole, "init_data", lambda flags: seen.append("data") or "D")
    monkeypatch.setattr(hole, "run_training", lambda data, flags, **kw: seen.append(("train", data)))
    hole.main(BASE + ["--log_loss", "--batch_size", "511"])
    assert seen == ["data", ("train", "D")]


@pytest.mark.parametrize("trial", range(20))
def test_ranks_shares_concatenate_to_the_one_gpu_batches(trial):
    rng = np.random.default_rng(trial)
    world = int(rng.choice([1, 2, 3, 4, 8]))
    B = world * int(rng.integers(1, 40))
    T = int(rng.integers(0, 12 * B))
    perm = torch.randperm(T, generator=torch.Generator().manual_seed(trial))
    shares = [hole.rank_rows(perm, B, world, k) for k in range(world)]
    n, b = T // B, B // world
    assert all(s.shape == (n * b,) for s in shares)
    for step in range(n):
        got = torch.cat([s[step * b:(step + 1) * b] for s in shares])
        assert torch.equal(got, perm[step * B:(step + 1) * B])
    # a chunk of steps of one rank is contiguous in its share, as the multi-step call takes it
    if n >= 2:
        k = int(rng.integers(0, world))
        assert torch.equal(shares[k][b:2 * b], perm[B + k * b:B + (k + 1) * b])


@pytest.mark.parametrize("trial", range(20))
def test_validation_split_covers_the_file_exactly(trial):
    rng = np.random.default_rng(100 + trial)
    world = int(rng.integers(1, 17))
    V = int(rng.integers(0, 3 * world + 50))
    o = hole.valid_split(V, world)
    assert len(o) == world + 1 and o[0] == 0 and o[-1] == V
    assert all(a <= b for a, b in zip(o, o[1:]))
    covered = np.concatenate([np.arange(o[k], o[k + 1]) for k in range(world)])
    assert np.array_equal(covered, np.arange(V))          # index_base o_k: each row keeps its whole-file index
    assert max(b - a for a, b in zip(o, o[1:])) - min(b - a for a, b in zip(o, o[1:])) <= 1


def test_training_batch_split_is_the_rank_layout():
    """The next training batch's split (index_base = rank * B / world) is the validation split of B rows."""
    for world in (1, 2, 3, 8):
        B = 24 * world
        assert hole.valid_split(B, world) == [k * (B // world) for k in range(world + 1)]
