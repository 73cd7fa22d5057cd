"""The AdaGrad step (tests/adagrad_reference.py, what the library computes with hole_ctx_set_optimizer) against
torch.optim.Adagrad, on a hand-worked case and in fp32 against fp64; the checkpoint slot round trip; and the
command-line refusals.  No GPU needed."""
import os

import numpy as np
import pytest
import torch

import adagrad_reference as R
from graphembeddings_b200 import data as D
from graphembeddings_b200 import hole, tf_bundle
from oracle import hole_oracle as O


def _problem(seed, zipf, B=256, dim=20):
    kg = D.synthetic_kg(5, 300, 2048, 4, dim, seed=seed, trained_scale=True, zipf_entities=zipf)
    off, ids = D.build_type_csr(kg.type_of)
    pos = kg.triples[:B]
    side, neg = O.corrupt(pos, kg.type_of, off, ids, seed + 11, 3)
    return kg, pos, neg, side


@pytest.mark.parametrize("seed,zipf", [(0, False), (1, True), (2, True), (3, False)])
def test_fp64_step_matches_torch_adagrad_on_the_sparse_gradient_with_duplicates(seed, zipf):
    kg, pos, neg, side = _problem(seed, zipf)
    E = kg.E.astype(np.float64)
    init, lr, margin = 0.1, 0.3, 0.2
    A = np.full_like(E, init)
    # the six IndexedSlices, concatenated uncoalesced: torch coalesces (sums) the duplicates as TF dedups them
    slices, _, _, _ = O.indexed_slices(E, pos, neg, side, margin, np.float64)
    idx = np.concatenate([s[0] for s in slices]).astype(np.int64)
    val = np.concatenate([s[1] for s in slices], axis=0)
    assert len(np.unique(idx)) < len(idx)                      # duplicates are present
    p = torch.nn.Parameter(torch.from_numpy(E.copy()))
    opt = torch.optim.Adagrad([p], lr=lr, initial_accumulator_value=init, eps=0.0)
    p.grad = torch.sparse_coo_tensor(torch.from_numpy(idx)[None], torch.from_numpy(val), E.shape,
                                     check_invariants=True)
    opt.step()
    E1, A1 = E.copy(), A.copy()
    R.adagrad_step(E1, A1, pos, neg, side, margin, lr, np.float64)
    np.testing.assert_allclose(E1, p.detach().numpy(), rtol=0, atol=1e-13)
    np.testing.assert_allclose(A1, opt.state[p]["sum"].numpy(), rtol=1e-14, atol=0)
    untouched = np.setdiff1d(np.arange(len(E)), idx)
    assert np.array_equal(E1[untouched], E[untouched]) and np.all(A1[untouched] == init)


def test_hand_worked_two_rows():
    """Row 0 is used twice (gradients [1, 2] and [3, -1], summed to [4, 1]), row 1 once; row 2 is untouched."""
    E = np.array([[1.0, -1.0], [0.5, 0.25], [7.0, 7.0]])
    A = np.full_like(E, 0.1)
    idx = np.array([0, 1, 0])
    g = np.array([[1.0, 2.0], [0.5, 0.0], [3.0, -1.0]])
    acc = np.zeros_like(E)
    np.add.at(acc, idx, g)
    rows = np.unique(idx)
    R.adagrad_apply(E, A, rows, acc[rows], lr=0.5)
    np.testing.assert_allclose(A, [[16.1, 1.1], [0.35, 0.1], [0.1, 0.1]], rtol=1e-15)
    np.testing.assert_allclose(E, [[1.0 - 0.5 * 4 / np.sqrt(16.1), -1.0 - 0.5 * 1 / np.sqrt(1.1)],
                                   [0.5 - 0.5 * 0.5 / np.sqrt(0.35), 0.25],      # g = 0: unchanged
                                   [7.0, 7.0]], rtol=1e-15)


@pytest.mark.parametrize("seed,zipf", [(4, False), (5, True)])
def test_fp32_step_is_close_to_fp64(seed, zipf):
    kg, pos, neg, side = _problem(seed, zipf)
    E64 = kg.E.astype(np.float64)
    A64 = np.full_like(E64, 0.1)
    E32, A32 = kg.E.astype(np.float32), np.full(kg.E.shape, 0.1, dtype=np.float32)
    for step in range(3):
        l64 = R.adagrad_step(E64, A64, pos, neg, side, 0.2, 0.1, np.float64)
        l32 = R.adagrad_step(E32, A32, pos, neg, side, 0.2, 0.1, np.float32)
        assert np.abs(l64 - l32).max() < 1e-5
    assert np.abs(E32 - E64).max() < 1e-5 * (1 + np.abs(E64).max())
    assert np.abs(A32 - A64).max() < 1e-6 * np.abs(A64).max()


def test_bundle_round_trip_with_the_adagrad_slot(tmp_path):
    rng = np.random.default_rng(0)
    E = rng.normal(size=(37, 10)).astype(np.float32)
    A = rng.uniform(0.1, 3.0, size=(37, 10)).astype(np.float32)
    prefix = str(tmp_path / "model.ckpt")
    tf_bundle.save_bundle(prefix, {"embeddings": E, "batch/Variable": np.array(12, dtype=np.int32),
                                   hole.ADAGRAD_SLOT: A})
    keys = [k.decode() for k, _ in tf_bundle.read_index(prefix + ".index")]
    assert keys == ["", "batch/Variable", "embeddings", "embeddings/Adagrad"]
    b = tf_bundle.load_bundle(prefix)
    assert np.array_equal(b["embeddings"], E) and np.array_equal(b[hole.ADAGRAD_SLOT], A)
    E2, step = hole.load_checkpoint(str(tmp_path))
    assert np.array_equal(E2, E) and step == 12
    assert np.array_equal(hole.load_accumulator(str(tmp_path)), A)


def test_resume_without_the_slot_is_refused(tmp_path):
    tf_bundle.save_bundle(str(tmp_path / "model.ckpt"), {"embeddings": np.zeros((3, 4), np.float32)})
    with pytest.raises(SystemExit, match="no embeddings/Adagrad slot"):
        hole.load_accumulator(str(tmp_path))


@pytest.mark.parametrize("extra,msg", [
    (["--log_loss"], "no --log_loss branch"),
    (["--score_variant", "ccorr_tanh"], "not available with --score_variant ccorr_tanh"),
    (["--adagrad_initial_accumulator", "0"], "must be > 0"),
])
def test_cli_refusals(tmp_path, extra, msg):
    argv = ["--data_dir", str(tmp_path / "no_data"), "--output_dir", str(tmp_path / "out"),
            "--optimizer", "adagrad", *extra]
    with pytest.raises(SystemExit, match=msg):
        hole.main(argv)
    assert not os.path.exists(tmp_path / "out")


def test_cli_flag_defaults():
    f, _ = hole.build_parser().parse_known_args(["--data_dir", "d", "--output_dir", "o"])
    assert f.optimizer == "sgd" and f.adagrad_initial_accumulator == 0.1
