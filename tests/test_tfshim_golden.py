"""The oracle (NumPy and C) against tests/golden/tfshim_step.npz -- outputs of the REFERENCE's own
hot-path source (holE.py corrupt_batch / get_embedding / evaluate_triples / evaluate_batch /
minimize) executed on the torch-backed TensorFlow shim tests/golden/tfshim.py by
tests/golden/make_tfshim_golden.py.  This is what pins the floating-point oracle: fp64 to 1e-12,
fp32 (same op order as the TF graph) to a few ulp."""
import os

import numpy as np
import pytest

from oracle import hole_oracle as O
from oracle import hole_ref as R

HINGE_CASES = [("A", 3, 0.2), ("B", 2, 0.2), ("D", 2, 0.01)]


@pytest.fixture(scope="module")
def g(golden_dir):
    return np.load(os.path.join(golden_dir, "tfshim_step.npz"))


def test_fixture_covers_both_sides_clips_ties_and_inactive_hinges(g):
    sides = {int(g[f"{nm}_f64_side{s}"]) for nm, n, _ in HINGE_CASES for s in range(n)}
    assert sides == {0, 1}
    norms = np.linalg.norm(g["A_E0"].astype(np.float64), axis=1)
    assert (norms > 1).any() and (norms < 1).any() and (norms == 1.0).any()     # clip, no clip, the tie
    assert np.linalg.norm(g["B_E0"], axis=1).max() < 1                          # Xavier scale: never clipped
    frac = np.mean(g["D_f64_loss0"] > 0)
    assert 0.5 < frac < 0.95                                                    # some hinges inactive
    assert g["B_E0"].shape[1] == 150                                            # odd half-width


@pytest.mark.parametrize("nm,steps,margin", HINGE_CASES)
def test_corruption_fed_to_the_reference_is_the_philox_oracle(g, nm, steps, margin):
    off, ids = O.build_type_csr(g[nm + "_type_of"])
    seed = {"A": 5, "B": 6, "D": 8}[nm]
    for s in range(steps):
        side, neg = O.corrupt(g[nm + "_pos"], g[nm + "_type_of"], off, ids, seed, s)
        assert side == int(g[f"{nm}_f64_side{s}"]) and np.array_equal(neg, g[f"{nm}_f64_neg{s}"])


@pytest.mark.parametrize("nm,steps,margin", HINGE_CASES)
def test_sgd_step_fp64_matches_reference_source(g, nm, steps, margin):
    E = g[nm + "_E0"].astype(np.float64)
    for s in range(steps):
        lr = g[f"{nm}_f64_lr{s}"]
        assert lr == O.inverse_time_decay(0.1, s, 32 * 100, 0.5)                # holE.py:292-294
        loss, vp, vn = O.sgd_step(E, g[nm + "_pos"], g[f"{nm}_f64_neg{s}"], int(g[f"{nm}_f64_side{s}"]),
                                  margin, lr, np.float64, "tf")
        assert np.abs(vp - g[f"{nm}_f64_vp{s}"]).max() <= 1e-12
        assert np.abs(vn - g[f"{nm}_f64_vn{s}"]).max() <= 1e-12
        assert np.abs(loss - g[f"{nm}_f64_loss{s}"]).max() <= 1e-12
        assert np.abs(E - g[f"{nm}_f64_E{s}"]).max() <= 1e-12
    assert np.abs(E - g[nm + "_E0"]).max() > 1e-4


@pytest.mark.parametrize("nm,steps,margin", HINGE_CASES)
def test_sgd_step_fp32_matches_reference_source(g, nm, steps, margin):
    """Same op order as the fp32 TF graph: agreement to a few ulp, chained over the steps."""
    E = g[nm + "_E0"].copy()
    for s in range(steps):
        loss, vp, vn = O.sgd_step(E, g[nm + "_pos"], g[f"{nm}_f32_neg{s}"], int(g[f"{nm}_f32_side{s}"]),
                                  margin, g[f"{nm}_f32_lr{s}"], np.float32, "tf")
        assert np.abs(vp - g[f"{nm}_f32_vp{s}"]).max() <= 2e-7
        assert np.abs(loss - g[f"{nm}_f32_loss{s}"]).max() <= 4e-7
        assert np.abs(E - g[f"{nm}_f32_E{s}"]).max() <= 5e-7
        # and fp32 vs fp64 of the reference itself bounds what any fp32 implementation can claim
        assert np.abs(g[f"{nm}_f32_E{s}"] - g[f"{nm}_f64_E{s}"]).max() <= 2e-6


@pytest.mark.parametrize("nm,steps,margin", HINGE_CASES)
def test_merged_order_of_the_kernels_matches_reference_source(g, nm, steps, margin):
    """order="merged" (what the CUDA kernels do: +/- contributions of a shared row pre-added,
    per-row sum applied once) is the same real-number update."""
    E = g[nm + "_E0"].astype(np.float64)
    for s in range(steps):
        O.sgd_step(E, g[nm + "_pos"], g[f"{nm}_f64_neg{s}"], int(g[f"{nm}_f64_side{s}"]), margin,
                   g[f"{nm}_f64_lr{s}"], np.float64, "merged")
        assert np.abs(E - g[f"{nm}_f64_E{s}"]).max() <= 1e-12


@pytest.mark.parametrize("tag,dtype,tol", [("f64", np.float64, 1e-12), ("f32", np.float32, 5e-7)])
def test_logloss_step_matches_reference_source(g, tag, dtype, tol):
    E = g["C_E0"].astype(dtype)
    for s in range(2):
        sides, negs = g[f"C_{tag}_sides{s}"], g[f"C_{tag}_negs{s}"]
        l2_ref = float(g[f"C_{tag}_l2loss{s}"])
        loss, l2_loss = O.logloss_step(E, g["C_pos"], list(negs), list(sides), g[f"C_{tag}_lr{s}"], 1e-3, dtype)
        # the reference adds the scalar l2 * l2_loss(E) to every row (holE.py:196)
        want = g[f"C_{tag}_loss{s}"] - dtype(1e-3) * dtype(l2_ref)
        assert np.abs(loss - want).max() <= max(tol, 1e-12)
        assert abs(float(l2_loss) - l2_ref) <= 1e-5 * l2_ref
        assert np.abs(E - g[f"C_{tag}_E{s}"]).max() <= tol


@pytest.mark.parametrize("nm,steps,margin", HINGE_CASES)
def test_c_port_matches_reference_source(g, nm, steps, margin):
    """oracle/hole_ref.c (bench.py's CPU baseline) against the same fixture."""
    E = np.ascontiguousarray(g[nm + "_E0"], np.float32).copy()
    for s in range(steps):
        _, loss = R.train_step(E, g[nm + "_pos"], g[f"{nm}_f32_neg{s}"], int(g[f"{nm}_f32_side{s}"]), margin,
                               float(g[f"{nm}_f32_lr{s}"]))
        assert np.abs(loss - g[f"{nm}_f64_loss{s}"]).max() <= 2e-6
        assert np.abs(E - g[f"{nm}_f64_E{s}"]).max() <= 5e-6
