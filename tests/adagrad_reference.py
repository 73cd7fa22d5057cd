"""NumPy statement of the AdaGrad training step (include/hole_b200.h, hole_ctx_set_optimizer), shared by
tests/test_adagrad_oracle.py (held to torch.optim.Adagrad) and tests/test_gpu_adagrad.py (held against the device).
TEST INFRASTRUCTURE ONLY.

It restates TF 1.2's AdagradOptimizer(learning_rate, initial_accumulator_value) applied to holE.py's hinge loss:
  * Optimizer.apply_gradients -> _apply_sparse_duplicate_indices -> _deduplicate_indexed_slices sums the
    duplicate indices of the six IndexedSlices, so each touched row i gets one gradient g_i;
  * SparseApplyAdagrad (training_ops.cc) then applies, per touched row and in the variable's dtype,
        accum[i] += g_i * g_i;   var[i] -= lr * g_i * rsqrt(accum[i])
    with the NEW accumulator and no epsilon.
The gradient is the oracle's (oracle.hole_oracle.indexed_slices, pinned by tests/golden/tfshim_step.npz), merged
as sgd_step(order="merged") merges it; the two update lines are the only new arithmetic."""
import numpy as np

from oracle import hole_oracle as O


def merged_gradient(E, pos, neg_ent, side, margin, dtype=np.float64):
    """(rows int64[U] ascending, g [U, D], loss [B]): the summed gradient of every row the step touches, in the
    device's merge order (sgd_step(order="merged"))."""
    slices, loss, _, _ = O.indexed_slices(E, pos, neg_ent, side, margin, dtype)
    (ri, rp), (_, rn), (ti, tp), (tni, tn), (hi, hp), (hni, hn) = slices
    if side:  # heads corrupted: t and r shared
        merged = [(ri, rp + rn), (ti, tp + tn), (hi, hp), (hni, hn)]
    else:     # tails corrupted: h and r shared
        merged = [(ri, rp + rn), (ti, tp), (hi, hp + hn), (tni, tn)]
    idx = np.concatenate([m[0] for m in merged]).astype(np.int64)
    g = np.concatenate([m[1] for m in merged], axis=0)
    order_ix = np.argsort(idx, kind="stable")
    acc = np.zeros((E.shape[0], E.shape[1]), dtype=g.dtype)
    np.add.at(acc, idx[order_ix], g[order_ix])
    rows = np.unique(idx)
    return rows, acc[rows], loss


def adagrad_apply(E, A, rows, g, lr):
    """SparseApplyAdagrad of one summed gradient row per (unique) row, in place on E and A (their dtype)."""
    dt = E.dtype.type
    A[rows] += g * g
    E[rows] -= (dt(lr) * g) * (dt(1.0) / np.sqrt(A[rows]))


def adagrad_step(E, A, pos, neg_ent, side, margin, lr, dtype=np.float64):
    """One AdaGrad training step in place on E (table, checkpoint layout [N, dim]) and A (accumulator, same
    shape), both of `dtype`.  Returns the hinge loss [B]."""
    assert E.dtype == np.dtype(dtype) and A.dtype == np.dtype(dtype)
    rows, g, loss = merged_gradient(E, pos, neg_ent, side, margin, dtype)
    adagrad_apply(E, A, rows, g, lr)
    return loss
