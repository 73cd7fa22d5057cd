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


def tree_tolerance(G, absg, depth, A0, lr, E_ref):
    """(tolE, tolA) per element: how far the device's AdaGrad step may lie from the fp64 one (adagrad_step) on a
    row whose uses were combined by a depth-`depth` K3 tree (test_gpu_update_paths.tree_depth; 0 = K1 applied
    the row alone).  G is the fp64 summed gradient, absg = sum_i |g_i| over the per-use gradients, A0 the
    accumulator before the step, E_ref the fp64 row after it.

    The device sums fp32 per-use gradients (each within 1e-6 relative of fp64) in a fixed C-ary tree, 31 fp32
    adds per level and one at the leaf, so its sum is acc = G + e with
        |e| <= delta = absg * (1e-6 + (31 depth + 1) 2^-24)     (test_gpu_update_paths._tree_tol's bound).
    Accumulator: S = fma(acc, acc, A0) against A_ref = A0 + G^2.  |acc^2 - G^2| = |e| |2G + e| <= (2|G| + delta)
    delta, and the fma rounds once (2^-24 |S|; 2^-22 leaves a factor 4):
        tolA = 1e-7 + 2^-22 |A_ref| + (2|G| + delta) delta.
    Row: E - u(acc) against E - u(G), u(g) = lr g / sqrt(A0 + g^2).  u'(g) = lr A0 / (A0 + g^2)^(3/2) falls
    with |g|, so over [G - delta, G + delta] it is at most its value at max(|G| - delta, 0): the tree's error
    moves the row by at most delta lr A0 / (A0 + max(|G| - delta, 0)^2)^(3/2).  The fp32 products -lr acc and
    rsqrt(S) (correctly rounded), and the rounding of S under the rsqrt, add 2^-24 + 2^-24 + 2^-25 of |u|:
        tolE = 2e-6 + 1e-5 |E_ref| + delta lr A0 / (A0 + max(|G| - delta, 0)^2)^(3/2)
               + 2^-22 lr |G| / sqrt(A_ref).
    The constant terms are the one-step band of tests/test_gpu_adagrad.py (the final fma and the fp32 forward
    pass).  With A0 >> G^2 the row term is delta lr / sqrt(A0): _tree_tol at the effective rate lr / sqrt(A0).
    With A0 << G^2 it is ~ delta lr A0 / |G|^3, and the accumulator alone shows a wrong sum."""
    G, absg = np.abs(np.asarray(G, np.float64)), np.asarray(absg, np.float64)
    A0 = np.asarray(A0, np.float64)
    delta = absg * (1e-6 + (31 * np.asarray(depth, np.float64) + 1) * 2.0**-24)
    A_ref = A0 + G * G
    tolA = 1e-7 + 2.0**-22 * A_ref + (2 * G + delta) * delta
    tolE = (2e-6 + 1e-5 * np.abs(E_ref) + delta * lr * A0 / (A0 + np.maximum(G - delta, 0.0)**2)**1.5
            + 2.0**-22 * lr * G / np.sqrt(A_ref))
    return tolE, tolA
