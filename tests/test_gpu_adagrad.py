"""AdaGrad training on the device (hole_ctx_set_optimizer: K1 in DM 4, the AdaGrad K3 root) against the fp64
statement in tests/adagrad_reference.py.

Every step is checked re-synchronised: the device's table and accumulator before the step go through the fp64
reference, and the device's result after the step is held to
  rows         2e-6 + 1e-5 |x|     (the SGD step's one-step band)
  accumulator  1e-7 + 1e-5 |a|     (a = a0 + g^2 with g carrying fp32 rounding of ~1e-6 relative: 2e-6 |a| at
                                    most; the band leaves a factor 5 for the summation order of duplicates)
  loss         2e-6
Rows and accumulator elements the step does not touch must keep their bits."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import adagrad_reference as R
from graphembeddings_b200 import _lib
from graphembeddings_b200 import data as D
from graphembeddings_b200.engine import HoleEngine, HoleError
from oracle import hole_oracle as O

pytestmark = pytest.mark.gpu

ROW_ATOL, ROW_RTOL, ACC_ATOL, ACC_RTOL, LOSS_ATOL = 2e-6, 1e-5, 1e-7, 1e-5, 2e-6
MARGIN, INIT = 0.2, 0.1
# first and last dim of every K1 lane group (GS 8 / 16 / 32 x V 1, 2, 3): masked (with pad columns) and full
LANE_GROUP_DIMS = [2, 64, 66, 128, 130, 256, 258, 512, 514, 768]


def _engine(kg, init=INIT, sort_small=None, monkeypatch=None):
    if sort_small is not None:
        monkeypatch.setenv("HOLE_SORT_SMALL", sort_small)
    off, ids = D.build_type_csr(kg.type_of)
    e = HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E).set_types(kg.type_of, off, ids)
    e.set_relation_count(kg.n_relations)
    e.set_optimizer("adagrad", init)
    return e, off, ids


def _state(e):
    return e.embeddings().cpu().numpy(), e.accumulator().cpu().numpy()


def _check_step(e, pos, seed, step, lr):
    """One device step against the fp64 reference on the device's own state before it."""
    E0, A0 = _state(e)
    side, neg = e.corrupt_batch(pos, seed=seed, step=step)
    loss = e.train_step(pos, neg, side, MARGIN, lr).cpu().numpy()
    E1, A1 = _state(e)
    Er, Ar = E0.astype(np.float64), A0.astype(np.float64)
    lr_ = R.adagrad_step(Er, Ar, pos, neg.cpu().numpy(), side, MARGIN, lr, np.float64)
    assert np.abs(loss - lr_).max() < LOSS_ATOL
    assert np.all(np.abs(E1 - Er) <= ROW_ATOL + ROW_RTOL * np.abs(Er)), np.abs(E1 - Er).max()
    assert np.all(np.abs(A1 - Ar) <= ACC_ATOL + ACC_RTOL * np.abs(Ar)), np.abs(A1 - Ar).max()
    rows, _, _ = R.merged_gradient(E0.astype(np.float64), pos, neg.cpu().numpy(), side, MARGIN)
    untouched = np.setdiff1d(np.arange(len(E0)), rows)
    assert np.array_equal(E1[untouched], E0[untouched]) and np.array_equal(A1[untouched], A0[untouched])
    return side, float(np.abs(A1 - Ar).max() / max(np.abs(Ar).max(), 1e-30))


@pytest.mark.parametrize("dim", LANE_GROUP_DIMS)
def test_chained_steps_every_lane_group(dim):
    kg = D.synthetic_kg(6, 700, 4096, 4, dim, seed=dim, trained_scale=True, zipf_entities=True)
    e, _, _ = _engine(kg)
    sides = set()
    for step in range(4):
        pos = kg.triples[step * 512:(step + 1) * 512]
        side, rel_err = _check_step(e, pos, seed=dim + 1, step=step, lr=0.3 / (1 + step))
        sides.add(side)
    print(f"dim {dim}: accumulator max relative error {rel_err:.2e}")
    e.close()


@pytest.mark.parametrize("zipf", [False, True])
@pytest.mark.parametrize("sort_small", ["0", "2"])    # radix-chain plan / one-launch plan sort
def test_uniform_and_zipf_under_both_plan_sorts(zipf, sort_small, monkeypatch):
    kg = D.synthetic_kg(9, 3000, 20000, 5, 150, seed=7, trained_scale=True, zipf_entities=zipf)
    e, _, _ = _engine(kg, sort_small=sort_small, monkeypatch=monkeypatch)
    sides = set()
    for step in range(6):      # both corruption sides occur over these Philox steps
        pos = kg.triples[step * 2048:(step + 1) * 2048]
        side, _ = _check_step(e, pos, seed=11, step=step, lr=0.2)
        sides.add(side)
    assert sides == {0, 1}
    e.close()


def test_inactive_hinges_and_clipped_rows_keep_or_move_as_the_reference():
    """Margin 0 on a table whose even rows are clipped and odd rows are not: about half the hinges are inactive."""
    kg = D.synthetic_kg(4, 3000, 2048, 3, 40, seed=2, trained_scale=True)
    kg.E[:] *= np.where(np.arange(kg.n_rows)[:, None] % 2 == 0, 3.0, 0.2).astype(np.float32)   # clipped / not
    e, _, _ = _engine(kg)
    E0, A0 = _state(e)
    pos = kg.triples[:1024]
    side, neg = e.corrupt_batch(pos, seed=3, step=0)
    loss = e.train_step(pos, neg, side, 0.0, 0.5).cpu().numpy()
    E1, A1 = _state(e)
    Er, Ar = E0.astype(np.float64), A0.astype(np.float64)
    want = R.adagrad_step(Er, Ar, pos, neg.cpu().numpy(), side, 0.0, 0.5, np.float64)
    assert 0 < (want == 0).sum() < len(want)                               # active and inactive hinges
    assert np.abs(loss - want).max() < LOSS_ATOL
    assert np.all(np.abs(E1 - Er) <= ROW_ATOL + ROW_RTOL * np.abs(Er))
    assert np.all(np.abs(A1 - Ar) <= ACC_ATOL + ACC_RTOL * np.abs(Ar))
    # the rows only inactive triples use keep their bits
    neg_np = neg.cpu().numpy()
    off = want == 0
    used_active = set(pos[~off].ravel()) | set(neg_np[~off])
    only_inactive = sorted((set(pos[off].ravel()) | set(neg_np[off])) - used_active)
    assert np.array_equal(E1[only_inactive], E0[only_inactive]) and np.array_equal(A1[only_inactive], A0[only_inactive])
    e.close()


def _per_step(e, triples, B, n, seed, first, lrs):
    for k in range(n):
        pos = triples[k * B:(k + 1) * B]
        side, neg = e.corrupt_batch(pos, seed=seed, step=first + k)
        e.train_step(pos, neg, side, MARGIN, lrs[k])


@pytest.mark.parametrize("host", [False, True])
def test_multi_step_calls_across_a_chunk_boundary_equal_the_per_step_path(host):
    kg = D.synthetic_kg(5, 2000, 300 * 64, 4, 48, seed=5, trained_scale=True, zipf_entities=True)
    B, n, seed, first = 64, 300, 9, 17          # 300 steps > the 256-step plan chunk
    lrs = [float(0.2 / (1 + 0.01 * k)) for k in range(n)]
    a, _, _ = _engine(kg)
    b, _, _ = _engine(kg)
    if host:
        a.train_steps_host(kg.triples[:n * B], B, seed, first, MARGIN, lrs)
    else:
        a.train_steps(kg.triples[:n * B], B, seed, first, MARGIN, lrs)
    _per_step(b, kg.triples, B, n, seed, first, lrs)
    Ea, Aa = _state(a)
    Eb, Ab = _state(b)
    assert np.array_equal(Ea.view(np.uint32), Eb.view(np.uint32))
    assert np.array_equal(Aa.view(np.uint32), Ab.view(np.uint32))
    assert not np.array_equal(Aa, np.full_like(Aa, INIT))
    a.close(); b.close()


def test_two_runs_are_bit_identical():
    kg = D.synthetic_kg(7, 5000, 40000, 5, 256, seed=8, trained_scale=True, zipf_entities=True)
    out = []
    for _ in range(2):
        e, _, _ = _engine(kg)
        e.train_steps(kg.triples[:20 * 2000], 2000, 4, 0, MARGIN, [0.1] * 20)
        out.append(_state(e))
        e.close()
    assert np.array_equal(out[0][0].view(np.uint32), out[1][0].view(np.uint32))
    assert np.array_equal(out[0][1].view(np.uint32), out[1][1].view(np.uint32))


def test_pad_columns_stay_zero_after_training_from_a_restored_accumulator():
    kg = D.synthetic_kg(5, 800, 8192, 4, 130, seed=4, trained_scale=True, zipf_entities=True)   # H 65: 3 pad columns a half
    e, _, _ = _engine(kg, init=0.25)
    A = np.random.default_rng(0).uniform(0.1, 2.0, size=kg.E.shape).astype(np.float32)
    e.set_accumulator(A)
    assert np.array_equal(e.accumulator().cpu().numpy(), A)
    half, H = e.row_stride // 2, kg.dim // 2
    assert torch.all(e.accum[:, H:half] == 0.25) and torch.all(e.accum[:, half + H:] == 0.25)
    e.train_steps(kg.triples[:8 * 1024], 1024, 2, 0, MARGIN, [0.3] * 8)
    t = e.table
    assert torch.all(t[:, H:half] == 0) and torch.all(t[:, half + H:] == 0)
    assert torch.isfinite(t).all() and torch.isfinite(e.accum).all()
    assert torch.all(e.accum[:, H:half] == 0.25)
    e.close()


def _snapshot(e):
    return e.table.clone(), e.accum.clone()


def test_refusals_write_nothing_and_leave_the_context_usable():
    kg = D.synthetic_kg(5, 600, 4096, 4, 64, seed=6, trained_scale=True, zipf_entities=True)
    e, off, ids = _engine(kg)
    pos = kg.triples[:512]
    side, neg = e.corrupt_batch(pos, seed=1, step=0)
    p32 = e._triples(pos)
    delta = torch.zeros_like(e.table)
    t0, a0 = _snapshot(e)
    torch.cuda.synchronize()
    n0 = e.launch_count()
    calls = [
        lambda: e.train_step_delta(p32, neg, side, MARGIN, 0.1, delta),
        lambda: e.train_step_logloss(pos, 1, 0, 0.1),
        lambda: e.shard_step(p32, 1, 0, MARGIN, 0.1),
        lambda: e.shard_step(p32, 1, 0, MARGIN, 0.1, phase="apply"),
        lambda: e.shard_prepare(p32, 1, 0),
        lambda: e.shard_steps(p32, 512, 1, 0, MARGIN, [0.1]),
    ]
    for call in calls:
        with pytest.raises(HoleError, match="error -4"):
            call()
    e.set_score_mode("ccorr_tanh")
    for call in (lambda: e.train_step(pos, neg, side, MARGIN, 0.1),
                 lambda: e.train_steps(kg.triples[:1024], 512, 1, 0, MARGIN, [0.1, 0.1]),
                 lambda: e.train_steps_host(kg.triples[:1024], 512, 1, 0, MARGIN, [0.1, 0.1])):
        with pytest.raises(HoleError, match="error -4"):
            call()
    torch.cuda.synchronize()
    assert e.launch_count() == n0                          # nothing was launched
    assert torch.equal(e.table, t0) and torch.equal(e.accum, a0) and torch.count_nonzero(delta) == 0
    e.set_score_mode("complex")
    # still usable: an AdaGrad step runs and matches the reference
    _check_step(e, pos, seed=1, step=0, lr=0.1)
    # back to SGD: bit for bit the steps of a context that never used AdaGrad
    e.set_optimizer("sgd")
    assert e.accum is None
    f = HoleEngine(kg.n_rows, kg.dim).set_embeddings(e.embeddings()).set_types(kg.type_of, off, ids)
    f.set_relation_count(kg.n_relations)
    e.train_steps(kg.triples[:8 * 512], 512, 3, 5, MARGIN, [0.1] * 8)
    f.train_steps(kg.triples[:8 * 512], 512, 3, 5, MARGIN, [0.1] * 8)
    l1 = e.train_step(pos, neg, side, MARGIN, 0.1)
    l2 = f.train_step(pos, neg, side, MARGIN, 0.1)
    assert torch.equal(e.table, f.table) and torch.equal(l1, l2)
    e.close(); f.close()


def test_set_optimizer_arguments():
    kg = D.synthetic_kg(3, 100, 256, 2, 16, seed=1, trained_scale=True)
    e, _, _ = _engine(kg)
    lib = e.lib
    with pytest.raises(HoleError):
        _lib.check(lib.hole_ctx_set_optimizer(e._ctx, _lib.HOLE_OPT_ADAGRAD, None))
    with pytest.raises(HoleError):
        _lib.check(lib.hole_ctx_set_optimizer(e._ctx, _lib.HOLE_OPT_SGD, C.c_void_p(e.accum.data_ptr())))
    with pytest.raises(HoleError):
        _lib.check(lib.hole_ctx_set_optimizer(e._ctx, 2, C.c_void_p(e.accum.data_ptr())))
    with pytest.raises(HoleError):
        e.set_optimizer("adagrad", 0.0)
    with pytest.raises(HoleError):
        e.set_optimizer("adam")
    e.close()


def test_an_adagrad_step_invalidates_the_ranking_operand_cache():
    kg = D.synthetic_kg(6, 900, 4096, 4, 64, seed=12, trained_scale=True)
    e, off, ids = _engine(kg)
    q = kg.triples[:200]
    e.rank_prepare(kg.n_relations, kg.n_rows)
    e.rank(q, 0, kg.n_relations, kg.n_rows)
    e.train_steps(kg.triples[:4 * 1024], 1024, 1, 0, MARGIN, [0.5] * 4)
    raw, filt, ts = e.rank(q, 0, kg.n_relations, kg.n_rows)
    f = HoleEngine(kg.n_rows, kg.dim).set_embeddings(e.embeddings())
    raw2, filt2, ts2 = f.rank(q, 0, kg.n_relations, kg.n_rows)
    assert torch.equal(raw, raw2) and torch.equal(ts, ts2)
    e.close(); f.close()


def _rows_ckpt(e, t, rows_d):
    """Rows rows_d of a device-layout tensor, in checkpoint layout, as float64 numpy."""
    src = t[rows_d].contiguous()
    out = torch.empty((len(rows_d), e.dim), dtype=torch.float32, device=e.device)
    _lib.check(e.lib.hole_unpack_rows(e._ctx, C.c_void_p(src.data_ptr()), C.c_void_p(out.data_ptr()), len(rows_d),
                                      C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return out.cpu().numpy().astype(np.float64)


def test_config1_shape_touched_rows_against_the_reference():
    """Config 1's table (1,200,014 x 256) at B = 32768, 3 steps: the touched rows against the fp64 reference run on
    the touched rows alone; every other row and accumulator element keeps its bits."""
    kg = D.synthetic_kg(14, 1_200_000, 3 * 32768, 50, 256, seed=21, trained_scale=True, zipf_entities=True)
    e, _, _ = _engine(kg)
    B = 32768
    for step in range(3):
        pos = kg.triples[step * B:(step + 1) * B]
        side, neg = e.corrupt_batch(pos, seed=2, step=step)
        neg_np = neg.cpu().numpy()
        rows = np.unique(np.concatenate([pos.ravel(), neg_np]))
        rows_d = torch.from_numpy(rows).to(e.device)
        E0t, A0t = e.table.clone(), e.accum.clone()
        Er, Ar = _rows_ckpt(e, E0t, rows_d), _rows_ckpt(e, A0t, rows_d)
        loss = e.train_step(pos, neg, side, MARGIN, 0.1).cpu().numpy()
        d, a = _rows_ckpt(e, e.table, rows_d), _rows_ckpt(e, e.accum, rows_d)
        # fp64 reference on the touched rows, re-indexed into a compact table
        sub = lambda x: np.searchsorted(rows, x)
        want = R.adagrad_step(Er, Ar, sub(pos), sub(neg_np), side, MARGIN, 0.1, np.float64)
        assert np.abs(loss - want).max() < LOSS_ATOL
        assert np.all(np.abs(d - Er) <= ROW_ATOL + ROW_RTOL * np.abs(Er)), np.abs(d - Er).max()
        assert np.all(np.abs(a - Ar) <= ACC_ATOL + ACC_RTOL * np.abs(Ar)), np.abs(a - Ar).max()
        mask = torch.ones(kg.n_rows, dtype=torch.bool, device=e.device)
        mask[rows_d] = False
        assert torch.equal(e.table[mask], E0t[mask]) and torch.equal(e.accum[mask], A0t[mask])
    e.close()


def test_cli_adagrad_train_checkpoint_resume_infer(tmp_path):
    from graphembeddings_b200 import build, hole, tf_bundle
    from test_gpu_cli import _write_data_dir
    build.build()
    kg = D.synthetic_kg(8, 1500, 9000, 4, 64, seed=3, with_embeddings=False)
    d = tmp_path / "data"; d.mkdir()
    _write_data_dir(str(d), kg, 600, 400)
    out = str(tmp_path / "run")
    args = ["--data_dir", str(d), "--output_dir", out, "--batch_size", "256", "--embedding_dim", "64",
            "--num_epochs", "1", "--optimizer", "adagrad", "--adagrad_initial_accumulator", "0.2"]
    hole.main(args)
    b = tf_bundle.load_bundle(os.path.join(out, "model.ckpt"))
    A = b["embeddings/Adagrad"]
    assert A.shape == (kg.n_rows, 64) and np.all(A >= np.float32(0.2)) and np.any(A > np.float32(0.2))
    step0 = int(np.asarray(b["batch/Variable"]).reshape(-1)[0])
    hole.main(args + ["--resume_checkpoint", "--max_steps", "3"])
    b2 = tf_bundle.load_bundle(os.path.join(out, "model.ckpt"))
    assert np.all(b2["embeddings/Adagrad"] >= A)                   # resumed from the saved accumulator
    # SGD resumes the same checkpoint and ignores the slot; AdaGrad refuses a checkpoint without one
    hole.main(args[:-4] + ["--resume_checkpoint", "--max_steps", "2"])
    out2 = str(tmp_path / "sgd"); os.makedirs(out2)
    tf_bundle.save_bundle(os.path.join(out2, "model.ckpt"), {"embeddings": b["embeddings"],
                                                            "batch/Variable": np.array(step0, np.int32)})
    tf_bundle.write_checkpoint_state(out2)
    with pytest.raises(SystemExit, match="no embeddings/Adagrad slot"):
        hole.main(["--data_dir", str(d), "--output_dir", out2, "--batch_size", "256", "--embedding_dim", "64",
                   "--optimizer", "adagrad", "--resume_checkpoint"])
    cwd = os.getcwd()
    os.chdir(tmp_path)          # --infer writes inference_results.tsv to the working directory, as holE.py does
    try:
        m = hole.infer_triples(hole.build_parser().parse_args(args + ["--infer"]), log=lambda *a: None)
    finally:
        os.chdir(cwd)
    assert 0 < m["filtered_mrr"] <= 1
    assert os.path.exists(tmp_path / "inference_results.tsv")
