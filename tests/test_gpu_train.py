"""Parity of the CUDA training path (through the C ABI) against the oracle.

Standards (north_star / SURVEY 8c):
  * corruption ids, side coin: bit-exact;
  * sigma, loss: |d| <= 1e-6 vs the fp32 and fp64 oracle;
  * updated rows after one step: |d| <= 2e-6 + 1e-5*|x| vs the fp64 oracle (fp32 compute,
    fixed but different summation order than TF's sequential ScatterSub).
"""
import os

import numpy as np
import pytest
import torch

from graphembeddings_b200 import data as D
from oracle import hole_oracle as O

pytestmark = pytest.mark.gpu

SIGMA_ATOL = 1e-6
ROW_ATOL, ROW_RTOL = 2e-6, 1e-5


@pytest.fixture(scope="module")
def eng_mod():
    from graphembeddings_b200 import build
    build.build()
    from graphembeddings_b200 import engine
    return engine


def _engine(eng_mod, kg):
    e = eng_mod.HoleEngine(kg.n_rows, kg.dim)
    e.set_embeddings(kg.E)
    off, ids = D.build_type_csr(kg.type_of)
    e.set_types(kg.type_of, off, ids)
    return e, off, ids


# 20 .. 600: round dims; 2, 66, 130, 258, 768: the first or last dim of a K1 lane-group regime
# (tests/test_gpu_shapes.py lane_group)
DIMS = [20, 64, 128, 150, 256, 512, 600, 2, 66, 130, 258, 768]


@pytest.mark.parametrize("dim", DIMS)
def test_pack_unpack_roundtrip(eng_mod, dim):
    kg = D.synthetic_kg(5, 300, 10, 3, dim, seed=1)
    e, _, _ = _engine(eng_mod, kg)
    assert torch.equal(e.embeddings().cpu(), torch.from_numpy(kg.E))
    # padding lanes are zero
    H, Hp = dim // 2, e.row_stride // 2
    tab = e.table.cpu().numpy()
    assert np.all(tab[:, H:Hp] == 0) and np.all(tab[:, Hp + H:] == 0)


@pytest.mark.parametrize("dim", DIMS)
@pytest.mark.parametrize("trained", [False, True])
def test_score_matches_oracle(eng_mod, dim, trained):
    kg = D.synthetic_kg(9, 2000, 3000, 6, dim, seed=dim, trained_scale=trained, zipf_entities=True)
    e, _, _ = _engine(eng_mod, kg)
    got = e.evaluate_triples(kg.triples).cpu().numpy()
    want64 = O.evaluate_triples(kg.E.astype(np.float64), kg.triples, np.float64)
    want32 = O.evaluate_triples(kg.E, kg.triples, np.float32)
    assert np.abs(got - want64).max() <= SIGMA_ATOL
    assert np.abs(got - want32).max() <= SIGMA_ATOL
    if trained:
        assert got.std() > 1e-4      # not a degenerate all-0.5 comparison


def test_corruption_bit_exact(eng_mod):
    kg = D.make_config("fb15k_d150", n_triples=20000, with_embeddings=False)
    kg.E = D.init_embeddings(kg.n_rows, 8, np.random.default_rng(0))
    kg.dim = 8
    e, off, ids = _engine(eng_mod, kg)
    seen = set()
    for step in (0, 1, 2, 3, 2**33 + 5):
        side, neg = e.corrupt_batch(kg.triples, seed=0xC0FFEE123456789, step=step)
        oside, oneg = O.corrupt(kg.triples, kg.type_of, off, ids, 0xC0FFEE123456789, step)
        assert side == oside
        assert np.array_equal(neg.cpu().numpy(), oneg)
        seen.add(side)
    assert seen == {0, 1}


def _check_step(eng_mod, kg, B, side_force=None, seed=3, step=0, lr=0.1, margin=0.2):
    e, off, ids = _engine(eng_mod, kg)
    pos = kg.triples[:B]
    side, neg = O.corrupt(pos, kg.type_of, off, ids, seed, step)
    if side_force is not None:
        side = side_force
    loss, vp, vn = e.train_step(pos, neg, side, margin, lr, return_sigma=True)
    E64 = kg.E.astype(np.float64)
    l64, vp64, vn64 = O.sgd_step(E64, pos, neg, side, margin, lr, np.float64, "tf")
    E32 = kg.E.copy()
    l32, _, _ = O.sgd_step(E32, pos, neg, side, margin, lr, np.float32, "tf")
    assert np.abs(vp.cpu().numpy() - vp64).max() <= SIGMA_ATOL
    assert np.abs(vn.cpu().numpy() - vn64).max() <= SIGMA_ATOL
    assert np.abs(loss.cpu().numpy() - l64).max() <= 2 * SIGMA_ATOL
    got = e.embeddings().cpu().numpy()
    err = np.abs(got - E64)
    tol = ROW_ATOL + ROW_RTOL * np.abs(E64)
    assert (err <= tol).all(), float((err - tol).max())
    # also against the fp32 oracle in TF order
    assert np.abs(got - E32).max() <= 1e-5
    # the step did move the touched rows and nothing else
    touched = np.unique(np.concatenate([pos.ravel(), neg]))
    untouched = np.setdiff1d(np.arange(kg.n_rows), touched)
    assert np.array_equal(got[untouched], kg.E[untouched])
    assert np.abs(got - kg.E).max() > 1e-5
    return e


@pytest.mark.parametrize("dim", DIMS)
@pytest.mark.parametrize("side", [0, 1])
def test_train_step_matches_oracle(eng_mod, dim, side):
    kg = D.synthetic_kg(7, 500, 1024, 5, dim, seed=100 + dim, trained_scale=True, zipf_entities=True)
    _check_step(eng_mod, kg, 1024, side_force=side)


def test_train_step_xavier_init_all_hinges_active(eng_mod):
    kg = D.synthetic_kg(11, 4000, 2048, 5, 150, seed=5)
    e = _check_step(eng_mod, kg, 2048)


def test_train_step_heavy_duplicates(eng_mod):
    """3 relations, 40 entities, 6000 triples: every row has hundreds of occurrences, so the
    combine tree runs several levels deep."""
    kg = D.synthetic_kg(3, 40, 6000, 2, 64, seed=8, trained_scale=True, zipf_entities=True)
    _check_step(eng_mod, kg, 6000)


@pytest.mark.parametrize("B", [1, 2, 31, 33, 513])
def test_train_step_ragged_batches(eng_mod, B):
    kg = D.synthetic_kg(4, 200, 600, 3, 150, seed=B, trained_scale=True)
    _check_step(eng_mod, kg, B)


def test_empty_batch_is_a_noop(eng_mod):
    kg = D.synthetic_kg(4, 50, 10, 3, 16, seed=2)
    e, _, _ = _engine(eng_mod, kg)
    loss = e.train_step(np.zeros((0, 3), np.int32), np.zeros(0, np.int32), 0, 0.2, 0.1)
    assert loss.numel() == 0
    assert torch.equal(e.embeddings().cpu(), torch.from_numpy(kg.E))
    assert e.evaluate_triples(np.zeros((0, 3), np.int32)).numel() == 0


def test_train_step_is_deterministic(eng_mod):
    kg = D.synthetic_kg(3, 100, 4096, 2, 128, seed=21, trained_scale=True, zipf_entities=True)
    outs = []
    for _ in range(3):
        e, off, ids = _engine(eng_mod, kg)
        side, neg = O.corrupt(kg.triples, kg.type_of, off, ids, 1, 0)
        e.train_step(kg.triples, neg, side, 0.2, 0.1)
        outs.append(e.embeddings().cpu())
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])


def test_golden_fixture_step(eng_mod, golden_dir):
    z = np.load(os.path.join(golden_dir, "train_step_oracle.npz"))
    E0, pos = z["E0"], z["pos"]
    for step in (0, 1):
        e = eng_mod.HoleEngine(E0.shape[0], E0.shape[1])
        e.set_embeddings(E0)
        loss = e.train_step(pos, z[f"neg{step}"], int(z[f"side{step}"]), 0.2, 0.1)
        assert np.abs(loss.cpu().numpy() - z[f"loss64_{step}"]).max() <= 2 * SIGMA_ATOL
        got = e.embeddings().cpu().numpy()
        assert np.abs(got - z[f"E64_{step}"]).max() <= ROW_ATOL + ROW_RTOL


@pytest.mark.parametrize("nm,steps,margin", [("A", 3, 0.2), ("B", 2, 0.2), ("D", 2, 0.01)])
def test_reference_source_fixture_hinge_steps(eng_mod, golden_dir, nm, steps, margin):
    """tests/golden/tfshim_step.npz: the REFERENCE's own evaluate_batch + minimize (holE.py:205-234,
    291-296) executed on the TensorFlow shim (tests/golden/make_tfshim_golden.py).  Identical
    triples, identical corruption ids (checked bit-exact against the device sampler), chained
    steps: sigma / loss <= 1e-6 / 2e-6, rows <= 2e-6 + 1e-5|x| per step vs the fp64 reference run,
    and within 4e-6 of the reference's own fp32 run."""
    z = np.load(os.path.join(golden_dir, "tfshim_step.npz"))
    E0, pos, type_of = z[nm + "_E0"], z[nm + "_pos"], z[nm + "_type_of"]
    off, ids = D.build_type_csr(type_of)
    e = eng_mod.HoleEngine(E0.shape[0], E0.shape[1]).set_embeddings(E0).set_types(type_of, off, ids)
    seed = {"A": 5, "B": 6, "D": 8}[nm]
    for s in range(steps):
        side, neg = e.corrupt_batch(pos, seed, s)
        assert side == int(z[f"{nm}_f64_side{s}"]) and np.array_equal(neg.cpu().numpy(), z[f"{nm}_f64_neg{s}"])
        loss, vp, vn = e.train_step(pos, neg, side, margin, float(z[f"{nm}_f32_lr{s}"]), return_sigma=True)
        assert np.abs(vp.cpu().numpy() - z[f"{nm}_f64_vp{s}"]).max() <= SIGMA_ATOL
        assert np.abs(vn.cpu().numpy() - z[f"{nm}_f64_vn{s}"]).max() <= SIGMA_ATOL
        assert np.abs(loss.cpu().numpy() - z[f"{nm}_f64_loss{s}"]).max() <= 2 * SIGMA_ATOL
        got = e.embeddings().cpu().numpy()
        want = z[f"{nm}_f64_E{s}"]
        assert (np.abs(got - want) <= (s + 1) * (ROW_ATOL + ROW_RTOL * np.abs(want))).all()
        assert np.abs(got - z[f"{nm}_f32_E{s}"]).max() <= (s + 1) * 4e-6


def test_reference_source_fixture_logloss_steps(eng_mod, golden_dir):
    """Same fixture, --log_loss branch (holE.py:194-196, 206-220): k = 2, l2 = 1e-3, two chained steps."""
    z = np.load(os.path.join(golden_dir, "tfshim_step.npz"))
    E0, pos, type_of = z["C_E0"], z["C_pos"], z["C_type_of"]
    off, ids = D.build_type_csr(type_of)
    e = eng_mod.HoleEngine(E0.shape[0], E0.shape[1]).set_embeddings(E0).set_types(type_of, off, ids)
    for s in range(2):
        loss, l2_loss, sides, neg = e.train_step_logloss(pos, 7, s, float(z[f"C_f32_lr{s}"]), 1e-3, 2,
                                                         want_corruption=True)
        assert sides == [int(x) for x in z[f"C_f64_sides{s}"]]
        assert np.array_equal(neg.cpu().numpy(), z[f"C_f64_negs{s}"])
        l2_ref = float(z[f"C_f64_l2loss{s}"])
        assert abs(float(l2_loss) - l2_ref) <= 1e-5 * l2_ref
        want = z[f"C_f64_loss{s}"] - 1e-3 * l2_ref          # the reference adds the scalar to every row
        assert np.abs(loss.cpu().numpy() - want).max() <= 2e-6
        got = e.embeddings().cpu().numpy()
        assert (np.abs(got - z[f"C_f64_E{s}"]) <= (s + 1) * (ROW_ATOL + ROW_RTOL * np.abs(z[f"C_f64_E{s}"]))).all()


def test_logloss_golden_fixture_step(eng_mod, golden_dir):
    """The committed fixture of the oracle's --log_loss step (tests/golden/make_golden.py):
    corruption bit-exact, loss rows and updated table within the fp32 tolerances."""
    z = np.load(os.path.join(golden_dir, "logloss_step_oracle.npz"))
    E0, pos, type_of = z["E0"], z["pos"], z["type_of"]
    off, ids = D.build_type_csr(type_of)
    e = eng_mod.HoleEngine(E0.shape[0], E0.shape[1]).set_embeddings(E0).set_types(type_of, off, ids)
    loss, l2_loss, sides, neg = e.train_step_logloss(pos, int(z["seed"]), int(z["step"]), float(z["lr"]),
                                                     float(z["l2"]), int(z["k"]), want_corruption=True)
    assert sides == [int(x) for x in z["sides"]] and np.array_equal(neg.cpu().numpy(), z["negs"])
    assert np.abs(loss.cpu().numpy() - z["loss64"]).max() <= 2e-6
    assert abs(float(l2_loss) - float(z["l2_64"])) <= 1e-5 * float(z["l2_64"])
    assert np.abs(e.embeddings().cpu().numpy() - z["E64"]).max() <= ROW_ATOL + ROW_RTOL


@pytest.mark.parametrize("dim,B", [(150, 512), (256, 1000)])
def test_multi_step_matches_oracle_loop(eng_mod, dim, B):
    """hole_train_steps (device-side loop incl. Philox corruption) vs the oracle loop."""
    n_steps = 5
    kg = D.synthetic_kg(6, 3000, B * n_steps, 4, dim, seed=77, trained_scale=True)
    e, off, ids = _engine(eng_mod, kg)
    lrs = [eng_mod.inverse_time_decay(0.1, s, 32 * 100, 0.5) for s in range(n_steps)]
    sums, loss = e.train_steps(kg.triples, B, seed=9, first_step=0, margin=0.2, lrs=lrs, want_loss=True)
    E64 = kg.E.astype(np.float64)
    want = []
    for s in range(n_steps):
        pos = kg.triples[s * B:(s + 1) * B]
        side, neg = O.corrupt(pos, kg.type_of, off, ids, 9, s)
        l, _, _ = O.sgd_step(E64, pos, neg, side, 0.2, float(lrs[s]), np.float64, "tf")
        want.append(l)
    want = np.concatenate(want)
    assert np.abs(loss.cpu().numpy() - want).max() <= 5e-6
    assert np.abs(sums.cpu().numpy() - want.reshape(n_steps, B).sum(1)).max() <= 1e-3
    got = e.embeddings().cpu().numpy()
    assert np.abs(got - E64).max() <= 1e-5
    # host-buffer path gives the same table bit for bit
    e2, _, _ = _engine(eng_mod, kg)
    hs = e2.train_steps_host(kg.triples, B, seed=9, first_step=0, margin=0.2, lrs=lrs)
    assert np.array_equal(hs, sums.cpu().numpy())
    assert torch.equal(e2.embeddings().cpu(), e.embeddings().cpu())


def test_full_size_properties_config0(eng_mod):
    """BASELINE config 0 at full size (16,296 x 150, 483,142 triples, B = 8192): properties
    that need no oracle -- determinism across runs, untouched rows unchanged, loss in range,
    row norms finite."""
    kg = D.make_config("fb15k_d150")
    B = 8192
    n_steps = kg.triples.shape[0] // B
    lrs = [0.1] * n_steps
    res = []
    for _ in range(2):
        e, _, _ = _engine(eng_mod, kg)
        sums = e.train_steps(kg.triples, B, seed=1, first_step=0, margin=0.2, lrs=lrs)
        res.append((sums.cpu(), e.embeddings().cpu()))
    assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1])
    mean_loss = res[0][0].numpy() / B
    # at Xavier init every score is ~0, so the hinge sits at the margin and moves slowly
    assert np.all(np.abs(mean_loss - 0.2) < 0.05)
    assert not torch.equal(res[0][1], torch.from_numpy(kg.E))
    assert torch.isfinite(res[0][1]).all()


def test_sharded_trainer_single_rank_matches_engine(eng_mod):
    """RowShardedTrainer with one rank (no process group) routes everything through the
    step table W and the delta application; it must agree with the plain engine step."""
    from graphembeddings_b200.sharded import CudaBackend, RowShardedTrainer
    kg = D.synthetic_kg(6, 3000, 1500, 4, 150, seed=41, trained_scale=True, zipf_entities=True)
    off, ids = D.build_type_csr(kg.type_of)
    be = CudaBackend(kg.n_relations, kg.dim, 500, 0, kg.type_of, off, ids)
    tr = RowShardedTrainer(kg.n_relations, kg.n_entities, kg.dim, be, None).load_embeddings(kg.E)
    e, _, _ = _engine(eng_mod, kg)
    for s in range(3):
        pos = kg.triples[s * 500:(s + 1) * 500]
        loss_s = tr.train_step(torch.from_numpy(pos), 5, s, 0.2, 0.1)
        side, neg = e.corrupt_batch(pos, 5, s)
        loss_e = e.train_step(pos, neg, side, 0.2, 0.1)
        assert torch.allclose(loss_s, loss_e, atol=2e-6, rtol=0)
    got = tr.gather_embeddings().cpu().numpy()
    want = e.embeddings().cpu().numpy()
    assert np.abs(got - want).max() <= 1e-6
    assert np.abs(want - kg.E).max() > 1e-4


@pytest.mark.parametrize("dim,k,l2", [(150, 1, 0.0), (256, 3, 0.0), (64, 2, 1e-5), (600, 2, 0.0), (720, 2, 0.0),
                                      (66, 1, 1e-5), (56, 1, 0.0), (128, 2, 1e-5), (258, 2, 0.0), (512, 1, 1e-5),
                                      (768, 2, 0.0)])
def test_logloss_step_matches_oracle(eng_mod, dim, k, l2):
    """--log_loss branch (holE.py:194-196, 206-220): k corrupt batches drawn with virtual steps
    step*k + j (bit-exact vs the oracle's Philox), softplus rows, sparse gradients taken at the
    old table + dense L2 decay.  fp32 tolerances as for the hinge step."""
    kg = D.synthetic_kg(7, 4000, 900, 5, dim, seed=50 + k, trained_scale=True, zipf_entities=True)
    e, off, ids = _engine(eng_mod, kg)
    seed, B, lr = 21, 300, 0.05
    E = kg.E.copy()
    for step in range(3):
        pos = kg.triples[step * B:(step + 1) * B]
        loss, l2_loss, sides, neg = e.train_step_logloss(pos, seed, step, lr, l2, k, want_corruption=True,
                                                         want_l2_loss=True)
        neg_h = neg.cpu().numpy()
        for j in range(k):
            side_o, neg_o = O.corrupt(pos, kg.type_of, off, ids, seed, step * k + j)
            assert side_o == sides[j] and np.array_equal(neg_o, neg_h[j])
        want_l2 = 0.5 * float((E.astype(np.float64) ** 2).sum())
        want_loss, _ = O.logloss_step(E, pos, list(neg_h), sides, lr, l2, np.float32)
        assert np.abs(loss.cpu().numpy() - want_loss).max() <= 2e-6
        assert abs(float(l2_loss) - want_l2) <= 1e-5 * want_l2
    got = e.embeddings().cpu().numpy()
    assert np.allclose(got, E, atol=ROW_ATOL * 3, rtol=ROW_RTOL)
    assert np.abs(E - kg.E).max() > 1e-4
    assert not e._delta_ws.any()                 # the scratch delta table is handed back clean


def test_logloss_gradient_is_taken_at_the_old_table(eng_mod):
    """Heavy duplicates + k = 4: every pass must see the table as it was before the step
    (TF computes the whole gradient, then applies it once)."""
    kg = D.synthetic_kg(3, 40, 512, 2, 128, seed=77, trained_scale=True)
    e, off, ids = _engine(eng_mod, kg)
    E = kg.E.copy()
    pos = kg.triples[:512]
    loss, l2_loss, sides, neg = e.train_step_logloss(pos, 5, 0, 0.1, 0.0, 4, want_corruption=True)
    O.logloss_step(E, pos, list(neg.cpu().numpy()), sides, 0.1, 0.0, np.float32)
    got = e.embeddings().cpu().numpy()
    assert np.allclose(got, E, atol=2e-5, rtol=1e-4)


def test_logloss_training_reduces_the_loss(eng_mod):
    """96 consecutive --log_loss steps (k = 2): the loss of the positives falls, and by the
    same amount as in the oracle's loop."""
    kg = D.synthetic_kg(8, 1500, 4096, 4, 64, seed=4, trained_scale=True)
    e, off, ids = _engine(eng_mod, kg)
    E = kg.E.copy()

    def pos_loss(X):
        return float(np.log1p(np.exp(-O.score(X, kg.triples, np.float64))).mean())

    step = 0
    for epoch in range(6):
        for b in range(16):
            pos = kg.triples[b * 256:(b + 1) * 256]
            e.train_step_logloss(pos, 3, step, 0.5, 0.0, 2)
            drawn = [O.corrupt(pos, kg.type_of, off, ids, 3, step * 2 + j) for j in range(2)]
            O.logloss_step(E, pos, [d[1] for d in drawn], [d[0] for d in drawn], 0.5, 0.0, np.float32)
            step += 1
    got = pos_loss(e.embeddings().cpu().numpy())
    assert got < pos_loss(kg.E) - 0.02
    assert abs(got - pos_loss(E)) < 1e-4


@pytest.mark.parametrize("world,n_ent", [pytest.param(1, 1000, id="1"), pytest.param(2, 1000, id="2"),
                                         pytest.param(3, 1000, id="3"), pytest.param(2, 3 << 24, id="2-4pass")])
def test_shard_route_and_post_virtual_ranks(eng_mod, world, n_ent):
    """Request routing of the sharded step with `world` virtual ranks on one GPU (peer buffers are
    local tensors): route == np.unique / searchsorted, post delivers every owner's slice.  n_ent = 3 * 2^24:
    ids above 2^24 (the largest one included), so the routing sort takes 4 byte passes; routing reads ids
    only, so the engine's own table stays small."""
    from graphembeddings_b200.sharded import row_partition
    rng = np.random.default_rng(100 + world)
    dim, R, B = 150, 5, 257
    e = eng_mod.HoleEngine(R + 1000, dim)
    cap = 3 * B
    rows_per = row_partition(n_ent, world)
    dev = e.device
    inbox = [torch.full((world, cap), -7, dtype=torch.int32, device=dev) for _ in range(world)]
    meta = [torch.zeros((world, 2), dtype=torch.int32, device=dev) for _ in range(world)]
    pa = e.peer_array
    for k in range(world):
        pos = np.stack([R + rng.integers(0, n_ent, B), R + rng.integers(0, n_ent, B), rng.integers(0, R, B)], 1)
        pos[:5, 1] = pos[:5, 0]                                  # head == tail rows
        neg = R + rng.integers(0, n_ent, B)
        neg[7] = R + n_ent - 1
        pos_t = torch.from_numpy(pos.astype(np.int32)).to(dev)
        neg_t = torch.from_numpy(neg.astype(np.int32)).to(dev)
        uniq = torch.full((cap,), -1, dtype=torch.int32, device=dev)
        cuts = torch.zeros(world + 1, dtype=torch.int32, device=dev)
        pos_w = torch.zeros((B, 3), dtype=torch.int32, device=dev)
        neg_w = torch.zeros(B, dtype=torch.int32, device=dev)
        e.shard_route(pos_t, neg_t, R, R + n_ent, rows_per, world, uniq, cuts, pos_w, neg_w)
        want = np.unique(np.concatenate([pos[:, 0], pos[:, 1], neg]))
        U = len(want)
        cuts_h = cuts.cpu().numpy()
        assert cuts_h[world] == U and cuts_h[0] == 0
        uh = uniq.cpu().numpy()
        assert np.array_equal(uh[:U], want) and (uh[U:] == -1).all()
        bounds = R + rows_per * np.arange(world + 1)
        assert np.array_equal(cuts_h[:world], np.searchsorted(want, bounds[:world]))
        pw, nw = pos_w.cpu().numpy(), neg_w.cpu().numpy()
        assert np.array_equal(want[pw[:, 0] - R], pos[:, 0]) and np.array_equal(want[pw[:, 1] - R], pos[:, 1])
        assert np.array_equal(pw[:, 2], pos[:, 2]) and np.array_equal(want[nw - R], neg)
        e.shard_post(uniq, cuts, world, k, cap, pa(inbox), pa(meta))
        for o in range(world):
            lo, hi = cuts_h[o], cuts_h[o + 1]
            got = inbox[o][k].cpu().numpy()
            assert np.array_equal(got[:hi - lo], want[lo:hi]) and (got[hi - lo:] == -7).all()
            assert meta[o][k].tolist() == [hi - lo, lo]


class _VirtualRanks:
    """`world` ranks of the row-sharded step on ONE GPU: one engine (library context) per rank, every
    "peer" buffer a local tensor.  A step runs its compute half on every rank, then its apply half on
    every rank, all on one stream -- so every flag a kernel waits for has been set by an earlier
    kernel of the stream.  csr: the (offsets, ids) type table corruption draws from (default: built from
    kg.type_of).  Trailing ranks may own no rows (e.g. 20 entities over 16 ranks)."""

    def __init__(self, eng_mod, kg, world, B, csr=None):
        from graphembeddings_b200.sharded import row_partition
        self.world, self.B, self.R, self.n_rows = world, B, kg.n_relations, kg.n_rows
        off, ids = D.build_type_csr(kg.type_of) if csr is None else csr
        self.rows_per = row_partition(kg.n_entities, world)
        self.engs, self.bufs = [], []
        for k in range(world):
            e = eng_mod.HoleEngine(kg.n_relations + 3 * B, kg.dim).set_types(kg.type_of, off, ids)
            e.set_relation_count(kg.n_relations)
            dev, w, cap = e.device, e.row_stride, 3 * B
            shard = torch.zeros((self.R + self.rows_per, w), dtype=torch.float32, device=dev)
            b0, b1 = self._block(k)
            full = eng_mod.HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E)
            shard[: self.R] = full.table[: self.R]
            shard[self.R: self.R + (b1 - b0)] = full.table[b0:b1]
            full.close()
            self.bufs.append([shard,
                              torch.zeros((world, cap, w), dtype=torch.float32, device=dev),
                              torch.zeros((world, max(self.R, 1), w), dtype=torch.float32, device=dev),
                              torch.zeros((2, world, cap), dtype=torch.int32, device=dev),
                              torch.zeros((2, world, 2), dtype=torch.int32, device=dev),
                              torch.zeros((2, world), dtype=torch.int32, device=dev),
                              torch.zeros(1, dtype=torch.int32, device=dev)])
            self.engs.append(e)
        for k, e in enumerate(self.engs):
            pa = e.peer_array
            e.shard_init(world, k, self.R, kg.n_entities, self.rows_per, B, self.bufs[k][0],
                         *[pa([self.bufs[j][i] for j in range(world)]) for i in range(6)], self.bufs[k][6], 5.0)
        self.kg = kg

    def _block(self, k):
        """[b0, b1): the global rows rank k owns (empty for a trailing rank past the last entity)."""
        b0 = self.R + k * self.rows_per
        return b0, max(b0, min(self.n_rows, b0 + self.rows_per))

    def step(self, slices, seed, step, margin, lr, ahead=None):
        losses = []
        for k, e in enumerate(self.engs):
            if ahead is not None:
                e.shard_prepare(ahead[k], seed, step + 1)
            losses.append(e.shard_step(slices[k], seed, step, margin, lr, phase="compute"))
        for e in self.engs:
            e.shard_step(None, seed, step, margin, lr, phase="apply")
        return losses

    def table(self):
        """[N, dim] gathered from the shards; also checks that the relation replicas are bit-identical."""
        kg = self.kg
        rel = self.bufs[0][0][: self.R]
        ents = []
        for k in range(self.world):
            assert torch.equal(self.bufs[k][0][: self.R], rel)
            assert not self.engs[k].shard_poll()
            b0, b1 = self._block(k)
            ents.append(self.bufs[k][0][self.R: self.R + (b1 - b0)])
        tab = torch.cat([rel] + ents)
        tmp = self.engs[0].__class__(kg.n_rows, kg.dim)
        tmp.table = tab.contiguous()
        out = tmp.embeddings().cpu().numpy()
        tmp.table = None
        tmp.close()
        return out


@pytest.mark.parametrize("world,dim,B", [(1, 150, 300), (2, 256, 257), (3, 150, 129), (4, 64, 200), (8, 150, 65),
                                         (2, 512, 96)])
def test_sharded_step_virtual_ranks_matches_single_gpu(eng_mod, world, dim, B):
    """hole_shard_step (rows gathered from the owners' shards and deltas staged at the owners by the
    training kernel itself) with `world` virtual ranks against the single-GPU step on the concatenated
    global batch: identical corruption (global triple index), loss <= 2e-6, table <= 2e-6 after 3
    chained steps; heavy cross-rank duplicates (Zipf entities), ragged B, d not a multiple of 8."""
    steps = 3
    kg = D.synthetic_kg(7, 2000, steps * world * B, 5, dim, seed=500 + world, trained_scale=True, zipf_entities=True)
    vr = _VirtualRanks(eng_mod, kg, world, B)
    e, off, ids = _engine(eng_mod, kg)
    dev = e.device
    tri = torch.from_numpy(kg.triples).to(dev).view(steps, world, B, 3)
    for s in range(steps):
        slices = [tri[s, k].contiguous() for k in range(world)]
        ahead = [tri[s + 1, k].contiguous() for k in range(world)] if s + 1 < steps and s % 2 == 0 else None
        if ahead is not None:
            keep_ahead = ahead
        if s > 0 and s % 2 == 1:
            slices = keep_ahead                  # the tensors the step was prepared for
        losses = vr.step(slices, 11, s, 0.2, 0.1, ahead)
        gb = kg.triples[s * world * B:(s + 1) * world * B]
        side, neg = e.corrupt_batch(gb, 11, s)
        want = e.train_step(gb, neg, side, 0.2, 0.1).cpu().numpy().reshape(world, B)
        for k in range(world):
            assert np.abs(losses[k].cpu().numpy() - want[k]).max() <= 2e-6
    got = vr.table()
    ref = e.embeddings().cpu().numpy()
    assert np.abs(got - ref).max() <= 2e-6
    assert np.abs(ref - kg.E).max() > 1e-4


def test_sharded_steps_call_matches_step_by_step(eng_mod):
    """hole_shard_steps (the multi-step entry, one step prepared ahead) == hole_shard_step called per
    step, bit for bit, and its loss sums are the sums of the per-triple losses (world = 1)."""
    B, steps, dim = 500, 6, 150
    kg = D.synthetic_kg(7, 3000, steps * B, 5, dim, seed=61, trained_scale=True, zipf_entities=True)
    lrs = [0.1 / (1 + s) for s in range(steps)]
    a, b = _VirtualRanks(eng_mod, kg, 1, B), _VirtualRanks(eng_mod, kg, 1, B)
    tri = torch.from_numpy(kg.triples).to(a.engs[0].device)
    sums = a.engs[0].shard_steps(tri, B, 3, 10, 0.2, lrs).cpu().numpy()
    want = []
    for s in range(steps):
        loss = b.step([tri[s * B:(s + 1) * B]], 3, 10 + s, 0.2, lrs[s])[0]
        want.append(float(loss.double().sum()))
    assert np.abs(sums - np.array(want)).max() <= 1e-3
    assert np.array_equal(a.table(), b.table())
    host = _VirtualRanks(eng_mod, kg, 1, B)
    hs = host.engs[0].shard_steps_host(kg.triples, B, 3, 10, 0.2, lrs)
    assert np.array_equal(hs, sums) and np.array_equal(host.table(), a.table())


def test_delta_mode_writes_every_used_row(eng_mod):
    """hole_train_step_ex in delta mode must overwrite (not accumulate into) every row the
    step uses, zeros included for inactive hinges: the sharded trainer does not clear D."""
    kg = D.synthetic_kg(6, 3000, 600, 4, 150, seed=43, trained_scale=True)
    e, _, _ = _engine(eng_mod, kg)
    pos = torch.from_numpy(kg.triples[:600]).to(e.device)
    side, neg = e.corrupt_batch(pos, 9, 0)
    before = e.table.clone()
    e.train_step_plan(pos, neg)
    junk = torch.full_like(e.table, 7.0)
    e.train_step_delta(pos, neg, side, 0.0, 0.1, junk)           # margin 0: about half the hinges inactive
    e.train_step_plan(pos, neg)
    clean = torch.zeros_like(e.table)
    loss = e.train_step_delta(pos, neg, side, 0.0, 0.1, clean)
    assert torch.equal(e.table, before)
    used = torch.unique(torch.cat([pos[:, 0], pos[:, 1], pos[:, 2], neg.to(pos.dtype)]).long())
    assert torch.equal(junk[used], clean[used])
    assert (loss == 0).any() and (loss > 0).any()
    mask = torch.ones(e.table.shape[0], dtype=torch.bool, device=e.device)
    mask[used] = False
    assert (junk[mask] == 7.0).all()


def test_full_size_properties_config1(eng_mod):
    """BASELINE config 1 at full table size (1,200,014 x 256), B = 32768: determinism across
    runs, rows untouched by any step bit-identical, loss sums finite and equal between the
    device-resident and the host-buffer entry points."""
    kg = D.make_config("diffbot_d256", n_triples=32768 * 6)
    B, n_steps = 32768, 6
    lrs = [0.1] * n_steps
    off, ids = D.build_type_csr(kg.type_of)
    outs = []
    for mode in ("device", "device", "host"):
        e = eng_mod.HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E).set_types(kg.type_of, off, ids)
        e.set_relation_count(kg.n_relations)
        if mode == "device":
            sums = e.train_steps(kg.triples, B, 11, 0, 0.2, lrs).cpu().numpy()
        else:
            sums = e.train_steps_host(kg.triples, B, 11, 0, 0.2, lrs)
        outs.append((sums, e.embeddings().cpu()))
        e.close()
    assert np.array_equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    assert np.array_equal(outs[0][0], outs[2][0]) and torch.equal(outs[0][1], outs[2][1])
    assert np.isfinite(outs[0][0]).all() and np.all(np.abs(outs[0][0] / B - 0.2) < 0.01)
    E0 = torch.from_numpy(kg.E)
    changed = (outs[0][1] != E0).any(dim=1)
    used = torch.zeros(kg.n_rows, dtype=torch.bool)
    used[torch.from_numpy(kg.triples.reshape(-1).astype(np.int64))] = True
    # every changed row was used by a triple or drawn as a corrupt entity (same type => entity row)
    assert not bool(changed[: kg.n_relations][~used[: kg.n_relations]].any())
    assert int(changed.sum()) > 3 * B          # most touched rows really moved


@pytest.mark.parametrize("case", ["few_duplicates", "relation_hint", "all_duplicates"])
def test_update_plan_paths_give_identical_tables(eng_mod, monkeypatch, case):
    """The one-launch plan kernels (relation sort, row sort + segments: one block per step, shared memory) produce
    the plan of the multi-launch radix chain: training through either gives the same table bit for bit.
    HOLE_SORT_SMALL is read when a context is created: 0 = radix chain only, 1 = adaptive (radix chain in the
    first call, one-launch kernels from the second call on while the steps fit), 2 = one-launch row sort always
    (all_duplicates: 16,000 duplicated uses per step do not fit its shared memory -- its global-memory path)."""
    if case == "all_duplicates":
        kg = D.synthetic_kg(3, 60, 4000 * 4, 2, 64, seed=5, trained_scale=True, zipf_entities=True)
        B, calls, per_call = 4000, 2, 2
    else:
        kg = D.synthetic_kg(9, 50000, 3000 * 6, 4, 150, seed=6, trained_scale=True)
        B, calls, per_call = 3000, 3, 2
    outs = []
    for mode in ("0", "1", "2"):
        monkeypatch.setenv("HOLE_SORT_SMALL", mode)
        e, _, _ = _engine(eng_mod, kg)
        if case == "relation_hint":
            e.set_relation_count(kg.n_relations)          # one 8-bit pass in the relation sort
        sums = []
        for c in range(calls):
            k0 = c * per_call
            tri = kg.triples[k0 * B:(k0 + per_call) * B]
            sums.append(e.train_steps(tri, B, 3, k0, 0.2, [0.1] * per_call).cpu().numpy())
        outs.append((np.concatenate(sums), e.embeddings().cpu()))
        e.close()
    monkeypatch.delenv("HOLE_SORT_SMALL")
    for sums, table in outs[1:]:
        assert np.array_equal(sums, outs[0][0]) and torch.equal(table, outs[0][1])
    assert not torch.equal(outs[0][1], torch.from_numpy(kg.E))
