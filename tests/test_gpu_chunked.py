"""The multi-step training calls across their chunk boundaries.

hole_train_steps[_host] cut a call into plan chunks (plan_chunk / chunk_sizes in csrc/hole_train.cu): each
chunk's update plan is built on a side stream into one of two plan slots while the previous chunk trains, the
host path also stages the triples in one of two buffers, and every chunk carries its own offsets into the
learning rates, the Philox step, the per-triple losses and the loss sums.  hole_shard_steps[_host] prepare
16 steps at a time (SHARD_PREP_STEPS) and sum losses in 64-step blocks (SHARD_LOSS_CHUNK, csrc/hole_shard.cuh).

Reference method, used for every multi-step call below:
  1. bit-exact against the per-step path: a second engine on the same table takes the same steps one at a
     time (train_step with corrupt_batch(pos, seed, first_step + k) and lr[k]); tables and per-triple losses
     must be identical, loss sums within 1e-3 of the fp64 sums of those losses.  Both paths use the same
     plan (the sorts are bit-identical), the same triples per K1 lane group (a function of B and the
     context) and the same corruption, so nothing but a chunking fault can make them differ;
  2. re-synchronised oracle check: at the first and last step and on both sides of every chunk boundary,
     the per-step engine's table before step k goes through the fp32 C port (oracle/hole_ref.c) and the
     result is held to the one-step band (rows 2e-6 + 1e-5 |x|, loss 2e-6) of the table after step k.
     With 1. this pins the multi-step call to the oracle at every boundary without a band that grows with
     the step count.
The learning rate changes at every step and first_step != 0, so an offset that is off by a chunk changes
the result.
"""
import numpy as np
import pytest
import torch

from graphembeddings_b200 import data as D
from oracle import hole_oracle as O
from oracle import hole_ref as R

pytestmark = pytest.mark.gpu

ROW_ATOL, ROW_RTOL, LOSS_ATOL = 2e-6, 1e-5, 2e-6      # one step against the oracle
SUM_ATOL = 1e-3                                        # a step's loss sum against the fp64 sum of its losses
MARGIN = 0.2
SS_CAP = 11264                   # duplicated row uses the one-launch row sort keeps in shared memory (hole_train.cu)
SHARD_PREP_STEPS, SHARD_LOSS_CHUNK = 16, 64            # csrc/hole_shard.cuh
ENV_KEYS = ("HOLE_PLAN_RAMP", "HOLE_HOST_FIRST", "HOLE_SORT_SMALL")


@pytest.fixture(scope="module")
def eng_mod():
    from graphembeddings_b200 import build
    build.build()
    from graphembeddings_b200 import engine
    return engine


# ---------------------------------------------------------------- chunk layout (mirror of hole_train.cu)
def plan_chunk(B):
    """Mirror of plan_chunk() in csrc/hole_train.cu: steps per planned chunk."""
    return max(32, min(256, (1 << 23) // (4 * B)))


def chunk_sizes(B, n_steps, ramp=None, host_first=0, from_host=False):
    """Mirror of chunk_sizes() in csrc/hole_train.cu.  ramp: (first, factor) of HOLE_PLAN_RAMP, host_first:
    HOLE_HOST_FIRST (only read by the host-buffer entry, and ignored while a ramp is set)."""
    S = plan_chunk(B)
    ramp_first, ramp_factor = ramp if ramp else (0, 4)
    first = ramp_first
    if from_host and first <= 0 and host_first > 0 and n_steps > 2 * host_first:
        first = host_first
    cur = min(S, first) if first > 0 else S
    sizes, left = [], n_steps
    while left > 0:
        n = min(cur, left)
        sizes.append(n)
        left -= n
        cur = S if (from_host and ramp_first <= 0) else min(S, cur * max(2, ramp_factor))
    return sizes


def boundary_steps(sizes):
    """First and last step, and the steps on both sides of every chunk boundary."""
    starts = np.cumsum([0] + list(sizes))
    out = {0, int(starts[-1]) - 1}
    for k in starts[1:-1]:
        out.update((int(k) - 1, int(k)))
    return sorted(out)


def test_chunk_layout_mirror():
    """The layouts the tests below rely on (the mirror itself runs on the CPU)."""
    assert plan_chunk(64) == 256 and plan_chunk(8192) == 256
    assert plan_chunk(16384) == 128 and plan_chunk(32768) == 64 and plan_chunk(65536) == 32
    assert chunk_sizes(64, 600) == [256, 256, 88]
    assert chunk_sizes(16384, 300) == [128, 128, 44]
    assert chunk_sizes(32768, 140) == [64, 64, 12]
    assert chunk_sizes(1000, 40, ramp=(1, 2)) == [1, 2, 4, 8, 16, 9]
    assert chunk_sizes(1000, 40, ramp=(3, 3)) == [3, 9, 27, 1]
    assert chunk_sizes(1000, 40, host_first=4, from_host=True) == [4, 36]
    assert chunk_sizes(1000, 40, host_first=4) == [40]                          # the device entry ignores it
    assert chunk_sizes(1000, 40, ramp=(3, 3), host_first=4, from_host=True) == [3, 9, 27, 1]
    assert boundary_steps([3, 9, 27, 1]) == [0, 2, 3, 11, 12, 38, 39]


# ---------------------------------------------------------------- helpers
def _set_env(monkeypatch, env):
    for k in ENV_KEYS:
        monkeypatch.delenv(k, raising=False)
    for k, v in (env or {}).items():
        monkeypatch.setenv(k, str(v))


def _engine(eng_mod, monkeypatch, kg, env=None, n_rel_hint=None):
    """A context created under exactly `env` (the switches are read by hole_ctx_create)."""
    _set_env(monkeypatch, env)
    off, ids = D.build_type_csr(kg.type_of)
    e = eng_mod.HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E).set_types(kg.type_of, off, ids)
    if n_rel_hint is not None:
        e.set_relation_count(n_rel_hint)
    _set_env(monkeypatch, None)
    return e


def _lrs(eng_mod, first_step, n_steps):
    """A learning rate that changes at every step (inverse time decay over 8 steps)."""
    return np.array([eng_mod.inverse_time_decay(0.1, first_step + k, 8, 0.5) for k in range(n_steps)], np.float32)


def _oracle_step(k, before, pos, neg, side, lr, loss, after):
    """One step of the fp32 C port from the engine's table `before`, held to the one-step band."""
    E = np.ascontiguousarray(before, np.float32)
    _, want = R.train_step(E, pos, neg, side, MARGIN, float(lr))
    assert np.abs(loss - want).max() <= LOSS_ATOL, (k, float(np.abs(loss - want).max()))
    err, tol = np.abs(after - E), ROW_ATOL + ROW_RTOL * np.abs(E)
    assert (err <= tol).all(), (k, float((err - tol).max()))


def _per_step(eng, tri, B, seed, first_step, lrs, check_at=()):
    """The per-step path: corrupt_batch + train_step one step at a time.  At the steps in check_at, the
    step is also re-run by the oracle from this engine's table.  Returns the per-triple losses [n*B]."""
    n = tri.shape[0] // B
    losses, check_at = [], set(check_at)
    for k in range(n):
        pos = tri[k * B:(k + 1) * B]
        side, neg = eng.corrupt_batch(pos, seed, first_step + k)
        before = eng.embeddings().cpu().numpy() if k in check_at else None
        loss = eng.train_step(pos, neg, side, MARGIN, lrs[k])
        if before is not None:
            _oracle_step(first_step + k, before, pos.cpu().numpy(), neg.cpu().numpy(), side, lrs[k],
                         loss.cpu().numpy(), eng.embeddings().cpu().numpy())
        losses.append(loss)
    return torch.cat(losses)


def _fp64_sums(loss, B):
    return loss.double().view(-1, B).sum(1).cpu().numpy()


def _assert_matches_per_step(tag, table, ref_table, sums, ref_loss, B, loss=None):
    assert torch.equal(table, ref_table), f"{tag}: table differs from the per-step path"
    if loss is not None:
        assert torch.equal(loss, ref_loss), f"{tag}: per-triple losses differ from the per-step path"
    s = sums.cpu().numpy() if isinstance(sums, torch.Tensor) else np.asarray(sums)
    err = np.abs(s - _fp64_sums(ref_loss, B))
    assert err.max() <= SUM_ATOL, (tag, int(err.argmax()), float(err.max()))


# ---------------------------------------------------------------- 1. natural chunk boundaries
@pytest.mark.parametrize("B,dim,n_steps,n_ent,layout", [
    (64, 150, 600, 5000, [256, 256, 88]),
    (16384, 64, 300, 50000, [128, 128, 44]),
    (32768, 256, 140, 200000, [64, 64, 12]),
])
def test_natural_chunks_match_per_step_and_oracle(eng_mod, monkeypatch, B, dim, n_steps, n_ent, layout):
    """hole_train_steps (device loop) over 3 natural plan chunks, the last one ragged: B = 64 -> 256, 256, 88;
    B = 16384 -> 128, 128, 44; B = 32768 -> 64, 64, 12 (trained-scale rows, so the clip fires, and Zipf
    entities: hot rows used thousands of times a step).  Both plan slots are used, slot 0 twice."""
    assert chunk_sizes(B, n_steps) == layout and len(layout) == 3 and layout[-1] < layout[0]
    kg = D.synthetic_kg(14, n_ent, n_steps * B, 6, dim, seed=B + dim, trained_scale=True, zipf_entities=True)
    seed, first_step = 0x5EED + B, 1000 + B
    lrs = _lrs(eng_mod, first_step, n_steps)
    a = _engine(eng_mod, monkeypatch, kg)
    tri = torch.from_numpy(kg.triples).to(a.device)
    sums, loss = a.train_steps(tri, B, seed, first_step, MARGIN, lrs, want_loss=True)
    b = _engine(eng_mod, monkeypatch, kg)
    ref = _per_step(b, tri, B, seed, first_step, lrs, check_at=boundary_steps(layout))
    _assert_matches_per_step(f"B={B}", a.table, b.table, sums, ref, B, loss)
    assert not torch.equal(a.embeddings().cpu(), torch.from_numpy(kg.E))
    a.close(); b.close()


# ---------------------------------------------------------------- 2. ramped chunks and the host path
VARIANTS = [   # (entry, HOLE_PLAN_RAMP, HOLE_HOST_FIRST, chunk layout of 40 steps at B = 1000)
    ("device", (1, 2), 0, [1, 2, 4, 8, 16, 9]),
    ("device", (3, 3), 0, [3, 9, 27, 1]),
    ("host", (1, 2), 0, [1, 2, 4, 8, 16, 9]),
    ("host", (3, 3), 0, [3, 9, 27, 1]),
    ("host", None, 4, [4, 36]),
    ("host", (3, 3), 4, [3, 9, 27, 1]),
]


@pytest.mark.parametrize("entry,ramp,host_first,layout", VARIANTS)
def test_ramped_chunks_and_host_path(eng_mod, monkeypatch, entry, ramp, host_first, layout):
    """40 steps at B = 1000 cut by HOLE_PLAN_RAMP / HOLE_HOST_FIRST into many small chunks: 1,2,4,8,16,9
    (6 chunks: each plan slot and staging buffer used 3 times) and 3,9,27,1 (4 chunks: each used twice);
    HOLE_HOST_FIRST=4 without a ramp gives the host entry 4, 36, and is ignored while a ramp is set.
    hole_train_steps and hole_train_steps_host must equal the per-step path and the same call made with no
    switch set (one chunk of 40) bit for bit: tables, and loss sums (the host entry returns them per step)."""
    B, n_steps, dim = 1000, 40, 150
    from_host = entry == "host"
    assert chunk_sizes(B, n_steps, ramp, host_first, from_host) == layout and len(layout) > 1
    assert chunk_sizes(B, n_steps, None, 0, from_host) == [40]
    env = {}
    if ramp:
        env["HOLE_PLAN_RAMP"] = "%d,%d" % ramp
    if host_first:
        env["HOLE_HOST_FIRST"] = host_first
    kg = D.synthetic_kg(9, 20000, n_steps * B, 5, dim, seed=3 + len(layout), trained_scale=True, zipf_entities=True)
    seed, first_step = 77, 333
    lrs = _lrs(eng_mod, first_step, n_steps)

    def run(env):
        e = _engine(eng_mod, monkeypatch, kg, env)
        if from_host:
            sums, loss = e.train_steps_host(kg.triples, B, seed, first_step, MARGIN, lrs), None
        else:
            sums, loss = e.train_steps(kg.triples, B, seed, first_step, MARGIN, lrs, want_loss=True)
            sums = sums.cpu().numpy()
        return e, sums, loss

    a, sums, loss = run(env)
    plain, sums0, loss0 = run(None)
    b = _engine(eng_mod, monkeypatch, kg)
    ref = _per_step(b, torch.from_numpy(kg.triples).to(b.device), B, seed, first_step, lrs,
                    check_at=boundary_steps(layout))
    _assert_matches_per_step(f"{entry} {env}", a.table, b.table, sums, ref, B, loss)
    _assert_matches_per_step(f"{entry} plain", plain.table, b.table, sums0, ref, B, loss0)
    assert np.array_equal(sums, sums0)
    a.close(); plain.close(); b.close()


# ---------------------------------------------------------------- 3. adaptive plan sort inside a call
def _dup_uses(pos, neg):
    """Uses of entity rows that the step uses more than once (of its 3B entity uses)."""
    _, cnt = np.unique(np.concatenate([pos[:, 0], pos[:, 1], neg]), return_counts=True)
    return int(cnt[cnt > 1].sum())


def test_adaptive_plan_sort_switches_inside_a_call(eng_mod, monkeypatch):
    """HOLE_SORT_SMALL=1 picks the one-launch row sort while the last plan of each slot had at most SS_CAP
    duplicated row uses, reading the counts the plans report without waiting, so the choice can change
    between the chunks of one call.  B = 4096 (4B = 16,384 uses a step): steps [0, 16) and [28, 56) draw
    from 100,000 entities (few duplicates), steps [16, 28) from a type of 40 entities (heads, tails and
    corrupt entities all duplicated: 3B > SS_CAP).  A first call of 8 steps (chunks 1, 2, 4, 1) lets the
    plans report small steps; the second call of 48 steps has chunks 1, 2, 4, 8, 16, 17 and crosses both
    ways.  Radix chain only (0), adaptive (1) and one launch always (2) give the same tables and loss sums
    bit for bit, equal to the per-step path."""
    B, dim, n_rel, n_hub, n_spread = 4096, 64, 8, 40, 100000
    warm, n_steps, heavy = 8, 48, range(16, 28)
    assert chunk_sizes(B, warm, (1, 2)) == [1, 2, 4, 1]
    layout = chunk_sizes(B, n_steps, (1, 2))
    assert layout == [1, 2, 4, 8, 16, 17]
    total = warm + n_steps
    rng = np.random.default_rng(12)
    type_of = np.concatenate([np.zeros(n_rel), np.ones(n_hub), np.full(n_spread, 2)]).astype(np.int32)
    hub0, spread0 = n_rel, n_rel + n_hub
    tri = np.empty((total * B, 3), np.int32)
    tri[:, 2] = rng.integers(0, n_rel, total * B)
    for k in range(total):
        lo, hi = (hub0, hub0 + n_hub) if k in heavy else (spread0, spread0 + n_spread)
        tri[k * B:(k + 1) * B, :2] = rng.integers(lo, hi, (B, 2))
    E = D.init_embeddings(len(type_of), dim, rng, trained_scale=True)
    kg = D.SyntheticKG(n_rel, n_hub + n_spread, dim, tri, type_of, E)
    seed, first_step = 2024, 4000
    off, ids = D.build_type_csr(type_of)
    # the construction, checked: duplicated uses per step from the triples and the oracle's corruption
    # (relation keys add at most B more)
    dups = [_dup_uses(tri[k * B:(k + 1) * B], O.corrupt(tri[k * B:(k + 1) * B], type_of, off, ids, seed,
                                                        first_step + k)[1]) for k in range(total)]
    big = [d > SS_CAP for d in dups]
    assert all(big[k] for k in heavy)
    assert all(dups[k] + B <= SS_CAP for k in range(total) if k not in heavy)
    crossings = [k for k in range(warm + 1, total) if big[k] != big[k - 1]]
    assert crossings == [16, 28]
    lrs = _lrs(eng_mod, first_step, total)
    outs = []
    for mode in ("0", "1", "2"):
        e = _engine(eng_mod, monkeypatch, kg, {"HOLE_PLAN_RAMP": "1,2", "HOLE_SORT_SMALL": mode})
        t = torch.from_numpy(tri).to(e.device)
        s0, l0 = e.train_steps(t[:warm * B], B, seed, first_step, MARGIN, lrs[:warm], want_loss=True)
        s1, l1 = e.train_steps(t[warm * B:], B, seed, first_step + warm, MARGIN, lrs[warm:], want_loss=True)
        outs.append((mode, e, torch.cat([s0, s1]), torch.cat([l0, l1])))
    b = _engine(eng_mod, monkeypatch, kg)
    check = sorted({0, warm - 1} | {warm + k for k in boundary_steps(layout)} | {15, 16, 27, 28})
    ref = _per_step(b, torch.from_numpy(tri).to(b.device), B, seed, first_step, lrs, check_at=check)
    for mode, e, sums, loss in outs:
        _assert_matches_per_step(f"HOLE_SORT_SMALL={mode}", e.table, b.table, sums, ref, B, loss)
        assert torch.equal(sums, outs[0][2])
        e.close()
    b.close()


# ---------------------------------------------------------------- 4. sharded multi-step
@pytest.mark.parametrize("n_steps", [70, 130])
def test_sharded_steps_across_prep_and_loss_chunks(eng_mod, n_steps):
    """hole_shard_steps[_host] with one virtual rank, B = 97: 70 steps = prep chunks of 16 x 4 + 6 and loss
    blocks 64 + 6; 130 steps = 16 x 8 + 2 and 64 + 64 + 2 (the last block ragged in both).  Both entries
    equal a hole_shard_step loop bit for bit, with lr and step changing at every step; their loss sums match
    the per-step sums block by block; against the single-GPU hole_train_steps on the same batches the table
    stays within the virtual-rank test's per-step band times the step count.
    (A wrong offset in the preparation would only cost overlap: hole_shard_step prepares a step again when
    the prepared chunk does not match its (pos, seed, step).  Multi-rank calls of hole_shard_steps need one
    GPU per rank -- tests/test_gpu_multi.py.)"""
    from test_gpu_train import _VirtualRanks
    B, dim = 97, 150
    n_prep = -(-n_steps // SHARD_PREP_STEPS)
    blocks = [(l0, min(n_steps, l0 + SHARD_LOSS_CHUNK)) for l0 in range(0, n_steps, SHARD_LOSS_CHUNK)]
    assert n_prep * SHARD_PREP_STEPS > n_steps and len(blocks) >= 2 and blocks[-1][1] - blocks[-1][0] < 64
    kg = D.synthetic_kg(7, 3000, n_steps * B, 5, dim, seed=n_steps, trained_scale=True, zipf_entities=True)
    seed, first_step = 3, 500
    lrs = _lrs(eng_mod, first_step, n_steps)
    a, b, h = (_VirtualRanks(eng_mod, kg, 1, B) for _ in range(3))
    tri = torch.from_numpy(kg.triples).to(a.engs[0].device)
    sums = a.engs[0].shard_steps(tri, B, seed, first_step, MARGIN, lrs).cpu().numpy()
    hs = h.engs[0].shard_steps_host(kg.triples, B, seed, first_step, MARGIN, lrs)
    per = []
    for k in range(n_steps):
        loss = b.step([tri[k * B:(k + 1) * B]], seed, first_step + k, MARGIN, float(lrs[k]))[0]
        per.append(float(loss.double().sum()))
    per = np.array(per)
    ref = b.table()
    assert np.array_equal(a.table(), ref) and np.array_equal(h.table(), ref)
    for l0, l1 in blocks:
        err = np.abs(sums[l0:l1] - per[l0:l1])
        assert err.max() <= SUM_ATOL, ("loss block", l0, int(err.argmax()) + l0, float(err.max()))
    assert np.array_equal(hs, sums)
    # the single-GPU engine on the same batches
    e = eng_mod.HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E)
    off, ids = D.build_type_csr(kg.type_of)
    e.set_types(kg.type_of, off, ids)
    s1 = e.train_steps(tri, B, seed, first_step, MARGIN, lrs).cpu().numpy()
    assert np.abs(s1 - sums).max() <= SUM_ATOL
    single = e.embeddings().cpu().numpy()
    assert np.abs(single - ref).max() <= n_steps * 2e-6
    assert np.abs(ref - kg.E).max() > 1e-4
    e.close()


# ---------------------------------------------------------------- 5. a broken relation-count hint
@pytest.mark.parametrize("sort_small", ["0", "1"])
@pytest.mark.parametrize("hint", [4, 200, 300])
def test_relation_ids_above_the_hint_are_trained_right(eng_mod, monkeypatch, hint, sort_small):
    """include/hole_b200.h: a relation id >= the hole_ctx_set_relations hint is grouped with other relations,
    never mis-trained.  300 relations (ids above 255) under hints of 4 (HOLE_SORT_SMALL=1: the counting sort
    clamps ids to 3), 200 (one 8-bit pass on ids that need two) and 300 (honest, the control).  One step
    stays within the one-step band of the fp64 oracle; a call of 12 steps in chunks 1, 2, 4, 5 (HOLE_PLAN_RAMP
    =1,2) equals the per-step path bit for bit and passes the boundary oracle checks.  The grouping changes
    the order in which relation gradients are summed, so results are not compared across hints."""
    B, dim, n_rel, n_steps = 2000, 150, 300, 12
    layout = chunk_sizes(B, n_steps, (1, 2))
    assert layout == [1, 2, 4, 5]
    kg = D.synthetic_kg(n_rel, 4000, (n_steps + 1) * B, 5, dim, seed=hint, trained_scale=True, zipf_entities=True)
    kg.triples[::5, 2] = 256 + np.arange(len(kg.triples[::5])) % (n_rel - 256)      # every batch has ids > 255
    for k in range(n_steps + 1):
        r = kg.triples[k * B:(k + 1) * B, 2]
        assert (r > 255).sum() >= B // 5 and (r < 256).sum() > B // 2 and r.max() < n_rel
        assert hint == n_rel or (r >= hint).any()
    env = {"HOLE_SORT_SMALL": sort_small}
    # one step against the fp64 oracle
    e = _engine(eng_mod, monkeypatch, kg, env, n_rel_hint=hint)
    off, ids = D.build_type_csr(kg.type_of)
    pos = kg.triples[n_steps * B:]
    side, neg = O.corrupt(pos, kg.type_of, off, ids, 5, 9)
    loss = e.train_step(pos, neg, side, MARGIN, 0.1).cpu().numpy()
    E64 = kg.E.astype(np.float64)
    want, _, _ = O.sgd_step(E64, pos, neg, side, MARGIN, 0.1, np.float64, "tf")
    assert np.abs(loss - want).max() <= LOSS_ATOL
    got = e.embeddings().cpu().numpy()
    err, tol = np.abs(got - E64), ROW_ATOL + ROW_RTOL * np.abs(E64)
    assert (err <= tol).all(), float((err - tol).max())
    moved = np.abs(got - kg.E).max(axis=1) > 0
    assert moved[256:n_rel].any()                        # relations above 255 were trained
    e.close()
    # a multi-chunk call
    seed, first_step = 41, 7000
    lrs = _lrs(eng_mod, first_step, n_steps)
    tri = torch.from_numpy(kg.triples[:n_steps * B].copy())
    a = _engine(eng_mod, monkeypatch, kg, dict(env, HOLE_PLAN_RAMP="1,2"), n_rel_hint=hint)
    sums, loss = a.train_steps(tri, B, seed, first_step, MARGIN, lrs, want_loss=True)
    b = _engine(eng_mod, monkeypatch, kg, env, n_rel_hint=hint)
    ref = _per_step(b, tri.to(b.device), B, seed, first_step, lrs, check_at=boundary_steps(layout))
    _assert_matches_per_step(f"hint {hint}", a.table, b.table, sums, ref, B, loss)
    a.close(); b.close()
