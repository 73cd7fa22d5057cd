"""Type-constrained ranking and top-k (hole_rank_typed / hole_topk_typed) checked EXACTLY against the all-candidate
calls.

Restricting query q to the entities of its type tau_q is the all-candidate call with every entity of another type
filtered out, so, with C(q) = the entity rows outside tau_q:
    raw_typed  == filt of hole_rank over the entity range with filter C(q)
    filt_typed == filt of the same call with filter C(q) | known(q)
    true_score is bit-identical (both from the diagonal pass over the same packed rows)
    topk_typed == hole_topk with filter C(q) | known(q), ids and scores bit for bit.
That rests on the assumption test_gpu_rank_filter.py already makes: a candidate's tensor-core score does not
depend on its column (nor, here, a query's on its row).
"""
import ctypes as C

import numpy as np
import pytest
import torch

from graphembeddings_b200 import data as D

pytestmark = pytest.mark.gpu

TAIL, HEAD, BOTH, REL = 0, 1, 2, 3
BF16, BF16X3 = 0, 1


@pytest.fixture(scope="module")
def eng_mod():
    from graphembeddings_b200 import build
    build.build()
    from graphembeddings_b200 import engine
    return engine


def _types_from_hist(rng, n_rel, hist):
    """type_of over all rows: relations are type 0, the entities are shuffled into types 1.. of the given sizes."""
    ent = np.repeat(np.arange(1, len(hist) + 1), hist)
    rng.shuffle(ent)
    type_of = np.concatenate([np.zeros(n_rel, dtype=np.int64), ent]).astype(np.int32)
    off, ids = D.build_type_csr(type_of, len(hist) + 1)
    return type_of, off, ids


def _setup(eng_mod, n_rel, hist, dim=64, seed=0, mode="complex"):
    rng = np.random.default_rng(seed)
    n_ent = int(np.sum(hist))
    kg = D.synthetic_kg(n_rel, n_ent, 8, 4, dim, seed=seed, trained_scale=True)
    type_of, off, ids = _types_from_hist(rng, n_rel, hist)
    eng = eng_mod.HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E).set_types(type_of, off, ids)
    eng.set_score_mode(mode)
    return kg, eng, rng, type_of, off, ids


def _queries(rng, n_rel, n_rows, Q):
    h = rng.integers(n_rel, n_rows, size=Q)
    t = rng.integers(n_rel, n_rows, size=Q)
    r = rng.integers(0, n_rel, size=Q)
    return np.stack([h, t, r], axis=1).astype(np.int32)


def _known(rng, queries, side, n_rel, n_rows, type_of):
    """Per query: a few random entities of any type, now and then the true id itself, ascending."""
    out = []
    for q in queries:
        true = int(q[1] if side == TAIL else q[0])
        s = set(int(x) for x in rng.integers(n_rel, n_rows, size=int(rng.integers(0, 7))))
        same = np.flatnonzero(type_of == type_of[true])
        s |= set(int(x) for x in rng.choice(same, size=min(3, len(same)), replace=False))
        if rng.random() < 0.3:
            s.add(true)
        out.append(sorted(s))
    return out


def _csr(slices):
    off = np.zeros(len(slices) + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(s) for s in slices])
    ids = np.array([x for s in slices for x in s], dtype=np.int32)
    return off, ids


def _complement(tau, type_of, n_rel, extra=()):
    """Entity rows outside type tau, with `extra` merged in, ascending."""
    ent = np.arange(n_rel, len(type_of))
    c = ent[type_of[n_rel:] != tau]
    if len(extra):
        c = np.union1d(c, np.asarray(extra, dtype=np.int64))
    return c


def _check_exact(eng, kg, type_of, queries, side, prec, known, k=None, query_types=None):
    n_rel, n_rows = kg.n_relations, kg.n_rows
    tcol = 1 if side == TAIL else 0
    taus = type_of[queries[:, tcol]] if query_types is None else np.asarray(query_types)
    foff, fids = _csr(known)
    if k is None:
        raw_t, filt_t, ts_t = eng.rank_typed(queries, side, foff, fids, precision=prec)
        c_only = _csr([_complement(t, type_of, n_rel) for t in taus])
        c_known = _csr([_complement(t, type_of, n_rel, kn) for t, kn in zip(taus, known)])
        _, f1, ts_u = eng.rank(queries, side, n_rel, n_rows, *c_only, precision=prec)
        _, f2, _ = eng.rank(queries, side, n_rel, n_rows, *c_known, precision=prec)
        assert torch.equal(raw_t.cpu(), f1.cpu())
        assert torch.equal(filt_t.cpu(), f2.cpu())
        assert torch.equal(ts_t.cpu().view(torch.int32), ts_u.cpu().view(torch.int32))
        return raw_t, filt_t, ts_t
    ids_t, sc_t = eng.topk_typed(queries, side, taus, k, foff, fids, precision=prec)
    c_known = _csr([_complement(t, type_of, n_rel, kn) for t, kn in zip(taus, known)])
    ids_u, sc_u = eng.topk(queries, side, n_rel, n_rows, k, *c_known, precision=prec)
    assert torch.equal(ids_t.cpu(), ids_u.cpu())
    assert torch.equal(sc_t.cpu().view(torch.int32), sc_u.cpu().view(torch.int32))
    ids = ids_t.cpu().numpy()
    ok = ids >= 0
    assert (type_of[ids[ok]] == np.broadcast_to(taus[:, None], ids.shape)[ok]).all()
    return ids_t, sc_t


@pytest.mark.parametrize("mode", ["complex", "ccorr_tanh"])
@pytest.mark.parametrize("prec", [BF16, BF16X3])
@pytest.mark.parametrize("side", [TAIL, HEAD])
def test_exact_against_untyped(eng_mod, side, prec, mode):
    rng0 = np.random.default_rng(7)
    hist = rng0.multinomial(2000, rng0.dirichlet(np.ones(30)))
    hist[hist == 0] = 1
    hist[0] += 2000 - hist.sum()
    kg, eng, rng, type_of, _, _ = _setup(eng_mod, 8, hist, dim=64 if mode == "complex" else 48, seed=1, mode=mode)
    q = _queries(rng, kg.n_relations, kg.n_rows, 500)
    known = _known(rng, q, side, kg.n_relations, kg.n_rows, type_of)
    _check_exact(eng, kg, type_of, q, side, prec, known)
    _check_exact(eng, kg, type_of, q, side, prec, known, k=10)


def test_type_size_edges(eng_mod):
    """Types of 1, 255, 256, 257 rows, one of more tiles than a work item takes (the all-candidate shape of 5000
    rows splits into chunks of 10 tiles; this type has 16), and 127 / 128 / 129 queries of one type so that query
    windows begin mid-tile."""
    hist = [1, 255, 256, 257, 4000, 100, 131]
    kg, eng, rng, type_of, off, ids = _setup(eng_mod, 4, hist, seed=2)
    n_rel = kg.n_relations
    for side in (TAIL, HEAD):
        col = 1 if side == TAIL else 0
        parts = []
        for tau, nq in zip(range(1, len(hist) + 1), [3, 127, 128, 129, 150, 5, 40]):
            members = ids[off[tau]:off[tau + 1]]
            qq = _queries(rng, n_rel, kg.n_rows, nq)
            qq[:, col] = rng.choice(members, size=nq)
            parts.append(qq)
        q = np.concatenate(parts)
        q = q[rng.permutation(len(q))]                 # shuffled type order
        q = np.concatenate([q, q[:17]])                # duplicated queries
        known = _known(rng, q, side, n_rel, kg.n_rows, type_of)
        _check_exact(eng, kg, type_of, q, side, BF16, known)
        _check_exact(eng, kg, type_of, q, side, BF16X3, known, k=7)


def test_one_type_and_every_entity_its_own_type(eng_mod):
    kg, eng, rng, type_of, _, _ = _setup(eng_mod, 4, [900], seed=3)
    q = _queries(rng, kg.n_relations, kg.n_rows, 300)
    known = _known(rng, q, TAIL, kg.n_relations, kg.n_rows, type_of)
    raw_t, _, _ = _check_exact(eng, kg, type_of, q, TAIL, BF16, known)
    raw_all, _, _ = eng.rank(q, TAIL, kg.n_relations, kg.n_rows)
    assert torch.equal(raw_t.cpu(), raw_all.cpu())
    _check_exact(eng, kg, type_of, q, HEAD, BF16X3, known, k=5)
    # every row its own type: nothing ranks before the true entity, top-k is the query's own type's single row
    own = np.arange(kg.n_rows, dtype=np.int32)
    off, ids = D.build_type_csr(own, kg.n_rows)
    eng.set_types(own, off, ids)
    raw, filt, ts = eng.rank_typed(q, HEAD)
    assert int(raw.abs().sum()) == 0 and int(filt.abs().sum()) == 0
    _, _, ts_u = eng.rank(q, HEAD, kg.n_relations, kg.n_rows)
    assert torch.equal(ts.cpu().view(torch.int32), ts_u.cpu().view(torch.int32))
    ids_t, sc = eng.topk_typed(q, HEAD, own[q[:, 0]], 3)
    ids_t = ids_t.cpu().numpy()
    assert (ids_t[:, 0] == q[:, 0]).all() and (ids_t[:, 1:] == -1).all()
    assert torch.isinf(sc[:, 1:]).all()


def test_k_above_type_size_and_empty(eng_mod):
    kg, eng, rng, type_of, off, ids = _setup(eng_mod, 4, [5, 300, 40], seed=4)
    q = _queries(rng, kg.n_relations, kg.n_rows, 60)
    taus = rng.integers(1, 4, size=60)
    known = [sorted(set(int(x) for x in rng.choice(ids[off[t]:off[t + 1]], size=2, replace=False))) for t in taus]
    ids_t, sc = _check_exact(eng, kg, type_of, q, TAIL, BF16X3, known, k=20, query_types=taus)
    ids_t = ids_t.cpu().numpy()
    for row, t, kn in zip(ids_t, taus, known):
        n_left = int(off[t + 1] - off[t]) - len(kn)
        assert (row[:min(n_left, 20)] >= 0).all() and (row[min(n_left, 20):] == -1).all()
    raw, filt, ts = eng.rank_typed(q[:0], TAIL)
    assert raw.numel() == 0 and filt.numel() == 0 and ts.numel() == 0
    i0, s0 = eng.topk_typed(q[:0], TAIL, taus[:0], 5)
    assert i0.shape == (0, 5)


def test_refusals_write_nothing(eng_mod):
    kg, eng, rng, type_of, off, ids = _setup(eng_mod, 4, [100, 200], seed=5)
    lib, dev = eng.lib, eng.device
    q = torch.as_tensor(_queries(rng, kg.n_relations, kg.n_rows, 10)).to(dev)
    sent_i = torch.full((10,), 12345, dtype=torch.int32, device=dev)
    sent_f = torch.full((10,), 7.0, dtype=torch.float32, device=dev)
    p = lambda t: C.c_void_p(t.data_ptr())
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    n_types = off.shape[0] - 1
    for side in (BOTH, REL):
        rc = lib.hole_rank_typed(eng._ctx, p(eng.table), p(q), 10, side, BF16, p(eng.type_of), p(eng.csr_off),
                                 p(eng.csr_ids), n_types, None, None, p(sent_f), p(sent_i), p(sent_i), s)
        assert rc != 0
    qt = torch.full((10,), 1, dtype=torch.int32, device=dev)
    ids_o = torch.full((10, 129), 12345, dtype=torch.int32, device=dev)
    sc_o = torch.full((10, 129), 7.0, dtype=torch.float32, device=dev)
    for side, k in ((BOTH, 5), (REL, 5), (TAIL, 0), (TAIL, 129)):
        rc = lib.hole_topk_typed(eng._ctx, p(eng.table), p(q), p(qt), 10, side, BF16X3, k, p(eng.csr_off),
                                 p(eng.csr_ids), n_types, None, None, p(ids_o), p(sc_o), s)
        assert rc != 0
    torch.cuda.synchronize()
    assert (sent_i == 12345).all() and (sent_f == 7.0).all() and (ids_o == 12345).all() and (sc_o == 7.0).all()
    # dims past the smem budget: 642 (bf16), 322 (bf16x3)
    for dim, prec in ((642, BF16), (322, BF16X3)):
        e2 = eng_mod.HoleEngine(kg.n_rows, dim).set_embeddings(np.zeros((kg.n_rows, dim), np.float32))
        e2.set_types(type_of, off, ids)
        rc = lib.hole_rank_typed(e2._ctx, p(e2.table), p(q), 10, TAIL, prec, p(e2.type_of), p(e2.csr_off),
                                 p(e2.csr_ids), n_types, None, None, p(sent_f), p(sent_i), p(sent_i), s)
        assert rc == -4
        rc = lib.hole_topk_typed(e2._ctx, p(e2.table), p(q), p(qt), 10, TAIL, prec, 5, p(e2.csr_off),
                                 p(e2.csr_ids), n_types, None, None, p(ids_o), p(sc_o), s)
        assert rc == -4
        e2.close()
    torch.cuda.synchronize()
    assert (sent_i == 12345).all() and (sent_f == 7.0).all() and (ids_o == 12345).all()
    e3 = eng_mod.HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E)
    with pytest.raises(eng_mod.HoleError):
        e3.rank_typed(q.cpu().numpy(), TAIL)
    with pytest.raises(eng_mod.HoleError):
        e3.topk_typed(q.cpu().numpy(), TAIL, np.ones(10), 5)
    with pytest.raises(eng_mod.HoleError):
        eng.topk_typed(q.cpu().numpy(), TAIL, np.full(10, n_types), 5)
    # the context stays usable
    eng.rank_typed(q.cpu().numpy(), TAIL)


def test_typed_call_drops_the_prepared_operand(eng_mod):
    kg, eng, rng, type_of, _, _ = _setup(eng_mod, 4, [300, 500], seed=6)
    q = _queries(rng, kg.n_relations, kg.n_rows, 200)
    b, e = kg.n_relations, kg.n_rows
    eng.rank_prepare(b, e)
    before = [x.cpu() for x in eng.rank(q, TAIL, b, e)]
    eng.rank_typed(q, TAIL)
    eng.topk_typed(q, HEAD, type_of[q[:, 0]], 4)
    after = [x.cpu() for x in eng.rank(q, TAIL, b, e)]
    for x, y in zip(before, after):
        assert torch.equal(x, y)
