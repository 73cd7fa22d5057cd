"""Filtered rank counts (filt_before of hole_rank / hole_rank_ex) checked EXACTLY against the count pass's own
decisions.

include/hole_b200.h defines
    filt_before[q] = raw_before[q] - #{f in filter[q], f in range : (s_f, f) < (s_true, true_id)}
with s the score raw_before was counted with.  The oracle here needs no fp64 band: candidate f is "counted" for
row q when a call over the single-candidate range [f, f+1) -- the same query array (each query keeps its tile
row), compute_true = 0, the row's threshold -- counts it.  Then, exactly,
    filt[q] == raw[q] - sum over unique f in slice(q), f in range, of counted(q, f).
That rests on one assumption, which the diagonal pass already makes: a candidate's tensor-core score does not
depend on its column.  test_exact_ties_inside_the_filter checks it on bit-identical rows.
"""
import numpy as np
import pytest
import torch

from graphembeddings_b200 import data as D
from oracle import hole_oracle as O

pytestmark = pytest.mark.gpu

TAIL, HEAD, BOTH, REL = 0, 1, 2, 3
BF16, BF16X3 = 0, 1


@pytest.fixture(scope="module")
def eng_mod():
    from graphembeddings_b200 import build
    build.build()
    from graphembeddings_b200 import engine
    return engine


def _setup(eng_mod, n_rel, n_ent, n_q, dim, seed):
    kg = D.synthetic_kg(n_rel, n_ent, n_q, 4, dim, seed=seed, trained_scale=True)
    return kg, eng_mod.HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E)


def _range(kg, side):
    return (0, kg.n_relations) if side == REL else (kg.n_relations, kg.n_rows)


def _true_ids(queries, side):
    """Global id of each output row's true candidate (2Q rows for BOTH: tails, then heads)."""
    q = np.asarray(queries, dtype=np.int64)
    if side == BOTH:
        return np.concatenate([q[:, 1], q[:, 0]])
    return q[:, {TAIL: 1, HEAD: 0, REL: 2}[side]]


def _csr(slices):
    off = np.zeros(len(slices) + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(s) for s in slices])
    ids = np.array([x for s in slices for x in s], dtype=np.int32)
    return off, ids


def _pool_slices(rng, true_ids, b, en, pool_size=40, per_row=6, own=1.0):
    """Per row: a random subset of a shared pool of candidates, plus (with probability `own`) the row's own true
    column, plus now and then an id outside [b, en).  Ascending, duplicate-free."""
    pool = rng.choice(np.arange(b, en), size=min(pool_size, en - b), replace=False)
    slices = []
    for t in true_ids:
        s = set(int(x) for x in rng.choice(pool, size=int(rng.integers(0, per_row + 1)), replace=False))
        if rng.random() < own:
            s.add(int(t))
        if rng.random() < 0.1 and b > 0:
            s.add(b - 1)
        slices.append(sorted(s))
    return slices


def _rank_call(e, queries, side, precision):
    """call(lo, hi, foff, fids, thr, compute_true) -> (raw, filt, ts) numpy through HoleEngine.rank."""
    def call(lo, hi, foff=None, fids=None, thr=None, compute_true=True):
        ts = None if thr is None else torch.as_tensor(thr, dtype=torch.float32, device="cuda").clone()
        r, f, t = e.rank(queries, side, lo, hi, foff, fids, precision=precision, true_score=ts,
                         compute_true=compute_true)
        return r.cpu().numpy(), f.cpu().numpy(), t.cpu().numpy()
    return call


def _rank_ex_call(e, queries, side, precision, query_table):
    """The same through hole_rank_ex with a separate query table."""
    q = torch.as_tensor(queries, dtype=torch.int32, device="cuda").contiguous()
    rows = q.shape[0] * (2 if side == BOTH else 1)

    def call(lo, hi, foff=None, fids=None, thr=None, compute_true=True):
        raw = torch.zeros(rows, dtype=torch.int32, device="cuda")
        filt = torch.zeros(rows, dtype=torch.int32, device="cuda")
        ts = (torch.zeros(rows, dtype=torch.float32, device="cuda") if thr is None
              else torch.as_tensor(thr, dtype=torch.float32, device="cuda").clone())
        fo = fi = None
        if foff is not None and len(fids):
            fo = torch.as_tensor(foff, dtype=torch.int64, device="cuda").contiguous()
            fi = torch.as_tensor(fids, dtype=torch.int32, device="cuda").contiguous()
        e.rank_ex(q, side, lo, hi, query_table=query_table, filter_off=fo, filter_ids=fi, precision=precision,
                  true_score=ts, compute_true=compute_true, raw_before=raw, filt_before=filt)
        return raw.cpu().numpy(), filt.cpu().numpy(), ts.cpu().numpy()
    return call


def _counted(call, ids, thr):
    """counted[f] = int [rows]: 1 where candidate f alone, against the row's threshold, counts."""
    out = {}
    for f in sorted(set(int(x) for x in ids)):
        raw, _, _ = call(f, f + 1, thr=thr, compute_true=False)
        assert np.all((raw == 0) | (raw == 1))
        out[f] = raw
    return out


def _assert_filt_exact(call, raw, filt, thr, foff, fids, b, en):
    """filt == raw - the counted unique in-range ids of each slice; returns (counted, per-row subtraction)."""
    inr = fids[(fids >= b) & (fids < en)]
    counted = _counted(call, inr, thr)
    sub = np.zeros(len(raw), dtype=np.int64)
    for q in range(len(raw)):
        for f in set(int(x) for x in fids[foff[q]:foff[q + 1]]):
            if b <= f < en:
                sub[q] += counted[f][q]
    bad = np.nonzero(filt != raw - sub)[0]
    assert len(bad) == 0, (f"{len(bad)} rows differ, e.g. row {bad[0]}: raw {raw[bad[0]]} filt {filt[bad[0]]} "
                           f"want {raw[bad[0]] - sub[bad[0]]}")
    return counted, sub


# ---------------------------------------------------------------------------------------------------- own column
@pytest.mark.parametrize("precision", [BF16, BF16X3])
@pytest.mark.parametrize("side", [TAIL, HEAD, REL, BOTH])
def test_own_column_counts_with_a_foreign_threshold_everything_filtered(eng_mod, side, precision):
    """compute_true = 0, a threshold above every score, every candidate filtered: raw counts every candidate, the
    query's own column included, and the filter removes every one of them."""
    kg, e = _setup(eng_mod, 9, 700, 150, 64, seed=3 + side)
    b, en = _range(kg, side)
    rows = len(kg.triples) * (2 if side == BOTH else 1)
    foff, fids = _csr([list(range(b, en))] * rows)
    raw, filt, _ = _rank_call(e, kg.triples, side, precision)(b, en, foff, fids, thr=np.full(rows, 1e4),
                                                              compute_true=False)
    assert np.all(raw == en - b)
    assert np.all(filt == 0)


@pytest.mark.parametrize("precision", [BF16, BF16X3])
@pytest.mark.parametrize("side", [TAIL, HEAD, REL, BOTH])
def test_own_column_counts_with_another_rows_threshold(eng_mod, side, precision):
    """Each row gets the true score of a better-placed row; its own column is in-sample and scores below that
    threshold for most rows, so the count pass counts it and the filter must remove it."""
    kg, e = _setup(eng_mod, 9, 1500, 200, 150, seed=11 + side)
    b, en = _range(kg, side)
    call = _rank_call(e, kg.triples, side, precision)
    _, _, ts = call(b, en)
    order = np.argsort(ts, kind="stable")
    n = len(ts)
    thr = np.empty_like(ts)
    thr[order] = ts[order[np.minimum(np.arange(n) + n // 3, n - 1)]]
    tid = _true_ids(kg.triples, side)
    rng = np.random.default_rng(side)
    foff, fids = _csr(_pool_slices(rng, tid, b, en, pool_size=min(30, en - b), per_row=4, own=1.0))
    raw, filt, _ = call(b, en, foff, fids, thr=thr, compute_true=False)
    counted, _ = _assert_filt_exact(call, raw, filt, thr, foff, fids, b, en)
    own = np.array([counted[int(t)][q] for q, t in enumerate(tid)])
    assert own.sum() >= n // 2                  # the own column really is counted on most rows
    assert np.all(filt <= raw) and np.all(filt >= 0)


# ---------------------------------------------------------------------------------------------------- exact ties
def _tie_layout(kg, side, n_q, seed):
    """Queries whose true candidates t are spaced five rows apart with the four rows t-2 .. t+2 around each one
    free for copies; the queries' other entities lie beyond the spaced block."""
    rng = np.random.default_rng(seed)
    b = kg.n_relations
    t = b + 2 + 5 * np.arange(n_q)
    other = rng.integers(b + 5 * n_q, kg.n_rows, size=n_q)
    r = rng.integers(0, kg.n_relations, size=n_q)
    q = np.stack([other, t, r], 1) if side == TAIL else np.stack([t, other, r], 1)
    return q.astype(np.int32), t


@pytest.mark.parametrize("precision", [BF16, BF16X3])
@pytest.mark.parametrize("dim,side", [(64, TAIL), (150, HEAD), (258, TAIL)])
def test_exact_ties_inside_the_filter(eng_mod, dim, side, precision):
    """Filtered bit-identical copies of the true row at smaller and larger ids (test_gpu_rank's ragged-ties style):
    filt subtracts exactly the smaller-id copies plus the filtered rows that score strictly better."""
    kg = D.synthetic_kg(5, 2000, 10, 4, dim, seed=dim + side, trained_scale=True)
    q, t = _tie_layout(kg, side, 250, seed=dim)
    E = kg.E.copy()
    for d in (-2, -1, 1, 2):
        E[t + d] = E[t]
    e = eng_mod.HoleEngine(kg.n_rows, dim).set_embeddings(E)
    b, en = kg.n_relations, kg.n_rows
    call = _rank_call(e, q, side, precision)
    raw0, _, ts = call(b, en)
    cand, qp = e.rank_debug_operands()
    parts = 2 if precision == BF16X3 else 1
    K = cand.shape[1] // parts
    C = cand.double().cpu().numpy()[: en - b]
    Qm = qp.double().cpu().numpy()[: len(q)]
    if parts == 2:
        S = Qm[:, :K] @ C[:, :K].T + Qm[:, K:] @ C[:, :K].T + Qm[:, :K] @ C[:, K:].T
    else:
        S = Qm @ C.T
    tj = t - b
    thr64 = S[np.arange(len(q)), tj]
    # filters: the copies, the true id itself, and pool rows at least 1e-3 away from the threshold
    rng = np.random.default_rng(dim)
    slices, better = [], np.zeros(len(q), np.int64)
    far = np.abs(S - thr64[:, None]) > 1e-3
    for i in range(len(q)):
        pick = rng.choice(np.nonzero(far[i])[0][::7], size=5, replace=False)
        better[i] = int((S[i, pick] < thr64[i]).sum())
        slices.append(sorted(set((pick + b).tolist()) | {int(t[i]) + d for d in (-2, -1, 0, 1, 2)}))
    foff, fids = _csr(slices)
    raw, filt, ts2 = call(b, en, foff, fids)
    assert np.array_equal(raw, raw0) and np.array_equal(ts, ts2)
    counted, _ = _assert_filt_exact(call, raw, filt, ts, foff, fids, b, en)
    # the copies score exactly the threshold in a column of their own: the id rule decides (the oracle's
    # column-independence assumption), and the true column itself never counts
    for d in (-2, -1):
        assert np.all(np.array([counted[int(x) + d][i] for i, x in enumerate(t)]) == 1)
    for d in (0, 1, 2):
        assert np.all(np.array([counted[int(x) + d][i] for i, x in enumerate(t)]) == 0)
    assert np.array_equal(filt, raw - 2 - better)


@pytest.mark.parametrize("dim,side,precision", [(64, TAIL, BF16), (150, HEAD, BF16), (514, TAIL, BF16),
                                                 (64, TAIL, BF16X3), (150, HEAD, BF16X3), (320, TAIL, BF16X3)])
def test_near_ties_inside_the_filter(eng_mod, dim, side, precision):
    """Filtered rows built as the true row with one component moved by one bf16 ulp, up and down, where the
    query's |q_k| is smallest: the scores differ from the threshold by a few fp32 ulps at most, and filt must
    still follow the count pass's own decisions exactly."""
    kg = D.synthetic_kg(5, 2000, 10, 4, dim, seed=2 * dim + side, trained_scale=True)
    q, t = _tie_layout(kg, side, 250, seed=dim + 1)
    E = kg.E.copy()
    # the true rows: bf16-representable and of norm < 1, so the packer's clip leaves them exactly as they are
    Et = E[t] / np.linalg.norm(E[t], axis=1, keepdims=True) * 0.8
    E[t] = torch.from_numpy(Et).to(torch.bfloat16).float().numpy()
    e = eng_mod.HoleEngine(kg.n_rows, dim).set_embeddings(E)
    b, en = kg.n_relations, kg.n_rows
    e.rank(q, side, b, en)
    _, qp = e.rank_debug_operands()
    qv = qp.float().cpu().numpy()[: len(q), :dim]
    H = dim // 2
    stride = e.table.shape[1]
    # table row layout [Re | pad | Im | pad]: operand column k < H is row column k, k >= H is stride/2 + k - H
    colmap = np.concatenate([np.arange(H), stride // 2 + np.arange(H)])
    rows = E[t]
    ok = (np.abs(qv) > 0) & (np.abs(rows) > 1e-3)
    k = np.argmin(np.where(ok, np.abs(qv), np.inf), axis=1)
    tab = e.table.clone()
    for d, step in ((-2, 1), (-1, -1), (1, 1), (2, -1)):
        moved = torch.as_tensor(rows[np.arange(len(t)), k]).to(torch.bfloat16).view(torch.int16)
        moved = (moved + step).view(torch.bfloat16).float().to("cuda")
        tab[torch.as_tensor(t + d, device="cuda")] = tab[torch.as_tensor(t, device="cuda")]
        tab[torch.as_tensor(t + d, device="cuda"), torch.as_tensor(colmap[k], device="cuda")] = moved
    e.table = tab
    e.rank_invalidate()
    call = _rank_call(e, q, side, precision)
    rng = np.random.default_rng(dim)
    slices = []
    for i in range(len(q)):
        s = {int(t[i]) + d for d in (-2, -1, 1, 2) if rng.random() < 0.8}
        if rng.random() < 0.5:
            s.add(int(t[i]))
        s |= set(int(x) for x in rng.integers(b, en, size=3))
        slices.append(sorted(s))
    foff, fids = _csr(slices)
    raw, filt, ts = call(b, en, foff, fids)
    _assert_filt_exact(call, raw, filt, ts, foff, fids, b, en)


# ---------------------------------------------------------------------------------------------------- coverage
@pytest.mark.parametrize("dim,precision", [(d, BF16) for d in (2, 64, 150, 258, 514, 640)] +
                         [(d, BF16X3) for d in (2, 64, 150, 258, 320)])
def test_filtered_counts_exact_at_every_packer_iteration_and_ring_depth(eng_mod, dim, precision):
    """test_gpu_shapes' edges: query-packer iterations 1..3, ring depths 4..2, both precisions; filter slices mix
    a shared pool, the row's own true column and ids outside the range."""
    side = TAIL if dim % 4 else HEAD
    kg, e = _setup(eng_mod, 7, 1700, 300, dim, seed=100 + dim + precision)
    b, en = _range(kg, side)
    call = _rank_call(e, kg.triples, side, precision)
    rng = np.random.default_rng(dim)
    foff, fids = _csr(_pool_slices(rng, _true_ids(kg.triples, side), b, en, own=0.5))
    raw, filt, ts = call(b, en, foff, fids)
    _assert_filt_exact(call, raw, filt, ts, foff, fids, b, en)
    assert raw.max() > 100 and np.any(filt < raw)


@pytest.mark.parametrize("side", [TAIL, HEAD, REL])
def test_filtered_counts_exact_ccorr_tanh(eng_mod, side):
    kg, e = _setup(eng_mod, 13, 1200, 250, 150, seed=40 + side)
    e.set_score_mode("ccorr_tanh")
    b, en = _range(kg, side)
    for precision in (BF16, BF16X3):
        call = _rank_call(e, kg.triples, side, precision)
        rng = np.random.default_rng(side + 10 * precision)
        foff, fids = _csr(_pool_slices(rng, _true_ids(kg.triples, side), b, en, pool_size=min(40, en - b),
                                       own=0.5))
        raw, filt, ts = call(b, en, foff, fids)
        _assert_filt_exact(call, raw, filt, ts, foff, fids, b, en)
        assert np.any(filt < raw)


@pytest.mark.parametrize("precision", [BF16, BF16X3])
def test_filtered_counts_exact_relation_side(eng_mod, precision):
    """HOLE_SIDE_RELATION over 40 relation rows: slices of known relations of (h, t), the true one included on
    some rows, through build_filter_csr."""
    kg, e = _setup(eng_mod, 40, 1500, 400, 150, seed=7)
    rng = np.random.default_rng(8)
    q = kg.triples
    known = np.concatenate([np.stack([q[:, 0], q[:, 1], rng.integers(0, 40, len(q))], 1) for _ in range(4)] +
                           [q[rng.random(len(q)) < 0.3]])
    foff, fids = D.build_filter_csr(q, known, "relation")
    call = _rank_call(e, q, REL, precision)
    raw, filt, ts = call(0, 40, foff, fids)
    _assert_filt_exact(call, raw, filt, ts, foff, fids, 0, 40)
    assert np.any(filt < raw)


@pytest.mark.parametrize("side", [TAIL, HEAD, BOTH])
def test_filtered_counts_exact_rank_ex_with_query_table(eng_mod, side):
    """hole_rank_ex: candidates from the engine's table, query rows from another table of the same layout."""
    kg, e = _setup(eng_mod, 7, 1300, 250, 150, seed=60 + side)
    b, en = _range(kg, side)
    g = torch.Generator(device="cuda").manual_seed(side)
    qtab = (e.table * (0.5 + torch.rand(e.table.shape, device="cuda", generator=g))).contiguous()
    for precision in (BF16, BF16X3):
        call = _rank_ex_call(e, kg.triples, side, precision, qtab)
        rng = np.random.default_rng(side + 5 * precision)
        foff, fids = _csr(_pool_slices(rng, _true_ids(kg.triples, side), b, en, own=0.5))
        raw, filt, ts = call(b, en, foff, fids)
        _assert_filt_exact(call, raw, filt, ts, foff, fids, b, en)
        # the query table is really used: the same call on the engine's own table ranks differently
        raw_own, _, _ = _rank_call(e, kg.triples, side, precision)(b, en)
        assert not np.array_equal(raw, raw_own)


@pytest.mark.parametrize("precision", [BF16, BF16X3])
@pytest.mark.parametrize("side", [TAIL, BOTH])
def test_candidate_shards_with_filters_sum_to_one_call(eng_mod, side, precision):
    """Three candidate shards, true scores in phase 1, filtered counts in phase 2: the per-shard raw and filt
    accumulate to one whole-range call exactly, and that call meets the exact oracle."""
    kg, e = _setup(eng_mod, 6, 2600, 300, 150, seed=70 + side)
    b, en = _range(kg, side)
    call = _rank_call(e, kg.triples, side, precision)
    rng = np.random.default_rng(side)
    slices = _pool_slices(rng, _true_ids(kg.triples, side), b, en, pool_size=60, per_row=10, own=0.5)
    foff, fids = _csr(slices)
    raw1, filt1, ts1 = call(b, en, foff, fids)
    _assert_filt_exact(call, raw1, filt1, ts1, foff, fids, b, en)
    rows = len(raw1)
    cuts = [b, b + 700, b + 1601, en]                 # not tile-aligned
    ts = torch.zeros(rows, dtype=torch.float32, device="cuda")
    raw = torch.zeros(rows, dtype=torch.int32, device="cuda")
    filt = torch.zeros(rows, dtype=torch.int32, device="cuda")
    scratch_r, scratch_f = torch.zeros_like(raw), torch.zeros_like(filt)
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        e.rank(kg.triples, side, lo, hi, precision=precision, true_score=ts, compute_true=True,
               raw_before=scratch_r, filt_before=scratch_f)
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        e.rank(kg.triples, side, lo, hi, foff, fids, precision=precision, true_score=ts, compute_true=False,
               raw_before=raw, filt_before=filt)
    assert np.array_equal(ts.cpu().numpy(), ts1)
    assert np.array_equal(raw.cpu().numpy(), raw1)
    assert np.array_equal(filt.cpu().numpy(), filt1)


@pytest.mark.parametrize("precision", [BF16, BF16X3])
def test_repeated_filter_ids_subtract_once(eng_mod, precision):
    """A slice that lists an id twice (or three times) subtracts it once, as the reference's set does."""
    kg, e = _setup(eng_mod, 7, 1500, 300, 150, seed=80)
    b, en = _range(kg, TAIL)
    call = _rank_call(e, kg.triples, TAIL, precision)
    rng = np.random.default_rng(81)
    slices = _pool_slices(rng, _true_ids(kg.triples, TAIL), b, en, own=0.5)
    foff, fids = _csr(slices)
    raw, filt, ts = call(b, en, foff, fids)
    rep = [sorted(s + [x for x in s if rng.random() < 0.5] + [x for x in s[:1]]) for s in slices]
    foff2, fids2 = _csr(rep)
    assert len(fids2) > len(fids) + 100
    raw2, filt2, _ = call(b, en, foff2, fids2)
    assert np.array_equal(raw2, raw) and np.array_equal(filt2, filt)
    _assert_filt_exact(call, raw2, filt2, ts, foff2, fids2, b, en)
    assert np.any(filt < raw)


# ---------------------------------------------------------------------------------------------------- typed protocol
def test_typed_protocol_equals_the_heap_exactly():
    """hole.eval_link_prediction_typed (holE.py's own protocol) against the oracle's heap, exactly, on a table whose
    scores are exact in bf16 and fp32 and pairwise distinct within each head's candidate product.  Many items have
    an in-sample (h, r2, t*) or (h, r2, next tail) that scores better than the item: each counting row's own column
    is then a filtered candidate under another row's threshold."""
    from graphembeddings_b200 import build, hole
    from graphembeddings_b200.engine import HoleEngine
    build.build()
    n_rel, n_ent, dim = 5, 200, 2
    rels, heads = [1, 2, 4], [10, 20, 30, 40]
    tails = list(range(60, 60 + 48))
    for seed in range(200):
        rng = np.random.default_rng(seed)
        # entity components k / 256 with |k| <= 127 (norms < 1: the clip leaves them alone); relations with
        # power-of-two components, so that the query h * r has at most 8 significant bits per component and is
        # exact in bf16, and every score (two products of such numbers, summed) is exact in fp32
        E = (rng.integers(-127, 128, size=(n_rel + n_ent, dim)) / 256.0).astype(np.float32)
        E[:n_rel] = 0.0
        E[1], E[2], E[4] = (0.5, 0.0), (0.0, 0.5), (0.25, 0.25)
        vals = {h: O.score(E.astype(np.float64), np.array([(h, t, r) for t in tails for r in rels]), np.float64)
                for h in heads}
        if all(len(np.unique(v)) == len(v) for v in vals.values()):
            break
    else:
        pytest.fail("no table with distinct scores")
    eng = HoleEngine(n_rel + n_ent, dim).set_embeddings(E)
    cand = hole.InferenceCandidates(rels, tails, 3, 0.05)
    true_t, test_t = {}, {}
    n_better = 0
    for h in heads:
        v = vals[h].reshape(len(tails), len(rels))
        for ri, r in enumerate(rels):
            pick = rng.choice(len(tails), size=14, replace=False)
            test_t.setdefault(h, {})[r] = {tails[i] for i in pick[:6]}
            true_t.setdefault(h, {})[r] = {tails[i] for i in pick[4:]}       # two in-sample test tails
        # for every item (t*, r*): (t*, r2) and (next tail, r2) in-sample for the other relations r2
        for r in rels:
            for ts in test_t[h][r]:
                i = tails.index(ts)
                for r2 in rels:
                    if r2 == r:
                        continue
                    true_t[h][r2].add(ts)
                    if i + 1 < len(tails):
                        true_t[h][r2].add(tails[i + 1])
                    n_better += int(v[i, rels.index(r2)] < v[i, rels.index(r)])
    raw, filt = hole.eval_link_prediction_typed(eng, heads, cand, true_t, test_t)
    assert n_better > 10
    k = 0
    for h in heads:
        triples = [(h, t, r) for t in tails for r in rels]
        rr, ff = O.eval_link_prediction_heap(O.evaluate_triples(E, np.array(triples), np.float64), triples,
                                             true_t, test_t)
        n = len(rr)
        assert sorted(zip(raw[k:k + n], filt[k:k + n])) == sorted(zip(rr, ff))
        k += n
    assert k == len(raw) > 0
