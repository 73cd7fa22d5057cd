"""Type-constrained ranking and top-k against independent statements: the fp64 contract of tests/typed_reference.py
at the FB15k shape, the reference's own per-type-pool protocol (hole.eval_link_prediction_typed), and the
`--infer --type_constrained` driver."""
import os

import numpy as np
import pytest

import typed_reference as R
from graphembeddings_b200 import data as D
from oracle import hole_oracle as O

pytestmark = pytest.mark.gpu

TAIL, HEAD = 0, 1
BAND_X3 = 3e-5          # DESIGN §2: split-bf16 counts agree with fp64 outside +-3e-5 of the true score


@pytest.fixture(scope="module")
def eng_mod():
    from graphembeddings_b200 import build
    build.build()
    from graphembeddings_b200 import engine
    return engine


@pytest.fixture(scope="module")
def fb15k(eng_mod):
    """The rank_fb15k_d150 table (the FB15k type histogram: 815 types with the relation rows' own, 372 singletons)
    and 1,500 of the real FB15k test queries, filtered by the FB15k valid triples."""
    kg = D.make_config("rank_fb15k_d150", trained_scale=True)
    off, ids = D.build_type_csr(kg.type_of)
    assert len(off) - 1 == 815 and int((np.diff(off)[1:] == 1).sum()) == 372      # type 0: the relation rows
    npz = np.load(os.path.join(os.path.dirname(__file__), "golden", "fb15k_test_valid_triples.npz"))
    test, valid = npz["test"][:1500], npz["valid"]
    eng = eng_mod.HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E).set_types(kg.type_of, off, ids)
    return kg, eng, off, ids, test, valid


def _full_scores(kg, queries, side):
    """fp64 scores [Q, n_rows] of every entity row (relation columns +inf: no query's type holds them)."""
    S = np.full((len(queries), kg.n_rows), np.inf)
    S[:, kg.n_relations:] = O.all_scores(kg.E.astype(np.float64), queries, side, np.arange(kg.n_relations, kg.n_rows),
                                         np.float64)
    return S


@pytest.mark.parametrize("side", [TAIL, HEAD])
def test_counts_and_topk_match_fp64_at_fb15k_shape(eng_mod, fb15k, side):
    kg, eng, off, ids, test, valid = fb15k
    name = "tail" if side == TAIL else "head"
    tcol = 1 if side == TAIL else 0
    foff, fids = D.build_filter_csr(test, valid, name)
    flists = [fids[foff[q]:foff[q + 1]].astype(np.int64) for q in range(len(test))]
    S = _full_scores(kg, test, name)
    true = test[:, tcol].astype(np.int64)
    taus = kg.type_of[true]
    raw, filt, ts = eng.rank_typed(test, side, foff, fids, precision=eng_mod.HOLE_RANK_BF16X3)
    raw, filt, ts = raw.cpu().numpy(), filt.cpu().numpy(), ts.cpu().numpy()
    want_raw, want_filt = R.rank_counts(S, true, taus, off, ids, flists)
    st = S[np.arange(len(test)), true]
    assert np.all(np.abs(ts - st) <= BAND_X3)
    exact = 0
    for q in range(len(test)):
        cand = ids[off[taus[q]]:off[taus[q] + 1]].astype(np.int64)
        near = int(((np.abs(S[q, cand] - st[q]) <= BAND_X3) & (cand != true[q])).sum())
        assert abs(int(raw[q]) - want_raw[q]) <= near, q
        assert abs(int(filt[q]) - want_filt[q]) <= near, q
        exact += int(raw[q] == want_raw[q] and filt[q] == want_filt[q])
    assert exact >= 0.99 * len(test)
    # top-10 of the answer's type, filtered: nothing from beyond the band of the 10th fp64 score, everything
    # clearly inside it returned, scores rescored in fp32
    k = 10
    got_i, got_s = eng.topk_typed(test, side, taus, k, foff, fids)
    got_i, got_s = got_i.cpu().numpy(), got_s.cpu().numpy().astype(np.float64)
    want_i, want_s = R.topk(S, taus, off, ids, k, flists)
    for q in range(len(test)):
        n = int((want_i[q] >= 0).sum())
        g = got_i[q, :n].astype(np.int64)
        assert np.all(got_i[q, n:] == -1) and np.all(np.isinf(got_s[q, n:])), q
        assert np.all(kg.type_of[g] == taus[q]) and not np.isin(g, flists[q]).any(), q
        if n == 0:
            continue
        assert np.all(np.abs(got_s[q, :n] - S[q, g]) <= 2e-6 + 1e-5 * np.abs(S[q, g])), q
        kth = want_s[q, n - 1]
        assert np.all(S[q, g] <= kth + BAND_X3), q
        assert np.isin(want_i[q, :n][want_s[q, :n] < kth - BAND_X3], g).all(), q


def test_equals_the_reference_protocol(eng_mod):
    """Tail side, bf16: the ranks of hole.eval_link_prediction_typed (the reference's heap over a per-type pool,
    one relation per call) with the pool = the entities of the answer's type, exactly."""
    from graphembeddings_b200 import hole
    kg = D.synthetic_kg(4, 1500, 5000, 6, 64, seed=41, trained_scale=True)
    off, ids = D.build_type_csr(kg.type_of)
    eng = eng_mod.HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E).set_types(kg.type_of, off, ids)
    test, known = kg.triples[:300], kg.triples[300:]
    true_triples, test_triples = {}, {}
    for h, t, r in known.tolist():
        true_triples.setdefault(h, {}).setdefault(r, set()).add(t)
    for h, t, r in test.tolist():
        test_triples.setdefault(h, {}).setdefault(r, set()).add(t)
    n_checked = 0
    for r in sorted(set(test[:, 2].tolist())):
        for tau in sorted(set(kg.type_of[test[test[:, 2] == r, 1]].tolist())):
            pool = ids[off[tau]:off[tau + 1]].tolist()
            heads = sorted(set(test[test[:, 2] == r, 0].tolist()))
            cand = hole.InferenceCandidates({r}, pool, 0, 0.0)
            want_raw, want_filt = hole.eval_link_prediction_typed(eng, heads, cand, true_triples, test_triples)
            items, fl = [], []
            pset = set(pool)
            for h in heads:
                for t in sorted(test_triples.get(h, {}).get(r, ())):
                    if t in pset and t not in true_triples.get(h, {}).get(r, ()):
                        items.append((h, t, r))
                        fl.append(sorted(true_triples.get(h, {}).get(r, ())))
            assert len(items) == len(want_raw)
            if not items:
                continue
            foff = np.zeros(len(fl) + 1, np.int64)
            foff[1:] = np.cumsum([len(x) for x in fl])
            fids = np.array([x for s in fl for x in s], np.int32)
            raw, filt, _ = eng.rank_typed(np.array(items, np.int32), TAIL, foff, fids,
                                          precision=eng_mod.HOLE_RANK_BF16)
            assert (raw.cpu().numpy() + 1).tolist() == want_raw
            assert (filt.cpu().numpy() + 1).tolist() == want_filt
            n_checked += len(items)
    assert n_checked > 100


# ---------------------------------------------------------------------------------------------- CLI
def _write_data_dir(d, kg, n_valid, n_test):
    with open(os.path.join(d, "entity_metadata.tsv"), "w") as f:
        f.write("Index\tId\tName\tType\n")
        for i in range(kg.n_rows):
            f.write(f"{i}\tid{i}\tname{i}\t{'RELATION' if i < kg.n_relations else 'T%d' % kg.type_of[i]}\n")
    with open(os.path.join(d, "relation_ids.txt"), "w") as f:
        for r in range(kg.n_relations):
            f.write(f"rel{r}\t{r}\n")
    n = len(kg.triples)
    parts = {"triples.txt": kg.triples[: n - n_valid - n_test],
             "triples-valid.txt": kg.triples[n - n_valid - n_test: n - n_test],
             "test_positive_triples.txt": kg.triples[n - n_test:]}
    for name, tr in parts.items():
        np.savetxt(os.path.join(d, name), tr, fmt="%d", delimiter="\t")
    return parts


def test_cli_type_constrained(eng_mod, tmp_path):
    from graphembeddings_b200 import hole, tf_bundle
    kg = D.synthetic_kg(8, 1500, 9000, 7, 64, seed=5, with_embeddings=False)
    d = tmp_path / "data"
    d.mkdir()
    parts = _write_data_dir(str(d), kg, 600, 400)
    out = str(tmp_path / "run")
    args = ["--data_dir", str(d), "--output_dir", out, "--batch_size", "256", "--embedding_dim", "64",
            "--num_epochs", "2"]
    hole.main(args)
    runs = {}
    cwd = os.getcwd()
    for tag, extra in (("plain", []), ("typed", ["--type_constrained"])):
        wd = tmp_path / tag
        wd.mkdir()
        os.chdir(wd)
        lines = []
        try:
            res = hole.infer_triples(hole.build_parser().parse_args(args + ["--infer", "--predict_top_k", "4"] + extra),
                                     log=lambda *a: lines.append(" ".join(str(x) for x in a)))
        finally:
            os.chdir(cwd)
        runs[tag] = (res, lines, (wd / "inference_results.tsv").read_bytes(),
                     open(os.path.join(out, "predictions.tsv"), "rb").read(),
                     os.path.exists(os.path.join(out, "predictions_typed.tsv")))
    (res0, log0, inf0, pred0, typed0), (res1, log1, inf1, pred1, typed1) = runs["plain"], runs["typed"]
    # without the flag there is no typed output; with it the all-entity outputs are byte-identical and the block
    # follows them
    assert "typed" not in res0 and not typed0 and typed1
    assert inf1 == inf0 and pred1 == pred0 and log1[:len(log0)] == log0
    assert "\nType-constrained link prediction:" in log1[len(log0):]
    assert {k: v for k, v in res1.items() if k != "typed"} == res0
    # the block's MRR is the engine's computation
    E = tf_bundle.load_bundle(os.path.join(out, "model.ckpt"))["embeddings"]
    test = parts["test_positive_triples.txt"]
    known = np.concatenate([parts["triples.txt"], parts["triples-valid.txt"]])
    id_to_type = {i: ("RELATION" if i < kg.n_relations else "T%d" % kg.type_of[i]) for i in range(kg.n_rows)}
    type_of, off, ids = hole.type_tables(kg.n_rows, id_to_type)
    eng = eng_mod.HoleEngine(kg.n_rows, 64).set_embeddings(E).set_types(type_of, off, ids)
    q = np.unique(test, axis=0)
    q = q[~D.rows_in(q, known)]
    raws, filts = [], []
    for side, name in ((TAIL, "tail"), (HEAD, "head")):
        foff, fids = D.build_filter_csr(q, known, name)
        raw, filt, _ = eng.rank_typed(q, side, foff, fids, precision=eng_mod.HOLE_RANK_BF16X3)   # --rank_precision
        raws.append(raw.cpu().numpy() + 1)
        filts.append(filt.cpu().numpy() + 1)
    raws, filts = np.concatenate(raws), np.concatenate(filts)
    assert res1["typed"]["filtered_mrr"] == float(np.mean(1.0 / filts))
    assert res1["typed"]["raw_mrr"] == float(np.mean(1.0 / raws))
    # predictions_typed.tsv: predictions.tsv's columns; every line of the type of one of its pair's test answers,
    # never a known triple, positions 1.. by ascending score within each (pair, type)
    known_set = set(map(tuple, known.tolist()))
    answer_types = {}
    for h, t, r in test.tolist():
        answer_types.setdefault(("tail", h, r), set()).add(int(type_of[t]))
        answer_types.setdefault(("head", t, r), set()).add(int(type_of[h]))
    groups = {}
    rows = [line.rstrip("\n").split("\t") for line in open(os.path.join(out, "predictions_typed.tsv"))]
    assert rows and all(len(x) == 8 for x in rows)
    for side, h, t, r, pos, s, v, it in rows:
        h, t, r, pos, s = int(h), int(t), int(r), int(pos), float(s)
        pred, pair = (t, (side, h, r)) if side == "tail" else (h, (side, t, r))
        tau = int(type_of[pred])
        assert tau in answer_types[pair]
        assert (h, t, r) not in known_set
        groups.setdefault(pair + (tau,), []).append((pos, s, pred))
    for g in groups.values():
        assert [x[0] for x in g] == list(range(1, len(g) + 1)) and len(g) <= 4
        assert all((a[1], a[2]) < (b[1], b[2]) for a, b in zip(g, g[1:]))
