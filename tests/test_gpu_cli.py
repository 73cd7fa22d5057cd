"""End to end through the holE.py-compatible driver on a synthetic --data_dir."""
import os

import numpy as np
import pytest

from graphembeddings_b200 import data as D
from oracle import hole_oracle as O

pytestmark = pytest.mark.gpu


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


def test_train_checkpoint_resume_infer(tmp_path):
    from graphembeddings_b200 import build, hole, tf_bundle
    build.build()
    kg = D.synthetic_kg(8, 1500, 9000, 4, 64, seed=3, with_embeddings=False)
    d = tmp_path / "data"; d.mkdir()
    parts = _write_data_dir(str(d), kg, 600, 400)
    out = str(tmp_path / "run")
    args = ["--data_dir", str(d), "--output_dir", out, "--batch_size", "256", "--embedding_dim", "64",
            "--num_epochs", "2"]
    hole.main(args)
    for name in ("model.ckpt.index", "model.ckpt.data-00000-of-00001", "checkpoint",
                 "projector_config.pbtxt", "summaries.tsv"):
        assert os.path.exists(os.path.join(out, name)), name
    ev = [f for f in os.listdir(out) if f.startswith("events.out.tfevents.")]
    assert len(ev) == 1
    from graphembeddings_b200 import tf_events
    recs = tf_events.read_events(os.path.join(out, ev[0]))              # (both CRCs of every record checked)
    tags = {t for e in recs for t in list(e["scalars"]) + list(e["histograms"])}
    for want in ("validation/summaries/mean", "validation/positive/eval/summaries/stddev_1",
                 "validation/corrupt/eval/summaries/histogram", "batch/eval/summaries/max",
                 "batch/learn/learning_rate"):
        assert want in tags, (want, sorted(tags)[:5])
    assert recs[0]["file_version"] == "brain.Event:2" and len(recs) >= 3
    rows = [dict(kv.split("=") for kv in line.split("\t")) for line in open(os.path.join(out, "summaries.tsv"))]
    # the whole validation file is scored at every validation point (holE.py:350 TODO)
    assert abs(recs[1]["histograms"]["validation/summaries/histogram"]["num"] - 600) < 0.5
    assert abs(recs[1]["scalars"]["validation/summaries/mean"] - float(rows[0]["valid_loss_mean"])) < 1e-6
    b = tf_bundle.load_bundle(os.path.join(out, "model.ckpt"))
    assert b["embeddings"].shape == (kg.n_rows, 64) and np.isfinite(b["embeddings"]).all()
    # refuses to clobber an existing output_dir (holE.py:254-255) ...
    with pytest.raises(Exception, match="already exists"):
        hole.main(args)
    # ... unless resuming
    hole.main(args + ["--resume_checkpoint", "--max_steps", "5"])
    # --infer: all-entity filtered ranking, agrees with the oracle's heap on the saved table
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        flags = hole.build_parser().parse_args(args + ["--infer"])
        m = hole.infer_triples(flags, log=lambda *a: None)
    finally:
        os.chdir(cwd)
    assert 0 < m["filtered_mrr"] <= 1 and m["raw_mean_pos"] >= m["filtered_mean_pos"]
    assert os.path.exists(tmp_path / "inference_results.tsv")
    E = tf_bundle.load_bundle(os.path.join(out, "model.ckpt"))["embeddings"]
    test = np.unique(parts["test_positive_triples.txt"], axis=0)[:40]
    known = np.concatenate([parts["triples.txt"], parts["triples-valid.txt"]])
    cand = np.arange(kg.n_relations, kg.n_rows)
    S = O.sigmoid(O.all_scores(E, test, "tail", cand, np.float32))
    true_t, test_t = {}, {}
    for h, t, r in known.tolist():
        true_t.setdefault(h, {}).setdefault(r, set()).add(t)
    got_r, got_f = [], []
    from graphembeddings_b200.engine import HoleEngine
    eng = HoleEngine(kg.n_rows, 64).set_embeddings(E)
    raw, filt = hole.eval_link_prediction(eng, test, known, kg.n_relations, kg.n_rows, sides=("tail",))
    # oracle heap per query (single test tail per group so ranks are per-triple)
    keep = [tuple(q) not in set(map(tuple, known.tolist())) for q in test.tolist()]
    want_r, want_f = [], []
    for q, (h, t, r) in enumerate(test.tolist()):
        if not keep[q]:
            continue
        triples = [(h, int(c), r) for c in cand]
        rr, ff = O.eval_link_prediction_heap(S[q], triples, true_t, {h: {r: {t}}})
        want_r += rr; want_f += ff
    assert len(raw) == len(want_r)
    # split-bf16 scores (the --infer default) vs the fp32-sigma heap: a rank may differ only by candidates
    # whose fp64 score lies within 3e-5 of the true one (band check, per query, raw and filtered)
    S64 = O.all_scores(E.astype(np.float64), test, "tail", cand, np.float64)
    k = 0
    for q, (h, t, r) in enumerate(test.tolist()):
        if not keep[q]:
            continue
        thr = S64[q, t - kg.n_relations]
        lo = int((S64[q] < thr - 3e-5).sum())
        hi = int((S64[q] <= thr + 3e-5).sum()) - 1
        fl = np.array(sorted(true_t.get(h, {}).get(r, ())), dtype=np.int64) - kg.n_relations
        f_sure = int((S64[q, fl] < thr - 3e-5).sum()) if len(fl) else 0
        f_maybe = int((S64[q, fl] <= thr + 3e-5).sum()) if len(fl) else 0
        for got, ref in ((raw[k], want_r[k]),):
            assert lo + 1 <= got <= hi + 1 and lo + 1 <= ref <= hi + 1
        for got, ref in ((filt[k], want_f[k]),):
            assert lo - f_maybe + 1 <= got <= hi - f_sure + 1 and lo - f_maybe + 1 <= ref <= hi - f_sure + 1
        k += 1
    assert k == len(raw)


def test_log_loss_branch_trains_and_logs(tmp_path):
    """--log_loss --negative_ratio 2 (holE.py:194-196, 206-220) through the driver, resumed
    from a trained-scale checkpoint: summaries and the pocket checkpoint are written (that the loss falls is
    tests/test_gpu_train.py::test_logloss_training_reduces_the_loss)."""
    from graphembeddings_b200 import build, hole, tf_bundle
    build.build()
    kg = D.synthetic_kg(8, 1500, 9000, 4, 64, seed=4, trained_scale=True)
    d = tmp_path / "data"; d.mkdir()
    parts = _write_data_dir(str(d), kg, 600, 400)
    out = str(tmp_path / "run")
    os.makedirs(out)
    tf_bundle.save_bundle(os.path.join(out, "model.ckpt"),
                          {"embeddings": kg.E, "batch/Variable": np.array(0, dtype=np.int32)})
    args = ["--data_dir", str(d), "--output_dir", out, "--batch_size", "256", "--embedding_dim", "64",
            "--num_epochs", "4", "--log_loss", "--negative_ratio", "2", "--l2_regularization", "0",
            "--learning_rate", "0.5", "--resume_checkpoint"]
    hole.main(args)
    rows = [dict(kv.split("=") for kv in line.split("\t")) for line in open(os.path.join(out, "summaries.tsv"))]
    assert len(rows) >= 8 and all(np.isfinite(float(r["valid_loss_mean"])) for r in rows)
    E1 = tf_bundle.load_bundle(os.path.join(out, "model.ckpt"))["embeddings"]
    assert np.isfinite(E1).all() and np.abs(E1 - kg.E).max() > 1e-4
    # the first validation row is the logistic loss of the restored table: positives and two
    # corrupt batches of near-random scores -> close to log 2
    assert abs(float(rows[0]["valid_loss_mean"]) - np.log(2.0)) < 0.05


def test_typed_candidate_protocol_matches_heap_restatement():
    """holE.py's own inference protocol: per head, product(tails, relations) ranked jointly
    (holE.py:564-573, 427-469) -- tensor-core counts vs the oracle's heap restatement, which is
    pinned against the reference's eval_link_prediction in tests/test_oracle.py."""
    from graphembeddings_b200 import build, hole
    from graphembeddings_b200.engine import HoleEngine
    build.build()
    rng = np.random.default_rng(4)
    kg = D.synthetic_kg(6, 900, 10, 3, 64, seed=9, trained_scale=True)
    eng = HoleEngine(kg.n_rows, kg.dim).set_embeddings(kg.E)
    heads = [int(x) for x in rng.choice(np.arange(6, 300), size=25, replace=False)]
    tails = sorted(int(x) for x in rng.choice(np.arange(300, 906), size=200, replace=False))
    rels = [1, 3, 4]
    cand = hole.InferenceCandidates(rels, tails, 3, 0.05)
    true_t, test_t = {}, {}
    for h in heads:
        for r in rels:
            ts = rng.choice(tails, size=12, replace=False)
            true_t.setdefault(h, {})[r] = set(int(x) for x in ts[:7])
            test_t.setdefault(h, {})[r] = set(int(x) for x in ts[5:])     # overlap: 2 in-sample test tails
    raw, filt = hole.eval_link_prediction_typed(eng, heads, cand, true_t, test_t)
    want_r, want_f = [], []
    for h in heads:
        triples = [(h, t, r) for t in tails for r in rels]
        vals = O.evaluate_triples(kg.E, np.array(triples), np.float32)
        rr, ff = O.eval_link_prediction_heap(vals, triples, true_t, test_t)
        want_r += sorted(rr); want_f += sorted(ff)
    # per head the GPU path emits items in (relation, tail) order, the heap in score order:
    # compare as multisets per head
    assert len(raw) == len(want_r) == 25 * 3 * 5
    got_r, got_f, k = [], [], 0
    for h in heads:
        n = 15
        got_r += sorted(raw[k:k + n]); got_f += sorted(filt[k:k + n]); k += n
    # band check per recorded item, in the order the GPU path emits them (per head: relation, then tail):
    # bf16 operands move a score by at most 4e-3 |q||e| <= 4e-3, so a rank may differ from the exact one only
    # by candidates within 8e-3 of the item's own fp64 score
    E64 = kg.E.astype(np.float64)
    k = n_exact = 0
    for h in heads:
        triples = np.array([(h, t, r) for t in tails for r in rels])
        s64 = O.score(E64, triples, np.float64)
        insample = np.array([t in true_t[h][r] for (_, t, r) in triples.tolist()])
        for r in sorted(rels):
            for t in sorted(test_t[h][r]):
                if t in true_t[h][r]:
                    continue
                me = s64[(triples[:, 1] == t) & (triples[:, 2] == r)][0]
                lo = int((s64 < me - 8e-3).sum())
                hi = int((s64 <= me + 8e-3).sum()) - 1
                assert lo + 1 <= raw[k] <= hi + 1
                f_sure = int(((s64 < me - 8e-3) & insample).sum())
                f_maybe = int(((s64 <= me + 8e-3) & insample).sum())
                assert lo - f_maybe + 1 <= filt[k] <= hi - f_sure + 1
                if hi == lo:                   # no other candidate inside the band: both ranks are exact
                    assert raw[k] == lo + 1 and filt[k] == lo - f_sure + 1
                    n_exact += 1
                k += 1
    assert k == len(raw) and n_exact > 0
    m = hole.score_mrr(raw, filt, log=lambda *a: None)
    mw = O.score_mrr(want_r, want_f)
    assert abs(m["filtered_mrr"] - mw["filtered_mrr"]) < 5e-3


def test_archived_ccorr_tanh_variant_trains_through_the_driver(tmp_path):
    """--score_variant ccorr_tanh --margin 1.0 (the archived holE-20170724 run's score and margin) through the
    training loop: the validation loss of the hinge on tanh scores falls, the checkpoint is written."""
    from graphembeddings_b200 import build, hole, tf_bundle
    build.build()
    kg = D.synthetic_kg(8, 1500, 9000, 4, 64, seed=5)
    d = tmp_path / "data"; d.mkdir()
    _write_data_dir(str(d), kg, 600, 400)
    out = str(tmp_path / "run")
    args = ["--data_dir", str(d), "--output_dir", out, "--batch_size", "256", "--embedding_dim", "64",
            "--num_epochs", "12", "--score_variant", "ccorr_tanh", "--margin", "1.0", "--learning_rate", "0.5"]
    hole.main(args)
    rows = [dict(kv.split("=") for kv in line.split("\t")) for line in open(os.path.join(out, "summaries.tsv"))]
    v = [float(r["valid_loss_mean"]) for r in rows]
    assert all(np.isfinite(v)) and abs(v[0] - 1.0) < 0.05          # near-zero scores at the Xavier start: loss = margin
    assert min(v) < v[0] - 0.02                                      # the pocket checkpoint keeps the best one
    E1 = tf_bundle.load_bundle(os.path.join(out, "model.ckpt"))["embeddings"]
    assert np.isfinite(E1).all()
    # --infer in the archived mode: the same all-entity filtered ranking on the raw score
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        flags = hole.build_parser().parse_args(args + ["--infer"])
        m = hole.infer_triples(flags, log=lambda *a: None)
    finally:
        os.chdir(cwd)
    assert 0 < m["filtered_mrr"] <= 1 and m["raw_mean_pos"] >= m["filtered_mean_pos"]
