"""Host-side mirror of holE.py: loaders, flags, metrics (no GPU needed)."""
import json
import os
import re

import numpy as np
import pytest

from graphembeddings_b200 import data as D
from graphembeddings_b200 import hole


def test_load_triples_real_fb15k_head(golden_dir):
    t = D.load_triples(os.path.join(golden_dir, "fb15k_test_positive_triples_head.txt"))
    assert t.dtype == np.int32 and t.shape == (2000, 3)
    assert tuple(t[0]) == (13839, 4403, 733)              # diffbot_data/FB15k/test_positive_triples.txt:1
    # column order (head, tail, relation): relations are rows 0..1344, entities 1345..16295
    assert t[:, 2].max() < 1345 and t[:, :2].min() >= 1345


def test_load_triples_empty_file(tmp_path):
    p = tmp_path / "triples-valid.txt"                    # prepareSubset-20170712/triples-valid.txt is empty
    p.write_text("")
    assert D.load_triples(str(p)).shape == (0, 3)


def test_metadata_accepts_4_and_6_columns(golden_dir, tmp_path):
    md = D.load_entity_metadata(os.path.join(golden_dir, "fb15k_metadata_head.tsv"))
    assert md.entity_count == 100 and md.id_to_type[0] == "RELATION"
    assert all(v == 0 for v in md.mentions.values())
    p = tmp_path / "entity_metadata.tsv"
    p.write_text("Index\tId\tName\tType\tMentions\tIsTail\n0\t!r0\trel\t!\t0\tfalse\n1\tP1\tAnn\tP\t70000\ttrue\n")
    md6 = D.load_entity_metadata(str(p))
    assert md6.entity_count == 2 and md6.mentions[1] == 70000 and md6.id_to_type[1] == "P"


def test_type_csr_and_filter_csr():
    type_of = np.array([0, 0, 1, 2, 1, 1, 2], dtype=np.int32)
    off, ids = D.build_type_csr(type_of)
    assert off.tolist() == [0, 2, 5, 7] and ids.tolist() == [0, 1, 2, 4, 5, 3, 6]
    q = np.array([[10, 20, 1], [11, 21, 2]])
    known = np.array([[10, 22, 1], [10, 23, 1], [10, 22, 1], [12, 21, 2], [10, 24, 3]])
    fo, fi = D.build_filter_csr(q, known, "tail")
    assert fo.tolist() == [0, 2, 2] and fi.tolist() == [22, 23]
    fo, fi = D.build_filter_csr(q, known, "head")
    assert fo.tolist() == [0, 0, 1] and fi.tolist() == [12]


def test_flags_match_reference_defaults():
    f = hole.build_parser().parse_args(["--output_dir", "o", "--data_dir", "d"])
    want = dict(learning_rate=0.1, learning_decay_steps=32, learning_decay_rate=0.5, batch_size=512,
                num_epochs=1000, embedding_dim=128, log_loss=False, l2_regularization=0.1,
                negative_ratio=1, margin=0.2, padded_size=1024, reader_threads=4,
                resume_checkpoint=False, save_embeddings=False, infer=False, infer_threshold=0.05,
                min_mentions=50000)                       # holE.py:598-619
    for k, v in want.items():
        assert getattr(f, k) == v, k


def test_score_mrr_matches_reference_stdout(golden_dir):
    g = json.load(open(os.path.join(golden_dir, "ranking_ref.json")))
    raw = [x for c in g["cases"] for x in c["raw_positions"]]
    filt = [x for c in g["cases"] for x in c["filtered_positions"]]
    lines = []
    hole.score_mrr(raw, filt, log=lines.append)
    assert "\n".join(lines) + "\n" == g["score_mrr_stdout"]      # byte-identical report


def test_init_inference_data_semantics(tmp_path):
    d = tmp_path
    (d / "entity_metadata.tsv").write_text(
        "Index\tId\tName\tType\tMentions\tIsTail\n"
        "0\t!a\tr0\t!\t0\tf\n1\tP1\tAnn\tP\t0\tt\n2\tS2\tjava\tS\t60000\tt\n3\tS3\tcobol\tS\t10\tt\n")
    (d / "relation_ids.txt").write_text("r0\t0\n")
    (d / "triples.txt").write_text("1\t2\t0\n3\t2\t0\n")
    (d / "triples-valid.txt").write_text("")
    (d / "test_positive_triples.txt").write_text("1\t3\t0\n")
    flags = hole.build_parser().parse_args(["--output_dir", "o", "--data_dir", str(d)])
    inf = hole.init_inference_data(flags)
    assert inf.relation_count == 1 and inf.entity_count == 4
    assert inf.type_to_ids["S"] == [2]                    # min_mentions filter (holE.py:397)
    assert inf.type_to_ids["P"] == [1]                    # ids starting with 'P' always kept
    assert inf.test_triples[1][0] == {3}
    assert inf.true_triples[1][0] == {2}                  # only (h, r) pairs present in test (holE.py:421)
    assert 3 not in inf.true_triples


def test_lr_schedule_matches_oracle():
    from graphembeddings_b200.engine import inverse_time_decay
    from oracle import hole_oracle as O
    for step in (0, 1, 1000, 123456):
        assert inverse_time_decay(0.1, step, 32 * 943, 0.5) == O.inverse_time_decay(0.1, step, 32 * 943, 0.5)


def test_native_triple_parser_matches_numpy(tmp_path, golden_dir):
    from graphembeddings_b200 import build
    build.build()
    src = os.path.join(golden_dir, "fb15k_triples-valid_head.txt")
    want = np.loadtxt(src, dtype=np.int64, delimiter="\t").astype(np.int32)
    got = D.load_triples(src)
    assert got.dtype == np.int32 and np.array_equal(got, want)
    # no trailing newline, CRLF, blank line at the end
    p = tmp_path / "t.txt"
    p.write_bytes(b"1\t2\t3\r\n40\t50\t6\n\n7\t8\t9")
    assert D.load_triples(str(p)).tolist() == [[1, 2, 3], [40, 50, 6], [7, 8, 9]]
    bad = tmp_path / "bad.txt"
    bad.write_text("1\t2\n")
    with pytest.raises(ValueError):
        D.load_triples(str(bad))
    neg = tmp_path / "neg.txt"
    neg.write_text("1\t-2\t3\n")
    with pytest.raises(ValueError):
        D.load_triples(str(neg))


def test_event_file_round_trip_and_tensorboard_can_read_it(tmp_path):
    """The events file of --output_dir (holE.py:317, 353): TFRecord framing with masked CRC32C, Event /
    Summary protos encoded by hand -- parsed back by our reader and by TensorBoard's own proto classes."""
    from graphembeddings_b200 import tf_events as T
    rng = np.random.default_rng(0)
    vals = rng.uniform(0.27, 0.73, 1000)
    w = T.EventFileWriter(str(tmp_path))
    sc, hi = T.summarize_tags("validation/positive/eval", vals)          # holE.py:237-246
    sc["batch/learn/learning_rate"] = 0.1
    w.add_summary(7, sc, hi)
    w.add_summary(123456789012, {"x": -1.5})
    w.close()
    ev = T.read_events(w.path)
    assert [e["step"] for e in ev] == [0, 7, 123456789012] and ev[0]["file_version"] == "brain.Event:2"
    assert abs(ev[1]["scalars"]["validation/positive/eval/summaries/mean"] - vals.mean()) < 1e-6
    assert abs(ev[1]["scalars"]["validation/positive/eval/summaries/stddev_1"] - vals.std()) < 1e-6
    assert ev[2]["scalars"] == {"x": -1.5}
    h = ev[1]["histograms"]["validation/positive/eval/summaries/histogram"]
    assert h["num"] == 1000 and h["min"] == vals.min() and h["max"] == vals.max()
    assert abs(h["sum"] - vals.sum()) < 1e-9 and h["bucket"].sum() == 1000
    assert len(h["bucket"]) == len(h["bucket_limit"]) and np.all(np.diff(h["bucket_limit"]) > 0)
    # every value falls in the bucket whose limit is the first one >= value
    assert h["bucket_limit"][-1] >= vals.max() and h["bucket_limit"][0] >= vals.min()
    event_pb2 = pytest.importorskip("tensorboard.compat.proto.event_pb2")
    import struct
    buf = open(w.path, "rb").read()
    pos, n_ok = 0, 0
    while pos < len(buf):
        (n,) = struct.unpack_from("<Q", buf, pos)
        e = event_pb2.Event()
        e.ParseFromString(buf[pos + 12:pos + 12 + n])
        if n_ok == 1:
            got = {v.tag: v.simple_value for v in e.summary.value if v.HasField("simple_value")}
            assert abs(got["batch/learn/learning_rate"] - 0.1) < 1e-7 and e.step == 7
            hp = [v for v in e.summary.value if v.HasField("histo")][0].histo
            assert hp.num == 1000 and len(hp.bucket) == len(h["bucket"])
        pos += 16 + n
        n_ok += 1
    assert n_ok == 3
    # a flipped byte is caught by the record CRC
    bad = bytearray(buf)
    bad[40] ^= 1
    p2 = tmp_path / "bad"
    p2.write_bytes(bytes(bad))
    with pytest.raises(ValueError):
        T.read_events(str(p2))


def test_rows_in_and_id_checks():
    known = np.array([[1, 2, 0], [1, 3, 0], [4, 2, 1], [1, 2, 0]], dtype=np.int32)
    q = np.array([[1, 2, 0], [1, 2, 1], [4, 2, 1], [9, 9, 0]], dtype=np.int32)
    assert D.rows_in(q, known).tolist() == [True, False, True, False]
    assert D.rows_in(q, np.zeros((0, 3), np.int32)).tolist() == [False] * 4
    rng = np.random.default_rng(1)
    a = rng.integers(0, 50, size=(300, 3)).astype(np.int32)
    b = rng.integers(0, 50, size=(5000, 3)).astype(np.int32)
    want = [tuple(x) in set(map(tuple, b.tolist())) for x in a.tolist()]
    assert D.rows_in(a, b).tolist() == want
    D.check_triple_ids(np.array([[5, 6, 1]]), 7, 2)
    for bad in ([[5, 7, 1]], [[-1, 6, 1]], [[5, 6, 2]], [[5, 6, 9]]):
        with pytest.raises(ValueError):
            D.check_triple_ids(np.array(bad), 7, 2)
    D.check_triple_ids(np.zeros((0, 3), np.int32), 7, 2)               # an empty file is fine


@pytest.mark.parametrize("W", [1, 2, 3, 5, 8])
def test_bench_warm_up_issues_exactly_w_steps_in_order(W):
    """bench.py's warm-up is W steps, issued as two calls (the second training call of a context still carries
    one-time costs): consecutive triples, consecutive step numbers, nothing skipped or repeated."""
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench

    class Rows:                      # stands in for the device triple tensor: records the slices taken
        def __getitem__(self, sl):
            return (sl.start, sl.stop)

    class Eng:
        calls = []

        def train_steps(self, tri, B, seed, first_step, margin, lrs):
            self.calls.append((tri, first_step, len(lrs)))

    B, e = 64, Eng()
    bench.warm_up(e, Rows(), B, W, 7, 1000)
    assert 1 <= len(e.calls) <= 2
    nxt = 0
    for (lo, hi), first_step, n in e.calls:
        assert lo == nxt * B and hi == (nxt + n) * B and first_step == 7 + nxt and n >= 1
        nxt += n
    assert nxt == W


def test_bench_dump_outputs_are_seeded_and_bounded(tmp_path):
    """bench.py --dump-outputs: the same rows on every run, every relation row among them, under 64 MB at the
    headline shape (1,200,014 rows x d=256, B=32768), written as float32 / float64 .npy files."""
    import sys
    import types
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench

    kg = types.SimpleNamespace(n_relations=14, n_rows=1_200_014)
    last = np.random.default_rng(0).integers(14, kg.n_rows, size=(32768, 3))
    rows = bench.dump_rows(kg, last)
    assert np.array_equal(rows, bench.dump_rows(kg, last))
    assert np.array_equal(rows[:14], np.arange(14)) and rows[-1] < kg.n_rows
    assert np.isin(rows, last[:, :2]).sum() >= bench.DUMP_SAMPLE
    assert len(rows) * 256 * 4 + 8 * len(rows) < 64 << 20
    table_rows = np.random.default_rng(1).standard_normal((len(rows), 256)).astype(np.float32)
    bench.write_dump(str(tmp_path), np.arange(5, dtype=np.float32), rows, table_rows)
    got = {p.stem: np.load(p) for p in tmp_path.iterdir()}
    assert sorted(got) == ["embedding_rows", "embeddings", "loss_sums"]
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert np.array_equal(got["embedding_rows"], rows) and np.array_equal(got["embeddings"], table_rows)
