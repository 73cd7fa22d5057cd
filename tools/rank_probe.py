"""Ranking kernel probe: times the ranking call on config 2 (FB15k shape) and a reduced config 3.

PROBE_ZERO=1 ranks all-zero tables, PROBE_Q3 sets the config 3 query count (default 20000) and PROBE_ENV is a
label printed on the timing line (tools/rank_ab.sh passes the library's name)."""
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from graphembeddings_b200 import data as D
from graphembeddings_b200.engine import HOLE_SIDE_BOTH, HOLE_SIDE_TAIL, HoleEngine
from graphembeddings_b200.rank_bench import time_rank


def main():
    kg2 = D.make_config("rank_fb15k_d150", trained_scale=True)
    e2 = HoleEngine(kg2.n_rows, kg2.dim).set_embeddings(kg2.E)
    kg3 = D.make_config("diffbot_d256", n_triples=100000)
    e3 = HoleEngine(kg3.n_rows, kg3.dim).set_embeddings(kg3.E)
    if os.environ.get("PROBE_ZERO") == "1":       # all-zero operands: the same instruction stream at minimal switching power
        e2.set_embeddings(np.zeros_like(kg2.E))
        e3.set_embeddings(np.zeros_like(kg3.E))
    rng = np.random.default_rng(1)
    q3 = kg3.triples[rng.integers(0, len(kg3.triples), size=int(os.environ.get("PROBE_Q3", "20000")))]
    extra = os.environ.get("PROBE_ENV", "")
    ms2, _, _ = time_rank(e2, kg2.triples, kg2.n_relations, kg2.n_rows, sides=(HOLE_SIDE_BOTH,))
    ms3, _, _ = time_rank(e3, q3, kg3.n_relations, kg3.n_rows, sides=(HOLE_SIDE_TAIL,), reps=2)
    tf2 = 2 * len(kg2.triples) * kg2.n_entities * 2 * kg2.dim / ms2 / 1e9
    tf3 = len(q3) * kg3.n_entities * 2 * kg3.dim / ms3 / 1e9
    print(f"rank {extra}: cfg2 {ms2:.3f} ms {tf2:.0f} TF/s | cfg3 {ms3:.3f} ms {tf3:.0f} TF/s", flush=True)
    print(json.dumps({"cfg2_ms": ms2, "cfg2_tflops": tf2, "cfg3_ms": ms3, "cfg3_tflops": tf3}))


if __name__ == "__main__":
    main()
