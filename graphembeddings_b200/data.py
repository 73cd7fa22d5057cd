"""Host-side data preparation for the HolE path: file loaders, type->entity CSR, ranking
filter CSR, and the seeded synthetic knowledge graphs BASELINE.json's configs name.

Mirrors holE.py's ``init_data`` (holE.py:44-94) and ``init_inference_data``
(holE.py:381-424).  File formats: SURVEY.md App. C.  Triple column order is
(head, tail, relation) -- holE.py:80-81, 407.
"""
import json
import os
from collections import defaultdict
from dataclasses import dataclass, field

import numpy as np

# --------------------------------------------------------------------------------------
# file loaders
# --------------------------------------------------------------------------------------


def load_triples(path):
    """``head<TAB>tail<TAB>relation`` per line, decimal, no header (holE.py:76-81).

    Returns int32 [T, 3].  An empty file gives shape (0, 3) (the 0712 subset's
    triples-valid.txt is empty)."""
    if os.path.getsize(path) == 0:
        return np.zeros((0, 3), dtype=np.int32)
    fast = _load_triples_native(path)
    if fast is not None:
        return fast
    arr = np.loadtxt(path, dtype=np.int64, delimiter="\t", ndmin=2)
    if arr.shape[1] != 3:
        raise ValueError(f"{path}: expected 3 tab-separated columns, found {arr.shape[1]}")
    if arr.min() < 0 or arr.max() > np.iinfo(np.int32).max:
        raise ValueError(f"{path}: ids out of int32 range")
    return arr.astype(np.int32)


def _load_triples_native(path):
    """The library's mmap parser (hole_parse_triples): ~100x np.loadtxt on 30 M-line files.
    Returns None when the library has not been built (pure-Python fallback for the loader
    only -- this is file parsing, not the compute path)."""
    try:
        import ctypes
        from . import _lib
        lib = _lib.load()
    except Exception:
        return None
    n = lib.hole_parse_triples(path.encode(), None, 0)
    if n < 0:
        raise ValueError(lib.hole_last_error().decode())
    out = np.empty((n, 3), dtype=np.int32)
    m = lib.hole_parse_triples(path.encode(), out.ctypes.data_as(ctypes.c_void_p), n)
    if m != n:
        raise ValueError(f"{path}: changed while reading")
    return out


def check_triple_ids(triples, entity_count, relation_count=None, what="triples"):
    """The reference's embedding_lookup raises InvalidArgument on an out-of-range id; the kernels index
    the table unchecked, so the host checks once per file (one numpy pass)."""
    t = np.asarray(triples)
    if t.size == 0:
        return
    if t.min() < 0:
        raise ValueError(f"{what}: negative id {int(t.min())}")
    if int(t[:, :2].max()) >= entity_count:
        raise ValueError(f"{what}: entity id {int(t[:, :2].max())} >= entity_count {entity_count} "
                         "(entity_metadata.tsv has fewer rows than the triples use)")
    rmax = int(t[:, 2].max())
    if rmax >= entity_count:                  # relations are rows of the same table (holE.py:186, 263-264)
        raise ValueError(f"{what}: relation id {rmax} outside the table of {entity_count} rows")
    if relation_count and rmax >= relation_count:
        raise ValueError(f"{what}: relation id {rmax} >= relation_count {relation_count} (relation_ids.txt)")


def rows_in(a, b):
    """Boolean mask: which triples of `a` [n,3] (a few 1e5 rows) occur in `b` [m,3] (up to 1e8 rows) --
    without walking `b` in Python: `b` is first cut down to the rows whose (head, relation) occurs in `a`
    (one sort-based np.isin over int64 keys)."""
    a = np.asarray(a, dtype=np.int64).reshape(-1, 3)
    b = np.asarray(b, dtype=np.int64).reshape(-1, 3)
    if len(a) == 0 or len(b) == 0:
        return np.zeros(len(a), dtype=bool)
    ka = (a[:, 0] << 32) | a[:, 2]
    kb = (b[:, 0] << 32) | b[:, 2]
    near = b[np.isin(kb, ka)]
    seen = set(map(tuple, near.tolist()))
    return np.fromiter((tuple(x) in seen for x in a.tolist()), dtype=bool, count=len(a))


def count_lines(path):
    """holE.py:52-53 count lines with ``sum(1 for line in open(f))``."""
    with open(path, "rb") as f:
        return sum(1 for _ in f)


@dataclass
class EntityMetadata:
    """Parsed entity_metadata.tsv (holE.py:55-62, 390-399)."""
    entity_count: int = 0                     # every row, relations included (holE.py:58)
    id_to_type: dict = field(default_factory=dict)            # index -> type string
    type_to_ids: dict = field(default_factory=lambda: defaultdict(list))
    id_to_metadata: dict = field(default_factory=dict)        # index -> "id name"
    mentions: dict = field(default_factory=dict)


def load_entity_metadata(path):
    """Header skipped; tab-separated.  The script unpacks 6 columns
    (index, id, name, type, mentions, is_tail -- holE.py:59) but every committed file has 4
    (Index, Id, Name, Type); both are accepted, ``mentions`` defaults to 0."""
    md = EntityMetadata()
    with open(path, "r") as f:
        next(f)
        for line in f:
            cols = line.rstrip("\n").split("\t")
            if len(cols) < 4:
                raise ValueError(f"{path}: metadata row with {len(cols)} columns: {line!r}")
            index = int(cols[0])
            md.entity_count += 1
            md.type_to_ids[cols[3]].append(index)
            md.id_to_type[index] = cols[3]
            md.id_to_metadata[index] = cols[1] + " " + cols[2]
            md.mentions[index] = int(cols[4]) if len(cols) > 4 and cols[4] != "" else 0
    return md


# --------------------------------------------------------------------------------------
# device-table builders (host side; the arrays are uploaded once)
# --------------------------------------------------------------------------------------


def type_arrays(md_or_types, n_rows=None):
    """Dense ``type_of[N] int32`` plus the type-name list, from EntityMetadata (or pass a
    ready type_of array through)."""
    if isinstance(md_or_types, EntityMetadata):
        md = md_or_types
        names = list(md.type_to_ids.keys())
        code = {n: i for i, n in enumerate(names)}
        n = md.entity_count if n_rows is None else n_rows
        type_of = np.zeros(n, dtype=np.int32)
        for idx, t in md.id_to_type.items():
            type_of[idx] = code[t]
        return type_of, names
    return np.asarray(md_or_types, dtype=np.int32), None


def build_type_csr(type_of, n_types=None):
    """type -> entity-id CSR (replaces holE.py's ``type_to_ids`` dict and its per-step
    ``padded_size`` subsample, holE.py:343-347).  ids ascend within a type."""
    type_of = np.asarray(type_of, dtype=np.int64)
    T = int(type_of.max()) + 1 if n_types is None else int(n_types)
    order = np.argsort(type_of, kind="stable")
    counts = np.bincount(type_of, minlength=T)
    off = np.zeros(T + 1, dtype=np.int64)
    np.cumsum(counts, out=off[1:])
    return off, order.astype(np.int32)


def build_filter_csr(queries, known_triples, side):
    """Per-query list of known-true candidates to filter (holE.py:413-422, 454-461).

    side "tail": for query (h, t, r) the known tails of (h, r); side "head": the known
    heads of (t, r); side "relation": the known relations of (h, t).  ``known_triples`` = train +
    valid triples [K, 3].  Returns (off int64[Q+1], ids int32[.]) with ids ascending and
    de-duplicated per query."""
    queries = np.asarray(queries, dtype=np.int64)
    known = np.asarray(known_triples, dtype=np.int64).reshape(-1, 3)
    # (first key column, second key column, value column)
    cols = {"tail": (0, 2, 1), "head": (1, 2, 0), "relation": (0, 1, 2)}.get(side)
    if cols is None:
        raise ValueError(side)
    a, b, v = cols
    kv = known[:, v]
    big = np.int64(1) << 32
    kkey = known[:, a] * big + known[:, b]
    qkey = queries[:, a] * big + queries[:, b]
    order = np.lexsort((kv, kkey))
    kkey, kv = kkey[order], kv[order]
    if len(kkey):                                   # drop repeated (key, value) pairs once, globally
        keep = np.ones(len(kkey), dtype=bool)
        keep[1:] = (kkey[1:] != kkey[:-1]) | (kv[1:] != kv[:-1])
        kkey, kv = kkey[keep], kv[keep]
    lo = np.searchsorted(kkey, qkey, side="left")
    hi = np.searchsorted(kkey, qkey, side="right")
    cnt = hi - lo
    off = np.zeros(len(queries) + 1, dtype=np.int64)
    np.cumsum(cnt, out=off[1:])
    # ids = concatenation of kv[lo[q]:hi[q]] over q, without a Python loop
    take = np.arange(off[-1], dtype=np.int64) - np.repeat(off[:-1] - lo, cnt)
    return off, kv[take].astype(np.int32)


# --------------------------------------------------------------------------------------
# synthetic knowledge graphs (SURVEY.md section 8d)
# --------------------------------------------------------------------------------------


@dataclass
class SyntheticKG:
    n_relations: int
    n_entities: int
    dim: int
    triples: np.ndarray        # int32 [T, 3] (h, t, r); entity ids offset by n_relations
    type_of: np.ndarray        # int32 [N]; type 0 = relation rows
    E: np.ndarray              # float32 [N, dim]

    @property
    def n_rows(self):
        return self.n_relations + self.n_entities


def xavier_stddev(n_rows, dim):
    """holE.py:263-264 via xavier_initializer(uniform=False): sqrt(2.6 / (N + D))."""
    return float(np.sqrt(2.6 / (n_rows + dim)))


def init_embeddings(n_rows, dim, rng, trained_scale=False):
    """Truncated-normal Xavier init (holE.py:263-264), or a "trained-scale" table whose row
    norms are ~U(0.5, 1.5) so that the norm clip and its backward are exercised."""
    sd = xavier_stddev(n_rows, dim)
    x = rng.standard_normal((n_rows, dim), dtype=np.float32)
    bad = np.abs(x) > 2.0
    while bad.any():
        x[bad] = rng.standard_normal(int(bad.sum()), dtype=np.float32)
        bad = np.abs(x) > 2.0
    if trained_scale:
        norms = np.linalg.norm(x, axis=1, keepdims=True)
        target = rng.uniform(0.5, 1.5, size=(n_rows, 1)).astype(np.float32)
        return (x / norms * target).astype(np.float32)
    return (x * np.float32(sd)).astype(np.float32)


def _zipf_choice(rng, n, size, s=1.0):
    w = 1.0 / np.arange(1, n + 1, dtype=np.float64) ** s
    cdf = np.cumsum(w / w.sum())
    return np.minimum(np.searchsorted(cdf, rng.random(size)), n - 1).astype(np.int64)


def synthetic_kg(n_relations, n_entities, n_triples, n_types, dim, seed, zipf_entities=False,
                 trained_scale=False, type_histogram=None, dominant_type_frac=None,
                 with_embeddings=True):
    """Seeded synthetic KG.  Rows 0..n_relations-1 are relations (type 0), entity rows
    follow (SURVEY.md section 0, surprise 3).  Relations ~ Zipf(1); entities uniform or
    Zipf(1) (duplicate-index stress)."""
    rng = np.random.default_rng(seed)
    N = n_relations + n_entities
    if type_histogram is not None:
        hist = np.asarray(type_histogram, dtype=np.int64)
        assert hist.sum() == n_entities
        ent_type = np.repeat(np.arange(1, len(hist) + 1), hist)
        rng.shuffle(ent_type)
    elif dominant_type_frac is not None:
        p = np.full(n_types, (1.0 - dominant_type_frac) / max(n_types - 1, 1))
        p[0] = dominant_type_frac
        ent_type = 1 + rng.choice(n_types, size=n_entities, p=p)
    else:
        ent_type = 1 + rng.integers(0, n_types, size=n_entities)
    type_of = np.concatenate([np.zeros(n_relations, dtype=np.int64), ent_type]).astype(np.int32)
    r = _zipf_choice(rng, n_relations, n_triples)
    if zipf_entities:
        perm = rng.permutation(n_entities)
        h = perm[_zipf_choice(rng, n_entities, n_triples)]
        t = perm[_zipf_choice(rng, n_entities, n_triples)]
    else:
        h = rng.integers(0, n_entities, size=n_triples)
        t = rng.integers(0, n_entities, size=n_triples)
    triples = np.stack([h + n_relations, t + n_relations, r], axis=1).astype(np.int32)
    E = init_embeddings(N, dim, rng, trained_scale) if with_embeddings else None
    return SyntheticKG(n_relations, n_entities, dim, triples, type_of, E)


def fb15k_type_histogram():
    """The 815-class entity type histogram of the real FB15k metadata (372 singletons): package data,
    written by tests/golden/make_golden.py from diffbot_data/FB15k/entity_metadata.tsv."""
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "fb15k_types.json")) as f:
        return json.load(f)["entity_type_histogram"]


#: BASELINE.json configs -> generator arguments (SURVEY.md section 8d; seeds 20170903+k)
CONFIGS = {
    "fb15k_d150": dict(n_relations=1345, n_entities=14951, n_triples=483142, n_types=815,
                       dim=150, seed=20170903),
    "diffbot_d256": dict(n_relations=14, n_entities=1200000, n_triples=30000000, n_types=12,
                         dim=256, seed=20170904, dominant_type_frac=0.99),
    "rank_fb15k_d150": dict(n_relations=1345, n_entities=14951, n_triples=59071, n_types=815,
                            dim=150, seed=20170905),
    "rank_diffbot_d256": dict(n_relations=14, n_entities=1200000, n_triples=100000,
                              n_types=12, dim=256, seed=20170906, dominant_type_frac=0.99),
    "sharded_d512": dict(n_relations=32, n_entities=20000000, n_triples=500000000,
                         n_types=12, dim=512, seed=20170907, dominant_type_frac=0.99),
}


def make_config(name, n_triples=None, **overrides):
    """Instantiate one of BASELINE.json's configs (optionally with fewer triples)."""
    kw = dict(CONFIGS[name])
    if n_triples is not None:
        kw["n_triples"] = n_triples
    kw.update(overrides)
    if name in ("fb15k_d150", "rank_fb15k_d150") and "type_histogram" not in kw:
        kw["type_histogram"] = fb15k_type_histogram()
    return synthetic_kg(**kw)
