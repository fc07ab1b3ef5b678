"""Golden-case catalogue shared by ``make_golden.py`` (which runs the unmodified
reference over each case, in the build container) and by the tests (which re-create the
identical inputs from seeds and compare the oracle / the CUDA path with the recorded
reference outputs).

Inputs are never stored except the real-data Episode-53 excerpt; everything else is
regenerated from ``numpy.random.default_rng(seed)`` exactly as the reference's own
benchmark does (tools/benchmark_vectorbase.py:80-94).
"""

from __future__ import annotations

import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
EPISODE53_FILE = os.path.join(HERE, "episode53_excerpt.npy")
GOLDEN_FILE = os.path.join(HERE, "golden_cases.json")

# rows of tests/testdata/Episode_53_AdrianTchaikovsky_index_embeddings.bin kept in the
# excerpt (150 x 1536 float32, under 1 MB): the first 100 related-term rows and the first 50 of
# the 106 message-chunk rows (1188..1293)
EPISODE53_TERMS = 100
EPISODE53_ROWS = list(range(EPISODE53_TERMS)) + list(range(1188, 1238))


def unit_rows(rng, n, d):
    v = rng.standard_normal((n, d)).astype(np.float32)
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    return v


def _bf16(x):
    bits = np.ascontiguousarray(x, np.float32).view(np.uint32).astype(np.uint64)
    r = ((bits + 0x7FFF + ((bits >> 16) & 1)) >> 16) << 16
    return (r & 0xFFFFFFFF).astype(np.uint32).view(np.float32).reshape(x.shape)


def synthetic(n, d, seed, nq=1, storage="float32"):
    rng = np.random.default_rng(seed)
    v = unit_rows(rng, n, d)
    q = unit_rows(rng, nq, d)
    if storage == "bfloat16":
        v, q = _bf16(v), _bf16(q)
    elif storage == "float16":
        v = v.astype(np.float16).astype(np.float32)
        q = q.astype(np.float16).astype(np.float32)
    return v, q


def episode53():
    v = np.load(EPISODE53_FILE)
    # queries: a few term rows and a few message rows, slightly perturbed so that the
    # best hit is not a trivial exact duplicate with score 1.0 only
    rng = np.random.default_rng(53)
    picks = [0, 7, 61, 99, 100, 125, 149]
    q = v[picks] + 0.05 * unit_rows(rng, len(picks), v.shape[1])
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    return v, q.astype(np.float32)


def _mod3(i: int) -> bool:
    return i % 3 == 0


def _odd(i: int) -> bool:
    return i % 2 == 1


PREDICATES = {"mod3": _mod3, "odd": _odd}


# Each case: name, how to build (vectors, queries), and the lookups to record.
# A lookup is (kind, kwargs): kind in {"lookup", "subset", "predicate"}.
CASES: list[dict] = [
    dict(name="bench_1k", make=("synthetic", dict(n=1000, d=384, seed=42)),
         lookups=[("lookup", dict(max_hits=10, min_score=0.0))]),
    dict(name="bench_10k", make=("synthetic", dict(n=10000, d=384, seed=43)),
         lookups=[("lookup", dict(max_hits=10, min_score=0.0)),
                  ("lookup", dict(max_hits=None, min_score=None)),
                  ("lookup", dict(max_hits=50, min_score=0.55)),
                  ("lookup", dict(max_hits=10, min_score=0.58)),
                  ("lookup", dict(max_hits=100, min_score=0.0)),
                  ("lookup", dict(max_hits=10, min_score=0.99)),
                  ("subset", dict(subset=("choice", 99, 10000, 1000), max_hits=10, min_score=0.0)),
                  ("subset", dict(subset=("choice", 7, 10000, 37), max_hits=50, min_score=0.5)),
                  ("predicate", dict(predicate="mod3", max_hits=10, min_score=0.5)),
                  # max_hits=0 on the predicate path slices [:0]: nothing (the argpartition path returns everything)
                  ("predicate", dict(predicate="mod3", max_hits=0, min_score=0.5))]),
    dict(name="tiny_k_exceeds_n", make=("synthetic", dict(n=7, d=5, seed=5)),
         lookups=[("lookup", dict(max_hits=10, min_score=0.0)),
                  ("lookup", dict(max_hits=3, min_score=0.0)),
                  ("lookup", dict(max_hits=1, min_score=0.0))]),
    dict(name="quirk_k0_returns_all_passing", make=("synthetic", dict(n=50, d=8, seed=8)),
         lookups=[("lookup", dict(max_hits=0, min_score=0.5))]),
    dict(name="odd_dims", make=("synthetic", dict(n=333, d=17, seed=17, nq=3)),
         lookups=[("lookup", dict(max_hits=5, min_score=0.0)),
                  ("subset", dict(subset=("list", [5, 5, 9, 332, 0, 5]), max_hits=4, min_score=0.0))]),
    dict(name="dim_1536_batch", make=("synthetic", dict(n=2000, d=1536, seed=1536, nq=4)),
         lookups=[("lookup", dict(max_hits=32, min_score=0.0))]),
    dict(name="dim_100_unaligned", make=("synthetic", dict(n=4100, d=100, seed=100, nq=2)),
         lookups=[("lookup", dict(max_hits=20, min_score=0.45))]),
    dict(name="bf16_768", make=("synthetic", dict(n=4096, d=768, seed=768, nq=8, storage="bfloat16")),
         lookups=[("lookup", dict(max_hits=32, min_score=0.0))]),
    dict(name="f16_384_terms", make=("synthetic", dict(n=5000, d=384, seed=384, nq=8, storage="float16")),
         lookups=[("lookup", dict(max_hits=5, min_score=0.0)),
                  ("lookup", dict(max_hits=5, min_score=0.56))]),
    dict(name="episode53", make=("episode53", dict()),
         lookups=[("lookup", dict(max_hits=50, min_score=0.85)),
                  ("lookup", dict(max_hits=10, min_score=0.7)),
                  ("lookup", dict(max_hits=25, min_score=0.0)),
                  ("subset", dict(subset=("range", EPISODE53_TERMS, len(EPISODE53_ROWS)), max_hits=25,
                                  min_score=0.7))]),
]


def build_inputs(case: dict):
    kind, kw = case["make"]
    if kind == "synthetic":
        return synthetic(**kw)
    if kind == "episode53":
        return episode53()
    raise ValueError(kind)


def build_subset(spec) -> list[int]:
    tag = spec[0]
    if tag == "choice":
        _, seed, n, size = spec
        return np.random.default_rng(seed).choice(n, size=size, replace=False).tolist()
    if tag == "list":
        return list(spec[1])
    if tag == "range":
        return list(range(spec[1], spec[2]))
    raise ValueError(tag)


def reference_lookup(base, q, kind, kw):
    """One recorded lookup through a reference ``VectorBase``."""
    kw = dict(kw)
    if kind == "lookup":
        return base.fuzzy_lookup_embedding(q, **kw)
    if kind == "subset":
        return base.fuzzy_lookup_embedding_in_subset(q, build_subset(kw.pop("subset")), **kw)
    if kind == "predicate":
        return base.fuzzy_lookup_embedding(q, predicate=PREDICATES[kw.pop("predicate")], **kw)
    raise ValueError(kind)


def as_record(hits) -> dict:
    return {"items": [h.item for h in hits], "scores": [h.score for h in hits]}


# Randomised shapes (corpus size and dimension drawn from the seed).  Some lookups return half
# the corpus, so their recorded outputs are kept as arrays in RANDOM_FILE (see random_record).
RANDOM_SEEDS = [1, 2, 3]
RANDOM_FILE = os.path.join(HERE, "random_cases.npz")


def random_key(seed, query, lookup) -> str:
    return f"s{seed}_q{query}_l{lookup}"


def random_record(arrays, seed, query, lookup) -> dict:
    key = random_key(seed, query, lookup)
    return {"items": arrays[key + "_items"].tolist(), "scores": arrays[key + "_scores"].tolist()}


def random_case(seed):
    """(vectors, queries, lookups): lookups[i] is the list of (kind, kwargs) run for query i."""
    from oracle.vectorbase_oracle import make_corpus

    rng = np.random.default_rng(seed)
    n, d = int(rng.integers(50, 3000)), int(rng.choice([3, 64, 384, 769]))
    v, q = make_corpus(n, d, seed, n_queries=3)
    lookups = []
    for _ in q:
        per = [("lookup", dict(max_hits=k, min_score=ms))
               for k, ms in ((10, 0.0), (None, None), (5, 0.5), (n + 5, 0.49), (0, 0.52))]
        subset = rng.choice(n, size=min(n, 40), replace=True).tolist()
        per.append(("subset", dict(subset=("list", subset), max_hits=7, min_score=0.3)))
        per.append(("predicate", dict(predicate="odd", max_hits=6, min_score=0.4)))
        lookups.append(per)
    return v, q, lookups


# Lookups of the Episode-53 excerpt stored as an embedding-file pair: (which part, max_hits,
# min_score), recorded per query under GOLDEN["embedding_file_pair"].
EMBEDDING_FILE_LOOKUPS = [("related", 50, 0.85), ("messages", 10, 0.7), ("messages", 25, 0.0)]


def embedding_file_key(part, max_hits, min_score) -> str:
    return f"{part}/{max_hits}/{min_score}"
