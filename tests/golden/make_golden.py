#!/usr/bin/env python3
"""Generate the committed golden vectors by running the UNMODIFIED reference.

Run in the build container only (needs /root/reference):

    python tests/golden/make_golden.py

Writes ``golden_cases.json`` (reference outputs: items + float32 scores as Python
floats, which round-trip exactly through JSON) and ``episode53_excerpt.npy`` (150 of
the 1294 real embedding rows of the reference's Episode-53 test fixture).  Also records
the reference's own known-answer tests as literal cases, and the outputs of the randomised
cases as arrays in ``random_cases.npz``.
"""

from __future__ import annotations

import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle.ref_loader import make_reference_vectorbase  # noqa: E402
from tests.golden import cases as C  # noqa: E402

EP53_BIN = "/root/reference/tests/testdata/Episode_53_AdrianTchaikovsky_index_embeddings.bin"


def main() -> None:
    full = np.fromfile(EP53_BIN, dtype=np.float32).reshape(-1, 1536)
    assert full.shape == (1294, 1536), full.shape
    np.save(C.EPISODE53_FILE, np.ascontiguousarray(full[C.EPISODE53_ROWS]))

    out: dict = {"numpy": np.__version__, "cases": {}}
    for case in C.CASES:
        vectors, queries = C.build_inputs(case)
        base = make_reference_vectorbase(vectors)
        recorded = [[C.as_record(C.reference_lookup(base, q, kind, kw)) for q in queries]
                    for kind, kw in case["lookups"]]
        out["cases"][case["name"]] = recorded
        print(f"{case['name']}: {len(recorded)} lookups x {len(queries)} queries")

    arrays = {}
    for seed in C.RANDOM_SEEDS:
        vectors, queries, lookups = C.random_case(seed)
        base = make_reference_vectorbase(vectors)
        for qi, (q, per) in enumerate(zip(queries, lookups)):
            for li, (kind, kw) in enumerate(per):
                hits = C.reference_lookup(base, q, kind, kw)
                key = C.random_key(seed, qi, li)
                arrays[key + "_items"] = np.array([h.item for h in hits], np.int32)
                arrays[key + "_scores"] = np.array([h.score for h in hits], np.float32)   # exact: float32 scores
    np.savez_compressed(C.RANDOM_FILE, **arrays)

    # Episode-53 excerpt split as an embedding-file pair (related terms, message chunks)
    ep, epq = C.episode53()
    parts = {"related": make_reference_vectorbase(ep[:C.EPISODE53_TERMS]),
             "messages": make_reference_vectorbase(ep[C.EPISODE53_TERMS:])}
    out["embedding_file_pair"] = {
        C.embedding_file_key(part, k, ms): [C.as_record(parts[part].fuzzy_lookup_embedding(q, max_hits=k, min_score=ms))
                                            for q in epq]
        for part, k, ms in C.EMBEDDING_FILE_LOOKUPS}

    # state of a VectorBase after the calls of test_oracle_class_matches_reference_class_api
    base = make_reference_vectorbase()
    base.add_embedding(None, [0.7, 0.8, 0.9])
    base.add_embeddings(None, np.array([[0.1, 0.2, 0.3], [0.4, 0.5, 0.6]], np.float32))
    out["class_api_serialized"] = base.serialize().tolist()

    # The reference's own known-answer test (tests/test_vectorbase.py:239-252).
    base = make_reference_vectorbase()
    for row in ([1.0, 0.0], [0.0, 1.0], [-1.0, 0.0]):
        base.add_embedding(None, np.array(row, dtype=np.float32))
    hits = base.fuzzy_lookup_embedding(np.array([1.0, 0.0], dtype=np.float32), max_hits=3, min_score=0.0)
    kat = {"items": [h.item for h in hits], "scores": [h.score for h in hits]}
    assert kat == {"items": [0, 1, 2], "scores": [1.0, 0.5, 0.0]}, kat
    out["known_answer_score_scale"] = kat

    with open(C.GOLDEN_FILE, "w") as f:
        json.dump(out, f)
    print("wrote", C.GOLDEN_FILE, os.path.getsize(C.GOLDEN_FILE), "bytes")


if __name__ == "__main__":
    main()
