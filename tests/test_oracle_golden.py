"""Pin the CPU oracle (oracle/vectorbase_oracle.py) against the reference.

1. committed golden vectors generated from the unmodified reference
   (tests/golden/make_golden.py);
2. the reference's own known-answer tests (tests/test_vectorbase.py:239-252, :209-236);
3. the reference on randomised shapes and through its class API: recorded outputs, and the live
   reference as well where its sources can be loaded (``oracle/ref_loader.py``).
"""

from __future__ import annotations

import json

import numpy as np
import pytest

from oracle import vectorbase_oracle as O
from oracle.ref_loader import make_reference_vectorbase, reference_available
from tests.golden import cases as C
from tests.parity import assert_hits_match

with open(C.GOLDEN_FILE) as _f:
    GOLDEN = json.load(_f)


def run_oracle_lookup(vectors, q, kind, kw):
    kw = dict(kw)
    if kind == "lookup":
        return O.lookup(vectors, q, **kw)
    if kind == "subset":
        subset = C.build_subset(kw.pop("subset"))
        return O.lookup_in_subset(vectors, q, subset, **kw)
    if kind == "predicate":
        pred = C.PREDICATES[kw.pop("predicate")]
        return O.lookup(vectors, q, predicate=pred, **kw)
    raise ValueError(kind)


@pytest.mark.parametrize("case", C.CASES, ids=[c["name"] for c in C.CASES])
def test_oracle_matches_golden(case):
    vectors, queries = C.build_inputs(case)
    recorded = GOLDEN["cases"][case["name"]]
    for (kind, kw), per_query in zip(case["lookups"], recorded):
        for qi, (q, want) in enumerate(zip(queries, per_query)):
            got = run_oracle_lookup(vectors, q, kind, kw)
            # same numpy primitives in the same order: agreement to summation-order noise
            # (bit-exact on the machine that generated the goldens)
            assert_hits_match(got, want, score_tol=2e-6, min_score=kw.get("min_score"),
                              what=f"{case['name']}/{kind}/{kw}/q{qi}")


def test_known_answer_score_scale():
    """reference tests/test_vectorbase.py:239-252: exact [1.0, 0.5, 0.0]."""
    v = np.array([[1, 0], [0, 1], [-1, 0]], dtype=np.float32)
    hits = O.lookup(v, np.array([1, 0], dtype=np.float32), max_hits=3, min_score=0.0)
    assert [h.item for h in hits] == [0, 1, 2]
    assert [h.score for h in hits] == [1.0, 0.5, 0.0]
    assert GOLDEN["known_answer_score_scale"] == {"items": [0, 1, 2], "scores": [1.0, 0.5, 0.0]}


def test_known_answer_subset_cases():
    """reference tests/test_vectorbase.py:209-236."""
    v = np.array([[0.1, 0.2, 0.3], [0.4, 0.5, 0.6], [0.7, 0.8, 0.9]], dtype=np.float32)
    q = v[0]
    assert 0 in [h.item for h in O.lookup_in_subset(v, q, [0, 1, 2])]
    one = O.lookup_in_subset(v, q, [1])
    assert len(one) == 1 and one[0].item == 1
    assert O.lookup_in_subset(v, q, []) == []
    assert O.lookup(np.zeros((0, 3), np.float32), q) == []


def test_bf16_rounding_is_rne_and_idempotent():
    x = np.array([1.0, 1.00390625, 1.005859375, -0.3333333, 3.0e-39, 65504.0], np.float32)
    r = O.round_to_bfloat16(x)
    assert np.all((r.view(np.uint32) & 0xFFFF) == 0)
    np.testing.assert_array_equal(O.round_to_bfloat16(r), r)
    # 1 + 2^-8 is exactly half-way between bf16 neighbours 1.0 and 1+2^-7: ties to even -> 1.0
    assert r[1] == np.float32(1.0)
    # 1 + 2^-8 + 2^-9 rounds up
    assert r[2] == np.float32(1.0078125)
    try:
        import torch
        t = torch.from_numpy(x).to(torch.bfloat16).to(torch.float32).numpy()
        np.testing.assert_array_equal(t, r)
    except ImportError:
        pass


def test_sharded_equals_unsharded():
    v, q = O.make_corpus(3001, 64, seed=11, n_queries=3)
    for qq in q:
        want = O.lookup(v, qq, 20, 0.4)
        for g in (1, 2, 3, 8):
            got = O.lookup_sharded(v, qq, g, 20, 0.4)
            assert_hits_match(got, want, score_tol=2e-6, min_score=0.4, what=f"shards={g}")


def test_fake_embedding_known_values():
    """model_adapters.py:375-404: 'a' -> hash 97 -> 97/1961 in every component -> unit vector."""
    e = O.fake_text_embedding("a", 4)
    np.testing.assert_allclose(e, np.full(4, 0.5, np.float32), rtol=1e-6)
    e2 = O.fake_text_embedding("ab", 2)
    h_ab = (97 * 31 + 98) % 1961 / 1961
    h_ba = (98 * 31 + 97) % 1961 / 1961
    want = np.array([h_ab, h_ba], np.float32)
    want /= np.linalg.norm(want)
    np.testing.assert_allclose(e2, want, rtol=1e-6)
    with pytest.raises(ValueError):
        O.fake_text_embedding("", 3)


@pytest.mark.parametrize("seed", C.RANDOM_SEEDS)
def test_oracle_matches_live_reference(seed):
    """Randomised shapes: the oracle against the reference's recorded outputs and, where the
    reference sources can be loaded, against the live reference bit for bit."""
    v, q, lookups = C.random_case(seed)
    ref = make_reference_vectorbase(v) if reference_available() else None
    with np.load(C.RANDOM_FILE) as arrays:
        for qi, (qq, per) in enumerate(zip(q, lookups)):
            for li, (kind, kw) in enumerate(per):
                got = run_oracle_lookup(v, qq, kind, kw)
                assert_hits_match(got, C.random_record(arrays, seed, qi, li), score_tol=2e-6,
                                  min_score=kw.get("min_score"), what=f"seed {seed}/q{qi}/{kind}/{kw}")
                if ref is not None:
                    want = C.reference_lookup(ref, qq, kind, kw)
                    assert [(h.item, h.score) for h in got] == [(h.item, h.score) for h in want]


def test_oracle_class_matches_reference_class_api():
    """Same state after the same calls as the reference (recorded, and live where its sources can
    be loaded); same errors (tests/test_vectorbase.py:72-102,255-277)."""
    from types import SimpleNamespace

    model = O.FakeEmbeddingModel()
    mine = O.OracleVectorBase(SimpleNamespace(embedding_model=model, min_score=0.85, max_matches=None))
    ref = make_reference_vectorbase() if reference_available() else None
    rows = np.array([[0.1, 0.2, 0.3], [0.4, 0.5, 0.6]], np.float32)
    for b in (mine, ref) if ref is not None else (mine,):
        assert len(b) == 0 and bool(b) is True
        b.add_embedding(None, [0.7, 0.8, 0.9])
        b.add_embeddings(None, rows)
        with pytest.raises(ValueError, match="Embedding size mismatch"):
            b.add_embedding(None, np.zeros(5, np.float32))
        with pytest.raises(ValueError, match="Expected 2D"):
            b.add_embeddings(None, rows[0])
        with pytest.raises(IndexError):
            b.get_embedding_at(3)
        assert b.serialize_embedding_at(9) is None
    np.testing.assert_array_equal(mine.serialize(), np.array(GOLDEN["class_api_serialized"], np.float32))
    if ref is not None:
        np.testing.assert_array_equal(mine.serialize(), ref.serialize())
        ref.clear()
        assert ref.serialize().shape == (0, 3)
    mine.clear()
    assert mine.serialize().shape == (0, 3)
