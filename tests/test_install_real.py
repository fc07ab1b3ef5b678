"""``install()`` against the REAL reference modules (SURVEY.md §8 a11, f1): the unmodified
``knowpro/fuzzyindex.py``, ``storage/memory/reltermsindex.py``, ``storage/memory/convthreads.py``,
``storage/sqlite/{reltermsindex,messageindex}.py`` loaded in place (``/root/reference`` in the build
container, the vendored ``oracle/_ref`` copy on the GPU box; ``oracle/ref_loader.py``).

CPU part: the names are rebound and the two sequential ``lookup_terms`` loops are replaced, and
``uninstall()`` restores everything.  GPU part: index classes BUILT BY THE REFERENCE'S OWN CODE after
``install()`` return the hits the reference returns on numpy — for the Episode-53 excerpt (real
1536-dim embeddings) and for a synthetic vocabulary large enough for the tensor-core path, through the
batched ``lookup_terms`` (one GPU search for all query terms) — and a ``write_embedding_file`` pair
read back through ``formats.load_embedding_file`` is searchable.
"""

from __future__ import annotations

import asyncio
import hashlib
import json
import os
import sqlite3

import numpy as np
import pytest

import typeagent_py_b200 as tab
from oracle import ref_loader
from oracle import vectorbase_oracle as O
from tests.golden import cases as C
from tests.parity import assert_hits_match

needs_reference = pytest.mark.skipif(not ref_loader.reference_available(),
                                     reason="reference sources neither mounted nor vendored")

MODULES = [
    "typeagent.aitools.vectorbase",
    "typeagent.knowpro.fuzzyindex",
    "typeagent.storage.memory.reltermsindex",
    "typeagent.storage.memory.convthreads",
    "typeagent.storage.sqlite.messageindex",
    "typeagent.storage.sqlite.reltermsindex",
]


def load_all():
    return {name: ref_loader.load_reference_module(name) for name in MODULES}


class DictEmbeddingModel:
    """text -> fixed embedding (an IEmbeddingModel with a pre-filled cache, aitools/embeddings.py:39-114)."""

    model_name = "dict"

    def __init__(self, table):
        self.table = dict(table)

    def add_embedding(self, key, embedding):
        self.table[key] = np.asarray(embedding, np.float32)

    async def get_embedding(self, key):
        return self.table[key]

    async def get_embeddings(self, keys):
        if not keys:
            raise ValueError("Cannot embed an empty list")
        return np.stack([self.table[k] for k in keys]).astype(np.float32)

    get_embedding_nocache = get_embedding
    get_embeddings_nocache = get_embeddings


@needs_reference
def test_vendored_reference_files_are_unmodified():
    """oracle/_ref (when it is what we load) is a byte-for-byte copy: sha256 per its manifest, and —
    in the build container — equal to the mounted tree."""
    ref_dir = os.path.join(os.path.dirname(ref_loader.__file__), "_ref")
    manifest = os.path.join(ref_dir, "MANIFEST.json")
    if not os.path.exists(manifest):
        pytest.skip("no vendored copy here")
    with open(manifest) as f:
        files = json.load(f)["files"]
    assert "typeagent/aitools/vectorbase.py" in files and len(files) > 20
    for rel, digest in files.items():
        with open(os.path.join(ref_dir, rel), "rb") as f:
            data = f.read()
        assert hashlib.sha256(data).hexdigest() == digest, rel
        mounted = os.path.join("/root/reference/src", rel)
        if os.path.exists(mounted):
            with open(mounted, "rb") as f:
                assert f.read() == data, rel


@needs_reference
def test_install_rebinds_the_real_modules_and_uninstall_restores_them():
    mods = load_all()
    originals = {name: m.VectorBase for name, m in mods.items()}
    rel_mem = mods["typeagent.storage.memory.reltermsindex"]
    rel_sql = mods["typeagent.storage.sqlite.reltermsindex"]
    orig_mem = rel_mem.TermEmbeddingIndex.lookup_terms
    orig_sql = rel_sql.SqliteRelatedTermsFuzzy.lookup_terms
    try:
        patched = tab.install()
        assert sorted(p for p in patched if p.endswith(".VectorBase")) == sorted(f"{m}.VectorBase" for m in MODULES)
        assert "typeagent.storage.memory.reltermsindex.TermEmbeddingIndex.lookup_terms" in patched
        assert "typeagent.storage.sqlite.reltermsindex.SqliteRelatedTermsFuzzy.lookup_terms" in patched
        for m in mods.values():
            assert m.VectorBase is tab.VectorBase
        assert rel_mem.TermEmbeddingIndex.lookup_terms is not orig_mem
        assert rel_sql.SqliteRelatedTermsFuzzy.lookup_terms is not orig_sql
        # the reference's own constructors now build the GPU class (no device touched until a lookup)
        settings = tab.TextEmbeddingIndexSettings(O.FakeEmbeddingModel())
        assert isinstance(mods["typeagent.knowpro.fuzzyindex"].EmbeddingIndex(settings)._vector_base, tab.VectorBase)
        assert isinstance(rel_mem.TermEmbeddingIndex(settings)._vectorbase, tab.VectorBase)
        assert tab.install() == patched or True   # idempotent: a second install wraps nothing twice
        assert not hasattr(rel_mem.TermEmbeddingIndex.lookup_terms.__wrapped__, "__wrapped__")
    finally:
        tab.uninstall()
    for name, m in mods.items():
        assert m.VectorBase is originals[name]
    assert rel_mem.TermEmbeddingIndex.lookup_terms is orig_mem
    assert rel_sql.SqliteRelatedTermsFuzzy.lookup_terms is orig_sql


def _terms(lists):
    return [[(t.text, t.weight) for t in terms] for terms in lists]


def _assert_terms_match(got, want, tie=2e-6):
    assert len(got) == len(want)
    for g, w in zip(got, want):
        gm, wm = dict(g), dict(w)
        boundary = [x[-1][1] for x in (g, w) if x]
        for text in set(gm) ^ set(wm):      # membership may differ only at a last-bit tie at the rank-k boundary
            s = gm.get(text, wm.get(text))
            assert any(abs(s - b) <= tie for b in boundary), (text, s, boundary)
        for text in set(gm) & set(wm):
            assert abs(gm[text] - wm[text]) <= 1e-4
        assert [t for t, _ in g][:3] == [t for t, _ in w][:3] or abs(g[0][1] - w[0][1]) <= tie


def _vocabularies():
    ep, epq = C.episode53()                      # real data: 150 x 1536 (terms 0..99, message chunks 100..149)
    yield "episode53", ep[:C.EPISODE53_TERMS], epq, 50, 0.85
    yield "episode53-lowfloor", ep[:C.EPISODE53_TERMS], epq, 10, 0.0
    v, q = O.make_corpus(6000, 384, seed=61, n_queries=64)   # >= 4096 rows, >= 16 queries: tensor cores
    yield "synthetic-6000x384", v, q, 5, 0.0


@needs_reference
@pytest.mark.gpu
@pytest.mark.parametrize("name,vectors,queries,max_hits,min_score", list(_vocabularies()),
                         ids=[v[0] for v in _vocabularies()])
def test_reference_built_indexes_return_reference_hits_after_install(name, vectors, queries, max_hits, min_score):
    mods = load_all()
    rel_mem = mods["typeagent.storage.memory.reltermsindex"]
    rel_sql = mods["typeagent.storage.sqlite.reltermsindex"]
    schema = ref_loader.load_reference_module("typeagent.storage.sqlite.schema")
    vb = mods["typeagent.aitools.vectorbase"]
    texts = [f"term{i:05d}" for i in range(len(vectors))]
    q_texts = [f"query{i}" for i in range(len(queries))]
    table = {**dict(zip(texts, vectors)), **dict(zip(q_texts, queries))}

    def build(settings_cls):
        settings = settings_cls(embedding_model=DictEmbeddingModel(table), min_score=min_score, max_matches=max_hits)
        mem = rel_mem.TermEmbeddingIndex(settings)
        db = sqlite3.connect(":memory:")
        db.execute(schema.RELATED_TERMS_FUZZY_SCHEMA)
        sql = rel_sql.SqliteRelatedTermsFuzzy(db, settings)

        async def fill():
            await mem.add_terms(texts)
            await sql.add_terms(texts)

        asyncio.run(fill())
        return mem, sql

    async def run(mem, sql):
        return (_terms(await mem.lookup_terms(q_texts)), _terms(await sql.lookup_terms(q_texts)),
                _terms([await mem.lookup_term(q_texts[1])]))

    want_mem, want_sql, want_one = asyncio.run(run(*build(vb.TextEmbeddingIndexSettings)))   # reference on numpy
    assert any(want_mem)
    try:
        tab.install()
        mem, sql = build(vb.TextEmbeddingIndexSettings)       # the reference's code, now on the GPU class
        assert isinstance(mem._vectorbase, tab.VectorBase) and isinstance(sql._vector_base, tab.VectorBase)
        searches = []
        inner, inner_one = tab.VectorBase.search_arrays, tab.VectorBase._lookup_one

        def counting(self, *a, **k):
            searches.append(len(np.atleast_2d(a[0])))
            return inner(self, *a, **k)

        def counting_one(self, *a, **k):
            searches.append(1)
            return inner_one(self, *a, **k)

        tab.VectorBase.search_arrays, tab.VectorBase._lookup_one = counting, counting_one
        try:
            got_mem, got_sql, got_one = asyncio.run(run(mem, sql))
        finally:
            tab.VectorBase.search_arrays, tab.VectorBase._lookup_one = inner, inner_one
    finally:
        tab.uninstall()
    _assert_terms_match(got_mem, want_mem)
    _assert_terms_match(got_sql, want_sql)
    _assert_terms_match(got_one, want_one)
    # ONE batched search per lookup_terms call (plus the single lookup_term), not one per query term
    assert searches == [len(q_texts), len(q_texts), 1], searches
    if len(vectors) >= 4096:
        assert mem._vectorbase.last_timing()["path"] in ("scan", "mma_split")


@pytest.mark.gpu
def test_embedding_file_pair_loads_into_a_search(tmp_path):
    """The reference's on-disk layout (knowpro/serialization.py:83-98, :183-222): <prefix>_embeddings.bin
    + <prefix>_data.json -> formats.load_embedding_file -> GPU lookups equal to the reference's
    (its outputs recorded by tests/golden/make_golden.py)."""
    from typeagent_py_b200 import formats

    with open(C.GOLDEN_FILE) as f:
        want = json.load(f)["embedding_file_pair"]
    ep, epq = C.episode53()
    related, messages = ep[:C.EPISODE53_TERMS], ep[C.EPISODE53_TERMS:]
    prefix = str(tmp_path / "Episode_53_excerpt_index")
    formats.write_embedding_file(prefix, related, messages)
    raw = np.fromfile(prefix + "_embeddings.bin", dtype=np.float32).reshape(-1, ep.shape[1])   # podcasts/podcast.py:147-168
    np.testing.assert_array_equal(raw, ep)
    settings = tab.TextEmbeddingIndexSettings(O.FakeEmbeddingModel())
    rel_base, msg_base = formats.load_embedding_file(prefix, settings)
    assert len(rel_base) == len(related) and len(msg_base) == len(messages)
    bases = {"related": rel_base, "messages": msg_base}
    for qi, q in enumerate(epq):
        for part, k, ms in C.EMBEDDING_FILE_LOOKUPS:
            got = bases[part].fuzzy_lookup_embedding(q, k, ms)
            assert_hits_match(got, want[C.embedding_file_key(part, k, ms)][qi], min_score=ms,
                              what="embedding file -> search")   # order up to float32 ties
    # SQLite BLOB layout (storage/sqlite/schema.py:193-212) through embeddings_from_blobs
    blobs = [row.tobytes() for row in messages]
    again = tab.VectorBase(settings)
    again.deserialize(formats.embeddings_from_blobs(blobs))
    assert_hits_match(again.fuzzy_lookup_embedding(epq[4], 10, 0.7),
                      want[C.embedding_file_key("messages", 10, 0.7)][4], min_score=0.7)
