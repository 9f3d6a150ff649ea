"""Call-surface compatibility with the reference classes (CPU).  The device store is replaced by a test double that
answers through the oracle, so what is exercised here is the seam itself: method rebinding, coroutine signature,
id <-> row bookkeeping, return types and the error convention -- compared with what the reference's own methods
return on the same inputs: live, on the UNMODIFIED classes, when a checkout of the reference project is present
(oracle/ref_import.py; skipped otherwise), and on the reference outputs stored in tests/golden/ always."""
import asyncio
import os
import types

import numpy as np
import pytest

from oracle import oracle, ref_import, synth

needs_reference = pytest.mark.skipif(not ref_import.available(), reason="reference checkout not present (see oracle/ref_import.py)")


from doubles import OracleBackedStore


def _oracle_cosine_pairs(a, b, zero_rule=0, sum_mode=None, device=0):
    """Stands in for vidmem_b200.store.cosine_pairs: the device kernel's GPU parity is a GPU test."""
    a, b = np.atleast_2d(np.asarray(a, np.float64)), np.atleast_2d(np.asarray(b, np.float64))
    return np.array([oracle.cosine(x, y, variant=("injector", "retriever", "utils")[zero_rule]) for x, y in zip(a, b)])


def test_injector_seam_matches_stored_reference_lists(monkeypatch, golden_dir):
    """The adapter bound onto an injector returns, on the store dict and queries of tests/golden/batch_small.npz
    (an Exception-valued query, None and [] embeddings, duplicate and zero rows and a zero query), exactly the lists
    the reference's own _calculate_batch_similarities returned there."""
    from vidmem_b200 import adapters
    import vidmem_b200.store as vstore
    monkeypatch.setattr(vstore, "EmbeddingStore", OracleBackedStore)
    g = np.load(os.path.join(golden_dir, "batch_small.npz"))
    X, Q, row_ok, query_ok = g["X"], g["Q"], g["row_ok"], g["query_ok"]
    store = {f"c{i}": [float(v) for v in X[i]] if row_ok[i] else (None if i == 8 else []) for i in range(len(X))}
    queries = [[float(v) for v in Q[i]] if query_ok[i] else RuntimeError("embed failed") for i in range(len(Q))]

    async def fake_get(_handler):
        return store

    for k in (3, 10, 200):
        inj = types.SimpleNamespace(embedder_config=types.SimpleNamespace(top_k_chunk_with_batch_similarity=k, top_k_similar_batch=2),
                                    _get_chunk_embeddings=fake_get)
        adapters.install_injector(inj)
        got = asyncio.run(inj._calculate_batch_similarities(queries, object()))
        want = [[(f"c{int(r)}", float(s)) for r, s in zip(g[f"idx_k{k}"][qi, :c], g[f"score_k{k}"][qi, :c])]
                for qi, c in enumerate(g[f"count_k{k}"])]
        assert got == want, k
        assert got[3] == [] and all(isinstance(cid, str) and isinstance(s, float) for lst in got for cid, s in lst)


def test_ragged_rows_queries_and_growth_follow_stored_reference_lists(monkeypatch, golden_dir):
    """Stored rows and queries of the wrong length, rows inserted one to four at a time into a store that starts at 4
    rows and grows many times, and the same dict mirrored through the injector seam.  The expected lists come from the
    reference's own outputs in batch_small.npz: its k=200 lists rank every truthy row with its score; a wrong-length row
    scores 0.0 (the reference's `len(vec1) != len(vec2)` branch, :378-379, pinned by cosine_kat.npz), and ties keep store
    order (its stable sort, pinned by the zero query 4).  An empty query, or one whose length no stored row has, scores
    every row 0.0 by the same branch, which is the zero query's case.  (The reference compares each query with each row
    by their own two lengths, so a query would score a real cosine against rows of its own wrong length: the wrong
    query lengths here, d-3 and d+3, are ones no ragged row has.)"""
    from vidmem_b200 import adapters
    import vidmem_b200.store as vstore
    monkeypatch.setattr(vstore, "EmbeddingStore", OracleBackedStore)
    g = np.load(os.path.join(golden_dir, "batch_small.npz"))
    X, Q, row_ok, query_ok = g["X"], g["Q"], g["row_ok"], g["query_ok"]
    n, d = X.shape
    assert all(g["count_k200"][qi] == row_ok.sum() for qi in range(len(Q)) if query_ok[qi])    # every truthy row ranked
    rng = np.random.default_rng(20261020)
    ragged = sorted(int(r) for r in rng.choice(np.flatnonzero(row_ok[1:]) + 1, 16, replace=False))   # row 0 sets the dim
    lengths = (1, d - 1, d + 1, 2 * d)

    def row(i):
        if not row_ok[i]:
            return None if i == 8 else []
        v = [float(x) for x in np.concatenate([X[i], X[(i + 1) % n]])]
        return v[:lengths[ragged.index(i) % 4]] if i in ragged else v[:d]

    store = {f"c{i}": row(i) for i in range(n)}
    queries = [[float(v) for v in Q[i]] if query_ok[i] else RuntimeError("embed failed") for i in range(len(Q))]
    queries += [[float(v) for v in Q[0][:d - 3]], [], [float(v) for v in Q[2]] + [0.5, -0.25, 0.125]]   # wrong-length queries
    assert not {len(q) for q in queries[len(Q):]} & {len(r) for r in store.values() if r}

    def want(k):
        out = []
        for qi in list(range(len(Q))) + [4, 4, 4]:
            if not query_ok[qi]:
                out.append([])
                continue
            full = [(int(r), 0.0 if r in ragged else float(s)) for r, s in zip(g["idx_k200"][qi], g["score_k200"][qi][:g["count_k200"][qi]])]
            out.append([(f"c{r}", s) for r, s in sorted(full, key=lambda t: (-t[1], t[0]))[:k]])
        return out

    async def fake_get(_handler):
        return store

    for k in (1, 3, 10, 200):
        inj = types.SimpleNamespace(embedder_config=types.SimpleNamespace(top_k_chunk_with_batch_similarity=k, top_k_similar_batch=2),
                                    _get_chunk_embeddings=fake_get)
        adapters.install_injector(inj)
        assert asyncio.run(inj._calculate_batch_similarities(queries, object())) == want(k), k
    for batch in (1, 3, 4):
        res = adapters.ResidentChunkStore(initial_capacity=4)                    # grows many times
        res.upsert([("c0", store["c0"])])                                        # the store dimension is set by a good row
        for i in range(1, n, batch):                                             # ragged rows also first in a batch
            res.upsert([(f"c{j}", store[f"c{j}"]) for j in range(i, min(i + batch, n))])
        assert res.ids == list(store)
        for k in (3, 10):
            assert res.topk(queries, k) == want(k), (batch, k)


def test_first_batch_dimension_is_the_modal_length(monkeypatch):
    """A first insert batch with one malformed vector in front: the modal length sets the store dimension and the
    malformed row scores 0.0."""
    from vidmem_b200 import adapters
    import vidmem_b200.store as vstore
    monkeypatch.setattr(vstore, "EmbeddingStore", OracleBackedStore)
    res = adapters.ResidentChunkStore()
    res.upsert([("a", [1.0] * 9), ("b", [1.0, 0.0, 0.0]), ("c", [0.0, 1.0, 0.0])])
    assert res.dim == 3 and res.topk([[1.0, 0.0, 0.0]], 3) == [[("b", 1.0), ("a", 0.0), ("c", 0.0)]]


def test_scalar_cosine_seams_match_stored_reference(monkeypatch, golden_dir):
    """S2 / S4 and EmbeddingUtils.cosine_similarity through the adapters against what the reference's three methods
    returned on tests/golden/cosine_kat.npz: different lengths, zero vectors, magnitudes whose product underflows."""
    from vidmem_b200 import adapters
    import vidmem_b200.store as vstore
    monkeypatch.setattr(vstore, "cosine_pairs", _oracle_cosine_pairs)
    g = np.load(os.path.join(golden_dir, "cosine_kat.npz"))
    backend = adapters.ChunkSimilarityBackend(store=adapters.ResidentChunkStore())
    vs_backend = adapters.VectorSearchBackend(adapters.ResidentChunkStore())
    eu_backend = adapters.EmbeddingUtilsBackend()
    assert (g["len_a"] != g["len_b"]).any()
    for i in range(len(g["out"])):
        v1 = [float(v) for v in g["a"][i, :g["len_a"][i]]]
        v2 = [float(v) for v in g["b"][i, :g["len_b"][i]]]
        assert backend._cosine_similarity(v1, v2) == g["out"][i, 0], i
        assert vs_backend._cosine_similarity(v1, v2) == g["out"][i, 1], i
        assert eu_backend.cosine_similarity(v1, v2) == pytest.approx(g["out"][i, 2], rel=1e-15, abs=0), i


@needs_reference
def test_install_on_real_reference_injector(monkeypatch):
    from oracle import ref_import
    from vidmem_b200 import adapters
    import vidmem_b200.store as vstore
    monkeypatch.setattr(vstore, "EmbeddingStore", OracleBackedStore)
    n, d, k = 120, 64, 3
    X = synth.synth_rows(7, 0, n, d)
    store = {f"u_{i // 4}_{i % 4}": [float(v) for v in X[i]] for i in range(n)}
    store["u_bad"] = []                                                   # falsy embedding is skipped (:363)
    Q = synth.synth_queries(8, 4, d, 7, n)
    queries = [[float(v) for v in q] for q in Q] + [RuntimeError("embed failed")]

    # what the reference itself returns
    want = ref_import.run_batch_similarities(queries, store, k)

    # the same, through the adapter bound onto an unmodified PreLLMInjector instance
    inj = ref_import.make_injector(k)

    async def fake_get(_handler):
        return store

    inj._get_chunk_embeddings = fake_get                                   # the reference's own fetch seam (:390-412)
    backend = adapters.install_injector(inj)
    assert asyncio.iscoroutinefunction(inj._calculate_batch_similarities)
    got = asyncio.run(inj._calculate_batch_similarities(queries, object()))
    assert got == want and got[-1] == []
    assert all(isinstance(cid, str) and isinstance(s, float) for lst in got for cid, s in lst)
    assert len(backend.store) == n + 1 and backend.store.ids[-1] == "u_bad"


@needs_reference
def test_ragged_queries_and_growth_match_the_reference(monkeypatch):
    """Wrong-length, empty and Exception queries, falsy rows, and a store that outgrows its capacity several
    times: the adapter returns what the UNMODIFIED reference method returns on the same dict."""
    from hypothesis import given, settings, strategies as st
    from oracle import ref_import
    from vidmem_b200 import adapters
    import vidmem_b200.store as vstore
    monkeypatch.setattr(vstore, "EmbeddingStore", OracleBackedStore)
    d = 6
    vec = st.lists(st.integers(-3, 3).map(float), min_size=d, max_size=d)
    anyq = st.one_of(vec, st.lists(st.integers(-3, 3).map(float), min_size=0, max_size=d + 2), st.just(RuntimeError("embed failed")))
    rows = st.lists(st.one_of(vec, st.just([])), min_size=1, max_size=40)

    @settings(max_examples=40, deadline=None)
    @given(rows, st.lists(anyq, min_size=1, max_size=4), st.integers(1, 5))
    def run(row_list, queries, k):
        store = {f"u_{i}": list(r) for i, r in enumerate(row_list)}
        want = ref_import.run_batch_similarities(queries, store, k)
        res = adapters.ResidentChunkStore(initial_capacity=4)                    # forces repeated growth
        for i in range(0, len(row_list), 3):                                     # rows arrive in small insert batches
            res.upsert([(f"u_{j}", row_list[j]) for j in range(i, min(i + 3, len(row_list)))])
        assert res.topk(queries, k) == want
        assert res.ids == list(store)

    run()


@needs_reference
def test_scalar_cosine_seams_ragged_lengths_match_the_reference(monkeypatch):
    """S2 / S4 with vectors of different lengths, zero vectors and empty vectors: the adapters' length handling
    (0.0 on mismatch for the injector; zip-truncation == zero padding for the retriever) against the reference's
    own methods.  The device kernel behind cosine_pairs is replaced by the oracle (its GPU parity is a GPU test)."""
    from hypothesis import given, settings, strategies as st
    from oracle import ref_import
    from vidmem_b200 import adapters
    import vidmem_b200.store as vstore

    monkeypatch.setattr(vstore, "cosine_pairs", _oracle_cosine_pairs)
    ref = ref_import.load()
    inj = ref_import.make_injector(3)
    backend = adapters.ChunkSimilarityBackend(store=adapters.ResidentChunkStore())
    vs_backend = adapters.VectorSearchBackend(adapters.ResidentChunkStore())
    eu_backend = adapters.EmbeddingUtilsBackend()
    vec = st.lists(st.one_of(st.integers(-5, 5).map(float), st.floats(-1e3, 1e3, allow_nan=False, width=32)), min_size=0, max_size=9)

    @settings(max_examples=150, deadline=None)
    @given(vec, vec)
    def run(v1, v2):
        assert backend._cosine_similarity(v1, v2) == inj._cosine_similarity(v1, v2)
        assert vs_backend._cosine_similarity(v1, v2) == ref["HybridRetriever"]._cosine_similarity(v1, v2)
        assert eu_backend.cosine_similarity(v1, v2) == pytest.approx(ref["EmbeddingUtils"].cosine_similarity(v1, v2), rel=1e-15, abs=0)

    run()


@needs_reference
def test_ragged_rows_follow_the_length_mismatch_rule(monkeypatch):
    """Stored vectors of the wrong length score 0.0 like the reference's `len(vec1) != len(vec2)` branch (:378-379),
    wherever they sit in an insert batch -- also first in a batch while the store already exists (round-1 ADVICE)."""
    from hypothesis import given, settings, strategies as st
    from oracle import ref_import
    from vidmem_b200 import adapters
    import vidmem_b200.store as vstore
    monkeypatch.setattr(vstore, "EmbeddingStore", OracleBackedStore)
    d = 6
    good = st.lists(st.integers(-3, 3).map(float), min_size=d, max_size=d)
    odd = st.lists(st.integers(-3, 3).map(float), min_size=d + 3, max_size=d + 3)   # a length no query uses
    rows = st.lists(st.one_of(good, good, odd, st.just([])), min_size=2, max_size=30)
    anyq = st.one_of(good, st.lists(st.integers(-3, 3).map(float), min_size=0, max_size=d + 2))

    @settings(max_examples=60, deadline=None)
    @given(good, rows, st.lists(anyq, min_size=1, max_size=3), st.integers(1, 4), st.integers(1, 4))
    def run(first, row_list, queries, k, batch):
        row_list = [first] + row_list                                            # the store dimension is set by a good row
        store = {f"u_{i}": list(r) for i, r in enumerate(row_list)}
        want = ref_import.run_batch_similarities(queries, store, k)
        res = adapters.ResidentChunkStore(initial_capacity=4)
        res.upsert([("u_0", row_list[0])])                                       # ... which arrives first
        for i in range(1, len(row_list), batch):
            res.upsert([(f"u_{j}", row_list[j]) for j in range(i, min(i + batch, len(row_list)))])
        assert res.topk(queries, k) == want

    run()


class _Splitter:
    """Deterministic stand-in for langchain's RecursiveCharacterTextSplitter (absent here): fixed-width pieces."""

    def __init__(self, chunk_size=256, chunk_overlap=32, separators=None):
        self.w = 12

    def split_text(self, text):
        return [text[i:i + self.w] for i in range(0, len(text), self.w)]


class _TextEmbedder:
    """Deterministic 'embedding service': a vector derived from the text; one text makes it fail."""

    def __init__(self, d=8):
        self.d, self.calls = d, 0

    async def aembed_query(self, text):
        self.calls += 1
        if "FAIL" in text:
            raise RuntimeError("embedding service down")
        rng = np.random.default_rng(abs(hash(text)) % (2 ** 32))
        v = rng.integers(-4, 5, self.d).astype(float)
        return [float(x) for x in (v if "SHORT" not in text else v[:5])]       # a segment vector of another length


@needs_reference
def test_install_retriever_rebinds_s4_and_post_compression_on_the_real_class(monkeypatch):
    """S4 and its caller on the UNMODIFIED HybridRetriever: after install_retriever, _cosine_similarity and
    _post_compress_chunks (retriever_hybrid.py:465-514, 655-664) return exactly what the reference's own methods
    return -- same kept segments, order, dict shape, compression_score, [:top_k] cut, failed and ragged segments."""
    import sys
    import types
    from oracle import ref_import
    from vidmem_b200 import adapters
    import vidmem_b200.store as vstore

    def oracle_pairs(a, b, zero_rule=0, sum_mode=None, device=0):
        a, b = np.atleast_2d(np.asarray(a, np.float64)), np.atleast_2d(np.asarray(b, np.float64))
        return np.array([oracle.cosine(x, y, variant="injector" if zero_rule == 0 else "retriever") for x, y in zip(a, b)])

    monkeypatch.setattr(vstore, "cosine_pairs", oracle_pairs)
    monkeypatch.setattr(vstore, "EmbeddingStore", OracleBackedStore)
    ref = ref_import.load()
    cls = ref["HybridRetriever"]
    monkeypatch.setattr(sys.modules[cls.__module__], "RecursiveCharacterTextSplitter", _Splitter)
    chunks = [{"id": f"c{i}", "time": float(i), "score": 0.5, "source": "vector",
               "content": " ".join(f"w{i}{j}" for j in range(9)) + (" FAIL now" if i == 1 else "") + (" SHORT one!" if i == 2 else "")}
              for i in range(5)]
    for thr, top_k in ((-1.0, 100), (0.0, 6), (0.2, 3), (2.0, 5)):
        retr = object.__new__(cls)
        retr.embedder = _TextEmbedder()
        retr.config = types.SimpleNamespace(compression_threshold=thr, top_k=top_k, top_k_chunks=4)
        retr.neo4j_handler = types.SimpleNamespace(embedder=retr.embedder, run_uuid="g")
        want = asyncio.run(retr._post_compress_chunks("the query", chunks))
        backend = adapters.install_retriever(retr, adapters.ResidentChunkStore())
        got = asyncio.run(retr._post_compress_chunks("the query", chunks))
        assert got == want
        assert all(isinstance(g["compression_score"], float) for g in got)
        if thr < 0:
            assert len(got) > 10 and any(g["content"] != c["content"] for g, c in zip(got, chunks))
        assert retr._cosine_similarity([1.0, 2.0, 3.0], [0.5, -1.0]) == cls._cosine_similarity([1.0, 2.0, 3.0], [0.5, -1.0])
    # error convention (:512-514): a failing query embedding returns the chunks unchanged; no embedder -> unchanged
    retr.embedder = types.SimpleNamespace(aembed_query=None)
    assert asyncio.run(retr._post_compress_chunks("q", chunks)) is chunks
    retr.embedder = None
    assert asyncio.run(retr._post_compress_chunks("q", chunks)) is chunks


def test_vector_search_meta_in_mirror_and_hydrated_modes(monkeypatch):
    """Round-1 ADVICE: a mirror-mode store has no content/time, is capped at 5000 rows and refreshed at ingest only.
    The adapter therefore (a) serves S3 from HBM only when the store is known to be complete, falling back to the
    instance's own Cypher scan otherwise, (b) fetches content/time of the hits it does not hold, (c) hydrates time."""
    import types
    from test_hydrate_cpu import _Handler, _Result
    from vidmem_b200 import adapters
    import vidmem_b200.store as vstore
    monkeypatch.setattr(vstore, "EmbeddingStore", OracleBackedStore)
    n, d = 30, 16
    X = synth.synth_rows(3, 0, n, d)
    recs = [{"chunk_id": f"u_{i}", "embedding": [float(v) for v in X[i]], "content": f"text {i}", "time": f"00:{i:02d}"} for i in range(n)]
    q = [float(v) for v in X[7]]

    class Embedder:
        async def aembed_query(self, text):
            return q

    calls = []

    class Retr:
        neo4j_handler = types.SimpleNamespace(embedder=Embedder(), run_uuid="uuid-1")
        config = types.SimpleNamespace(top_k_chunks=3)

        async def _vector_search_chunks(self, session, query):
            calls.append(query)
            return [{"id": "from-neo4j"}]

    class Session:
        def __init__(self):
            self.queries = []

        async def run(self, query, **params):
            self.queries.append((query, params))
            return _Result([{"chunk_id": c, "chunk_time": "T" + c, "content": "C" + c} for c in params["ids"]])

    # (c) hydrated: time and content come from the hydration query, nothing else is fetched
    backend = adapters.ChunkSimilarityBackend()
    asyncio.run(backend.hydrate(_Handler(recs)))
    retr, sess = Retr(), Session()
    adapters.install_retriever(retr, backend.store)
    got = asyncio.run(retr._vector_search_chunks(sess, "what?"))
    assert got[0] == {"id": "u_7", "time": "00:07", "content": "text 7", "score": 1.0, "source": "vector"}
    assert not sess.queries and not calls and backend.store.complete
    # (b) rows that arrived without metadata: the hits' content/time are read through the caller's session
    bare = adapters.ResidentChunkStore()
    bare.upsert([(r["chunk_id"], r["embedding"]) for r in recs])
    retr, sess = Retr(), Session()
    adapters.install_retriever(retr, bare)
    got = asyncio.run(retr._vector_search_chunks(sess, "what?"))
    assert [g["id"] for g in got][0] == "u_7" and got[0]["content"] == "Cu_7" and got[0]["time"] == "Tu_7"
    assert len(sess.queries) == 1 and "c.id IN $ids" in sess.queries[0][0] and sess.queries[0][1]["graph_uuid"] == "uuid-1"
    asyncio.run(retr._vector_search_chunks(sess, "again"))
    assert len(sess.queries) == 1                                             # cached after the first fetch
    # (a) mirror mode: LIMIT-5000 ingest-time snapshot -> the reference's own exhaustive scan answers
    mirror = adapters.ResidentChunkStore()
    mirror.sync_from_dict({r["chunk_id"]: r["embedding"] for r in recs})
    assert mirror.complete is False
    retr = Retr()
    adapters.install_retriever(retr, mirror)
    assert asyncio.run(retr._vector_search_chunks(Session(), "mirror?")) == [{"id": "from-neo4j"}] and calls == ["mirror?"]
