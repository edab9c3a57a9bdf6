"""Host logic of the plugin (no GPU): the catalogue, the doc_ids/app_id filter, tombstones + compaction, and the
B200MultiVectorStore contract (core/vector_store/base_vector_store.py:7-65) exercised with an injected index whose
scores come from the oracle -- test wiring only; the product always constructs the CUDA MaxSimIndex."""
import asyncio

import numpy as np
import pytest
import torch

from morphik_core_b200.catalog import PageCatalog, PageRecord
from morphik_core_b200.models import DocumentChunk
from morphik_core_b200.store import B200MultiVectorStore, as_query_matrix, build_store_metrics
from oracle import maxsim_oracle as orc


class OracleIndex:
    """Stands in for MaxSimIndex in host-logic tests (binary semantics = the Postgres provider)."""

    row_bytes = 16

    def __init__(self):
        self.pages = []

    def add_pages(self, pages):
        first = len(self.pages)
        self.pages.extend(np.asarray(p, np.float32) for p in pages)
        return first, len(pages)

    def compact(self, keep):
        self.pages = [self.pages[int(i)] for i in keep]

    def search_host(self, queries, k, allow_mask=None):
        lens = [len(p) for p in self.pages]
        d = orc.sign_pack_c(np.concatenate(self.pages)) if sum(lens) else np.zeros((0, 16), np.uint8)
        off = orc.page_offsets(lens)
        ts = np.full((len(queries), k), -np.inf, np.float32)
        ti = np.full((len(queries), k), -1, np.int64)
        tc = np.zeros(len(queries), np.int32)
        for qi, q in enumerate(queries):
            s, _ = orc.binary_maxsim_c(orc.sign_pack_c(q), d, off)
            a, b = orc.topk_c(s, k, allow_mask)
            ts[qi, :len(a)], ti[qi, :len(b)], tc[qi] = a, b, len(a)
        return ts, ti, tc


def run(coro):
    return asyncio.run(coro)


def chunk(doc, num, emb, content="c", meta=None):
    return DocumentChunk(document_id=doc, chunk_number=num, content=content, embedding=emb, metadata=meta or {})


def test_catalog_mask_delete_compact():
    cat = PageCatalog()
    for d, n in [("a", 0), ("a", 1), ("b", 0), ("c", 0), ("c", 1), ("c", 2)]:
        cat.add(PageRecord(d, n, f"{d}{n}", {}, app_id="app1" if d != "b" else None, n_rows=3))
    assert len(cat) == 6 and cat.allow_mask() is None
    assert cat.allow_mask(["a", "zzz"]).tolist() == [1, 1, 0, 0, 0, 0]
    assert cat.allow_mask([]).tolist() == [0] * 6
    assert cat.allow_mask(None, app_id="other").tolist() == [0, 0, 1, 0, 0, 0]  # only the app-less page is visible
    assert cat.allow_mask(None, app_id="app1") is None
    words = PageCatalog.mask_words(np.array([1, 0, 1] + [0] * 30 + [1], dtype=bool))
    assert words.tolist() == [0b101, 0b10]
    assert cat.delete_document("a") == [0, 1] and cat.n_live == 4 and cat.lookup("a", 1) is None
    assert cat.allow_mask().tolist() == [0, 0, 1, 1, 1, 1]
    keep, remap = cat.compaction_plan()
    assert keep.tolist() == [2, 3, 4, 5] and remap.tolist() == [-1, -1, 0, 1, 2, 3]
    cat.apply_compaction(keep)
    assert len(cat) == 4 and cat.lookup("c", 2) == 3 and cat.pages_of("b") == [0]


def test_as_query_matrix_accepts_reference_input_forms():
    import torch

    q = np.random.default_rng(0).standard_normal((5, 128)).astype(np.float32)
    for form in (q, torch.from_numpy(q), [r for r in q], [torch.from_numpy(r) for r in q], q.tolist(), q.astype(np.float64)):
        np.testing.assert_array_equal(as_query_matrix(form), q)
    assert as_query_matrix(q[0]).shape == (1, 128)
    with pytest.raises(ValueError):
        as_query_matrix(np.zeros((3, 64)))


def test_store_contract_matches_reference_tests():
    store = B200MultiVectorStore(auto_initialize=False, index=OracleIndex(), compact_dead_fraction=0.3)
    # test_multivector.py:206-211: empty list
    assert run(store.store_embeddings([])) == (True, [], build_store_metrics())
    # test_multivector.py:214-256: pattern page ranks first
    e1 = np.ones((3, 128)); e1[:, 64:] = -1
    e2 = -e1
    ok, ids, metrics = run(store.store_embeddings([chunk("similarity_test_1", 1, e1), chunk("similarity_test_2", 2, e2)]))
    assert ok and ids == ["similarity_test_1-1", "similarity_test_2-2"] and metrics["vector_store_rows"] == 2
    qe = np.ones(128); qe[64:] = -1
    res = run(store.query_similar(np.array([qe]), k=2))
    assert [r.document_id for r in res] == ["similarity_test_1", "similarity_test_2"]
    assert [r.score for r in res] == [1.0, 0.0] and all(r.embedding == [] for r in res)
    # test_multivector.py:184-202: doc_ids filter
    res = run(store.query_similar(np.array([qe]), k=5, doc_ids=["similarity_test_2"]))
    assert [r.document_id for r in res] == ["similarity_test_2"]
    assert run(store.query_similar(np.array([qe]), k=5, doc_ids=["nope"])) == []
    # test_multivector.py:259-294: metadata round trip + get_chunks_by_id
    run(store.store_embeddings([chunk("meta_doc", 7, e1, content="payload", meta={"page": 7, "is_image": True})], app_id="app"))
    got = run(store.get_chunks_by_id([("meta_doc", 7), ("meta_doc", 7), ("missing", 0)]))
    assert len(got) == 1 and got[0].metadata == {"page": 7, "is_image": True} and got[0].content == "payload" and got[0].score == 0.0
    assert run(store.get_chunks_by_id([("meta_doc", 7)], app_id="other")) == []
    # chunks without embeddings are skipped (multi_vector_store.py:632-636)
    ok, ids, _ = run(store.store_embeddings([chunk("noemb", 0, None)]))
    assert ok and ids == []
    # delete + automatic compaction keep ids and scores consistent
    assert run(store.delete_chunks_by_document_id("similarity_test_1")) is True
    res = run(store.query_similar(np.array([qe]), k=5))
    assert [r.document_id for r in res] == ["meta_doc", "similarity_test_2"] and res[0].score == 1.0
    assert len(store.catalog) == 2  # compaction ran (1/3 dead > 0.3)
    assert run(store.delete_chunks_by_document_id("never_existed")) is True
    # batched extension returns one list per query, k larger than the corpus is fine
    out = run(store.query_similar_batch([np.array([qe]), np.array([-qe])], k=10))
    assert [len(o) for o in out] == [2, 2] and out[1][0].document_id == "similarity_test_2"
    # min_score (accepted but ignored by the reference, document_service.py:381-383) cuts the sorted list
    out = run(store.query_similar_batch([np.array([qe])], k=10, min_score=0.5))
    assert [r.document_id for r in out[0]] == ["meta_doc"]
    assert run(store.query_similar_batch([np.array([qe])], k=10, min_score=2.0)) == [[]]


def test_as_page_matrix_host_forms():
    from morphik_core_b200.store import as_page_matrix

    a = as_page_matrix([[0.5] * 128, [1.0] * 128])
    assert a.dtype == np.float32 and a.shape == (2, 128)
    assert as_page_matrix(np.ones(128, dtype=np.float64)).shape == (1, 128)
    t = torch.ones((3, 128), dtype=torch.bfloat16)  # CPU tensor: host float32, like the reference (multi_vector_store.py:334-337)
    b = as_page_matrix(t)
    assert isinstance(b, np.ndarray) and b.dtype == np.float32 and b.shape == (3, 128)


def test_concurrent_queries_are_coalesced_and_each_gets_its_own_filter():
    """Concurrent query_similar coroutines (different users: different doc_ids / app_id / k) share GPU passes; every caller
    gets exactly what a lone call returns.  (Host logic with the injected index; the CUDA per-query-mask path is covered by
    tests/test_gpu_store.py.)"""
    rng = np.random.default_rng(12)
    store = B200MultiVectorStore(auto_initialize=False, index=OracleIndex())
    calls = {"n": 0}
    inner = store._index.search_host

    def counting(queries, k, allow_mask=None):
        calls["n"] += 1
        return inner(queries, k, allow_mask=allow_mask)

    store._index.search_host = counting
    embs = [rng.standard_normal((int(rng.integers(3, 40)), 128)).astype(np.float32) for _ in range(30)]
    run(store.store_embeddings([chunk(f"doc{i % 10}", i // 10, e) for i, e in enumerate(embs[:20])], app_id="a"))
    run(store.store_embeddings([chunk(f"doc{i % 10}", i // 10, e) for i, e in enumerate(embs[20:], start=20)], app_id="b"))
    reqs = []
    for i in range(18):
        q = embs[i][:8] + 0.01 * rng.standard_normal((min(8, len(embs[i])), 128)).astype(np.float32)
        doc_ids = None if i % 3 == 0 else [f"doc{j}" for j in range(i % 10 + 1)]
        reqs.append(dict(query_embedding=q, k=1 + i % 5, doc_ids=doc_ids, app_id=("a", "b", None)[i % 3]))
    reqs.append(dict(query_embedding=embs[0][:4], k=3, doc_ids=["nope"], app_id=None))  # empty filter -> []
    lone = [run(store.query_similar(**r)) for r in reqs]
    calls["n"] = 0

    async def many():
        return await asyncio.gather(*[store.query_similar(**r) for r in reqs])

    together = run(many())
    key = lambda res: [(c.document_id, c.chunk_number, c.score) for c in res]  # noqa: E731
    assert [key(r) for r in together] == [key(r) for r in lone]
    assert together[-1] == [] and all(len(r) <= q["k"] for r, q in zip(together, reqs))
    assert store.last_coalesced_batch == len(reqs)  # one batch ...
    assert calls["n"] < len(reqs) - 1  # ... and one index call per DISTINCT filter (13 here), not one per request (19)
    # opting out restores one call per request
    plain = B200MultiVectorStore(auto_initialize=False, index=store._index, coalesce_queries=False)
    plain.catalog = store.catalog
    assert key(run(plain.query_similar(**reqs[1]))) == key(lone[1])


def test_allow_words_cache_follows_catalogue_mutations():
    """The mask LRU is keyed by the catalogue version: adds, deletes and compaction never serve a stale filter."""
    c = PageCatalog()
    for i in range(70):
        c.add(PageRecord(f"d{i % 7}", i // 7, "", {}, "a" if i % 2 else None, 5))
    vis, w = c.allow_words(["d1", "d3"], None)
    assert vis and w.shape == (3,) and np.array_equal(w, PageCatalog.mask_words(c.allow_mask(["d1", "d3"], None)))
    assert c.allow_words(["d1", "d3"], None)[1] is w  # LRU hit returns the cached array
    assert c.allow_words(None, None) == (True, None)  # nothing filtered: no mask upload
    assert c.allow_words(["nope"], None)[0] is False
    # app_id: pages stored under another app are hidden, pages without one stay visible
    m = c.allow_mask(None, "b")
    assert m is not None and m.sum() == 35 and not m[1]
    c.add(PageRecord("d1", 99, "", {}, None, 5))  # mutation -> new version -> recomputed, now 71 pages
    vis2, w2 = c.allow_words(["d1", "d3"], None)
    assert w2 is not w and np.array_equal(w2, PageCatalog.mask_words(c.allow_mask(["d1", "d3"], None))) and (w2[2] >> 6) & 1
    c.delete_document("d3")
    m3 = c.allow_mask(["d1", "d3"], None)
    assert np.array_equal(c.allow_words(["d1", "d3"], None)[1], PageCatalog.mask_words(m3)) and m3.sum() == 11
    keep, _ = c.compaction_plan()
    c.apply_compaction(keep)
    assert len(c) == 61 and c.allow_mask(["d3"], None).sum() == 0
    assert np.array_equal(c.allow_words(["d1"], None)[1], PageCatalog.mask_words(c.allow_mask(["d1"], None)))


def test_coalesced_query_errors_reach_every_waiter():
    class Boom(OracleIndex):
        def search_host(self, queries, k, allow_mask=None):
            raise RuntimeError("device lost")

    store = B200MultiVectorStore(auto_initialize=False, index=Boom())
    run(store.store_embeddings([chunk("d", 0, np.ones((3, 128)))]))

    async def many():
        return await asyncio.gather(*[store.query_similar(np.ones((2, 128)), k=1) for _ in range(3)], return_exceptions=True)

    res = run(many())
    assert len(res) == 3 and all(isinstance(r, RuntimeError) and "device lost" in str(r) for r in res)
    # the queue recovers: a later healthy call works
    store._index = OracleIndex()
    store._index.add_pages([np.ones((3, 128), np.float32)])
    assert [r.document_id for r in run(store.query_similar(np.ones((2, 128)), k=1))] == ["d"]


def test_batch_query_mask_search_and_chunks_are_one_critical_section():
    """ADVICE r1 (store.py:321): with coalescing off, an ingest between mask construction and the search used to hand a
    stale (too short) mask to the GPU call.  Now mask, search and chunk resolution happen under the store lock in one worker
    thread: an index that checks the mask length on every search never sees a mismatch while writers run concurrently."""
    import threading

    class CheckingIndex(OracleIndex):
        def __init__(self):
            super().__init__()
            self.bad = 0

        def search_host(self, queries, k, allow_mask=None):
            if allow_mask is not None and len(allow_mask) != (len(self.pages) + 31) // 32:
                self.bad += 1
            return super().search_host(queries, k, allow_mask)

    idx = CheckingIndex()
    store = B200MultiVectorStore(index=idx, mode="binary", auto_initialize=False, coalesce_queries=False)
    rng = np.random.default_rng(3)
    run(store.store_embeddings([chunk("seed", j, rng.standard_normal((4, 128)).astype(np.float32)) for j in range(40)], app_id="a"))
    stop = threading.Event()

    def writer():
        i = 0
        while not stop.is_set():
            run(store.store_embeddings([chunk(f"w{i}", 0, rng.standard_normal((3, 128)).astype(np.float32))], app_id="b"))
            i += 1

    t = threading.Thread(target=writer)
    t.start()
    try:
        q = rng.standard_normal((5, 128)).astype(np.float32)
        for _ in range(60):
            res = run(store.query_similar(q, k=5, app_id="a"))  # app filter => a real mask every time
            assert len(res) == 5 and all(r.document_id == "seed" for r in res)
    finally:
        stop.set()
        t.join()
    assert idx.bad == 0


def test_reference_dual_store_calls_replay_over_this_store(golden_dir):
    """SURVEY row a-11: the reference's DualMultiVectorStore (core/vector_store/dual_multivector_store.py) drives two stores as
    its fast / slow members.  tests/golden/dual_store_calls.json holds every member call it made (method, positional and
    keyword arguments) and every member attribute it read in this scenario (tests/golden/make_golden.py ran it over
    recording members).  Replayed as recorded on two B200MultiVectorStore instances -- the calls of one operation awaited
    together, as the dual store does -- each call is accepted, returns what the dual store unpacks, and the scenario holds."""
    import json
    import os

    with open(os.path.join(golden_dir, "dual_store_calls.json")) as f:
        ops = json.load(f)["operations"]
    members = {"fast": B200MultiVectorStore(index=OracleIndex(), mode="binary", auto_initialize=False, uri="b200://fast"),
               "slow": B200MultiVectorStore(index=OracleIndex(), mode="binary", auto_initialize=False, uri="b200://slow",
                                            storage="the-storage")}
    rng = np.random.default_rng(8)
    chunks = [chunk(f"d{i // 2}", i % 2, rng.standard_normal((3, 128)).astype(np.float32), content=f"c{i}", meta={"i": i})
              for i in range(8)]
    refs = {"chunks": chunks, "query": chunks[5].embedding}

    def arg(a):
        if isinstance(a, dict):
            return refs[a["ref"]]
        if isinstance(a, list):  # chunk identifiers are (document_id, chunk_number) tuples
            return [tuple(x) if isinstance(x, list) else x for x in a]
        return a

    async def replay(calls):
        out, pending = [None] * len(calls), []
        for j, c in enumerate(calls):
            m = members[c["member"]]
            if "attribute" in c:
                out[j] = getattr(m, c["attribute"])
                continue
            r = getattr(m, c["method"])(*[arg(a) for a in c["args"]], **{k: arg(v) for k, v in c["kwargs"].items()})
            if asyncio.iscoroutine(r):
                pending.append((j, r))
            else:
                out[j] = r
        for (j, _), r in zip(pending, await asyncio.gather(*(r for _, r in pending))):
            out[j] = r
        return [(c["member"], res) for c, res in zip(calls, out)]

    got = {op["label"]: run(replay(op["calls"])) for op in ops}
    assert got["initialize"] == [("fast", True), ("slow", True)]
    assert got["uri"] == [("slow", "b200://slow")] and got["storage"] == [("slow", "the-storage")]
    assert [m for m, _ in got["store_embeddings"]] == ["fast", "slow"]
    for _, (ok, ids, metrics) in got["store_embeddings"]:  # the dual store unpacks (success, ids, metrics) from each member
        assert ok is True and ids == [f"d{i // 2}-{i % 2}" for i in range(8)] and isinstance(metrics, dict) and metrics
    assert len(members["fast"].catalog) == len(members["slow"].catalog) == 8
    [(m, res)] = got["query_similar"]
    assert m == "slow" and len(res) == 3 and (res[0].document_id, res[0].chunk_number) == ("d2", 1) and res[0].metadata == {"i": 5}
    [(m, res)] = got["get_chunks_by_id"]
    assert m == "slow" and [(c.document_id, c.chunk_number) for c in res] == [("d1", 0)]
    assert got["delete_chunks_by_document_id"] == [("fast", True), ("slow", True)]
    assert members["fast"].catalog.pages_of("d2") == [] and members["slow"].catalog.pages_of("d2") == []
    [(m, res)] = got["query_similar_after_delete"]
    assert m == "slow" and len(res) == 6 and all(r.document_id != "d2" for r in res)
    assert [m for m, _ in got["close"]] == ["fast", "slow"]
