"""Exact maximal-marginal-relevance search, host side: the oracle (oracle/mmr.py) against langchain's algorithm, a
known answer, the NaN and short-list rules, the retriever's three search types (langchain-core 0.3's
`VectorStoreRetriever` dispatch over the stand-ins in tests/stubs, and the duck-typed `GpuRetriever`) and the daemon op --
all with an oracle-backed fake index, no GPU."""
import asyncio
import os
import subprocess
import sys
import textwrap
import uuid

import numpy as np
import pytest

from oracle import cosine_topk as O
from oracle.mmr import mmr_exact, mmr_select

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def langchain_mmr(query, embeddings, lambda_mult, k):
    """Literal float64 transcription of langchain-core's `maximal_marginal_relevance` (vectorstores/utils.py)."""
    def cosine_similarity(X, Y):
        X, Y = np.asarray(X, np.float64), np.asarray(Y, np.float64)
        return (X / np.linalg.norm(X, axis=1, keepdims=True)) @ (Y / np.linalg.norm(Y, axis=1, keepdims=True)).T
    if min(k, len(embeddings)) <= 0:
        return []
    query = np.expand_dims(query, axis=0)
    similarity_to_query = cosine_similarity(query, embeddings)[0]
    idxs = [int(np.argmax(similarity_to_query))]
    selected = np.array([embeddings[idxs[0]]])
    while len(idxs) < min(k, len(embeddings)):
        best_score, idx_to_add = -np.inf, -1
        similarity_to_selected = cosine_similarity(embeddings, selected)
        for i, query_score in enumerate(similarity_to_query):
            if i in idxs:
                continue
            redundant_score = max(similarity_to_selected[i])
            equation_score = lambda_mult * query_score - (1 - lambda_mult) * redundant_score
            if equation_score > best_score:
                best_score, idx_to_add = equation_score, i
        idxs.append(idx_to_add)
        selected = np.append(selected, [embeddings[idx_to_add]], axis=0)
    return idxs


def unit(*xs):
    v = np.zeros(O.DIM, np.float32)
    v[:len(xs)] = xs
    return v


# q = e0; r0 = e0, r1 = e0 (duplicate, higher id), r2 = (0.8, 0.6, 0), r3 = (0.6, 0, 0.8)
KNOWN_X = np.stack([unit(1), unit(1), unit(0.8, 0.6), unit(0.6, 0, 0.8)])
KNOWN_Q = unit(1)


@pytest.mark.parametrize("lam", [0.0, 0.25, 0.5, 0.8, 1.0])
@pytest.mark.parametrize("k", [1, 4, 12])
def test_oracle_picks_what_langchain_picks_on_tie_free_data(lam, k):
    rng = np.random.default_rng(int(lam * 100) + k)
    base = rng.standard_normal((6, O.DIM)).astype(np.float32)
    X = (base[rng.integers(0, 6, 300)] + 0.6 * rng.standard_normal((300, O.DIM))).astype(np.float32)   # clusters
    ids = O.ids_arange(0, 300)
    for j in range(3):
        q = (base[j] + rng.standard_normal(O.DIM)).astype(np.float32)
        c_ids, c_d = O.topk_exact(X, ids, q, 40)
        rows = X[[int(i) for i in c_ids[:, 1]]]
        assert mmr_select(c_d, rows, k, lam) == langchain_mmr(q, rows, lam, k)
        g_ids, g_d = mmr_exact(X, ids, q, k, 40, lam)
        picks = mmr_select(c_d, rows, k, lam)
        assert np.array_equal(g_ids, c_ids[picks]) and np.array_equal(g_d, c_d[picks])


def test_known_answer():
    ids = O.ids_arange(0, 4)
    got, d = mmr_exact(KNOWN_X, ids, KNOWN_Q, 2, 4, 0.7)
    assert O.ids_to_ints(got) == [0, 1] and d[0] == 0.0 and d[1] == 0.0
    got, _ = mmr_exact(KNOWN_X, ids, KNOWN_Q, 3, 4, 0.3)
    assert O.ids_to_ints(got) == [0, 3, 2]


def test_nan_rows_come_last_in_position_order_and_short_lists():
    X = np.concatenate([KNOWN_X, np.zeros((2, O.DIM), np.float32)])
    ids = O.ids_arange(0, 6)
    got, d = mmr_exact(X, ids, KNOWN_Q, 6, 6, 0.5)
    assert O.ids_to_ints(got)[:4] == O.ids_to_ints(mmr_exact(KNOWN_X, ids[:4], KNOWN_Q, 4, 4, 0.5)[0])
    assert O.ids_to_ints(got)[4:] == [4, 5] and np.isnan(d[4:]).all()
    # a zero query: every distance is NaN, every score too -> position order = the fetch order
    got, d = mmr_exact(X, ids, np.zeros(O.DIM, np.float32), 3, 6, 0.5)
    assert O.ids_to_ints(got) == [0, 1, 2] and np.isnan(d).all()
    # k >= m: every candidate once; empty table: nothing
    got, _ = mmr_exact(KNOWN_X, ids[:4], KNOWN_Q, 12, 20, 0.5)
    assert sorted(O.ids_to_ints(got)) == [0, 1, 2, 3]
    assert mmr_exact(np.zeros((0, O.DIM), np.float32), ids[:0], KNOWN_Q, 4, 20, 0.5)[0].shape == (0, 2)
    assert mmr_select([], np.zeros((0, O.DIM), np.float32), 4, 0.5) == []


def test_argument_errors_need_no_gpu():
    from outline_rag_b200 import _lib
    q = np.zeros((1, O.DIM), np.float32)
    assert _lib.lib.orx_search_mmr(None, q.ctypes.data, 1, O.DIM, 4, 20, 0.5, None, None, None) == _lib.ORX_ERR_INVALID
    assert "index is null" in _lib.last_error()
    assert _lib.lib.orx_search_mmr_filtered(None, q.ctypes.data, 1, O.DIM, 4, 20, 0.5, None, 0, None, None, None) \
        == _lib.ORX_ERR_INVALID
    assert _lib.lib.orx_search_mmr_with_filter(None, None, q.ctypes.data, 1, O.DIM, 4, 20, 0.5, None, None, None) \
        == _lib.ORX_ERR_INVALID


# ------------------------------------------------------------------ an oracle-backed index with the MMR surface
class FakeMmrIndex:
    def __init__(self, X, ids):
        self.X, self.ids, self.calls = np.asarray(X, np.float32), np.asarray(ids, np.uint64), []

    def _rows(self, allow):
        if allow is None:
            return self.X, self.ids
        from outline_rag_b200.engine import ids_to_array
        ok = {tuple(map(int, r)) for r in ids_to_array(allow)}
        keep = np.array([tuple(map(int, r)) in ok for r in self.ids], bool)
        return self.X[keep], self.ids[keep]

    def search(self, Q, k):
        return self.search_filtered(Q, k, None)

    def search_filtered(self, Q, k, allow):
        self.calls.append(("search", k))
        X, ids = self._rows(allow)
        Q = np.asarray(Q, np.float32).reshape(-1, O.DIM)
        out = (np.zeros((len(Q), k, 2), np.uint64), np.full((len(Q), k), np.nan), np.zeros(len(Q), np.int32))
        for j, q in enumerate(Q):
            a, b = O.topk_exact(X, ids, q, k)
            out[0][j, :len(b)], out[1][j, :len(b)], out[2][j] = a, b, len(b)
        return out

    def search_mmr(self, Q, k, fetch_k=20, lambda_mult=0.5, allow_ids=None):
        self.calls.append(("mmr", k, fetch_k, lambda_mult))
        X, ids = self._rows(allow_ids)
        Q = np.asarray(Q, np.float32).reshape(-1, O.DIM)
        out = (np.zeros((len(Q), k, 2), np.uint64), np.full((len(Q), k), np.nan), np.zeros(len(Q), np.int32))
        for j, q in enumerate(Q):
            a, b = mmr_exact(X, ids, q, k, fetch_k, lambda_mult)
            out[0][j, :len(b)], out[1][j, :len(b)], out[2][j] = a, b, len(b)
        return out


class Emb:
    """the query text 'q' embeds to the known-answer query"""
    vecs = {"q": KNOWN_Q}

    def embed_query(self, t):
        return self.vecs[t]

    async def aembed_query(self, t):
        return self.vecs[t]


def _known_store():
    from outline_rag_b200 import vectorstore as vs
    sids = [str(uuid.UUID(int=i)) for i in range(4)]
    doc_store = vs.MemoryDocStore()
    doc_store.put_many(sids, [f"r{i}" for i in range(4)], [{"source_id": "a" if i < 2 else "b"} for i in range(4)])
    return vs.GpuVectorStore(FakeMmrIndex(KNOWN_X, O.ids_arange(0, 4)), Emb(), doc_store)


def test_store_mmr_relevance_and_the_duck_typed_retriever():
    from outline_rag_b200 import vectorstore as vs
    store = _known_store()
    # MMR picks r0, r3, r2 at lambda 0.3; the store returns them in distance order (the fetch order)
    docs = store.max_marginal_relevance_search("q", k=3, fetch_k=4, lambda_mult=0.3)
    assert [d.page_content for d in docs] == ["r0", "r2", "r3"]
    # k is clamped to fetch_k; lambda 0 is pure diversity, not the default
    assert store.index.calls[-1] == ("mmr", 3, 4, 0.3)
    store.max_marginal_relevance_search("q", k=9, fetch_k=2, lambda_mult=0.0)
    assert store.index.calls[-1] == ("mmr", 2, 2, 0.0)
    # filter= as a metadata predicate: resolved in the doc store, MMR over the eligible rows only
    docs = store.max_marginal_relevance_search("q", k=2, fetch_k=4, filter={"source_id": "b"})
    assert [d.page_content for d in docs] == ["r2", "r3"]
    pairs = asyncio.run(store.amax_marginal_relevance_search_with_score_by_vector(KNOWN_Q, k=2, fetch_k=4,
                                                                                  lambda_mult=0.7))
    assert [(d.page_content, s) for d, s in pairs] == [("r0", 0.0), ("r1", 0.0)]
    # relevance = 1 - distance, thresholded
    assert store._select_relevance_score_fn()(0.25) == 0.75
    rel = store.similarity_search_with_relevance_scores("q", k=4, score_threshold=0.7)
    assert [d.page_content for d, _ in rel] == ["r0", "r1", "r2"] and rel[2][1] == 1.0 - float(
        O.canon_distance(KNOWN_X[2:3], KNOWN_Q)[0])
    arel = asyncio.run(store.asimilarity_search_with_relevance_scores("q", k=4, score_threshold=0.7))
    assert [(d.page_content, s) for d, s in arel] == [(d.page_content, s) for d, s in rel]
    # the duck-typed retriever (no langchain in this interpreter) dispatches the three search types
    if vs.HAVE_LANGCHAIN:
        return
    r = store.as_retriever(search_type="mmr", search_kwargs={"k": 3, "fetch_k": 4, "lambda_mult": 0.3})
    assert isinstance(r, vs.GpuRetriever) and [d.page_content for d in r.invoke("q")] == ["r0", "r2", "r3"]
    assert [d.page_content for d in asyncio.run(r.ainvoke("q"))] == ["r0", "r2", "r3"]
    r = store.as_retriever(search_type="similarity_score_threshold", search_kwargs={"k": 4, "score_threshold": 0.7})
    assert [d.page_content for d in r.invoke("q")] == ["r0", "r1", "r2"]
    assert [d.page_content for d in asyncio.run(r.ainvoke("q"))] == ["r0", "r1", "r2"]
    r = store.as_retriever(search_kwargs={"k": 2})
    assert r.search_type == "similarity" and [d.page_content for d in r.invoke("q")] == ["r0", "r1"]
    with pytest.raises(ValueError, match="not allowed"):
        store.as_retriever(search_type="nearest")
    with pytest.raises(ValueError, match="score_threshold"):
        store.as_retriever(search_type="similarity_score_threshold", search_kwargs={"k": 4})


STUB_SCRIPT = textwrap.dedent('''
    import asyncio, sys
    sys.path.insert(0, {stubs!r})
    sys.path.insert(0, {root!r})
    from typing import Any, ClassVar
    import pydantic
    import langchain_core.vectorstores as lcv

    class VectorStoreRetriever(lcv.VectorStoreRetriever):
        """the stand-in retriever with langchain-core 0.3's search-type check and dispatch"""
        allowed_search_types: ClassVar[tuple] = ("similarity", "similarity_score_threshold", "mmr")

        @pydantic.model_validator(mode="after")
        def _check_search_type(self):
            if self.search_type not in self.allowed_search_types:
                raise ValueError(f"search_type of {{self.search_type}} not allowed.")
            if self.search_type == "similarity_score_threshold" and not isinstance(
                    self.search_kwargs.get("score_threshold"), float):
                raise ValueError("`score_threshold` is not specified with a float value(0~1) in `search_kwargs`.")
            return self

        def _get_relevant_documents(self, query, *, run_manager: Any = None, **kwargs: Any):
            kw = {{**self.search_kwargs, **kwargs}}
            if self.search_type == "similarity":
                return self.vectorstore.similarity_search(query, **kw)
            if self.search_type == "similarity_score_threshold":
                return [d for d, _ in self.vectorstore.similarity_search_with_relevance_scores(query, **kw)]
            return self.vectorstore.max_marginal_relevance_search(query, **kw)

        async def _aget_relevant_documents(self, query, *, run_manager: Any = None, **kwargs: Any):
            kw = {{**self.search_kwargs, **kwargs}}
            if self.search_type == "similarity":
                return await self.vectorstore.asimilarity_search(query, **kw)
            if self.search_type == "similarity_score_threshold":
                return [d for d, _ in await self.vectorstore.asimilarity_search_with_relevance_scores(query, **kw)]
            return await self.vectorstore.amax_marginal_relevance_search(query, **kw)

    lcv.VectorStoreRetriever = VectorStoreRetriever        # what VectorStore.as_retriever constructs
    from tests.test_mmr import _known_store
    store = _known_store()
    r = store.as_retriever(search_type="mmr", search_kwargs={{"k": 3, "fetch_k": 4, "lambda_mult": 0.3}})
    assert isinstance(r, VectorStoreRetriever)
    assert [d.page_content for d in r.invoke("q")] == ["r0", "r2", "r3"]
    assert [d.page_content for d in asyncio.run(r.ainvoke("q"))] == ["r0", "r2", "r3"]
    r = store.as_retriever(search_type="similarity_score_threshold", search_kwargs={{"k": 4, "score_threshold": 0.7}})
    assert [d.page_content for d in r.invoke("q")] == ["r0", "r1", "r2"]
    assert [d.page_content for d in asyncio.run(r.ainvoke("q"))] == ["r0", "r1", "r2"]
    r = store.as_retriever(search_kwargs={{"k": 2}})
    assert [d.page_content for d in asyncio.run(r.ainvoke("q"))] == ["r0", "r1"]
    for bad in ({{"search_type": "nearest"}}, {{"search_type": "similarity_score_threshold", "search_kwargs": {{"k": 4}}}}):
        try:
            store.as_retriever(**bad)
        except (ValueError, pydantic.ValidationError):
            pass
        else:
            raise AssertionError(bad)
    print("DISPATCH-OK")
''')


def test_langchain_retriever_dispatches_the_three_search_types():
    code = STUB_SCRIPT.format(stubs=os.path.join(ROOT, "tests", "stubs"), root=ROOT)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0 and "DISPATCH-OK" in out.stdout, out.stdout[-1500:] + out.stderr[-3000:]


def test_daemon_search_mmr_round_trip(small_table, tmp_path, monkeypatch):
    from outline_rag_b200.daemon import RemoteIndex, serve_in_thread
    monkeypatch.chdir(tmp_path)                  # a unix socket path may hold at most 107 bytes: name it relatively
    X, Q, _ = small_table
    owner = FakeMmrIndex(X[:400], O.ids_arange(0, 400))
    srv = serve_in_thread(owner, "orx.sock", batch_window_ms=5.0)
    try:
        cli = RemoteIndex("orx.sock")
        ids, dist, cnt = cli.search_mmr(Q[:2], 4, 20, 0.3)
        for j in range(2):
            w_ids, w_d = mmr_exact(X[:400], O.ids_arange(0, 400), Q[j], 4, 20, 0.3)
            assert cnt[j] == 4 and np.array_equal(ids[j], w_ids) and np.array_equal(dist[j], w_d)
        assert owner.calls == [("mmr", 4, 20, 0.3)]         # one call, not through the batcher
        ids, dist, cnt = cli.search_mmr(Q[0], 3, 10, 0.5, allow_ids=O.ids_arange(100, 140))
        w_ids, w_d = mmr_exact(X[100:140], O.ids_arange(100, 140), Q[0], 3, 10, 0.5)
        assert np.array_equal(ids[0], w_ids) and np.array_equal(dist[0], w_d)
        cli.close()
    finally:
        srv.stop()
