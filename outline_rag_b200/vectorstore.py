"""`GpuVectorStore`: the drop-in for the object bound to ``rag.vector_store``.

The reference builds ``AsyncPGVectorStore.create(engine, embedding_service,
table_name="langchain_pg_embedding", metadata_columns=[...])`` (reference app/rag.py:69-79)
and uses exactly five things on it (SURVEY.md 8b):

* ``.as_retriever(search_kwargs={"k": TOP_K})``            rag.py:85-87  (-> ``asimilarity_search``)
* ``await .adelete(ids=[uuid, ...])``                       rag.py:231, :371
* ``await .aadd_documents(chunks)``                         rag.py:235
* (implied) ``asimilarity_search_with_score_by_vector(embedding, k)`` -> ``[(Document, distance)]``

This class keeps those names, argument meanings, return shapes and error behaviour
(exceptions propagate; api.py:125-127 turns them into "no documents").  The similarity
arithmetic + ORDER BY ... LIMIT k run on the B200 through the C-ABI; document text and the
four metadata columns stay in a `DocStore` (Postgres in production -- see INTEGRATION.md;
an in-memory dict here and in tests) and are hydrated by id in rank order.

Blocking C calls run in ``asyncio.to_thread`` so the uvicorn event loop is never stalled.
"""
from __future__ import annotations

import asyncio
import uuid
from dataclasses import dataclass, field
from typing import Any, Iterable, Optional, Sequence

import numpy as np

from ._lib import ORX_DIM, ORX_ERR_DIM, ORX_ERR_NONFINITE, OrxValueError
from .batcher import QueryBatcher
from .engine import Filter, Index, ids_to_array, ids_to_uuid_strs


def _is_handle(flt) -> bool:
    """A prepared filter (engine.Filter, daemon.RemoteFilter) rather than a metadata predicate."""
    return bool(getattr(flt, "is_filter_handle", False))

# The reference's seam is typed: `rag.vector_store: AsyncPGVectorStore` (a langchain VectorStore), its
# `.as_retriever(...)` result is handed to the pydantic-validated `ContextualCompressionRetriever(base_retriever=...)`
# (reference app/rag.py:28-31, :85-99).  So when the host application has langchain-core, GpuVectorStore IS a
# `langchain_core.vectorstores.VectorStore` and `as_retriever` returns langchain's own `VectorStoreRetriever`
# (a `BaseRetriever` / Runnable).  Without langchain (this image; tests) the same class stands on `object` and
# `as_retriever` returns the duck-typed `GpuRetriever`.
try:
    from langchain_core.documents import Document  # type: ignore
    from langchain_core.vectorstores import VectorStore as _VectorStoreBase  # type: ignore
    HAVE_LANGCHAIN = True
except Exception:
    HAVE_LANGCHAIN = False
    _VectorStoreBase = object

    @dataclass
    class Document:  # same three fields `rag.py` / `api.py` touch
        page_content: str
        metadata: dict = field(default_factory=dict)
        id: Optional[str] = None


DEFAULT_METADATA_COLUMNS = ["source_id", "title", "outline_updated_at_str", "url"]   # rag.py:73-78


class MemoryDocStore:
    """``langchain_id -> (content, metadata[, embedding])``: what stays in Postgres in production
    (columns ``content``, ``embedding`` + the 4 metadata columns, reference app/database.py:118-131).
    Postgres remains the source of truth for the embeddings too (`stores_embeddings`): the device table is
    rebuilt from it on restart (`copy_binary` = what `GpuVectorStore.COPY_SQL` streams)."""

    stores_embeddings = True

    def __init__(self):
        self._rows: dict[str, tuple[str, dict]] = {}
        self._emb: dict[str, np.ndarray] = {}

    def put_many(self, ids: Sequence[str], contents: Sequence[str], metadatas: Sequence[dict], embeddings=None) -> None:
        for n, (i, c, m) in enumerate(zip(ids, contents, metadatas)):
            self._rows[i] = (c, dict(m))
            if embeddings is not None:
                self._emb[i] = np.array(embeddings[n], dtype=np.float32)
            else:
                self._emb.pop(i, None)                       # INSERT ... DO UPDATE without a vector: NULL

    def get_many(self, ids: Sequence[str]) -> list[Optional[tuple[str, dict]]]:
        return [self._rows.get(i) for i in ids]

    def delete_many(self, ids: Iterable[str]) -> None:
        for i in ids:
            self._rows.pop(i, None)
            self._emb.pop(i, None)

    def copy_binary(self, rows_per_chunk: int = 256):
        """Yield what `COPY (SELECT langchain_id, embedding FROM langchain_pg_embedding) TO STDOUT (FORMAT
        binary)` streams for this store (PostgreSQL COPY binary format; pgvector's vector_send image; a row
        without an embedding is a NULL field), in chunks -- the stand-in for psycopg's `cursor.copy()`."""
        import struct
        yield b"PGCOPY\n\xff\r\n\x00" + bytes(8)
        buf = []
        for i in self._rows:
            buf.append(struct.pack(">hi", 2, 16) + uuid.UUID(i).bytes)
            e = self._emb.get(i)
            if e is None:
                buf.append(struct.pack(">i", -1))
            else:
                buf.append(struct.pack(">ihh", 4 + 4 * e.shape[0], e.shape[0], 0) + e.astype(">f4").tobytes())
            if len(buf) >= 2 * rows_per_chunk:
                yield b"".join(buf)
                buf = []
        yield b"".join(buf) + b"\xff\xff"

    def ids_for_filter(self, flt: dict) -> list[str]:
        """Resolve a metadata predicate to chunk ids -- `SELECT langchain_id ... WHERE <filter>` in
        production.  Supported: {"col": value}, {"col": {"$in": [...]}}, {"col": {"$eq": v}},
        {"$and": [f1, f2, ...]}, {"$or": [...]} (the subset of the upstream filter grammar that a
        `source_id` / `title` / `url` predicate needs)."""
        def match(meta: dict, f: dict) -> bool:
            for key, cond in f.items():
                if key == "$and":
                    if not all(match(meta, c) for c in cond):
                        return False
                elif key == "$or":
                    if not any(match(meta, c) for c in cond):
                        return False
                elif isinstance(cond, dict):
                    v = meta.get(key)
                    for op, arg in cond.items():
                        if op == "$in":
                            ok = v in arg
                        elif op == "$eq":
                            ok = v == arg
                        elif op == "$ne":
                            ok = v != arg
                        else:
                            raise NotImplementedError(f"filter operator {op}")
                        if not ok:
                            return False
                elif meta.get(key) != cond:
                    return False
            return True
        return [i for i, (_, m) in self._rows.items() if match(m, flt)]

    def ids_for_source(self, source_ids: Iterable[str]) -> list[str]:
        """``SELECT langchain_id ... WHERE source_id = ANY(:ids)`` (reference app/rag.py:216-224)."""
        want = set(source_ids)
        return [i for i, (_, m) in self._rows.items() if m.get("source_id") in want]


def _canon_uuid(v) -> str:
    if isinstance(v, uuid.UUID):
        return str(v)
    if isinstance(v, int):
        return str(uuid.UUID(int=v))
    return str(uuid.UUID(str(v)))


SEARCH_TYPES = ("similarity", "similarity_score_threshold", "mmr")     # langchain-core's VectorStoreRetriever


class GpuRetriever:
    """``VectorStoreRetriever`` stand-in for hosts WITHOUT langchain-core (with it, `GpuVectorStore.as_retriever`
    returns langchain's own ``VectorStoreRetriever``).  Same three search types and the same dispatch:
    ``similarity`` -> ``similarity_search``, ``mmr`` -> ``max_marginal_relevance_search`` (never micro-batched),
    ``similarity_score_threshold`` -> ``similarity_search_with_relevance_scores`` (``score_threshold`` required)."""

    def __init__(self, store: "GpuVectorStore", search_kwargs: Optional[dict] = None, search_type: str = "similarity"):
        if search_type not in SEARCH_TYPES:
            raise ValueError(f"search_type of {search_type} not allowed. Valid values are: {SEARCH_TYPES}")
        self.vectorstore = store
        self.search_type = search_type
        self.search_kwargs = dict(search_kwargs or {})
        if search_type == "similarity_score_threshold" and not isinstance(self.search_kwargs.get("score_threshold"), float):
            raise ValueError("`score_threshold` is not specified with a float value(0~1) in `search_kwargs`.")

    async def ainvoke(self, query: str, **_: Any) -> list:
        if self.search_type == "mmr":
            return await self.vectorstore.amax_marginal_relevance_search(query, **self.search_kwargs)
        if self.search_type == "similarity_score_threshold":
            return [d for d, _ in await self.vectorstore.asimilarity_search_with_relevance_scores(query, **self.search_kwargs)]
        return await self.vectorstore.asimilarity_search(query, **self.search_kwargs)

    def invoke(self, query: str, **_: Any) -> list:
        if self.search_type == "mmr":
            return self.vectorstore.max_marginal_relevance_search(query, **self.search_kwargs)
        if self.search_type == "similarity_score_threshold":
            return [d for d, _ in self.vectorstore.similarity_search_with_relevance_scores(query, **self.search_kwargs)]
        return self.vectorstore.similarity_search(query, **self.search_kwargs)


class GpuVectorStore(_VectorStoreBase):
    def __init__(self, index: Index, embedding_service, doc_store=None,
                 metadata_columns: Optional[list[str]] = None, table_name: str = "langchain_pg_embedding",
                 batch_window_ms: Optional[float] = None, max_batch: int = 256):
        self.index = index
        # micro-batching of concurrent by-vector searches (SURVEY.md 8f-3); None = one scan per request
        self.batcher = QueryBatcher(index, max_batch, batch_window_ms) if batch_window_ms is not None else None
        self.embedding_service = embedding_service
        self.doc_store = doc_store if doc_store is not None else MemoryDocStore()
        self.metadata_columns = list(metadata_columns or DEFAULT_METADATA_COLUMNS)
        self.table_name = table_name

    # ---------------------------------------------------------------- construction
    @classmethod
    async def create(cls, engine=None, embedding_service=None, table_name: str = "langchain_pg_embedding",
                     metadata_columns: Optional[list[str]] = None, *, dtype: str = "fp32", capacity: int = 0,
                     device: Optional[int] = None, devices: Optional[Sequence[int]] = None, doc_store=None,
                     batch_window_ms: Optional[float] = None, max_batch: int = 256, **_: Any) -> "GpuVectorStore":
        """Same call shape as ``AsyncPGVectorStore.create`` (reference app/rag.py:69-79).
        ``engine`` (the PGEngine) is accepted and handed to the doc store factory if it is
        callable; the vector column itself now lives in HBM.  ``devices=[0..7]`` row-shards the table over
        those GPUs inside this process (`orx_create_multi`): same object, same methods."""
        if embedding_service is None:
            raise ValueError("embedding_service is required")
        if callable(doc_store):
            doc_store = doc_store(engine)
        index = await asyncio.to_thread(lambda: Index(dtype, capacity, device, devices=devices))
        return cls(index, embedding_service, doc_store, metadata_columns, table_name, batch_window_ms, max_batch)

    @classmethod
    def create_sync(cls, embedding_service, **kw) -> "GpuVectorStore":
        doc_store = kw.pop("doc_store", None)
        index = Index(kw.pop("dtype", "fp32"), kw.pop("capacity", 0), kw.pop("device", None), devices=kw.pop("devices", None))
        return cls(index, embedding_service, doc_store, kw.pop("metadata_columns", None),
                   kw.pop("table_name", "langchain_pg_embedding"))

    def as_retriever(self, **kwargs: Any):
        """``vector_store.as_retriever(search_kwargs={"k": TOP_K})`` (reference app/rag.py:85-87).  With
        langchain-core: the inherited ``VectorStore.as_retriever`` -> a real ``VectorStoreRetriever`` (``BaseRetriever``,
        accepted by ``ContextualCompressionRetriever(base_retriever=...)``, rag.py:96-99) that calls
        ``asimilarity_search(query, **search_kwargs)``.  Without it: the duck-typed `GpuRetriever`."""
        if HAVE_LANGCHAIN:
            return super().as_retriever(**kwargs)
        return GpuRetriever(self, kwargs.get("search_kwargs"), kwargs.get("search_type", "similarity"))

    # -- the rest of langchain's abstract VectorStore surface
    @property
    def embeddings(self):
        return self.embedding_service

    def add_texts(self, texts, metadatas: Optional[Sequence[dict]] = None, *, ids: Optional[Sequence] = None,
                  **_: Any) -> list[str]:
        texts = list(texts)
        if not texts:
            return []
        return self.add_embeddings(texts, self.embedding_service.embed_documents(texts), metadatas, ids)

    async def aadd_texts(self, texts, metadatas: Optional[Sequence[dict]] = None, *, ids: Optional[Sequence] = None,
                         **_: Any) -> list[str]:
        texts = list(texts)
        if not texts:
            return []
        emb = await self.embedding_service.aembed_documents(texts)
        return await self.aadd_embeddings(texts, emb, metadatas, ids)

    @classmethod
    def from_texts(cls, texts, embedding, metadatas: Optional[Sequence[dict]] = None, **kw: Any) -> "GpuVectorStore":
        ids = kw.pop("ids", None)
        store = cls.create_sync(embedding, **kw)
        store.add_texts(texts, metadatas, ids=ids)
        return store

    # ---------------------------------------------------------------- writes
    def add_embeddings(self, texts: Sequence[str], embeddings, metadatas: Optional[Sequence[dict]] = None,
                       ids: Optional[Sequence] = None) -> list[str]:
        n = len(texts)
        if ids is None:
            ids = [None] * n
        ids = [_canon_uuid(i) if i is not None else str(uuid.uuid4()) for i in ids]   # `doc.id or uuid4()`
        metadatas = list(metadatas) if metadatas is not None else [{} for _ in range(n)]
        if n == 0:
            return []
        try:
            emb = np.asarray(embeddings, dtype=np.float32)
        except ValueError:                                # ragged: some vector has another length
            lens = sorted({len(e) for e in embeddings} - {ORX_DIM})
            raise OrxValueError(ORX_ERR_DIM, f"expected {ORX_DIM} dimensions, not {lens[0] if lens else '?'}") from None
        # pgvector's input checks, before anything is written anywhere (the reference's INSERT fails as a
        # whole for such a batch, rag.py:237-239 re-raises): same conditions and messages as orx_upsert
        if emb.ndim != 2 or emb.shape[0] != n or emb.shape[1] != ORX_DIM:
            got = emb.shape[-1] if emb.ndim >= 1 and emb.size else 0
            raise OrxValueError(ORX_ERR_DIM, f"expected {ORX_DIM} dimensions, not {got}")
        if not np.isfinite(emb).all():
            raise OrxValueError(ORX_ERR_NONFINITE, "NaN or infinite value not allowed in vector")
        # durable copy first (Postgres stays the source of truth; if this raises, the device table is untouched),
        # then the device table, which is a cache of it: a failure there is healed by a reload
        if getattr(self.doc_store, "stores_embeddings", False):
            self.doc_store.put_many(ids, list(texts), metadatas, embeddings=emb)
        else:
            self.doc_store.put_many(ids, list(texts), metadatas)
        self.index.upsert(ids, emb)
        return ids

    async def aadd_embeddings(self, texts, embeddings, metadatas=None, ids=None) -> list[str]:
        return await asyncio.to_thread(self.add_embeddings, texts, embeddings, metadatas, ids)

    async def aadd_documents(self, documents: Sequence, ids: Optional[Sequence] = None, **_: Any) -> list[str]:
        """reference app/rag.py:235.  ids default to ``doc.id or uuid4()``; texts are embedded with
        ``embedding_service.aembed_documents`` (remote bge-m3 in the reference)."""
        texts = [d.page_content for d in documents]
        metas = [dict(getattr(d, "metadata", {}) or {}) for d in documents]
        if ids is None:
            ids = [getattr(d, "id", None) for d in documents]
        if not texts:
            return []
        emb = await self.embedding_service.aembed_documents(texts)
        return await self.aadd_embeddings(texts, emb, metas, ids)

    def add_documents(self, documents: Sequence, ids: Optional[Sequence] = None, **_: Any) -> list[str]:
        texts = [d.page_content for d in documents]
        metas = [dict(getattr(d, "metadata", {}) or {}) for d in documents]
        if ids is None:
            ids = [getattr(d, "id", None) for d in documents]
        if not texts:
            return []
        return self.add_embeddings(texts, self.embedding_service.embed_documents(texts), metas, ids)

    def delete(self, ids: Optional[Sequence] = None, **_: Any) -> bool:
        """reference app/rag.py:231, :371.  Unknown ids are ignored (SQL DELETE semantics)."""
        if not ids:
            return False
        sids = [_canon_uuid(i) for i in ids]
        self.doc_store.delete_many(sids)                 # source of truth first; if it raises nothing changed
        self.index.delete(sids)
        return True

    async def adelete(self, ids: Optional[Sequence] = None, **kw: Any) -> bool:
        return await asyncio.to_thread(self.delete, ids, **kw)

    # ---------------------------------------------------------------- cold start (SURVEY.md 8f-1)
    COPY_SQL = ("COPY (SELECT langchain_id, embedding FROM {table} WHERE embedding IS NOT NULL) "
                "TO STDOUT (FORMAT binary)")

    def load_pgcopy(self, chunks) -> tuple[int, int]:
        """Rebuild the device table from a COPY BINARY stream of ``(langchain_id, embedding)``
        (`COPY_SQL`); content and metadata stay where they are (Postgres).  -> (rows_loaded, rows_null)."""
        return self.index.load_pgcopy(chunks)

    async def aload_pgcopy(self, chunks, feed_bytes: int = 8 << 20) -> tuple[int, int]:
        """Same, for an async iterator such as psycopg 3's ``async with cur.copy(sql) as copy: async for
        data in copy``.  Driver chunks are small (tens of KB); they are coalesced to `feed_bytes` so the
        event loop pays one thread hop per 8 MB, not per chunk."""
        ld = self.index.pgcopy_loader()
        pending = bytearray()
        try:
            async for data in chunks:
                pending += data
                if len(pending) >= feed_bytes:
                    block, pending = pending, bytearray()
                    await asyncio.to_thread(ld.feed, block)
            if pending:
                await asyncio.to_thread(ld.feed, pending)
        except BaseException:
            try:
                ld.close()
            except Exception:
                pass
            raise
        return await asyncio.to_thread(ld.close)

    # ---------------------------------------------------------------- reads
    def _hydrate(self, ids_row: np.ndarray, dist_row: np.ndarray, count: int) -> list[tuple[Any, float]]:
        sids = ids_to_uuid_strs(ids_row[:count])
        rows = self.doc_store.get_many(sids)
        out = []
        for sid, row, d in zip(sids, rows, dist_row[:count]):
            if row is None:      # the chunk left the source of truth after the scan (a delete in flight): the SQL
                continue         # would not have returned it either
            content, meta = row
            out.append((Document(page_content=content, metadata=dict(meta), id=sid), float(d)))
        return out

    def similarity_search_with_score_by_vector(self, embedding, k: int = 4, filter=None, **_: Any):
        """-> ``[(Document, cosine distance)]`` ascending, exactly the SQL's ORDER BY ... LIMIT k."""
        q = np.asarray(embedding, dtype=np.float32).reshape(1, -1)
        if filter is not None:
            # the metadata predicate is resolved where the metadata lives (doc store / Postgres), the
            # similarity ordering of the eligible chunks runs on the GPU (orx_search_filtered); a prepared
            # filter (`prepare_filter`) skips both the look-up and the id -> row resolution
            allow = filter if _is_handle(filter) else self.doc_store.ids_for_filter(filter)
            ids, dist, cnt = self.index.search_filtered(q, k, allow)
        else:
            ids, dist, cnt = self.index.search(q, k)
        return self._hydrate(ids[0], dist[0], int(cnt[0]))

    def prepare_filter(self, filter: dict):
        """Resolve a metadata predicate ONCE into a device-resident `Filter` (a `RemoteFilter` when the index is a
        `daemon.RemoteIndex`: the handle then lives in the owner process) that can be passed as `filter=`
        to every later search (a collection- or source-scoped assistant asks the same predicate each time).
        It denotes the chunk ids matching NOW; chunks added later need a new `prepare_filter`."""
        return self.index.make_filter(self.doc_store.ids_for_filter(filter))

    def batch_search_by_vector(self, embeddings, k: int = 4):
        """Many queries in one scan (the micro-batching front end of SURVEY.md 8f-3 calls this)."""
        ids, dist, cnt = self.index.search(np.asarray(embeddings, dtype=np.float32), k)
        return [self._hydrate(ids[i], dist[i], int(cnt[i])) for i in range(ids.shape[0])]

    async def asimilarity_search_with_score_by_vector(self, embedding, k: int = 4, filter=None, **kw: Any):
        if self.batcher is not None and (filter is None or _is_handle(filter)):
            # coalesced with concurrent requests (those carrying the same prepared filter share one filtered pass)
            ids, dist = await self.batcher.search(embedding, k, filter)
            return await asyncio.to_thread(self._hydrate, ids, dist, len(dist))
        return await asyncio.to_thread(self.similarity_search_with_score_by_vector, embedding, k, filter)

    async def asimilarity_search_by_vector(self, embedding, k: int = 4, **kw: Any):
        return [d for d, _ in await self.asimilarity_search_with_score_by_vector(embedding, k, **kw)]

    async def asimilarity_search_with_score(self, query: str, k: int = 4, **kw: Any):
        emb = await self.embedding_service.aembed_query(query)
        return await self.asimilarity_search_with_score_by_vector(emb, k, **kw)

    async def asimilarity_search(self, query: str, k: int = 4, **kw: Any):
        """What the retriever calls (reference app/rag.py:85-87 via api.py:122): the distance is dropped."""
        return [d for d, _ in await self.asimilarity_search_with_score(query, k, **kw)]

    def similarity_search(self, query: str, k: int = 4, **kw: Any):
        emb = self.embedding_service.embed_query(query)
        return [d for d, _ in self.similarity_search_with_score_by_vector(emb, k, **kw)]

    # ---------------------------------------------------------------- relevance scores
    @staticmethod
    def _cosine_relevance(distance: float) -> float:
        return 1.0 - distance

    def _select_relevance_score_fn(self):
        """Cosine distance -> relevance, as langchain-postgres does for its default (cosine) strategy: 1 - distance."""
        return self._cosine_relevance

    @staticmethod
    def _apply_threshold(pairs, score_threshold: Optional[float]):
        return pairs if score_threshold is None else [(d, s) for d, s in pairs if s >= score_threshold]

    def similarity_search_with_relevance_scores(self, query: str, k: int = 4, score_threshold: Optional[float] = None,
                                                **kw: Any):
        """-> ``[(Document, 1 - distance)]`` in distance order, keeping those with relevance >= `score_threshold`."""
        fn = self._select_relevance_score_fn()
        emb = self.embedding_service.embed_query(query)
        pairs = [(d, fn(s)) for d, s in self.similarity_search_with_score_by_vector(emb, k, **kw)]
        return self._apply_threshold(pairs, score_threshold)

    async def asimilarity_search_with_relevance_scores(self, query: str, k: int = 4,
                                                       score_threshold: Optional[float] = None, **kw: Any):
        fn = self._select_relevance_score_fn()
        pairs = [(d, fn(s)) for d, s in await self.asimilarity_search_with_score(query, k, **kw)]
        return self._apply_threshold(pairs, score_threshold)

    # ---------------------------------------------------------------- maximal marginal relevance
    def max_marginal_relevance_search_with_score_by_vector(self, embedding, k: int = 4, fetch_k: int = 20,
                                                           lambda_mult: float = 0.5, filter=None, **_: Any):
        """``[(Document, cosine distance)]``: the `k` rows MMR picks among the exact top-`fetch_k` (`Index.search_mmr`,
        on the GPU), returned in distance order as langchain-postgres returns them.  `k` is clamped to `fetch_k`;
        ``lambda_mult=0`` means pure diversity (not replaced by the default)."""
        q = np.asarray(embedding, dtype=np.float32).reshape(1, -1)
        k = min(int(k), int(fetch_k))
        allow = None
        if filter is not None:
            allow = filter if _is_handle(filter) else self.doc_store.ids_for_filter(filter)
        ids, dist, cnt = self.index.search_mmr(q, k, fetch_k, lambda_mult, allow)
        n = int(cnt[0])
        d = dist[0, :n]
        nan = np.isnan(d)
        # fetch order = the ordering contract (distance ASC, NaN last, id ASC)
        order = np.lexsort((ids[0, :n, 1], ids[0, :n, 0], np.where(nan, 0.0, d), nan))
        return self._hydrate(ids[0, :n][order], d[order], n)

    def max_marginal_relevance_search_by_vector(self, embedding, k: int = 4, fetch_k: int = 20,
                                                lambda_mult: float = 0.5, **kw: Any):
        return [d for d, _ in self.max_marginal_relevance_search_with_score_by_vector(embedding, k, fetch_k,
                                                                                     lambda_mult, **kw)]

    def max_marginal_relevance_search(self, query: str, k: int = 4, fetch_k: int = 20, lambda_mult: float = 0.5,
                                      **kw: Any):
        """What ``as_retriever(search_type="mmr", search_kwargs={"k": 12, "fetch_k": 48})`` calls."""
        emb = self.embedding_service.embed_query(query)
        return self.max_marginal_relevance_search_by_vector(emb, k, fetch_k, lambda_mult, **kw)

    async def amax_marginal_relevance_search_with_score_by_vector(self, embedding, k: int = 4, fetch_k: int = 20,
                                                                  lambda_mult: float = 0.5, **kw: Any):
        return await asyncio.to_thread(self.max_marginal_relevance_search_with_score_by_vector, embedding, k, fetch_k,
                                       lambda_mult, **kw)

    async def amax_marginal_relevance_search_by_vector(self, embedding, k: int = 4, fetch_k: int = 20,
                                                       lambda_mult: float = 0.5, **kw: Any):
        return [d for d, _ in await self.amax_marginal_relevance_search_with_score_by_vector(embedding, k, fetch_k,
                                                                                            lambda_mult, **kw)]

    async def amax_marginal_relevance_search(self, query: str, k: int = 4, fetch_k: int = 20,
                                             lambda_mult: float = 0.5, **kw: Any):
        emb = await self.embedding_service.aembed_query(query)
        return await self.amax_marginal_relevance_search_by_vector(emb, k, fetch_k, lambda_mult, **kw)


__all__ = ["GpuVectorStore", "GpuRetriever", "SEARCH_TYPES", "MemoryDocStore", "Document", "DEFAULT_METADATA_COLUMNS", "HAVE_LANGCHAIN"]
