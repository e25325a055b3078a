"""`Index`: the Python face of one device-resident embedding table (one GPU).

Thin wrapper over the C-ABI (`include/orx.h`) -- every method is one `orx_*` call; no
arithmetic happens in Python.  PyTorch is used only for tensor hand-off (device pointers,
current stream).  Ids are 128-bit (``langchain_id UUID``, reference app/database.py:119)
carried as ``uint64 [n, 2]`` (hi, lo) arrays; helpers convert UUID strings / ints.
"""
from __future__ import annotations

import ctypes as C
import uuid
import weakref
from typing import Iterable, Sequence

import numpy as np

from . import _lib
from ._lib import DTYPE_BF16, DTYPE_F32, ORX_DIM, OrxError, OrxId, OrxStats, check, lib

try:  # tensor hand-off only
    import torch
except Exception:  # pragma: no cover - torch is part of the image
    torch = None

_DTYPES = {"fp32": DTYPE_F32, "f32": DTYPE_F32, "float32": DTYPE_F32,
           "bf16": DTYPE_BF16, "bfloat16": DTYPE_BF16, DTYPE_F32: DTYPE_F32, DTYPE_BF16: DTYPE_BF16}


# ----------------------------------------------------------------------------- ids
def ids_to_array(ids) -> np.ndarray:
    """Anything id-like -> contiguous ``uint64 [n, 2]`` (hi, lo).

    Accepts a ``uint64 [n, 2]`` array, a 1-D integer array (ids < 2**64), or a sequence of
    ``int`` / ``uuid.UUID`` / UUID strings (what ``adelete(ids=[...])`` receives,
    reference app/rag.py:231)."""
    if isinstance(ids, np.ndarray):
        if ids.ndim == 2 and ids.shape[1] == 2:
            return np.ascontiguousarray(ids, dtype=np.uint64)
        if ids.ndim == 1 and ids.dtype.kind in "iu":
            out = np.zeros((ids.shape[0], 2), np.uint64)
            out[:, 1] = ids.astype(np.uint64)
            return out
    ids = list(ids)
    out = np.empty((len(ids), 2), np.uint64)
    for i, v in enumerate(ids):
        if isinstance(v, str):
            v = uuid.UUID(v).int
        elif isinstance(v, uuid.UUID):
            v = v.int
        else:
            v = int(v)
        if v < 0 or v >> 128:
            raise ValueError(f"id {v} does not fit 128 bits")
        out[i, 0] = v >> 64
        out[i, 1] = v & 0xFFFFFFFFFFFFFFFF
    return out


def ids_to_ints(ids: np.ndarray) -> list[int]:
    a = np.asarray(ids, dtype=np.uint64).reshape(-1, 2)
    return [(int(h) << 64) | int(l) for h, l in a]


def ids_to_uuid_strs(ids: np.ndarray) -> list[str]:
    return [str(uuid.UUID(int=v)) for v in ids_to_ints(ids)]


def _is_cuda_tensor(x) -> bool:
    return torch is not None and isinstance(x, torch.Tensor) and x.is_cuda


def _fence_producer(t) -> None:
    """A multi-GPU index launches on its own per-device streams: work that torch still has in flight on the tensor's
    current stream (the kernel that PRODUCES a query batch or a row block) must be finished before the library reads it.
    (A single-GPU index shares torch's stream after `use_torch_stream()`, or the legacy default stream.)"""
    torch.cuda.current_stream(t.device).synchronize()


def _host_f32(x, what: str) -> np.ndarray:
    if torch is not None and isinstance(x, torch.Tensor):
        x = x.detach().cpu().numpy()
    a = np.asarray(x)
    if a.ndim == 1:
        a = a.reshape(1, -1)
    if a.ndim != 2:
        raise _lib.OrxValueError(_lib.ORX_ERR_DIM, f"{what} must be [n, {ORX_DIM}]")
    return np.ascontiguousarray(a, dtype=np.float32)


def _host_result(nq: int, k: int):
    """Host result triple ``(ids uint64 [nq,k,2], dist float64 [nq,k], counts int32 [nq])``: zero ids, NaN distances."""
    k = max(k, 0)
    return np.zeros((nq, k, 2), np.uint64), np.full((nq, k), np.nan, np.float64), np.zeros(nq, np.int32)


def _device_result(nq: int, k: int, device):
    """Uninitialised CUDA result triple ``(ids int64 [nq,k,2], dist float64 [nq,k], counts int32 [nq])``."""
    return (torch.empty((nq, k, 2), dtype=torch.int64, device=device),
            torch.empty((nq, k), dtype=torch.float64, device=device),
            torch.empty((nq,), dtype=torch.int32, device=device))


def parse_vector_text(text, dim: int = ORX_DIM) -> np.ndarray:
    """pgvector's text input (``'[0.1, 0.2, ...]'`` -> fp32 ``[dim]``) with its checks: the format the
    reference sends the query vector and the stored embeddings in.  One rounding, decimal -> fp32
    (``np.asarray(list_of_python_floats, float32)`` rounds twice; the two differ only when the double
    sits on an fp32 rounding boundary).  Host-only; raises OrxValueError like pgvector raises."""
    raw = text.encode("ascii", "replace") if isinstance(text, str) else bytes(text)
    out = np.empty(int(dim), np.float32)
    check(lib.orx_parse_vector_text(raw, len(raw), C.c_void_p(out.ctypes.data), int(dim)))
    return out


class Filter:
    """A reusable predicate on chunk ids (`orx_filter_*`): the id -> row resolution and the row bitmap stay
    on the device between searches and follow upserts / deletes.  Pass it to `Index.search_filtered`."""

    is_filter_handle = True       # what `GpuVectorStore` / `QueryBatcher` look for (daemon.RemoteFilter has it too)

    def __init__(self, index: "Index", allow_ids):
        self._f = C.c_void_p()
        self._index = index
        ida = ids_to_array(allow_ids)
        check(lib.orx_filter_create(index._h, C.c_void_p(ida.ctypes.data), ida.shape[0], C.byref(self._f)))

    def handle_for(self, index: "Index"):
        """The C handle, once it is checked to be open and to belong to `index`."""
        if self._index is not index or not self._f:
            raise _lib.OrxValueError(_lib.ORX_ERR_INVALID, "filter is closed or belongs to another index")
        return self._f

    def close(self) -> None:
        if getattr(self, "_f", None) is not None and self._f:
            lib.orx_filter_destroy(self._f)
            self._f = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


class PgCopyLoader:
    """Streaming cold-start load from ``COPY (SELECT langchain_id, embedding FROM langchain_pg_embedding)
    TO STDOUT (FORMAT binary)`` (`orx_pgcopy_*`; table: reference app/database.py:118-131).

    ``feed`` takes the stream in chunks of any size (bytes / bytearray / memoryview, e.g. what psycopg 3's
    ``async for data in copy`` yields); ``close`` flushes and returns ``(rows_loaded, rows_null)``.
    ``index=None`` is a dry run that only validates the stream on the host (no GPU).  ``world`` / ``rank``:
    keep only the rows this rank owns under ``sharded.shard_of`` (every rank feeds the same stream)."""

    def __init__(self, index: "Index | None" = None, world: int = 1, rank: int = 0):
        self._ld = C.c_void_p()
        self._index = index          # keeps the table alive while the loader holds its handle
        self.result = None           # (rows_loaded, rows_null) once closed
        check(lib.orx_pgcopy_open_sharded(index._h if index is not None else None, int(world), int(rank),
                                          C.byref(self._ld)))
        if index is not None:
            index._loaders.add(self)     # Index.close() settles the batch this loader may have in flight first

    def _abandon(self) -> None:
        """The index is being closed under an open loader: wait for its batch in flight, free it, load nothing more."""
        if self._ld:
            ld, self._ld = self._ld, C.c_void_p()
            lib.orx_pgcopy_close(ld, None, None)

    def feed(self, data) -> None:
        if not self._ld:
            raise _lib.OrxValueError(_lib.ORX_ERR_INVALID, "loader is closed")
        if self._index is not None and not self._index._h:
            raise _lib.OrxValueError(_lib.ORX_ERR_INVALID, "the index of this loader was closed")
        a = np.frombuffer(data, dtype=np.uint8)          # zero-copy view of any contiguous buffer
        if a.size:
            check(lib.orx_pgcopy_feed(self._ld, C.c_void_p(a.ctypes.data), a.size))

    def close(self) -> tuple[int, int]:
        if not self._ld:
            return (0, 0)
        rows, nulls = C.c_uint64(0), C.c_uint64(0)
        ld, self._ld = self._ld, C.c_void_p()
        if self._index is not None and not self._index._h:
            raise _lib.OrxValueError(_lib.ORX_ERR_INVALID, "the index of this loader was closed before the loader")
        rc = lib.orx_pgcopy_close(ld, C.byref(rows), C.byref(nulls))
        self.result = (int(rows.value), int(nulls.value))
        check(rc)
        return self.result

    def __enter__(self):
        return self

    def __exit__(self, exc_type, *exc):
        if exc_type is None:
            self.close()
        else:                         # already failing: free the loader, keep the original exception
            try:
                self.close()
            except OrxError:
                pass

    def __del__(self):
        try:
            if self._ld:
                lib.orx_pgcopy_close(self._ld, None, None)
                self._ld = C.c_void_p()
        except Exception:
            pass


class Index:
    """One GPU's share of ``langchain_pg_embedding.embedding`` (reference app/database.py:118-131).

    ``dtype``: ``"fp32"`` keeps rows verbatim (bit-exact ids vs the oracle), ``"bf16"`` stores
    RNE-bf16 of the normalised row (half the HBM traffic; recall@k is reported)."""

    def __init__(self, dtype="fp32", capacity: int = 0, device: int | None = None, dim: int = ORX_DIM,
                 devices: Sequence[int] | None = None):
        """``devices=[0, 1, ..., 7]``: ONE table row-sharded over those GPUs, driven by this process
        (`orx_create_multi`; rows placed by ``mix64(id) mod len(devices)``; searches run on all GPUs at once and the
        k candidates per query meet on ``devices[0]`` over NVLink).  Same methods as a single-GPU index."""
        self._h = C.c_void_p()
        self._loaders = weakref.WeakSet()        # open COPY loaders (engine.PgCopyLoader)
        if devices is not None:
            devs = [int(d) for d in devices]
            if not devs:
                raise _lib.OrxValueError(_lib.ORX_ERR_INVALID, "devices must not be empty")
            arr = (C.c_int * len(devs))(*devs)
            self.device = devs[0]
            self.devices = devs
            check(lib.orx_create_multi(C.byref(self._h), int(dim), _DTYPES[dtype], int(capacity), arr, len(devs)))
        else:
            if device is None:
                device = torch.cuda.current_device() if (torch is not None and torch.cuda.is_available()) else 0
            self.device = int(device)
            self.devices = [self.device]
            check(lib.orx_create(C.byref(self._h), int(dim), _DTYPES[dtype], int(capacity), self.device))
        self.dtype = "fp32" if _DTYPES[dtype] == DTYPE_F32 else "bf16"

    # -- lifetime
    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h:
            for ld in list(getattr(self, "_loaders", ())):     # a COPY loader commits its batches on a helper thread
                ld._abandon()
            lib.orx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):  # noqa: D401
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __len__(self) -> int:
        return int(lib.orx_size(self._h))

    @property
    def capacity(self) -> int:
        return int(lib.orx_capacity(self._h))

    @property
    def shard_count(self) -> int:
        return int(lib.orx_shard_count(self._h))

    def use_torch_stream(self) -> None:
        """Launch on torch's current stream so ``torch.cuda.Event`` timing sees the kernels (single-GPU index; a
        multi-GPU index runs on its own per-device streams and every call returns only when its result is there)."""
        if len(self.devices) > 1 or self.shard_count > 1:
            return
        check(lib.orx_set_stream(self._h, C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)))

    def set_stream(self, cuda_stream: int) -> None:
        check(lib.orx_set_stream(self._h, C.c_void_p(cuda_stream)))

    def set_option(self, option: int, value: int) -> None:
        check(lib.orx_set_option(self._h, int(option), int(value)))

    def stats(self) -> dict:
        st = OrxStats()
        check(lib.orx_get_stats(self._h, C.byref(st)))
        return {name: getattr(st, name) for name, _ in OrxStats._fields_ if name != "reserved"}

    # -- writes
    def upsert(self, ids, vecs) -> None:
        """``aadd_documents`` -> INSERT ... ON CONFLICT DO UPDATE (reference app/rag.py:235)."""
        ida = ids_to_array(ids)
        if _is_cuda_tensor(vecs):
            if vecs.dim() != 2 or vecs.dtype != torch.float32:
                raise _lib.OrxValueError(_lib.ORX_ERR_DIM, "device vecs must be a float32 [n, dim] tensor")
            v = vecs.contiguous()
            if len(self.devices) > 1:
                _fence_producer(v)
            n, dim, ptr = v.shape[0], v.shape[1], v.data_ptr()
        else:
            v = _host_f32(vecs, "vecs")
            n, dim, ptr = v.shape[0], v.shape[1], v.ctypes.data
        if ida.shape[0] != n:
            raise _lib.OrxValueError(_lib.ORX_ERR_INVALID, f"{ida.shape[0]} ids for {n} vectors")
        check(lib.orx_upsert(self._h, C.c_void_p(ida.ctypes.data), C.c_void_p(ptr), n, dim))

    def delete(self, ids) -> int:
        """``adelete(ids=[...])`` -> DELETE ... WHERE langchain_id IN (...) (reference app/rag.py:231)."""
        ida = ids_to_array(ids)
        removed = C.c_uint64(0)
        check(lib.orx_delete(self._h, C.c_void_p(ida.ctypes.data), ida.shape[0], C.byref(removed)))
        return int(removed.value)

    def contains(self, one_id) -> bool:
        a = ids_to_array([one_id])
        return bool(lib.orx_contains(self._h, OrxId(int(a[0, 0]), int(a[0, 1]))))

    def fetch(self, ids):
        """Stored rows as fp32 ``[n, dim]`` + found mask (debugging / snapshots)."""
        ida = ids_to_array(ids)
        n = ida.shape[0]
        out = np.zeros((n, ORX_DIM), np.float32)
        found = np.zeros(n, np.int32)
        check(lib.orx_fetch(self._h, C.c_void_p(ida.ctypes.data), n, C.c_void_p(out.ctypes.data),
                            C.c_void_p(found.ctypes.data)))
        return out, found.astype(bool)

    # -- reads
    def search(self, queries, k: int = 12, out=None):
        """Exact ``ORDER BY embedding <=> :q LIMIT :k`` for each query row.

        Host input (NumPy / CPU tensor) -> NumPy ``(ids uint64 [nq,k,2], dist float64 [nq,k],
        counts int32 [nq])``.  CUDA tensor input -> the same as device tensors (ids int64 bit
        patterns), no host copies of the results; ``out`` = (ids, dist, counts) CUDA tensors to write into
        (a closed loop of searches then allocates nothing)."""
        if _is_cuda_tensor(queries):
            q = queries.contiguous()
            if q.dim() == 1:
                q = q.unsqueeze(0)
            if q.dtype != torch.float32:
                raise _lib.OrxValueError(_lib.ORX_ERR_INVALID, "device queries must be float32")
            nq, dim = q.shape
            if len(self.devices) > 1:
                _fence_producer(q)
            ids, dist, cnt = out if out is not None else _device_result(nq, k, q.device)
            check(lib.orx_search(self._h, C.c_void_p(q.data_ptr()), nq, dim, int(k), C.c_void_p(ids.data_ptr()),
                                 C.c_void_p(dist.data_ptr()), C.c_void_p(cnt.data_ptr())))
            return ids, dist, cnt
        q = _host_f32(queries, "queries")
        nq, dim = q.shape
        ids, dist, cnt = _host_result(nq, k)
        check(lib.orx_search(self._h, C.c_void_p(q.ctypes.data), nq, dim, int(k), C.c_void_p(ids.ctypes.data),
                             C.c_void_p(dist.ctypes.data), C.c_void_p(cnt.ctypes.data)))
        return ids, dist, cnt

    def debug_coarse_scores(self, queries, use_pairs: bool = False):
        """Diagnostic (`orx_debug_coarse_scores`): float32 CUDA tensor [live rows, nq] of the tcgen05 pass's coarse
        scores, rows in table order."""
        q = _host_f32(queries, "queries") if not _is_cuda_tensor(queries) else queries.contiguous()
        nq = q.shape[0]
        out = torch.empty((len(self), nq), dtype=torch.float32, device=f"cuda:{self.device}")
        ptr = q.data_ptr() if _is_cuda_tensor(q) else q.ctypes.data
        check(lib.orx_debug_coarse_scores(self._h, C.c_void_p(ptr), nq, int(bool(use_pairs)), C.c_void_p(out.data_ptr())))
        return out

    def debug_fast_scores(self, queries):
        """Diagnostic (`orx_debug_fast_scores`): float32 CUDA tensor [live rows, nq] of the GEMV scans' fast scores,
        rows in table order."""
        q = _host_f32(queries, "queries") if not _is_cuda_tensor(queries) else queries.contiguous()
        nq = q.shape[0]
        out = torch.empty((len(self), nq), dtype=torch.float32, device=f"cuda:{self.device}")
        ptr = q.data_ptr() if _is_cuda_tensor(q) else q.ctypes.data
        check(lib.orx_debug_fast_scores(self._h, C.c_void_p(ptr), nq, C.c_void_p(out.data_ptr())))
        return out

    def debug_image_scores(self, queries):
        """Diagnostic (`orx_debug_image_scores`): float32 CUDA tensor [live rows, nq] of the fast scores the GEMV scans
        over an fp32 table's bf16 image key on, rows in table order.  Raises when the index has no image."""
        q = _host_f32(queries, "queries") if not _is_cuda_tensor(queries) else queries.contiguous()
        nq = q.shape[0]
        out = torch.empty((len(self), nq), dtype=torch.float32, device=f"cuda:{self.device}")
        ptr = q.data_ptr() if _is_cuda_tensor(q) else q.ctypes.data
        check(lib.orx_debug_image_scores(self._h, C.c_void_p(ptr), nq, C.c_void_p(out.data_ptr())))
        return out

    def debug_image8_scores(self, queries):
        """Diagnostic (`orx_debug_image8_scores`): float32 CUDA tensor [live rows, nq] of the scores the scans over an fp32
        table's 8-bit image key on, rows in table order.  Raises when the index has no 8-bit image."""
        q = _host_f32(queries, "queries") if not _is_cuda_tensor(queries) else queries.contiguous()
        nq = q.shape[0]
        out = torch.empty((len(self), nq), dtype=torch.float32, device=f"cuda:{self.device}")
        ptr = q.data_ptr() if _is_cuda_tensor(q) else q.ctypes.data
        check(lib.orx_debug_image8_scores(self._h, C.c_void_p(ptr), nq, C.c_void_p(out.data_ptr())))
        return out

    # -- two searches in flight (orx_search_submit / orx_search_wait)
    def search_submit(self, queries, k: int, out, sharded: bool = False) -> int:
        """Launch a search of a float32 CUDA tensor `queries` into the caller-owned CUDA tensors `out` =
        (ids int64 [nq,k,2], dist float64 [nq,k], counts int32 [nq]) and return a ticket at once; at most two
        tickets may be outstanding.  `search_wait(ticket)` completes it (`out` is filled then).  `sharded=True`:
        the collective row-sharded search (every rank submits and waits in the same order)."""
        q = queries if queries.dim() == 2 else queries.unsqueeze(0)
        t = C.c_int(-1)
        fn = lib.orx_search_sharded_submit if sharded else lib.orx_search_submit
        check(fn(self._h, C.c_void_p(q.data_ptr()), q.shape[0], q.shape[1], int(k), C.c_void_p(out[0].data_ptr()),
                 C.c_void_p(out[1].data_ptr()), C.c_void_p(out[2].data_ptr()), C.byref(t)))
        return int(t.value)

    def search_wait(self, ticket: int) -> None:
        check(lib.orx_search_wait(self._h, int(ticket)))

    def make_filter(self, allow_ids) -> Filter:
        return Filter(self, allow_ids)

    def search_filtered(self, queries, k: int, allow_ids):
        """Exact top-k among the given chunk ids only (`WHERE langchain_id IN (...)`); NumPy in/out.
        `allow_ids`: ids (resolved on every call) or a `Filter` (resolved once, kept on the device)."""
        q = _host_f32(queries, "queries")
        nq, dim = q.shape
        ids, dist, cnt = _host_result(nq, k)
        if isinstance(allow_ids, Filter):
            check(lib.orx_search_with_filter(self._h, allow_ids.handle_for(self), C.c_void_p(q.ctypes.data), nq, dim, int(k),
                                             C.c_void_p(ids.ctypes.data), C.c_void_p(dist.ctypes.data),
                                             C.c_void_p(cnt.ctypes.data)))
            return ids, dist, cnt
        allow = ids_to_array(allow_ids)
        check(lib.orx_search_filtered(self._h, C.c_void_p(q.ctypes.data), nq, dim, int(k),
                                      C.c_void_p(allow.ctypes.data), allow.shape[0], C.c_void_p(ids.ctypes.data),
                                      C.c_void_p(dist.ctypes.data), C.c_void_p(cnt.ctypes.data)))
        return ids, dist, cnt

    def search_mmr(self, queries, k: int = 4, fetch_k: int = 20, lambda_mult: float = 0.5, allow_ids=None):
        """Maximal marginal relevance over the exact top-`fetch_k` (`orx_search_mmr*`): `min(k, candidates)` rows per
        query, picked greedily by `lambda_mult * (1 - distance) - (1 - lambda_mult) * max cosine to the rows picked so
        far` (include/orx.h states the exact rule).  `allow_ids`: None, ids or a `Filter`, as in `search_filtered`.
        NumPy in / out: ``(ids uint64 [nq,k,2], dist float64 [nq,k], counts int32 [nq])`` in SELECTION order, each
        row with its query distance.  Not served by the micro-batcher or the row-sharded `ShardedIndex`."""
        q = _host_f32(queries, "queries")
        nq, dim = q.shape
        ids, dist, cnt = _host_result(nq, k)
        outs = (C.c_void_p(ids.ctypes.data), C.c_void_p(dist.ctypes.data), C.c_void_p(cnt.ctypes.data))
        head = (C.c_void_p(q.ctypes.data), nq, dim, int(k), int(fetch_k), float(lambda_mult))
        if allow_ids is None:
            check(lib.orx_search_mmr(self._h, *head, *outs))
        elif isinstance(allow_ids, Filter):
            check(lib.orx_search_mmr_with_filter(self._h, allow_ids.handle_for(self), *head, *outs))
        else:
            allow = ids_to_array(allow_ids)
            check(lib.orx_search_mmr_filtered(self._h, *head, C.c_void_p(allow.ctypes.data), allow.shape[0], *outs))
        return ids, dist, cnt

    def search_into(self, queries, k: int, ids_out, dist_out, counts_out) -> None:
        """`search` of a float32 CUDA tensor writing into caller-owned CUDA tensors (views of one
        result block in the row-sharded path: no allocation, no packing kernels)."""
        q = queries if queries.dim() == 2 else queries.unsqueeze(0)
        check(lib.orx_search(self._h, C.c_void_p(q.data_ptr()), q.shape[0], q.shape[1], int(k),
                             C.c_void_p(ids_out.data_ptr()), C.c_void_p(dist_out.data_ptr()),
                             C.c_void_p(counts_out.data_ptr())))

    def merge_blocks(self, gathered, n_lists: int, nq: int, k: int, stride_bytes: int, ids_out, dist_out,
                     counts_out) -> None:
        """Merge the per-rank result blocks an all_gather left in `gathered` (int64 CUDA tensor; each
        block = ids [nq,k,2] | distance bits [nq,k] | counts int32 [nq]) into the global top-k."""
        base = gathered.data_ptr()
        check(lib.orx_merge_topk_strided(self._h, int(n_lists), int(nq), int(k), C.c_void_p(base),
                                         C.c_void_p(base + nq * k * 16), C.c_void_p(base + nq * k * 24),
                                         int(stride_bytes), C.c_void_p(ids_out.data_ptr()),
                                         C.c_void_p(dist_out.data_ptr()), C.c_void_p(counts_out.data_ptr())))

    # -- cold start from Postgres (SURVEY.md 8f-1)
    def pgcopy_loader(self, world: int = 1, rank: int = 0) -> PgCopyLoader:
        return PgCopyLoader(self, world, rank)

    def load_pgcopy(self, chunks, world: int = 1, rank: int = 0) -> tuple[int, int]:
        """Feed an iterable of COPY BINARY chunks (or one bytes object); -> (rows_loaded, rows_null)."""
        if isinstance(chunks, (bytes, bytearray, memoryview)):
            chunks = (chunks,)
        ld = PgCopyLoader(self, world, rank)
        with ld:
            for c in chunks:
                ld.feed(c)
        return ld.result

    # -- snapshot / cold start (SURVEY.md 8f-2)
    SNAPSHOT_CHUNK = 65536

    def export_rows(self, row_start: int, n: int, ids_out: np.ndarray, rows_out: np.ndarray) -> None:
        """Live rows [row_start, row_start+n) VERBATIM in the table dtype + their ids into caller-owned host
        buffers (`orx_export_rows`; pinned buffers make it a PCIe-rate copy).  Row order is table order."""
        rb = ORX_DIM * (4 if self.dtype == "fp32" else 2)
        if ids_out.nbytes < n * 16 or rows_out.nbytes < n * rb or not ids_out.flags.c_contiguous or not rows_out.flags.c_contiguous:
            raise _lib.OrxValueError(_lib.ORX_ERR_INVALID, "export buffers too small or not contiguous")
        check(lib.orx_export_rows(self._h, int(row_start), int(n), C.c_void_p(ids_out.ctypes.data),
                                  C.c_void_p(rows_out.ctypes.data)))

    def save(self, path: str, retries: int = 3) -> dict:
        """Write `manifest.json`, `ids.npy` (uint64 [n,2]) and `vecs.npy` (rows verbatim in the table dtype, uint8
        [n, row_bytes]) under `path`.  Postgres stays the source of truth; this avoids re-loading 41 GB of vectors
        through SQL text on restart.

        The snapshot is CONSISTENT and ATOMIC: the export runs in chunks (searches and writes of other threads are not
        locked out), the index's mutation counter is read before and after, and a snapshot during which a write
        landed is discarded and retried (`retries` times, then `OrxError`); files are written into a temporary
        sibling directory that replaces `path` with one rename, so a crash leaves either the old snapshot or the new
        one, never a mixture."""
        import json
        import os
        import shutil
        path = os.path.abspath(path)
        tmp = f"{path}.tmp-{os.getpid()}"
        rb = ORX_DIM * (4 if self.dtype == "fp32" else 2)
        for _attempt in range(max(1, retries)):
            shutil.rmtree(tmp, ignore_errors=True)
            os.makedirs(tmp)
            m0 = int(lib.orx_mutation_count(self._h))
            n = len(self)
            manifest = {"format": "orx-snapshot-1", "dtype": self.dtype, "dim": ORX_DIM, "rows": n, "row_bytes": rb}
            ids = np.lib.format.open_memmap(os.path.join(tmp, "ids.npy"), mode="w+", dtype=np.uint64, shape=(n, 2))
            vecs = np.lib.format.open_memmap(os.path.join(tmp, "vecs.npy"), mode="w+", dtype=np.uint8, shape=(n, rb))
            ok = True
            try:
                for s in range(0, n, self.SNAPSHOT_CHUNK):
                    m = min(self.SNAPSHOT_CHUNK, n - s)
                    ci = np.empty((m, 2), np.uint64)
                    cv = np.empty((m, rb), np.uint8)
                    check(lib.orx_export_rows(self._h, s, m, C.c_void_p(ci.ctypes.data), C.c_void_p(cv.ctypes.data)))
                    ids[s:s + m] = ci
                    vecs[s:s + m] = cv
            except OrxError:
                ok = False                       # a concurrent delete shrank the table under the export
            ids.flush()
            vecs.flush()
            del ids, vecs
            if ok and int(lib.orx_mutation_count(self._h)) == m0 and len(self) == n:
                with open(os.path.join(tmp, "manifest.json"), "w") as f:
                    json.dump(manifest, f)
                old = f"{path}.old-{os.getpid()}"
                if os.path.exists(path):
                    os.replace(path, old)
                os.replace(tmp, path)
                shutil.rmtree(old, ignore_errors=True)
                return manifest
        shutil.rmtree(tmp, ignore_errors=True)
        raise OrxError(_lib.ORX_ERR_INVALID, "the index kept changing while the snapshot was taken; pause the writer or retry")

    @classmethod
    def load(cls, path: str, device: int | None = None, capacity: int = 0) -> "Index":
        import json
        import os
        with open(os.path.join(path, "manifest.json")) as f:
            man = json.load(f)
        if man.get("format") != "orx-snapshot-1" or man["dim"] != ORX_DIM:
            raise _lib.OrxValueError(_lib.ORX_ERR_INVALID, f"not an orx snapshot: {path}")
        n = int(man["rows"])
        ix = cls(man["dtype"], max(capacity, n), device)
        ids = np.load(os.path.join(path, "ids.npy"), mmap_mode="r")
        vecs = np.load(os.path.join(path, "vecs.npy"), mmap_mode="r")
        if ids.shape != (n, 2) or vecs.shape != (n, man["row_bytes"]):
            raise _lib.OrxValueError(_lib.ORX_ERR_INVALID, "snapshot files do not match the manifest")
        for s in range(0, n, cls.SNAPSHOT_CHUNK):
            m = min(cls.SNAPSHOT_CHUNK, n - s)
            ci = np.ascontiguousarray(ids[s:s + m])
            cv = np.ascontiguousarray(vecs[s:s + m])
            check(lib.orx_import_rows(ix._h, C.c_void_p(ci.ctypes.data), C.c_void_p(cv.ctypes.data), m))
        return ix

    # -- row-sharded search over NVLink peer memory (collective; see sharded.ShardedIndex)
    def shard_export(self, world: int, rank: int) -> bytes:
        buf = C.create_string_buffer(_lib.ORX_IPC_HANDLE_BYTES)
        check(lib.orx_shard_export(self._h, int(world), int(rank), buf))
        return buf.raw

    def shard_connect(self, handles: Sequence[bytes]) -> None:
        blob = b"".join(handles)
        check(lib.orx_shard_connect(self._h, C.c_char_p(blob), len(handles)))

    def search_sharded(self, queries, k: int = 12, out=None):
        """COLLECTIVE exact top-k over all ranks' shards (`orx_search_sharded`): same calling
        convention and result layout as :meth:`search`; `out` = reusable (ids, dist, counts) CUDA
        tensors for the device path."""
        if _is_cuda_tensor(queries):
            q = queries if queries.dim() == 2 else queries.unsqueeze(0)
            nq, dim = q.shape
            if out is None:
                out = _device_result(nq, k, q.device)
            check(lib.orx_search_sharded(self._h, C.c_void_p(q.data_ptr()), nq, dim, int(k),
                                         C.c_void_p(out[0].data_ptr()), C.c_void_p(out[1].data_ptr()),
                                         C.c_void_p(out[2].data_ptr())))
            return out
        q = _host_f32(queries, "queries")
        nq, dim = q.shape
        ids, dist, cnt = _host_result(nq, k)
        check(lib.orx_search_sharded(self._h, C.c_void_p(q.ctypes.data), nq, dim, int(k), C.c_void_p(ids.ctypes.data),
                                     C.c_void_p(dist.ctypes.data), C.c_void_p(cnt.ctypes.data)))
        return ids, dist, cnt

    def merge_topk(self, ids, dist, counts, k: int):
        """Merge ``[n_lists, nq, k]`` shard results (NumPy or CUDA tensors) into the global top-k."""
        if _is_cuda_tensor(ids):
            n_lists, nq = ids.shape[0], ids.shape[1]
            oi, od, oc = _device_result(nq, k, ids.device)
            check(lib.orx_merge_topk(self._h, n_lists, nq, int(k), C.c_void_p(ids.contiguous().data_ptr()),
                                     C.c_void_p(dist.contiguous().data_ptr()),
                                     C.c_void_p(counts.contiguous().data_ptr()), C.c_void_p(oi.data_ptr()),
                                     C.c_void_p(od.data_ptr()), C.c_void_p(oc.data_ptr())))
            return oi, od, oc
        ids = np.ascontiguousarray(ids, np.uint64)
        dist = np.ascontiguousarray(dist, np.float64)
        counts = np.ascontiguousarray(counts, np.int32)
        n_lists, nq = ids.shape[0], ids.shape[1]
        oi, od, oc = _host_result(nq, k)
        check(lib.orx_merge_topk(self._h, n_lists, nq, int(k), C.c_void_p(ids.ctypes.data),
                                 C.c_void_p(dist.ctypes.data), C.c_void_p(counts.ctypes.data),
                                 C.c_void_p(oi.ctypes.data), C.c_void_p(od.ctypes.data),
                                 C.c_void_p(oc.ctypes.data)))
        return oi, od, oc


__all__ = ["Index", "Filter", "PgCopyLoader", "parse_vector_text", "OrxError", "ids_to_array", "ids_to_ints", "ids_to_uuid_strs"]
