"""One device table, several worker processes (SURVEY.md 8f-2, second half).

The reference starts `uvicorn --workers ${UVICORN_WORKERS:-2}` (reference app/entrypoint.sh:16-18)
and every worker PROCESS builds its own `rag.vector_store` handle onto the shared Postgres
(reference app/rag.py:36-44).  A GPU-resident table must have ONE owner, so the owner runs
`IndexServer` (an asyncio unix-socket server around one `Index`) and every worker talks to it
through `RemoteIndex`, which has the same `search / upsert / delete / __len__` surface as
`Index` and can be handed to `GpuVectorStore` as its index.

Searches arriving from different workers within the batching window are coalesced by the
server's `QueryBatcher` into one tcgen05 scan -- cross-process micro-batching for free.
Writes are applied in arrival order on the owner's single stream, so a search issued after an
upsert was acknowledged sees it (same guarantee as in-process use).

Wire format: 4-byte big-endian length + msgpack map {"op", "rid", ...}; arrays travel as raw bytes with
shape / dtype fields; every response echoes the request id ("rid").  Errors come back as
{"err": code, "msg": text} and are re-raised as `OrxError` / `OrxValueError` on the client, so
`api.py:125-127`'s "log and return no documents" behaviour is unchanged.

The client keeps a small POOL of connections: concurrent searches of one worker travel on different connections (so
the owner's batcher can coalesce them too), and a connection on which anything went wrong -- a timeout, a partial
read, a decode error, a response whose id is not the request's -- is CLOSED and never reused: a later caller can never
read the tail of somebody else's response.
"""
from __future__ import annotations

import asyncio
import os
import socket
import struct
import threading
from typing import Optional

import msgpack
import numpy as np

from ._lib import ORX_ERR_INVALID, OrxError, OrxValueError
from .batcher import QueryBatcher


def _pack_arr(a: np.ndarray) -> dict:
    a = np.ascontiguousarray(a)
    return {"shape": list(a.shape), "dtype": a.dtype.str, "data": a.tobytes()}


def _unpack_arr(d: dict) -> np.ndarray:
    return np.frombuffer(d["data"], dtype=np.dtype(d["dtype"])).reshape(d["shape"]).copy()


def _err_payload(e: Exception) -> dict:
    code = getattr(e, "code", -100)
    return {"err": int(code), "msg": getattr(e, "message", str(e)), "value_error": isinstance(e, ValueError)}


def _raise_from(resp: dict):
    cls = OrxValueError if resp.get("value_error") else OrxError
    raise cls(resp["err"], resp["msg"])


# --------------------------------------------------------------------------------- server
class IndexServer:
    """Owns `index`; serve with `await server.start()` / `await server.serve_forever()`."""

    def __init__(self, index, path: str, batch_window_ms: Optional[float] = 1.0, max_batch: int = 256):
        self.index = index
        self.path = path
        self.batcher = QueryBatcher(index, max_batch, batch_window_ms) if batch_window_ms is not None else None
        self._server: Optional[asyncio.AbstractServer] = None
        self._write_lock = asyncio.Lock()
        self._filters: dict[int, object] = {}        # prepared filters (device-resident in this process) by id
        self._next_fid = 0

    async def start(self) -> None:
        if os.path.exists(self.path):
            os.unlink(self.path)
        self._server = await asyncio.start_unix_server(self._client, path=self.path)

    async def serve_forever(self) -> None:
        async with self._server:
            await self._server.serve_forever()

    async def close(self) -> None:
        if self.batcher is not None:
            await self.batcher.drain()
        if self._server is not None:
            self._server.close()
            await self._server.wait_closed()
        if os.path.exists(self.path):
            os.unlink(self.path)

    async def _client(self, reader: asyncio.StreamReader, writer: asyncio.StreamWriter) -> None:
        try:
            while True:
                head = await reader.readexactly(4)
                body = await reader.readexactly(struct.unpack(">I", head)[0])
                req = msgpack.unpackb(body, raw=False)
                # requests of one connection are answered in order; different connections interleave
                resp = await self._handle(req)
                resp["rid"] = req.get("rid")
                out = msgpack.packb(resp, use_bin_type=True)
                writer.write(struct.pack(">I", len(out)) + out)
                await writer.drain()
        except (asyncio.IncompleteReadError, ConnectionResetError, BrokenPipeError):
            pass
        finally:
            writer.close()

    @staticmethod
    def _pack_rows(res, k: int) -> dict:
        """Per-query results of the batcher -> the padded arrays of `Index.search`; the first failure is raised."""
        for r in res:
            if isinstance(r, Exception):
                raise r
        ids = np.zeros((len(res), k, 2), np.uint64)
        dist = np.full((len(res), k), np.nan)
        cnt = np.zeros(len(res), np.int32)
        for i, (a, b) in enumerate(res):
            ids[i, :len(b)], dist[i, :len(b)], cnt[i] = a, b, len(b)
        return {"ids": _pack_arr(ids), "dist": _pack_arr(dist), "cnt": _pack_arr(cnt)}

    async def _handle(self, req: dict) -> dict:
        try:
            op = req.get("op")
            if op == "search":
                Q = _unpack_arr(req["q"])
                k = int(req["k"])
                if self.batcher is not None:
                    res = await asyncio.gather(*[self.batcher.search(q, k) for q in Q], return_exceptions=True)
                    return self._pack_rows(res, k)
                ids, dist, cnt = await asyncio.to_thread(self.index.search, Q, k)
                return {"ids": _pack_arr(ids), "dist": _pack_arr(dist), "cnt": _pack_arr(cnt)}
            if op == "search_filtered":
                Q, k = _unpack_arr(req["q"]), int(req["k"])
                if "fid" in req:
                    flt = self._filters.get(int(req["fid"]))
                    if flt is None:
                        return {"err": ORX_ERR_INVALID, "msg": f"unknown filter {req['fid']}", "value_error": True}
                    if self.batcher is not None:
                        # searches under the same prepared filter, from any worker, share one filtered pass
                        res = await asyncio.gather(*[self.batcher.search(q, k, flt) for q in Q], return_exceptions=True)
                        return self._pack_rows(res, k)
                    ids, dist, cnt = await asyncio.to_thread(self.index.search_filtered, Q, k, flt)
                else:
                    ids, dist, cnt = await asyncio.to_thread(self.index.search_filtered, Q, k, _unpack_arr(req["allow"]))
                return {"ids": _pack_arr(ids), "dist": _pack_arr(dist), "cnt": _pack_arr(cnt)}
            if op == "search_mmr":
                # never through the batcher: one MMR call per request, on the owner's index
                Q, k = _unpack_arr(req["q"]), int(req["k"])
                allow = None
                if "fid" in req:
                    allow = self._filters.get(int(req["fid"]))
                    if allow is None:
                        return {"err": ORX_ERR_INVALID, "msg": f"unknown filter {req['fid']}", "value_error": True}
                elif "allow" in req:
                    allow = _unpack_arr(req["allow"])
                ids, dist, cnt = await asyncio.to_thread(self.index.search_mmr, Q, k, int(req["fetch_k"]),
                                                         float(req["lambda_mult"]), allow)
                return {"ids": _pack_arr(ids), "dist": _pack_arr(dist), "cnt": _pack_arr(cnt)}
            if op == "filter_create":
                flt = await asyncio.to_thread(self.index.make_filter, _unpack_arr(req["allow"]))
                self._next_fid += 1
                self._filters[self._next_fid] = flt
                return {"fid": self._next_fid}
            if op == "filter_drop":
                flt = self._filters.pop(int(req["fid"]), None)
                if flt is not None and hasattr(flt, "close"):
                    await asyncio.to_thread(flt.close)
                return {"ok": True}
            if op == "upsert":
                async with self._write_lock:
                    await asyncio.to_thread(self.index.upsert, _unpack_arr(req["ids"]), _unpack_arr(req["vecs"]))
                return {"ok": True}
            if op == "delete":
                async with self._write_lock:
                    n = await asyncio.to_thread(self.index.delete, _unpack_arr(req["ids"]))
                return {"removed": int(n)}
            if op == "size":
                return {"size": len(self.index)}
            return {"err": ORX_ERR_INVALID, "msg": f"unknown op {op!r}", "value_error": True}
        except Exception as e:      # noqa: BLE001 -- every failure travels back to the caller
            return _err_payload(e)


def serve_in_thread(index, path: str, **kw) -> "ServerThread":
    """Run an `IndexServer` on its own event loop in a daemon thread (tests, single-binary deployments)."""
    t = ServerThread(index, path, **kw)
    t.start()
    t.ready.wait(10)
    return t


class ServerThread(threading.Thread):
    def __init__(self, index, path: str, **kw):
        super().__init__(daemon=True)
        self.index, self.path, self.kw = index, path, kw
        self.ready = threading.Event()
        self.loop: Optional[asyncio.AbstractEventLoop] = None
        self.server: Optional[IndexServer] = None

    def run(self) -> None:
        self.loop = asyncio.new_event_loop()
        asyncio.set_event_loop(self.loop)
        self.server = IndexServer(self.index, self.path, **self.kw)
        self.loop.run_until_complete(self.server.start())
        self.ready.set()
        try:
            self.loop.run_forever()
        finally:
            self.loop.run_until_complete(self.server.close())
            self.loop.close()

    def stop(self) -> None:
        if self.loop is not None:
            self.loop.call_soon_threadsafe(self.loop.stop)
        self.join(10)


# --------------------------------------------------------------------------------- client
class _Conn:
    def __init__(self, path: str, timeout: float):
        self.sock = socket.socket(socket.AF_UNIX, socket.SOCK_STREAM)
        self.sock.settimeout(timeout)
        self.sock.connect(path)

    def close(self) -> None:
        try:
            self.sock.close()
        except OSError:
            pass

    def recv_exact(self, n: int) -> bytes:
        buf = bytearray()
        while len(buf) < n:
            chunk = self.sock.recv(n - len(buf))
            if not chunk:
                raise OrxError(-100, "index server closed the connection")
            buf += chunk
        return bytes(buf)


class RemoteFilter:
    """A prepared filter that lives in the owner process (`engine.Filter` there); the worker holds its number."""

    is_filter_handle = True

    def __init__(self, index: "RemoteIndex", fid: int):
        self._index, self._fid = index, fid

    def close(self) -> None:
        fid, self._fid = self._fid, None
        if fid is not None:
            try:
                self._index._call({"op": "filter_drop", "fid": fid})
            except OrxError:
                pass                      # the owner is gone: so is the filter

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


class RemoteIndex:
    """`Index`-shaped proxy used by a worker process: blocking calls over a pool of unix-socket connections
    (thread-safe; `GpuVectorStore` already runs index calls in `asyncio.to_thread`)."""

    def __init__(self, path: str, timeout: float = 60.0, max_connections: int = 8):
        self.path, self.timeout = path, timeout
        self._idle: list[_Conn] = [_Conn(path, timeout)]          # fail at construction if the owner is not there
        self._lock = threading.Lock()
        self._slots = threading.BoundedSemaphore(max_connections)
        self._rid = 0
        self._closed = False

    def close(self) -> None:
        with self._lock:
            self._closed = True
            idle, self._idle = self._idle, []
        for c in idle:
            c.close()

    def _call(self, req: dict) -> dict:
        with self._slots:
            with self._lock:
                if self._closed:
                    raise OrxError(-100, "RemoteIndex is closed")
                self._rid += 1
                rid = self._rid
                conn = self._idle.pop() if self._idle else None
            if conn is None:
                conn = _Conn(self.path, self.timeout)
            ok = False
            try:
                out = msgpack.packb(dict(req, rid=rid), use_bin_type=True)
                conn.sock.sendall(struct.pack(">I", len(out)) + out)
                head = conn.recv_exact(4)
                resp = msgpack.unpackb(conn.recv_exact(struct.unpack(">I", head)[0]), raw=False)
                if not isinstance(resp, dict) or resp.get("rid") != rid:
                    raise OrxError(-100, "index server answered another request (framing lost): connection dropped")
                ok = True
            except OrxError:
                raise
            except Exception as e:       # noqa: BLE001 -- timeout, reset, decode error: the stream position is unknown
                raise OrxError(-100, f"index server call failed ({type(e).__name__}: {e}): connection dropped") from e
            finally:
                if ok:
                    with self._lock:
                        if self._closed:
                            conn.close()
                        else:
                            self._idle.append(conn)
                else:
                    conn.close()             # never reused: the next caller gets a fresh connection
        if "err" in resp:
            _raise_from(resp)
        return resp

    def __len__(self) -> int:
        return int(self._call({"op": "size"})["size"])

    def search(self, queries, k: int = 12):
        q = np.asarray(queries, dtype=np.float32)
        if q.ndim == 1:
            q = q.reshape(1, -1)
        r = self._call({"op": "search", "q": _pack_arr(q), "k": int(k)})
        return _unpack_arr(r["ids"]), _unpack_arr(r["dist"]), _unpack_arr(r["cnt"])

    def search_filtered(self, queries, k: int, allow_ids):
        """`Index.search_filtered` on the owner: with ids (resolved there on every call) or with a `RemoteFilter`
        (`make_filter`: resolved once, device-resident in the owner process; only its number crosses the socket)."""
        from .engine import ids_to_array
        q = np.asarray(queries, dtype=np.float32)
        if q.ndim == 1:
            q = q.reshape(1, -1)
        req = {"op": "search_filtered", "q": _pack_arr(q), "k": int(k)}
        if isinstance(allow_ids, RemoteFilter):
            if allow_ids._index is not self or allow_ids._fid is None:
                raise OrxValueError(ORX_ERR_INVALID, "filter is closed or belongs to another index")
            req["fid"] = allow_ids._fid
        else:
            req["allow"] = _pack_arr(ids_to_array(allow_ids))
        r = self._call(req)
        return _unpack_arr(r["ids"]), _unpack_arr(r["dist"]), _unpack_arr(r["cnt"])

    def search_mmr(self, queries, k: int = 4, fetch_k: int = 20, lambda_mult: float = 0.5, allow_ids=None):
        """`Index.search_mmr` on the owner; `allow_ids`: None, ids or a `RemoteFilter`."""
        from .engine import ids_to_array
        q = np.asarray(queries, dtype=np.float32)
        if q.ndim == 1:
            q = q.reshape(1, -1)
        req = {"op": "search_mmr", "q": _pack_arr(q), "k": int(k), "fetch_k": int(fetch_k),
               "lambda_mult": float(lambda_mult)}
        if isinstance(allow_ids, RemoteFilter):
            if allow_ids._index is not self or allow_ids._fid is None:
                raise OrxValueError(ORX_ERR_INVALID, "filter is closed or belongs to another index")
            req["fid"] = allow_ids._fid
        elif allow_ids is not None:
            req["allow"] = _pack_arr(ids_to_array(allow_ids))
        r = self._call(req)
        return _unpack_arr(r["ids"]), _unpack_arr(r["dist"]), _unpack_arr(r["cnt"])

    def make_filter(self, allow_ids) -> "RemoteFilter":
        from .engine import ids_to_array
        fid = int(self._call({"op": "filter_create", "allow": _pack_arr(ids_to_array(allow_ids))})["fid"])
        return RemoteFilter(self, fid)

    def upsert(self, ids, vecs) -> None:
        from .engine import ids_to_array
        self._call({"op": "upsert", "ids": _pack_arr(ids_to_array(ids)), "vecs": _pack_arr(np.asarray(vecs, np.float32))})

    def delete(self, ids) -> int:
        from .engine import ids_to_array
        return int(self._call({"op": "delete", "ids": _pack_arr(ids_to_array(ids))})["removed"])


__all__ = ["IndexServer", "RemoteFilter", "RemoteIndex", "ServerThread", "serve_in_thread"]
