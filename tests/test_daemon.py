"""`IndexServer` / `RemoteIndex`: one table owner, several worker processes (reference
app/entrypoint.sh:16 starts 2 uvicorn workers).  CPU: protocol, ordering, error transport and
cross-connection batching with an oracle-backed fake; GPU: a real index served to a child process."""
import json
import os
import subprocess
import sys
import threading

import numpy as np
import pytest

from oracle import cosine_topk as O
from tests.test_batcher import FakeIndex

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture
def sock_path(tmp_path, monkeypatch):
    """The owner's socket inside `tmp_path`, named relative to it: a unix socket path may hold at most 107 bytes,
    and `tmp_path` alone can be longer than that.  Server, clients and child processes resolve it from the working
    directory, which is `tmp_path` for the duration of the test."""
    monkeypatch.chdir(tmp_path)
    return "orx.sock"


class FakeOwner(FakeIndex):
    def __init__(self, X, ids):
        super().__init__(X.copy(), ids.copy())
        self.log = []

    def __len__(self):
        return self.ids.shape[0]

    def upsert(self, ids, vecs):
        self.log.append(("upsert", len(ids)))
        self.ids = np.concatenate([self.ids, np.asarray(ids, np.uint64).reshape(-1, 2)])
        self.X = np.concatenate([self.X, np.asarray(vecs, np.float32)])

    def search_filtered(self, Q, k, allow):
        self.log.append(("search_filtered", len(allow)))
        ok = {tuple(map(int, r)) for r in np.asarray(allow, np.uint64).reshape(-1, 2)}
        keep = np.array([tuple(map(int, r)) in ok for r in self.ids], bool)
        return FakeIndex(self.X[keep], self.ids[keep]).search(np.asarray(Q, np.float32), k)

    def delete(self, ids):
        kill = {tuple(map(int, r)) for r in np.asarray(ids, np.uint64).reshape(-1, 2)}
        keep = np.array([tuple(map(int, r)) not in kill for r in self.ids], bool)
        self.log.append(("delete", int((~keep).sum())))
        self.ids, self.X = self.ids[keep], self.X[keep]
        return int((~keep).sum())


def test_two_workers_share_one_owner(small_table, sock_path):
    import outline_rag_b200 as orx
    from outline_rag_b200.daemon import RemoteIndex, serve_in_thread
    X, Q, _ = small_table
    owner = FakeOwner(X[:500], O.ids_arange(0, 500))
    path = sock_path
    srv = serve_in_thread(owner, path, batch_window_ms=30.0, max_batch=64)
    try:
        a, b = RemoteIndex(path), RemoteIndex(path)
        assert len(a) == 500
        results = {}

        def worker(name, client, qs):
            results[name] = [client.search(Q[i], 12) for i in qs]

        t1 = threading.Thread(target=worker, args=("a", a, [0, 1, 2]))
        t2 = threading.Thread(target=worker, args=("b", b, [3, 4, 5]))
        t1.start(); t2.start(); t1.join(); t2.join()
        for name, qs in (("a", [0, 1, 2]), ("b", [3, 4, 5])):
            for (ids, dist, cnt), qi in zip(results[name], qs):
                w_ids, w_d = O.topk_exact(X[:500], O.ids_arange(0, 500), Q[qi], 12)
                assert cnt[0] == 12 and np.array_equal(ids[0], w_ids) and np.array_equal(dist[0], w_d)
        assert max(n for n, _ in owner.calls) >= 2            # requests of the two workers shared a scan
        # writes pass through in order; a search acknowledged after them sees them
        a.upsert(O.ids_arange(900, 903), X[600:603])
        assert b.delete(O.ids_arange(0, 2)) == 2 and len(b) == 501
        got = b.search(X[601], 1)
        assert O.ids_to_ints(got[0][0]) == [901]
        assert owner.log == [("upsert", 3), ("delete", 2)]
        # the WHERE-clause search crosses the socket too
        f_ids, f_d, f_c = a.search_filtered(Q[0], 5, O.ids_arange(100, 140))
        w_ids, w_d = O.topk_exact(X[100:140], O.ids_arange(100, 140), Q[0], 5)
        assert f_c[0] == 5 and np.array_equal(f_ids[0], w_ids) and np.array_equal(f_d[0], w_d)
        assert owner.log[-1] == ("search_filtered", 40)
        with pytest.raises(orx.OrxValueError, match="dimensions"):
            a.search(np.zeros((1, 100), np.float32), 12)
        with pytest.raises(orx.OrxValueError):
            a.search(Q[0], 1000)
        ok = a.search(Q[0], 3)                                  # the connection survives an error reply
        assert ok[2][0] == 3
        a.close(); b.close()
    finally:
        srv.stop()
    assert not os.path.exists(path)


def test_a_failed_call_never_desynchronises_the_next_one(small_table, sock_path):
    """ADVICE r1: after a timeout (or any exception between send and receive) the old client kept its socket, and the
    next caller read the tail of the previous response -- another query's ids.  Now the connection is dropped, a
    fresh one serves the next call, responses carry the request id, and concurrent calls of ONE client use several
    connections (so the owner can batch them)."""
    import time
    import outline_rag_b200 as orx
    from outline_rag_b200.daemon import RemoteIndex, serve_in_thread
    X, Q, _ = small_table
    ids = O.ids_arange(0, 400)

    class SlowOwner(FakeOwner):
        delay = 0.0

        def search(self, Qb, k):
            time.sleep(self.delay)
            return super().search(Qb, k)

    owner = SlowOwner(X[:400], ids)
    path = sock_path
    srv = serve_in_thread(owner, path, batch_window_ms=None)
    try:
        c = RemoteIndex(path, timeout=0.3)
        owner.delay = 1.0
        with pytest.raises(orx.OrxError, match="connection dropped"):
            c.search(Q[0], 12)                                  # times out; its late response must never be read
        owner.delay = 0.0
        time.sleep(1.2)                                         # the late response has been written to the dead socket
        for qi in (1, 2, 3):
            g = c.search(Q[qi], 12)
            w_ids, w_d = O.topk_exact(X[:400], ids, Q[qi], 12)
            assert np.array_equal(g[0][0], w_ids) and np.array_equal(g[1][0], w_d), "answer of another query"
        # concurrent searches of one client: several connections, every thread gets ITS answer
        owner.delay = 0.05
        out = {}

        def one(qi):
            out[qi] = c.search(Q[qi], 12)

        ts = [threading.Thread(target=one, args=(qi,)) for qi in range(8)]
        t0 = time.perf_counter()
        [t.start() for t in ts]
        [t.join() for t in ts]
        assert time.perf_counter() - t0 < 8 * 0.05 + 0.25        # not serialised behind one socket... (the fake owner is)
        for qi in range(8):
            w_ids, _ = O.topk_exact(X[:400], ids, Q[qi], 12)
            assert np.array_equal(out[qi][0][0], w_ids)
        c.close()
        with pytest.raises(orx.OrxError, match="closed"):
            c.search(Q[0], 12)
    finally:
        srv.stop()


CHILD = r"""
import json, sys, numpy as np
sys.path.insert(0, sys.argv[1])
from outline_rag_b200.daemon import RemoteIndex
from orx_testkit.synth import Synth
syn = Synth(1024)
Q, _ = syn.queries(4, 8192)
ix = RemoteIndex(sys.argv[2])
ids, dist, cnt = ix.search(Q, 12)
print(json.dumps([len(ix), ids[:, :, 1].tolist(), [float(d).hex() for d in dist[0]]]))
"""


@pytest.mark.gpu
def test_real_index_served_to_another_process(small_table, sock_path):
    import outline_rag_b200 as orx
    from outline_rag_b200.daemon import serve_in_thread
    X, Q, _ = small_table
    ids = O.ids_arange(0, X.shape[0])
    path = sock_path
    with orx.Index("fp32") as ix:
        ix.upsert(ids, X)
        srv = serve_in_thread(ix, path, batch_window_ms=2.0)
        try:
            out = subprocess.run([sys.executable, "-c", CHILD, ROOT, path], capture_output=True, text=True, timeout=120)
            assert out.returncode == 0, out.stderr[-1500:]
            size, got_ids, dist0 = json.loads(out.stdout.strip().splitlines()[-1])
        finally:
            srv.stop()
    assert size == X.shape[0]
    for i in range(4):
        w_ids, w_d = O.topk_exact(X, ids, Q[i], 12)
        assert got_ids[i] == O.ids_to_ints(w_ids)
    assert dist0 == [float(d).hex() for d in O.topk_exact(X, ids, Q[0], 12)[1]]


def test_prepared_filters_live_in_the_owner_and_their_searches_are_coalesced(small_table, sock_path):
    """`RemoteIndex.make_filter`: the allow-list crosses the socket once, the handle stays in the owner process, and
    searches of different workers under the same handle share one filtered pass of the owner's batcher.  A
    `GpuVectorStore` over a `RemoteIndex` prepares and uses such a filter like a local one."""
    import asyncio
    import outline_rag_b200 as orx
    from outline_rag_b200.daemon import RemoteFilter, RemoteIndex, serve_in_thread
    X, Q, _ = small_table
    ids = O.ids_arange(0, 500)

    class Handle:                                               # what FakeOwner.make_filter hands out
        def __init__(self, allow):
            self.allow, self.closed = np.asarray(allow, np.uint64).reshape(-1, 2), False

        def close(self):
            self.closed = True

    class Owner(FakeOwner):
        def __init__(self, *a):
            super().__init__(*a)
            self.handles = []

        def make_filter(self, allow):
            self.handles.append(Handle(allow))
            return self.handles[-1]

        def search_filtered(self, Q, k, allow):
            if isinstance(allow, Handle):
                self.log.append(("search_with_handle", int(np.asarray(Q).shape[0])))
                allow = allow.allow
            return super().search_filtered(Q, k, allow)

    owner = Owner(X[:500], ids)
    path = sock_path
    srv = serve_in_thread(owner, path, batch_window_ms=40.0, max_batch=64)
    try:
        a, b = RemoteIndex(path), RemoteIndex(path)
        flt = a.make_filter(ids[100:300])
        assert isinstance(flt, RemoteFilter) and len(owner.handles) == 1 and len(owner.handles[0].allow) == 200
        out = {}

        def worker(name, client, qs):
            out[name] = [client.search_filtered(Q[i], 7, flt if client is a else ids[100:300]) for i in qs]

        t1 = threading.Thread(target=worker, args=("a1", a, [0, 1]))
        t2 = threading.Thread(target=worker, args=("a2", a, [2, 3]))
        t1.start(); t2.start(); t1.join(); t2.join()
        for name, qs in (("a1", [0, 1]), ("a2", [2, 3])):
            for (g_ids, g_d, g_c), qi in zip(out[name], qs):
                w_ids, w_d = O.topk_exact(X[100:300], ids[100:300], Q[qi], 7)
                assert g_c[0] == 7 and np.array_equal(g_ids[0], w_ids) and np.array_equal(g_d[0], w_d)
        handle_calls = [n for op, n in owner.log if op == "search_with_handle"]
        assert sum(handle_calls) == 4 and max(handle_calls) >= 2        # two threads' searches shared a filtered pass
        with pytest.raises(orx.OrxValueError, match="another index"):
            b.search_filtered(Q[0], 3, flt)

        # the vector store of a worker process: prepare once, search under the handle
        class Emb:
            async def aembed_query(self, text):
                return X[int(text)]

        store = orx.GpuVectorStore(a, Emb(), batch_window_ms=None)
        store.doc_store.put_many([str(uuid_of(i)) for i in range(500)], [str(i) for i in range(500)],
                                 [{"source_id": f"d{i // 100}"} for i in range(500)])
        prepared = store.prepare_filter({"source_id": "d2"})
        assert isinstance(prepared, RemoteFilter)
        hits = asyncio.run(store.asimilarity_search("250", k=3, filter=prepared))
        assert [h.page_content for h in hits][0] == "250" and all(200 <= int(h.page_content) < 300 for h in hits)
        prepared.close()
        flt.close()
        assert all(h.closed for h in owner.handles)
        with pytest.raises(orx.OrxValueError, match="closed"):
            a.search_filtered(Q[0], 3, flt)
        a.close(); b.close()
    finally:
        srv.stop()


def uuid_of(i):
    import uuid
    return uuid.UUID(int=i)


@pytest.mark.gpu
def test_remote_prepared_filter_on_a_real_index(small_table, sock_path):
    """The same over a real device table: a worker prepares a filter that admits 5000 of 8192 rows (bitmap regime); 12
    concurrent searches under it are coalesced by the owner into filtered tensor-core passes; answers equal the oracle's."""
    import outline_rag_b200 as orx
    from outline_rag_b200.daemon import RemoteIndex, serve_in_thread
    X, Q, _ = small_table
    n = X.shape[0]
    ids = O.ids_arange(0, n)
    sel = np.sort(np.random.default_rng(8).choice(n, size=5000, replace=False))
    path = sock_path
    with orx.Index("fp32") as ix:
        ix.upsert(ids, X)
        srv = serve_in_thread(ix, path, batch_window_ms=30.0, max_batch=64)
        try:
            client = RemoteIndex(path, max_connections=16)
            with client.make_filter(ids[sel]) as flt:
                out = [None] * 12

                def one(i):
                    out[i] = client.search_filtered(Q[i], 12, flt)

                th = [threading.Thread(target=one, args=(i,)) for i in range(12)]
                for t in th:
                    t.start()
                for t in th:
                    t.join()
                st = ix.stats()
            client.close()
        finally:
            srv.stop()
    for i in range(12):
        w_ids, w_d = O.topk_exact(X[sel], ids[sel], Q[i], 12, exhaustive=True)
        assert np.array_equal(out[i][0][0], w_ids) and np.array_equal(out[i][1][0].view(np.uint64), w_d.view(np.uint64)), i
    assert st["searches"] < 12 and st["queries"] == 12 and st["last_path"] == 2      # coalesced, tensor-core pass
