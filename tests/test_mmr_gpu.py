"""Exact maximal-marginal-relevance search on the B200 (`orx_search_mmr*`): ids, selection order and distance bits
equal to oracle/mmr.py with tolerance 0, on every path that fetches the candidates."""
import asyncio
import ctypes as C

import numpy as np
import pytest

from oracle import cosine_topk as O
from oracle.mmr import mmr_exact
from tests._helpers import stored_bf16_rows
from tests.test_mmr import KNOWN_Q, KNOWN_X

pytestmark = pytest.mark.gpu

N = 6000


@pytest.fixture(scope="module")
def tables(small_table):
    import outline_rag_b200 as orx
    X, Q, _ = small_table
    X = X[:N]
    ids = O.ids_arange(0, N)
    out = {}
    for dtype in ("fp32", "bf16"):
        ix = orx.Index(dtype, device=0)
        ix.upsert(ids, X)
        out[dtype] = (ix, X if dtype == "fp32" else stored_bf16_rows(X), ids)
    yield out, Q
    for ix, _, _ in out.values():
        ix.close()


def queries(Q, nq):
    rng = np.random.default_rng(nq)
    return np.concatenate([Q, Q + 0.05 * rng.standard_normal(Q.shape).astype(np.float32)] * 5)[:nq].astype(np.float32)


def assert_oracle(got, X, ids, Q, k, fetch_k, lam, which):
    g_ids, g_d, g_c = got
    for j in which:
        w_ids, w_d = mmr_exact(X, ids, Q[j], k, fetch_k, lam)
        n = len(w_d)
        assert g_c[j] == n, (j, g_c[j], n)
        assert np.array_equal(g_ids[j, :n], w_ids), (j, "ids / selection order differ from the oracle")
        assert np.array_equal(g_d[j, :n].view(np.uint64), w_d.view(np.uint64)), (j, "distance bits differ")
        assert not g_ids[j, n:].any() and np.isnan(g_d[j, n:]).all()


@pytest.mark.parametrize("lam", [0.0, 0.3, 0.5, 1.0])
@pytest.mark.parametrize("k,fetch_k", [(1, 1), (4, 20), (12, 48), (12, 128), (128, 128)])
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_matrix_equals_oracle(tables, dtype, k, fetch_k, lam):
    t, Q = tables
    ix, X, ids = t[dtype]
    Qb = queries(Q, 7)
    got = ix.search_mmr(Qb, k, fetch_k, lam)
    assert_oracle(got, X, ids, Qb, k, fetch_k, lam, range(7) if k < 128 else (0, 6))
    if lam == 1.0:            # pure relevance: exactly the plain exact search
        s_ids, s_d, s_c = ix.search(Qb, k)
        assert np.array_equal(got[0], s_ids) and np.array_equal(got[1].view(np.uint64), s_d.view(np.uint64))
        assert np.array_equal(got[2], s_c)


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_one_query_and_one_past_the_chunk(tables, dtype):
    t, Q = tables
    ix, X, ids = t[dtype]
    Qb = queries(Q, 257)                   # MMR_QCHUNK = 256 queries per chunk
    got = ix.search_mmr(Qb, 12, 48, 0.5)
    assert_oracle(got, X, ids, Qb, 12, 48, 0.5, (0, 1, 255, 256))
    one = ix.search_mmr(Qb[256], 12, 48, 0.5)
    assert np.array_equal(one[0][0], got[0][256]) and np.array_equal(one[1][0].view(np.uint64), got[1][256].view(np.uint64))
    part = ix.search_mmr(Qb[:256], 12, 48, 0.5)
    assert np.array_equal(part[0], got[0][:256]) and np.array_equal(part[1].view(np.uint64), got[1][:256].view(np.uint64))


def test_known_answer_ties_and_small_tables():
    import outline_rag_b200 as orx
    ids = O.ids_arange(0, 4)
    for dtype in ("fp32", "bf16"):
        with orx.Index(dtype, device=0) as ix:
            ix.upsert(ids, KNOWN_X)
            g_ids, g_d, g_c = ix.search_mmr(KNOWN_Q, 2, 4, 0.7)
            assert O.ids_to_ints(g_ids[0]) == [0, 1] and g_c[0] == 2
            g_ids, _, _ = ix.search_mmr(KNOWN_Q, 3, 4, 0.3)
            assert O.ids_to_ints(g_ids[0]) == [0, 3, 2]
            # table smaller than fetch_k and than k
            g_ids, g_d, g_c = ix.search_mmr(KNOWN_Q, 12, 20, 0.5)
            w_ids, w_d = mmr_exact(KNOWN_X if dtype == "fp32" else stored_bf16_rows(KNOWN_X), ids, KNOWN_Q, 12, 20, 0.5)
            assert g_c[0] == 4 and np.array_equal(g_ids[0, :4], w_ids) and np.isnan(g_d[0, 4:]).all()
    # exact duplicates: s_dd = 1 after the clamp, equal scores -> the lowest position (lowest id) wins every tie
    rng = np.random.default_rng(5)
    base = rng.standard_normal((3, O.DIM)).astype(np.float32)
    X = np.concatenate([np.repeat(base[:1], 4, 0), np.repeat(base[1:2], 3, 0), base[2:], 3 * base[:1]])
    ids = O.ids_arange(0, X.shape[0])
    q = (base[0] + 0.5 * base[1]).astype(np.float32)
    with orx.Index("fp32", device=0) as ix:
        ix.upsert(ids, X)
        for lam in (0.0, 0.3, 0.5, 0.9):
            got = ix.search_mmr(q, X.shape[0], X.shape[0], lam)
            assert_oracle(got, X, ids, q[None], X.shape[0], X.shape[0], lam, (0,))
    # zero-norm rows (NaN distance) and an empty table
    X = np.concatenate([KNOWN_X, np.zeros((3, O.DIM), np.float32)])
    ids = O.ids_arange(0, 7)
    with orx.Index("fp32", device=0) as ix:
        g_ids, g_d, g_c = ix.search_mmr(KNOWN_Q, 2, 20, 0.5)
        assert g_c[0] == 0 and not g_ids.any() and np.isnan(g_d).all()
        ix.upsert(ids, X)
        for lam in (0.0, 0.5, 1.0):
            assert_oracle(ix.search_mmr(KNOWN_Q, 7, 7, lam), X, ids, KNOWN_Q[None], 7, 7, lam, (0,))
        assert_oracle(ix.search_mmr(np.zeros(O.DIM, np.float32), 5, 7, 0.5), X, ids, np.zeros((1, O.DIM), np.float32),
                      5, 7, 0.5, (0,))


def test_filtered_paths(tables):
    t, Q = tables
    ix, X, ids = t["fp32"]
    Qb = queries(Q, 5)
    for allow_rows in (np.arange(100, 1100, 3), np.arange(0, N, 7).tolist() + list(range(1, 4200))):
        rows = np.unique(np.asarray(allow_rows))
        for lam in (0.3, 1.0):
            got = ix.search_mmr(Qb, 12, 48, lam, allow_ids=ids[rows])
            assert_oracle(got, X[rows], ids[rows], Qb, 12, 48, lam, range(5))
        with ix.make_filter(ids[rows]) as flt:
            again = ix.search_mmr(Qb, 12, 48, 0.3, allow_ids=flt)
            base = ix.search_mmr(Qb, 12, 48, 0.3, allow_ids=ids[rows])
            assert np.array_equal(again[0], base[0]) and np.array_equal(again[1].view(np.uint64), base[1].view(np.uint64))


@pytest.mark.parametrize("devs", [[0, 0, 0], [0, 1]], ids=["three_shards_one_gpu", "two_gpus"])
def test_multi_gpu_handle_equals_single(tables, devs):
    import torch
    import outline_rag_b200 as orx
    from outline_rag_b200 import _lib
    if torch.cuda.device_count() < max(devs) + 1:
        pytest.skip(f"{max(devs) + 1} devices are not present")
    t, Q = tables
    ix, X, ids = t["fp32"]
    Qb = queries(Q, 9)
    with orx.Index("fp32", devices=devs) as mx:
        mx.upsert(ids, X)
        for k, fk, lam in ((4, 20, 0.5), (12, 128, 0.3)):
            a, b = ix.search_mmr(Qb, k, fk, lam), mx.search_mmr(Qb, k, fk, lam)
            assert np.array_equal(a[0], b[0]) and np.array_equal(a[1].view(np.uint64), b[1].view(np.uint64))
            assert np.array_equal(a[2], b[2])
        allow = ids[::5]
        a, b = ix.search_mmr(Qb, 12, 48, 0.5, allow), mx.search_mmr(Qb, 12, 48, 0.5, allow)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1].view(np.uint64), b[1].view(np.uint64))
        out = (np.zeros((1, 4, 2), np.uint64), np.zeros((1, 4)), np.zeros(1, np.int32))
        rc = _lib.lib.orx_search_mmr_with_filter(mx._h, None, C.c_void_p(Qb.ctypes.data), 1, O.DIM, 4, 20, 0.5,
                                                 *[C.c_void_p(o.ctypes.data) for o in out])
        assert rc == _lib.ORX_ERR_INVALID and "per GPU" in _lib.last_error()


def test_after_upsert_and_delete():
    import outline_rag_b200 as orx
    rng = np.random.default_rng(11)
    X = rng.standard_normal((3000, O.DIM)).astype(np.float32)
    ids = O.ids_arange(0, 3000)
    q = X[7] + 0.1 * rng.standard_normal(O.DIM).astype(np.float32)
    with orx.Index("fp32", device=0) as ix:
        ix.upsert(ids, X)
        dead = ids[:400]
        assert ix.delete(dead) == 400
        X2 = X.copy()
        X2[500:520] = X[7] + 0.01 * rng.standard_normal((20, O.DIM)).astype(np.float32)
        ix.upsert(ids[500:520], X2[500:520])
        got = ix.search_mmr(q, 12, 64, 0.5)
        assert not set(O.ids_to_ints(got[0][0])) & set(range(400))
        live = np.arange(400, 3000)
        # the table's row order changed with the delete; the oracle's row order does not matter (ids tie-break)
        assert_oracle(got, X2[live], ids[live], q[None], 12, 64, 0.5, (0,))


def test_argument_errors_leave_search_intact(tables):
    import outline_rag_b200 as orx
    from outline_rag_b200 import _lib
    t, Q = tables
    ix = t["fp32"][0]
    before = ix.search(Q[:3], 12)
    bad = [dict(k=0, fetch_k=20), dict(k=21, fetch_k=20), dict(k=4, fetch_k=129), dict(lambda_mult=-0.1),
           dict(lambda_mult=1.5), dict(lambda_mult=float("nan")), dict(lambda_mult=float("inf"))]
    for kw in bad:
        args = dict(k=4, fetch_k=20, lambda_mult=0.5)
        args.update(kw)
        with pytest.raises(orx.OrxValueError) as e:
            ix.search_mmr(Q[:3], **args)
        assert e.value.code == _lib.ORX_ERR_INVALID, kw
    with pytest.raises(orx.OrxValueError) as e:
        ix.search_mmr(np.zeros((1, 100), np.float32), 4)
    assert e.value.code == _lib.ORX_ERR_DIM
    q = Q[:2].copy()
    q[1, 3] = np.nan
    with pytest.raises(orx.OrxValueError) as e:
        ix.search_mmr(q, 4)
    assert e.value.code == _lib.ORX_ERR_NONFINITE
    # device buffers are refused
    import torch
    qd = torch.from_numpy(Q[:1]).cuda()
    ids = np.zeros((1, 4, 2), np.uint64)
    dist = np.zeros((1, 4))
    cnt = np.zeros(1, np.int32)
    rc = _lib.lib.orx_search_mmr(ix._h, C.c_void_p(qd.data_ptr()), 1, O.DIM, 4, 20, 0.5, C.c_void_p(ids.ctypes.data),
                                 C.c_void_p(dist.ctypes.data), C.c_void_p(cnt.ctypes.data))
    assert rc == _lib.ORX_ERR_INVALID and "host" in _lib.last_error()
    # a search in flight: rejected like orx_search_filtered
    out = (torch.empty((1, 12, 2), dtype=torch.int64, device="cuda:0"), torch.empty((1, 12), dtype=torch.float64,
           device="cuda:0"), torch.empty((1,), dtype=torch.int32, device="cuda:0"))
    ticket = ix.search_submit(qd, 12, out)
    with pytest.raises(orx.OrxValueError, match="in flight"):
        ix.search_mmr(Q[:1], 4)
    ix.search_wait(ticket)
    after = ix.search(Q[:3], 12)
    assert np.array_equal(before[0], after[0]) and np.array_equal(before[1].view(np.uint64), after[1].view(np.uint64))


def test_vector_store_and_remote_index(tables, tmp_path, monkeypatch):
    import outline_rag_b200 as orx
    from outline_rag_b200 import vectorstore as vs
    from outline_rag_b200.daemon import RemoteIndex, serve_in_thread
    t, Q = tables
    ix, X, ids = t["fp32"]

    class Emb:
        def embed_query(self, s):
            return Q[int(s)]

        async def aembed_query(self, s):
            return Q[int(s)]

    sids = orx.ids_to_uuid_strs(ids)
    docs = vs.MemoryDocStore()
    docs.put_many(sids, [f"c{i}" for i in range(N)], [{"source_id": f"s{i % 10}"} for i in range(N)])
    store = vs.GpuVectorStore(ix, Emb(), docs)
    w_ids, w_d = mmr_exact(X, ids, Q[3], 12, 48, 0.5)
    order = O.order_by_distance(w_d, w_ids)
    pairs = store.max_marginal_relevance_search_with_score_by_vector(Q[3], k=12, fetch_k=48)
    assert [d.id for d, _ in pairs] == orx.ids_to_uuid_strs(w_ids[order])
    assert [s for _, s in pairs] == [float(x) for x in w_d[order]]
    got = asyncio.run(store.amax_marginal_relevance_search("3", k=12, fetch_k=48))
    assert [d.id for d in got] == [d.id for d, _ in pairs]
    # filter= as a predicate and as a prepared handle
    allowed = np.array([i for i in range(N) if i % 10 == 4])
    w_ids, w_d = mmr_exact(X[allowed], ids[allowed], Q[3], 12, 48, 0.5)
    want = orx.ids_to_uuid_strs(w_ids[O.order_by_distance(w_d, w_ids)])
    assert [d.id for d in store.max_marginal_relevance_search("3", k=12, fetch_k=48, filter={"source_id": "s4"})] == want
    flt = store.prepare_filter({"source_id": "s4"})
    assert [d.id for d in store.max_marginal_relevance_search("3", k=12, fetch_k=48, filter=flt)] == want
    flt.close()
    # relevance scores: 1 - distance of the plain exact search, thresholded
    s_ids, s_d, _ = ix.search(Q[3:4], 12)
    rel = store.similarity_search_with_relevance_scores("3", k=12, score_threshold=float(1.0 - s_d[0, 5]))
    assert [s for _, s in rel] == [1.0 - float(x) for x in s_d[0, :6]]
    # the owner process serves it to workers
    monkeypatch.chdir(tmp_path)
    srv = serve_in_thread(ix, "orx.sock", batch_window_ms=1.0)
    try:
        cli = RemoteIndex("orx.sock")
        a, b = cli.search_mmr(Q[:4], 12, 48, 0.3), ix.search_mmr(Q[:4], 12, 48, 0.3)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1].view(np.uint64), b[1].view(np.uint64))
        rf = cli.make_filter(ids[allowed])
        a, b = cli.search_mmr(Q[:4], 12, 48, 0.3, rf), ix.search_mmr(Q[:4], 12, 48, 0.3, ids[allowed])
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1].view(np.uint64), b[1].view(np.uint64))
        rf.close()
        cli.close()
    finally:
        srv.stop()


def _clamp_sensitive_row():
    """x with s_dd(x, x) == 1 and a stored multiple c*x whose UNCLAMPED s_dd with x is 1 + 2^-52: only the clamp makes
    the two tie (found by a seeded search over the canonical arithmetic)."""
    from oracle.cosine_topk import canon_sum

    def s(a, b):
        a, b = a.astype(np.float64), b.astype(np.float64)
        return canon_sum(a * b) / np.sqrt(canon_sum(a * a) * canon_sum(b * b))
    rng = np.random.default_rng(0)
    for _ in range(4000):
        x = rng.standard_normal(O.DIM).astype(np.float32)
        if s(x, x) != 1.0:
            continue
        for c in rng.uniform(0.5, 3, 20).astype(np.float32):
            xb = (c * x).astype(np.float32)
            if s(xb, x) > 1.0:
                return x, xb
    raise AssertionError("no clamp-sensitive row in the seeded search")


def test_clamp_and_contraction_sensitive_tables():
    import outline_rag_b200 as orx
    # A = x, B = c*x, C = x, q = x: every distance is 0 (order = id).  At lambda 0 the score is -red; B and C tie only
    # because s_dd(B, A) is clamped to 1, and the tie goes to B, the lower position
    x, xb = _clamp_sensitive_row()
    X = np.stack([x, xb, x])
    ids = O.ids_arange(0, 3)
    with orx.Index("fp32", device=0) as ix:
        ix.upsert(ids, X)
        got = ix.search_mmr(x, 3, 3, 0.0)
        assert O.ids_to_ints(got[0][0]) == [0, 1, 2]
        assert_oracle(got, X, ids, x[None], 3, 3, 0.0, (0,))
    # a table (found by a search over small integer rows) on which evaluating the score with one fused multiply-add
    # instead of __dsub_rn(__dmul_rn(..), __dmul_rn(..)) swaps the last two picks at lambda 0.6
    pts = [[2, 0, 2], [1, 0, 0], [1, -3, 2], [3, 0, 0], [-1, -1, 0], [0, 1, 3], [-3, -3, -2], [3, -2, 0], [3, -3, 3]]
    X = np.zeros((len(pts), O.DIM), np.float32)
    X[:, :3] = pts
    q = np.zeros(O.DIM, np.float32)
    q[:3] = [-3, 0, 2]
    ids = O.ids_arange(0, len(pts))
    with orx.Index("fp32", device=0) as ix:
        ix.upsert(ids, X)
        assert_oracle(ix.search_mmr(q, len(pts), len(pts), 0.6), X, ids, q[None], len(pts), len(pts), 0.6, (0,))
