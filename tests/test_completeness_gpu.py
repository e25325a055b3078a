"""Forced rank inversions: the completeness proof of finalize (DESIGN.md section 2) must FAIL, and the exact fallbacks
must answer, whenever a true top-k row has a fast / coarse key that ranks outside the candidate list.

Each table holds a winner w at the LAST row and, at lower rows, more decoys than any candidate list holds; the decoys
tie w's fast and coarse scores bit for bit but have a strictly worse canonical distance (tests/adversarial.py
decoy_rows).  w's tcgen05 coarse score underestimates its cosine by ~1.8e-3 and its GEMV fast score by a little, so
every decoy's cosine lies above the tied score: a proof bound that loses its + eps, a cut that is too high or an
epsilon that is too small accepts a list without w.  Each test first checks that premise on the device (debug hooks),
then: ids and distance bits equal the exhaustive oracle, count == k, and the fallback counters moved -- the proof, not
luck, caught it.  The converse ("provable" tables, top-k separated from every other row by > 3 eps) must not move them.

Paths: scan_gemv (one query; finalize 1a), scan_gemv_batch (k > 64), the tcgen05 1-CTA and pair kernels with the
decoys spread over many row slots and concentrated in one, the filtered bitmap GEMV scan, the filtered masked-scale
tcgen05 pass, and a two-shard merge with the winner in one shard and the decoys in the other."""
import numpy as np
import pytest

from oracle import cosine_topk as O
from tests import adversarial as A

pytestmark = pytest.mark.gpu
KS = [1, 12, 16, 17, 32, 33, 64, 65, 96, 97, 128]
UMMA_KS = [k for k in KS if k <= 64]            # csrc/scan_umma.h UMMA_MAX_K
WIDE_KS = [k for k in KS if k > 64]
TILE = 256                                      # rows per tcgen05 table tile (one row slot of a CTA)
N_DECOYS = 192                                  # > 160: every candidate list of every path
N_ROWS = TILE * (N_DECOYS + 2)


def gemv_width(k):                              # finalize's K for the GEMV scans: 32 * slots_for_k (csrc/internal.h)
    return 32 * (1 if k <= 16 else 2 if k <= 32 else 4 if k <= 96 else 5)


def umma_width(k):                              # CAND / CAND_WIDE (csrc/scan_umma.cu), finalize's K for tcgen05
    return 64 if k <= 16 else 160


def _ordinary(n, seed, dtype):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, 1024)).astype(np.float32)
    return A.stored(X, dtype) if dtype == "bf16" else X


class Case:
    """One inversion table (stored rows in table order, ids = row numbers) and the exhaustive oracle of its query."""

    def __init__(self, dtype, layout):
        self.dtype, self.layout = dtype, layout
        self.q, w = A.inversion_case(dtype)
        decoys = A.decoy_rows(w, self.q, N_DECOYS)
        rows = _ordinary(N_ROWS, 7, dtype)
        self.decoy_rows = (np.arange(N_DECOYS) * TILE + 5 if layout == "spread" else np.arange(N_DECOYS))
        rows[self.decoy_rows] = decoys
        rows[-1] = w
        self.w_row = N_ROWS - 1
        self.rows = rows
        self.ids = O.ids_arange(0, N_ROWS)
        self.want_ids, self.want_d = O.topk_exact(rows, self.ids, self.q, max(KS), exhaustive=True)
        assert self.want_ids[0, 1] == self.w_row            # w is the true nearest row

    def allowed(self):
        """ids of a filter that excludes 100 ordinary rows (none of the oracle's top max(KS))"""
        out = np.setdiff1d(np.arange(1000, 1200), self.decoy_rows)[:100]
        assert not np.isin(out, self.want_ids[:, 1]).any()
        return np.delete(self.ids, out, axis=0)

    def index(self):
        import outline_rag_b200 as orx
        ix = orx.Index(self.dtype, N_ROWS, 0)
        A.import_stored(ix, self.ids, self.rows)
        return ix


_CASES = {}


def case(dtype, layout="concentrated"):
    if (dtype, layout) not in _CASES:
        _CASES[(dtype, layout)] = Case(dtype, layout)
    return _CASES[(dtype, layout)]


def key_rank(scores, row):
    """rank of `row`'s candidate key (score descending, then row ascending) among all rows"""
    s = scores[row]
    return int(np.sum(scores > s) + np.sum(scores[:row] == s))


def check_premise(c, scores, width, k):
    """w ranks outside the list, every decoy ties it on the device, w is in the oracle's top-k, and every listed decoy
    of the oracle's top-k has a cosine above the tied score (only + eps keeps the proof from accepting)."""
    assert (scores[c.decoy_rows] == scores[c.w_row]).all(), "the decoys do not tie the winner on the device"
    assert key_rank(scores, c.w_row) >= width, (key_rank(scores, c.w_row), width)
    assert c.w_row in c.want_ids[:k, 1]
    if k > 1:
        assert 1.0 - c.want_d[k - 1] > float(scores[c.w_row])


def check_answer(c, got, k, nq):
    g_ids, g_d, g_c = got
    for i in range(nq):
        assert g_c[i] == k
        assert np.array_equal(g_ids[i, :k], c.want_ids[:k]), f"query {i}: ids differ from the oracle"
        assert np.array_equal(g_d[i, :k].view(np.uint64), c.want_d[:k].view(np.uint64)), f"query {i}: distance bits"


def moved(before, after, name):
    return after[name] - before[name]


# ------------------------------------------------------------------------------------------------ GEMV scans
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("k", KS)
def test_gemv_single_query_inversion(dtype, k):
    c = case(dtype)
    with c.index() as ix:
        check_premise(c, ix.debug_fast_scores(c.q[None]).cpu().numpy()[:, 0], gemv_width(k), k)
        st0 = ix.stats()
        got = ix.search(c.q[None], k)
        st1 = ix.stats()
    assert st1["last_path"] == 1
    check_answer(c, got, k, 1)
    assert moved(st0, st1, "fallback_exhaustive") == 1


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("k", WIDE_KS)
def test_gemv_batch_inversion(dtype, k):
    c = case(dtype)
    Q = np.stack([c.q, c.q, c.q])
    with c.index() as ix:
        check_premise(c, ix.debug_fast_scores(c.q[None]).cpu().numpy()[:, 0], gemv_width(k), k)
        st0 = ix.stats()
        got = ix.search(Q, k)
        st1 = ix.stats()
    assert st1["last_path"] == 1
    check_answer(c, got, k, len(Q))
    assert moved(st0, st1, "fallback_exhaustive") == len(Q)


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("k", [1, 12, 17, 33, 65, 128])
def test_filtered_bitmap_gemv_inversion(dtype, k):
    c = case(dtype)
    allow = c.allowed()
    with c.index() as ix:
        check_premise(c, ix.debug_fast_scores(c.q[None]).cpu().numpy()[:, 0], gemv_width(k), k)
        st0 = ix.stats()
        got = ix.search_filtered(c.q[None], k, allow)
        st1 = ix.stats()
    assert st1["last_path"] == 1
    check_answer(c, got, k, 1)
    assert moved(st0, st1, "fallback_exhaustive") == 1


# ------------------------------------------------------------------------------------------------ tcgen05
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("layout", ["spread", "concentrated"])
@pytest.mark.parametrize("pairs", [False, True], ids=["one_cta", "pairs"])
@pytest.mark.parametrize("k", UMMA_KS)
def test_tcgen05_inversion(dtype, layout, pairs, k):
    c = case(dtype, layout)
    nq = 200 if pairs else 4                     # batches beyond one 128-query tile run on CTA pairs
    Q = np.repeat(c.q[None], nq, axis=0)
    with c.index() as ix:
        check_premise(c, ix.debug_coarse_scores(c.q[None], use_pairs=pairs).cpu().numpy()[:, 0], umma_width(k), k)
        assert float(ix.debug_coarse_scores(c.q[None], use_pairs=pairs)[c.w_row, 0]) < 1.0 - c.want_d[0] - 1.5e-3
        st0 = ix.stats()
        got = ix.search(Q, k)
        st1 = ix.stats()
    assert st1["last_path"] == 2
    check_answer(c, got, k, nq)
    assert moved(st0, st1, "fallback_gemv") == nq


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("k", [1, 16, 17, 64])
def test_filtered_tcgen05_inversion(dtype, k):
    c = case(dtype, "spread")
    allow = c.allowed()
    Q = np.repeat(c.q[None], 4, axis=0)
    with c.index() as ix:
        check_premise(c, ix.debug_coarse_scores(c.q[None]).cpu().numpy()[:, 0], umma_width(k), k)
        st0 = ix.stats()
        got = ix.search_filtered(Q, k, allow)
        st1 = ix.stats()
    assert st1["last_path"] == 2
    check_answer(c, got, k, len(Q))
    assert moved(st0, st1, "fallback_exhaustive") == len(Q)


# ------------------------------------------------------------------------------------------------ shard merge
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("k,nq", [(12, 1), (12, 4), (64, 4), (128, 1)])
def test_two_shard_merge_inversion(dtype, k, nq):
    """winner in shard 0, decoys in shard 1: shard 1 cannot prove its list, shard 0 finds w, the merge is exact"""
    import outline_rag_b200 as orx
    c = case(dtype, "spread")
    in0 = np.zeros(N_ROWS, bool)
    in0[c.w_row] = True
    in0[np.arange(0, N_ROWS, 2)] = True
    in0[c.decoy_rows] = False
    Q = np.repeat(c.q[None], nq, axis=0)
    parts = []
    shards = [orx.Index(dtype, N_ROWS, 0) for _ in range(2)]
    try:
        for s, sel in enumerate((in0, ~in0)):
            A.import_stored(shards[s], c.ids[sel], c.rows[sel])
            st0 = shards[s].stats()
            parts.append(shards[s].search(Q, k))
            st1 = shards[s].stats()
            if s == 1:
                assert moved(st0, st1, "fallback_exhaustive") + moved(st0, st1, "fallback_gemv") >= nq, \
                    "the decoy shard proved a list it cannot prove"
        merged = shards[0].merge_topk(np.stack([p[0] for p in parts]), np.stack([p[1] for p in parts]),
                                      np.stack([p[2] for p in parts]), k)
    finally:
        for ix in shards:
            ix.close()
    check_answer(c, merged, k, nq)


# ------------------------------------------------------------------------------------------------ provable tables
def _provable(dtype, k, seed):
    """k rows at cosine ~0.9 to a random query, every other row below 0.3: separated by far more than 3 eps"""
    rng = np.random.default_rng(seed)
    q = rng.standard_normal(1024).astype(np.float32)
    u = q / np.linalg.norm(q)
    rows = rng.standard_normal((8192, 1024)).astype(np.float32)
    noise = rng.standard_normal((k, 1024)).astype(np.float32)
    noise -= np.outer(noise @ u, u)
    noise /= np.linalg.norm(noise, axis=1, keepdims=True)
    top = 0.9 * u + np.sqrt(1 - 0.9 ** 2) * noise * rng.uniform(0.9, 1.1, (k, 1))
    rows[:k] = top                                # one tile: that CTA's threshold is the k-th best minus the margin
    rows = A.stored(rows, dtype) if dtype == "bf16" else rows
    ids = O.ids_arange(0, len(rows))
    cos = A.cosine(rows, q)
    assert np.sort(cos)[-k] - np.sort(cos)[-k - 1] > 0.5
    return q, rows, ids


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("path,k", [("gemv", 1), ("gemv", 12), ("gemv", 17), ("gemv", 64), ("gemv", 128),
                                    ("batch", 65), ("batch", 128),
                                    ("one_cta", 1), ("one_cta", 12), ("one_cta", 17), ("one_cta", 64),
                                    ("pairs", 12), ("pairs", 64)])
def test_provable_tables_need_no_fallback(dtype, path, k):
    import outline_rag_b200 as orx
    q, rows, ids = _provable(dtype, k, 100 + k)
    nq = {"gemv": 1, "batch": 3, "one_cta": 4, "pairs": 200}[path]
    Q = np.repeat(q[None], nq, axis=0)
    want_ids, want_d = O.topk_exact(rows, ids, q, k, exhaustive=True)
    with orx.Index(dtype, len(rows), 0) as ix:
        A.import_stored(ix, ids, rows)
        st0 = ix.stats()
        g_ids, g_d, g_c = ix.search(Q, k)
        st1 = ix.stats()
    assert st1["last_path"] == (2 if path in ("one_cta", "pairs") else 1)
    for i in range(nq):
        assert g_c[i] == k and np.array_equal(g_ids[i], want_ids)
        assert np.array_equal(g_d[i].view(np.uint64), want_d.view(np.uint64))
    assert moved(st0, st1, "fallback_gemv") == 0 and moved(st0, st1, "fallback_exhaustive") == 0, (st0, st1)
