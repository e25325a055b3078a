"""The image scans of fp32 tables where the other image tests do not reach (DESIGN.md section 2, "What the image tests
pin"): inversions whose answer depends on the SIZE of the image's eps, batched and chunked bitmap scans over either
image, adversarial tables on the images with the routing predicted row for row, and write sequences that walk rows
through every class of the 8-bit image while growth, compaction, imports, option flips and restores rebuild it.

The options force the image: IMAGE_MIN_ROWS 0 scans it from the first row on (-1: the fp32 rows, path 1);
IMAGE8_MIN_ROWS 0 makes it the 8-bit one (path 4), -1 the bf16 one (path 3).  The answers must equal the oracle bit for
bit, and last_path the path the routing of csrc/orx_api.cu (scan_pass, gemv_source) predicts, so a search that
silently fell through to the fp32 rows fails here."""
import numpy as np
import pytest
from hypothesis import HealthCheck, given, settings
from hypothesis import strategies as st

from oracle import cosine_topk as O
from tests import adversarial as A
from tests.test_image8_scan import image8_scores, quantise_rows
from tests.test_image8_scan_gpu import image8_in_step, stored_rows
from tests.test_image_scan_gpu import image_in_step

pytestmark = pytest.mark.gpu
D = 1024
IMAGE8_MAX_K = 12                  # csrc/internal.h
IMAGE8_MAX_CAPPED = 16
UMMA_MAX_K = 64                    # csrc/scan_umma.h
FILTER_SCAN_MIN_ROWS = 4096        # csrc/orx_api.cu
GEMV_QCHUNK = 64


def _L():
    from outline_rag_b200 import _lib
    return _lib


def use_image(ix, kind):
    """kind "8bit" / "bf16": that image, scanned from the first row on; "fp32": the fp32 rows"""
    L = _L()
    if kind == "fp32":
        ix.set_option(L.ORX_OPT_IMAGE_MIN_ROWS, -1)
        return ix
    ix.set_option(L.ORX_OPT_IMAGE8_MIN_ROWS, 0 if kind == "8bit" else -1)
    ix.set_option(L.ORX_OPT_IMAGE_MIN_ROWS, 0)
    return ix


def slots_for_k(k):
    return 1 if k <= 16 else 2 if k <= 32 else 4 if k <= 96 else 5


def capped8(rows):
    """the 8-bit image's over-cap count (table_ops.cu count_capped8_kernel) of the live rows `rows`"""
    if len(rows) == 0:
        return 0
    _, s8, _ = quantise_rows(rows)
    return int(np.sum(np.isinf(s8) & np.isfinite(A.row_scale(rows))))


def predict_path(n_live, nq, k, kind, n_capped, m=None):
    """last_path of a search by the documented routing (scan_pass, gemv_source): 2 the tcgen05 pass, 1 the fp32 rows,
    3 the bf16 image, 4 the 8-bit image.  m: the eligible rows of a filtered search; None when the filter rescores its
    rows without any scan (last_path is not touched then)."""
    if m is not None and not (m >= FILTER_SCAN_MIN_ROWS and m > 32 * slots_for_k(k)):
        return None
    if nq >= 2 and k <= UMMA_MAX_K and n_live >= 4096 and (m is None or nq * m >= n_live):
        return 2
    if kind == "fp32":
        return 1
    if kind == "bf16":
        return 3
    chunk = 1 if m is not None else min(nq, GEMV_QCHUNK)
    return 4 if chunk == 1 and k <= IMAGE8_MAX_K and n_capped <= IMAGE8_MAX_CAPPED else 1


def equal_oracle(got, i, rows, ids, q, k):
    """query i of a search result equals the oracle over (rows, ids) bit for bit, NaN distances in the same places"""
    w_ids, w_d = O.topk_exact(rows, ids, q, k)
    m = len(w_d)
    assert got[2][i] == m, (i, got[2][i], m)
    assert np.array_equal(got[0][i, :m], w_ids), i
    nan = np.isnan(w_d)
    assert np.array_equal(np.isnan(got[1][i, :m]), nan), i
    assert np.array_equal(got[1][i, :m][~nan].view(np.uint64), w_d[~nan].view(np.uint64)), i


def same(a, b):
    return (np.array_equal(a[0], b[0]) and np.array_equal(a[1].view(np.uint64), b[1].view(np.uint64))
            and np.array_equal(a[2], b[2]))


# ------------------------------------------------------------------------------ A. inversions that hang on eps
@pytest.mark.parametrize("k", [1, 12])
@pytest.mark.parametrize("kind", ["8bit", "bf16"])
def test_inversion_is_caught_only_by_the_image_eps(kind, k):
    """adversarial.image8_inversion / image_inversion: a smaller eps than the path's own proves k decoys in place of
    the winner (tests/test_image8_scan.py / test_image_scan.py pin that premise on the CPU, here it is checked again
    on the device's own scores); with the right eps every form falls back and answers the winner first."""
    import outline_rag_b200 as orx
    rows, q, w = (A.image8_inversion if kind == "8bit" else A.image_inversion)(k, seed=k)
    n = len(rows)
    ids = O.ids_arange(0, n)
    allow = np.concatenate([ids[:n - 601], ids[n - 1:]])               # 600 bulk rows out: a bitmap scan
    eps, smaller, width = ((1.662e-2, 3.92e-3, 160) if kind == "8bit"
                           else (3.92e-3, A.EPS_UMMA, 32 * (2 if k <= 16 else 4)))
    want = O.topk_exact(rows, ids, q, k)
    assert want[0][0, 1] == n - 1
    with use_image(orx.Index("fp32", n, 0), kind) as ix:
        ix.upsert(ids, rows)
        dev = (ix.debug_image8_scores(q[None]) if kind == "8bit" else ix.debug_image_scores(q[None])).cpu().numpy()[:, 0]
        cos = A.cosine(rows, q)
        assert not A.proof_holds(dev, cos, k, width, eps)[0]
        assert A.proof_holds(dev, cos, k, width, smaller)[0]
        with ix.make_filter(allow) as flt:
            for form, fn in (("single", lambda: ix.search(q, k)),
                             ("bitmap", lambda: ix.search_filtered(q[None], k, allow)),
                             ("handle", lambda: ix.search_filtered(q[None], k, flt))):
                st0 = ix.stats()
                got = fn()
                st1 = ix.stats()
                assert st1["last_path"] == (4 if kind == "8bit" else 3), form
                assert (st1["fallback_exhaustive"] + st1["fallback_gemv"]
                        > st0["fallback_exhaustive"] + st0["fallback_gemv"]), form
                assert got[0][0, 0, 1] == n - 1, form                 # the winner
                assert np.array_equal(got[0][0], want[0]), form
                assert np.array_equal(got[1][0].view(np.uint64), want[1].view(np.uint64)), form


# ------------------------------------------------------------------- B. batched and chunked bitmap scans
N_BULK = 600_000                   # > 130 queries x 4400 eligible rows: every batch below takes the bitmap scan
N_QB = 130


@pytest.fixture(scope="module")
def bitmap_table():
    """600k random rows outside the filter and a 4400-row eligible block: 80 rows near a common direction c, 12 near
    each query's own direction v_j, the rest random.  Query j = c + 1.5 v_j: its top rows are its own, then c's; a
    scan of query j with another query's quantisation or q^ would list that query's rows and c's -- which rescore well
    enough against query j to pass the proof with the wrong ids."""
    import torch
    import outline_rag_b200 as orx
    rng = np.random.default_rng(31)

    def unit(x):
        return x / np.linalg.norm(x, axis=-1, keepdims=True)
    c = unit(rng.standard_normal(D))
    v = unit(rng.standard_normal((N_QB, D)))
    Q = (c + 1.5 * v).astype(np.float32)
    near = [c + 0.2 * unit(rng.standard_normal((80, D)))]
    near += [v[j] + 0.2 * unit(rng.standard_normal((12, D))) for j in range(N_QB)]
    block = np.concatenate(near + [rng.standard_normal((4400 - 80 - 12 * N_QB, D))]).astype(np.float32)
    block = block[rng.permutation(len(block))]
    ix = orx.Index("fp32", N_BULK + len(block), 0)
    g = torch.Generator(device="cuda:0").manual_seed(7)
    for s in range(0, N_BULK, 131_072):
        m = min(131_072, N_BULK - s)
        ix.upsert(O.ids_arange(s, s + m), torch.randn((m, D), generator=g, device="cuda:0"))
    bids = O.ids_arange(N_BULK, N_BULK + len(block))
    ix.upsert(bids, block)
    yield ix, block, bids, Q
    ix.close()


@pytest.mark.parametrize("kind,k", [("8bit", 1), ("8bit", 12), ("bf16", 1), ("bf16", 12), ("bf16", 33), ("bf16", 65)])
def test_batched_bitmap_scans_equal_single_queries_fp32_rows_and_oracle(bitmap_table, kind, k):
    ix, block, bids, Q = bitmap_table
    path = 4 if kind == "8bit" else 3
    with ix.make_filter(bids) as flt:
        for form, allow in (("ids", bids), ("handle", flt)):
            use_image(ix, kind)
            alone = []
            for j in range(N_QB):
                alone.append(ix.search_filtered(Q[j:j + 1], k, allow))
                assert ix.stats()["last_path"] == path
            for j in range(N_QB):
                equal_oracle(alone[j], 0, block, bids, Q[j], k)
            for nq in (2, 7, 64, 65, 130):
                use_image(ix, kind)
                got = ix.search_filtered(Q[:nq], k, allow)
                assert ix.stats()["last_path"] == path, (form, nq)
                for j in range(nq):
                    assert same(tuple(a[j:j + 1] for a in got), alone[j]), (form, nq, j)
                use_image(ix, "fp32")
                ref = ix.search_filtered(Q[:nq], k, allow)
                assert ix.stats()["last_path"] == 1
                assert same(got, ref), (form, nq)
    use_image(ix, kind)


# ----------------------------------------------------------------------- C. adversarial tables on the images
def _capped_rows(rng, n):
    """rows over R8_CAP: one dominant element (the rest rounds to 0 or +-1) or every element just over half a step"""
    out = rng.standard_normal((n, D)).astype(np.float32) * np.float32(1e-3)
    half = rng.random(n) < 0.5
    out[half] = np.float32(0.5 / 127 * 1.0001) * np.sign(out[half])
    out[np.arange(n), rng.integers(0, D, n)] = np.float32(1.0)
    return out


def _band_rows(rng, n, inside):
    """unit rows scaled just inside (regular) or just outside (never trusted) |x| in [2^-40, 2^40]"""
    u = rng.standard_normal((n, D))
    u = u / np.linalg.norm(u, axis=1, keepdims=True)
    lo, hi = (2.0 ** -40 * 1.01, 2.0 ** 40 * 0.99) if inside else (2.0 ** -40 * 0.99, 2.0 ** 40 * 1.01)
    return (u * np.where(rng.random(n) < 0.5, lo, hi)[:, None]).astype(np.float32)


def _subnormal_rows(rng, n):
    out = rng.uniform(-1, 1, (n, D)).astype(np.float32) * np.float32(1e-39)
    out[:, 0] = np.float32(2.0 ** -30)
    return out


@st.composite
def image_tables(draw):
    """test_property_gpu.tables() plus what only the images treat specially"""
    from tests.test_property_gpu import tables
    X, ids, _, _, n_del, _ = draw(tables())
    rng = np.random.default_rng(draw(st.integers(0, 2**31 - 1)))
    extra = [rng.standard_normal((draw(st.sampled_from([0, 4200, 8400])), D)).astype(np.float32)]
    extra.append(_capped_rows(rng, draw(st.sampled_from([0, 5, 16, 17, 30]))))
    extra.append(_band_rows(rng, draw(st.integers(0, 20)), True))
    extra.append(_band_rows(rng, draw(st.sampled_from([0, 3, 17, 25])), False))
    extra.append(_subnormal_rows(rng, draw(st.integers(0, 4))))
    if draw(st.booleans()):                                          # more duplicates than a candidate list holds
        extra.append(np.repeat(X[rng.integers(0, len(X))][None], draw(st.integers(161, 240)), 0))
    E = np.concatenate(extra)
    perm = rng.permutation(len(X) + len(E))
    X = np.concatenate([X, E])[perm]
    ids = np.concatenate([ids, O.ids_from_ints([2**126 + i for i in range(len(E))])])[perm]
    k = draw(st.sampled_from([1, 5, 12, 13, 16, 17, 32, 33, 64, 65, 128]))
    nq = draw(st.sampled_from([1, 2, 7, 33]))
    src = rng.integers(0, len(X), nq)
    how = draw(st.sampled_from(["rows", "scaled", "negated", "noise", "zero"]))
    if how == "rows":
        Q = X[src].copy()
    elif how == "scaled":
        Q = X[src] * np.float32(2.0) ** rng.integers(-20, 21, (nq, 1)).astype(np.float32)
    elif how == "negated":
        Q = -X[src]
    else:
        Q = rng.standard_normal((nq, D)).astype(np.float32)
    if how == "zero":
        Q[0] = 0
    form = draw(st.sampled_from(["search", "filtered", "handle"]))
    kind = draw(st.sampled_from(["8bit", "bf16"]))
    return X, ids, np.ascontiguousarray(Q, np.float32), k, n_del, form, kind, draw(st.integers(0, 2**31 - 1))


@settings(max_examples=60, deadline=None, suppress_health_check=list(HealthCheck), derandomize=True)
@given(image_tables())
def test_image_scans_equal_oracle_and_predicted_path_on_adversarial_tables(case):
    import outline_rag_b200 as orx
    X, ids, Q, k, n_del, form, kind, seed = case
    rng = np.random.default_rng(seed)
    keep = np.ones(len(X), bool)
    keep[:n_del] = False
    with use_image(orx.Index("fp32", 0, 0), kind) as ix:
        ix.upsert(ids, X)
        if n_del:
            assert ix.delete(ids[:n_del]) == n_del
        live = stored_rows(ix)
        n_cap = capped8(live)
        m = None
        if form == "search":
            got = ix.search(Q, k)
            sel = keep
        else:
            sel = keep & (rng.random(len(X)) < rng.choice([0.02, 0.5, 0.97]))
            sel[np.nonzero(keep)[0][0]] = True
            m = int(sel.sum())
            if form == "filtered":
                got = ix.search_filtered(Q, k, ids[sel])
            else:
                with ix.make_filter(ids[sel]) as flt:
                    got = ix.search_filtered(Q, k, flt)
        want_path = predict_path(int(keep.sum()), len(Q), k, kind, n_cap, m)
        path = ix.stats()["last_path"]
    for i in range(len(Q)):
        equal_oracle(got, i, X[sel], ids[sel], Q[i], k)
    if want_path is not None:
        assert path == want_path, (path, want_path, kind, form, len(Q), k, n_cap, m)


# ------------------------------------------------------------------------------------- D. write sequences
def _class_rows(rng, cls, n):
    if cls == "regular":
        return rng.standard_normal((n, D)).astype(np.float32)
    if cls == "capped":
        return _capped_rows(rng, n)
    if cls == "zero":
        return np.zeros((n, D), np.float32)
    return _band_rows(rng, n, False)                                   # out of band


class Mirror:
    """what the table must hold: id (int) -> row"""

    def __init__(self):
        self.rows = {}

    def set(self, ids, rows):
        for i, r in zip(ids, rows):
            self.rows[int(i)] = r

    def arrays(self):
        keys = sorted(self.rows)
        return (O.ids_from_ints(keys), np.stack([self.rows[i] for i in keys]) if keys else np.zeros((0, D), np.float32))


def _check(ix, mir, rng, what, image8_min_rows):
    """after every write: the table equals the mirror, the image is in step, the routing and the answers are right"""
    ids, rows = mir.arrays()
    n = len(ids)
    assert len(ix) == n, what
    if n == 0:
        return
    got_ids = np.zeros((n, 2), np.uint64)
    raw = np.zeros((n, 4 * D), np.uint8)
    ix.export_rows(0, n, got_ids, raw)
    order = O.order_by_distance(np.zeros(n), got_ids)
    assert np.array_equal(got_ids[order], ids), what
    assert np.array_equal(raw.view(np.float32)[order].view(np.uint32), rows.view(np.uint32)), what
    n_cap = capped8(rows)
    kind = "8bit" if 0 <= image8_min_rows <= ix.capacity else "bf16"
    q = rows[rng.integers(0, n)] + np.float32(0.05) * rng.standard_normal(D).astype(np.float32)
    for k in (1, 12):
        got = ix.search(q, k)
        assert ix.stats()["last_path"] == predict_path(n, 1, k, kind, n_cap), (what, kind, n_cap, k)
        equal_oracle(got, 0, rows, ids, q, k)
    sel = rng.random(n) < 0.8
    m = int(sel.sum())
    got = ix.search_filtered(q[None], 12, ids[sel])
    want_path = predict_path(n, 1, 12, kind, n_cap, m)
    if want_path is not None:
        assert ix.stats()["last_path"] == want_path, (what, kind, n_cap, m)
    equal_oracle(got, 0, rows[sel], ids[sel], q, 12)
    Qs = np.stack([q, rng.standard_normal(D).astype(np.float32)])
    if kind == "8bit":
        image8_in_step(ix, Qs)
    else:
        image_in_step(ix, Qs)


def _options(ix, image8_min_rows):
    L = _L()
    ix.set_option(L.ORX_OPT_IMAGE_MIN_ROWS, 0)
    ix.set_option(L.ORX_OPT_IMAGE8_MIN_ROWS, image8_min_rows)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_write_sequences_keep_the_image_and_its_routing_in_step(seed, tmp_path):
    """3000 rows on a bf16 image (capacity < IMAGE8_MIN_ROWS = 4096), then random writes: fresh rows of every class
    (growth past 4096 switches to the 8-bit image), in-place rewrites between regular / capped / zero / out of band,
    deletes that compact (tail rows move into the holes), delete-all and refill, a rejected NaN batch, imports, option
    flips that make the next search switch the image kind, save + load.  Two scripted walks pin the capped count at
    its limit: exactly 16 capped rows beside 20 out-of-band ones, then a 17th appended as the last row; and capped
    rows appended at the tail, then moved into the holes of a delete."""
    import outline_rag_b200 as orx
    L = _L()
    rng = np.random.default_rng(100 + seed)
    mir = Mirror()
    next_id = [0]
    i8 = [4096]

    def fresh(n, cls=None):
        cls = cls or rng.choice(["regular", "regular", "capped", "zero", "band"])
        ids = list(range(next_id[0], next_id[0] + n))
        next_id[0] += n
        return ids, _class_rows(rng, cls, n)

    def put(ids, rows):
        ix.upsert(O.ids_from_ints(ids), rows)
        mir.set(ids, rows)

    def classes():
        keys = sorted(mir.rows)
        rows = np.stack([mir.rows[i] for i in keys])
        _, s8, _ = quantise_rows(rows)
        keys = np.array(keys, dtype=object)
        return keys[np.isinf(s8) & np.isfinite(A.row_scale(rows))], keys[np.isfinite(s8)]

    def set_capped(target):
        """in-place rewrites until exactly `target` live rows are over R8_CAP"""
        capped, regular = classes()
        if len(capped) > target:
            pick = [int(v) for v in capped[:len(capped) - target]]
            put(pick, _class_rows(rng, "regular", len(pick)))
        elif len(capped) < target:
            pick = [int(v) for v in rng.choice(regular, target - len(capped), replace=False)]
            put(pick, _class_rows(rng, "capped", len(pick)))

    def check(what):
        _check(ix, mir, rng, what, i8[0])

    ix = orx.Index("fp32", 3000, 0)
    try:
        _options(ix, i8[0])
        put(*fresh(2990, "regular"))
        check("start")
        for step in range(24):
            op = rng.choice(["fresh", "fresh", "inplace", "inplace", "delete", "nan", "import", "flip", "save",
                             "clear", "limit", "tail"] if step > 2 else ["fresh", "inplace"])
            if op == "fresh":
                put(*fresh(int(rng.choice([1, 7, 40, 700]))))
            elif op == "inplace":
                live = np.array(sorted(mir.rows), dtype=object)
                pick = [int(v) for v in rng.choice(live, min(len(live), int(rng.choice([1, 6, 20]))), replace=False)]
                put(pick, _class_rows(rng, rng.choice(["regular", "capped", "zero", "band"]), len(pick)))
            elif op == "delete":
                live = np.array(sorted(mir.rows), dtype=object)
                pick = [int(v) for v in rng.choice(live, min(len(live) - 1, int(rng.choice([1, 30, 400]))),
                                                   replace=False)]
                assert ix.delete(O.ids_from_ints(pick)) == len(pick)
                for i in pick:
                    del mir.rows[i]
            elif op == "clear":
                live = sorted(mir.rows)
                assert ix.delete(O.ids_from_ints(live)) == len(live)
                mir.rows.clear()
                check("cleared")
                put(*fresh(int(rng.choice([50, 3000])), "regular"))
            elif op == "nan":
                ids, rows = fresh(5, "regular")
                rows[2, 17] = np.nan
                live = sorted(mir.rows)[:3]                            # in place and fresh ids in one batch
                with pytest.raises(L.OrxValueError):
                    ix.upsert(O.ids_from_ints(live + ids), np.concatenate([_class_rows(rng, "capped", 3), rows]))
            elif op == "import":
                ids, rows = fresh(int(rng.choice([3, 300])))
                A.import_stored(ix, O.ids_from_ints(ids), rows)
                mir.set(ids, rows)
            elif op == "flip":
                i8[0] = int(rng.choice([0, -1, 4096]))
                _options(ix, i8[0])
            elif op == "limit":
                put(*fresh(20, "band"))
                set_capped(16)
                check(f"step {step}: 16 capped")
                put(*fresh(1, "capped"))                               # the 17th, as the last row
            elif op == "tail":
                set_capped(0)
                put(*fresh(10, "capped"))
                check(f"step {step}: 10 capped at the tail")
                _, regular = classes()
                pick = [int(v) for v in regular[:30]]                  # early rows: the tail fills their holes
                assert ix.delete(O.ids_from_ints(pick)) == len(pick)
                for i in pick:
                    del mir.rows[i]
            else:
                ix.save(str(tmp_path / f"snap{step}"))
                ix.close()
                ix = orx.Index.load(str(tmp_path / f"snap{step}"), device=0, capacity=int(rng.choice([0, 5000])))
                _options(ix, i8[0])
            check(f"step {step}: {op}")
    finally:
        ix.close()
