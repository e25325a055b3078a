"""The GEMV scans over the bf16 image of an fp32 table (DESIGN.md section 2, "bf16 image"): same answers as the fp32
scans, bit for bit, on every path and after every kind of write; the error bound EPS_GEMV_IMAGE measured on its worst
case; the completeness proof failing (and the fallback answering) when a forced rank inversion defeats the image scores.

ORX_OPT_IMAGE_MIN_ROWS switches the same index between the image scan (0: always, last_path 3) and the fp32 scan
(-1: never, last_path 1), so each comparison runs both on identical rows."""
import numpy as np
import pytest

from oracle import cosine_topk as O
from tests import adversarial as A

pytestmark = pytest.mark.gpu
KS = [1, 12, 16, 17, 32, 33, 64, 65, 96, 97, 128]
WIDE_KS = [k for k in KS if k > 64]
N_BIG = 1_100_000                 # above the default IMAGE_MIN_ROWS (2^20): the image path without any option
NQ = 8
EPS_GEMV_IMAGE = 3.92e-3          # csrc/internal.h
IMAGE_MIN_ROWS = 1 << 20


def _opt():
    from outline_rag_b200 import _lib
    return _lib.ORX_OPT_IMAGE_MIN_ROWS


def both(ix, fn):
    """fn() over the image (path 3) and over the fp32 rows (path 1) of the same index; option reset to its default"""
    ix.set_option(_opt(), 0)
    a = fn()
    pa = ix.stats()["last_path"]
    ix.set_option(_opt(), -1)
    b = fn()
    pb = ix.stats()["last_path"]
    ix.set_option(_opt(), IMAGE_MIN_ROWS)
    return a, b, pa, pb


def same(a, b):
    return (np.array_equal(a[0], b[0]) and np.array_equal(a[1].view(np.uint64), b[1].view(np.uint64))
            and np.array_equal(a[2], b[2]))


def agree(ix, Q, k, filtered=None, want_paths=(3, 1), no_fallback=False):
    fn = (lambda: ix.search(Q, k)) if filtered is None else (lambda: filtered(Q, k))
    st0 = ix.stats()
    a, b, pa, pb = both(ix, fn)
    st1 = ix.stats()
    assert (pa, pb) == want_paths, (pa, pb, k)
    assert same(a, b), k
    if no_fallback:
        assert st1["fallback_exhaustive"] == st0["fallback_exhaustive"], k
        assert st1["fallback_gemv"] == st0["fallback_gemv"], k
    return a


def image_in_step(ix, Q):
    """The image of every live row equals RNE-bf16 of the fp32 row now stored there: the image scores of `ix` equal, bit
    for bit, those of a fresh index whose image was built from the exported rows alone (orx_import_rows)"""
    import torch
    import outline_rag_b200 as orx
    n = len(ix)
    with orx.Index("fp32", n, ix.device) as fresh:
        chunk = 131_072
        for s in range(0, n, chunk):
            m = min(chunk, n - s)
            ids = np.zeros((m, 2), np.uint64)
            raw = np.zeros((m, 4096), np.uint8)
            ix.export_rows(s, m, ids, raw)
            A.import_stored(fresh, ids, raw.view(np.float32))
        want = fresh.debug_image_scores(Q)
    got = ix.debug_image_scores(Q)
    assert torch.equal(got.view(torch.int32), want.view(torch.int32))


@pytest.fixture(scope="module")
def big():
    import outline_rag_b200 as orx
    from oracle.synth_host import FastSynth
    from orx_testkit.device import synth_rows_device
    from orx_testkit.synth import SEED_TABLE, default_centres
    syn = FastSynth(default_centres(N_BIG))
    ix = orx.Index("fp32", N_BIG + 4096, 0)
    chunk = 262_144
    for s in range(0, N_BIG, chunk):
        m = min(chunk, N_BIG - s)
        ix.upsert(O.ids_arange(s, s + m), synth_rows_device(0, SEED_TABLE, syn.n_centres, s, m))
    Q, anchors = syn.queries(NQ, N_BIG)
    yield syn, ix, Q, anchors
    ix.close()


# ------------------------------------------------------------------------------------------- same answers, 1.1M rows
def test_large_fp32_table_takes_the_image_scan_by_default(big):
    syn, ix, Q, _ = big
    ix.search(Q[0], 12)
    assert ix.stats()["last_path"] == 3
    ix.set_option(_opt(), N_BIG + 1)
    ix.search(Q[0], 12)
    assert ix.stats()["last_path"] == 1
    ix.set_option(_opt(), IMAGE_MIN_ROWS)


@pytest.mark.parametrize("k", KS)
def test_single_query_image_equals_fp32_scan(big, k):
    _, ix, Q, _ = big
    for i in range(0, NQ, 3):
        agree(ix, Q[i], k)


@pytest.mark.parametrize("k", WIDE_KS)
def test_batch_wide_k_image_equals_fp32_scan(big, k):
    _, ix, Q, _ = big
    agree(ix, Q[:3], k)


@pytest.mark.parametrize("k", [1, 12, 33, 65, 128])
def test_filtered_bitmap_and_filter_handle_image_equals_fp32_scan(big, k):
    _, ix, Q, _ = big
    allow = O.ids_arange(0, N_BIG)[::3]
    agree(ix, Q[1:2], k, filtered=lambda q, kk: ix.search_filtered(q, kk, allow))
    with ix.make_filter(allow) as flt:
        agree(ix, Q[2:3], k, filtered=lambda q, kk: ix.search_filtered(q, kk, flt))


def test_image_scan_equals_the_full_oracle_pass_without_fallbacks(big):
    syn, ix, Q, anchors = big
    truth = O.StreamingTopK(Q, 12)
    for s in range(0, N_BIG, 65_536):
        m = min(65_536, N_BIG - s)
        truth.feed(syn.table(m, start=s), O.ids_arange(s, s + m))
    want = truth.result()
    st0 = ix.stats()
    for i in range(NQ):
        got = ix.search(Q[i], 12)
        assert ix.stats()["last_path"] == 3
        assert np.array_equal(got[0][0], want[i][0]), i
        assert np.array_equal(got[1][0].view(np.uint64), want[i][1].view(np.uint64)), i
        assert got[0][0, 0, 1] == anchors[i]
    st1 = ix.stats()
    assert st1["fallback_exhaustive"] == st0["fallback_exhaustive"]
    assert st1["fallback_gemv"] == st0["fallback_gemv"]


def test_in_place_upsert_and_delete_compaction_keep_the_image_in_step(big):
    """Runs last on the module table (it mutates it)."""
    syn, ix, Q, _ = big
    rng = np.random.default_rng(5)
    # in place: rows of the queries' best hits replaced by other synthetic rows, some by their own negation
    hits = ix.search(Q, 12)[0][:, :4, 1].reshape(-1)
    new = syn.rows(rng.integers(0, N_BIG, size=hits.size).astype(np.uint64))
    new[::2] = -syn.rows(hits[::2])
    ix.upsert(np.stack([np.zeros_like(hits), hits], 1), new)
    image_in_step(ix, Q[:4])
    for k in (12, 65):
        agree(ix, Q[0], k, no_fallback=True)
        agree(ix, Q[:3], 97)
    # delete with compaction: rows from the middle, refilled by the tail
    before = ix.stats()["rows_moved"]
    doomed = np.unique(np.concatenate([ix.search(Q, 12)[0][:, :3, 1].reshape(-1),
                                       rng.integers(0, N_BIG // 2, size=5000).astype(np.uint64)]))
    assert ix.delete(np.stack([np.zeros_like(doomed), doomed], 1)) == doomed.size
    assert ix.stats()["rows_moved"] > before
    image_in_step(ix, Q[:4])
    for i in range(NQ):
        agree(ix, Q[i], 12, no_fallback=True)
    agree(ix, Q[:3], 128)


# --------------------------------------------------------------------------------- small tables through the option
def _random_rows(n, seed):
    rng = np.random.default_rng(seed)
    return rng.standard_normal((n, 1024)).astype(np.float32), rng.standard_normal((4, 1024)).astype(np.float32)


def _against_oracle(ix, rows, ids, Q, k):
    got = agree(ix, Q, k, want_paths=(3, 1) if len(Q) == 1 or k > 64 else (2, 2), no_fallback=k <= 33)
    for i in range(len(Q)):
        w_ids, w_d = O.topk_exact(rows, ids, Q[i], k)
        assert np.array_equal(got[0][i], w_ids) and np.array_equal(got[1][i].view(np.uint64), w_d.view(np.uint64))


def test_growth_past_capacity_copies_the_image():
    import outline_rag_b200 as orx
    X, Q = _random_rows(40_000, 1)
    ids = O.ids_arange(0, len(X))
    with orx.Index("fp32", 1024, 0) as ix:
        ix.set_option(_opt(), 0)                         # small table: the image exists from the first growth on
        for s in range(0, len(X), 5000):                 # several growths, each with live rows to carry over
            ix.upsert(ids[s:s + 5000], X[s:s + 5000])
        assert ix.capacity >= len(X) > 1024
        image_in_step(ix, Q)
        for k in (12, 65):
            _against_oracle(ix, X, ids, Q[:1], k)
        _against_oracle(ix, X, ids, Q[:3], 97)


def test_snapshot_restore_and_copy_binary_load_rebuild_the_image(tmp_path):
    import outline_rag_b200 as orx
    from oracle import pgvector_wire as W
    X, Q = _random_rows(30_000, 2)
    ids = O.ids_arange(0, len(X))
    with orx.Index("fp32", len(X), 0) as ix:
        ix.upsert(ids, X)
        ix.save(str(tmp_path / "snap"))
    restored = orx.Index.load(str(tmp_path / "snap"), device=0, capacity=IMAGE_MIN_ROWS)   # image from the start
    with restored:
        image_in_step(restored, Q)
        _against_oracle(restored, X, ids, Q[:1], 12)
        _against_oracle(restored, X, ids, Q[:3], 128)
    with orx.Index("fp32", IMAGE_MIN_ROWS, 0) as ix:                                        # image from the start
        stream = W.copy_binary_stream(ids, X)
        assert ix.load_pgcopy([stream]) == (len(X), 0)
        image_in_step(ix, Q)
        _against_oracle(ix, X, ids, Q[:1], 33)
        _against_oracle(ix, X, ids, Q[:3], 65)


def test_two_shard_handle_merges_image_scans():
    import outline_rag_b200 as orx
    X, Q = _random_rows(30_000, 3)
    ids = O.ids_arange(0, len(X))
    with orx.Index("fp32", len(X), devices=[0, 0]) as ix:
        ix.upsert(ids, X)
        for k in (1, 12, 97):
            _against_oracle(ix, X, ids, Q[:1], k)


# ---------------------------------------------------------------------------------------------- the error bound
def _worst_query(seed, n_zero=0):
    """A unit query whose pattern elements are +-(1 + 2^-8) * 2^-5: the exact tie of RNE to bf16, which rounds to the
    even neighbour 1 -- 2^-8 / (1 + 2^-8), the largest relative error of the conversion (tests/test_image_scan.py
    checks every significand) -- and q^ keeps them bit for bit"""
    rng = np.random.default_rng(seed)
    pat = np.float32(1 + 2.0 ** -8)
    n_pat = 1024 - A.N_BALLAST - n_zero
    signs = rng.choice(np.array([-1.0, 1.0], np.float32), 1024)
    q = np.zeros(1024, np.float32)
    q[:n_pat] = signs[:n_pat] * pat * A.AMP
    s = float(O.canon_sqnorm(q[None])[0])
    q[n_pat:n_pat + A.N_BALLAST] = signs[n_pat:n_pat + A.N_BALLAST] * np.float32(np.sqrt((1.0 - s) / A.N_BALLAST))
    qh, _ = A.prep_qhat(q)
    assert np.array_equal(qh[:n_pat].view(np.uint32), q[:n_pat].view(np.uint32))
    return q


def test_image_error_is_below_eps_and_reaches_its_worst_case():
    import outline_rag_b200 as orx
    qs = [_worst_query(s) for s in range(4)]
    rng = np.random.default_rng(9)
    rows, expect_finite = [], []
    for q in qs:                                      # parallel / antiparallel (the error's sign pattern) / balanced
        for r in A.adversarial_rows(q, 1).values():
            rows.append(r)
            expect_finite.append(True)
    base = rng.standard_normal((64, 1024)).astype(np.float32)
    rows += list(base)
    expect_finite += [True] * len(base)
    for scale, finite in ((2.0 ** -40 * 1.01, True), (2.0 ** 40 * 0.99, True),       # inside the regular band
                          (2.0 ** -40 * 0.99, False), (2.0 ** 40 * 1.01, False)):    # outside: never trusted
        r = base[0] / np.float32(np.linalg.norm(base[0])) * np.float32(scale)
        rows.append(r.astype(np.float32))
        expect_finite.append(finite)
    sub = np.zeros(1024, np.float32)                  # subnormal elements beside one normal one
    sub[0] = np.float32(2.0 ** -30)
    sub[1:] = rng.uniform(-1, 1, 1023).astype(np.float32) * np.float32(1e-39)
    rows.append(sub)
    expect_finite.append(True)
    rows = np.stack(rows).astype(np.float32)
    Q = np.stack(qs + list(rng.standard_normal((4, 1024)).astype(np.float32)))
    with orx.Index("fp32", len(rows), 0) as ix:
        ix.upsert(O.ids_arange(0, len(rows)), rows)
        got = ix.debug_image_scores(Q).cpu().numpy()
        fast = ix.debug_fast_scores(Q).cpu().numpy()
    fin = np.array(expect_finite)
    assert np.isfinite(got[fin]).all() and not np.isfinite(got[~fin]).any()
    assert np.array_equal(np.isfinite(fast), np.isfinite(got))
    err = max(float(np.max(np.abs(got[fin, j].astype(np.float64) - A.cosine(rows[fin], Q[j])))) for j in range(len(Q)))
    print(f"\nmax |image score - cosine| = {err:.4e} (EPS_GEMV_IMAGE {EPS_GEMV_IMAGE:.3e})")
    assert err <= EPS_GEMV_IMAGE
    assert err > 0.95 * 2.0 ** -8                      # the construction reaches the bound: it is tight, not loose


# ---------------------------------------------------------------------------------------- forced rank inversions
N_DECOYS = 192
N_ROWS = 256 * (N_DECOYS + 2)


def image_width(k):                  # finalize's K for the image scans: 32 * image_slots_for_k (csrc/internal.h)
    return 32 * (2 if k <= 16 else 4 if k <= 32 else 5)


@pytest.fixture(scope="module")
def inversion():
    """Winner w = the worst-case query itself (its image score underestimates its cosine by ~3.8e-3), at the last row;
    192 decoys at the first rows raise one of the query's zero positions by a bf16-exact step: image and fp32 scores
    tie w's bit for bit, canonical distances are strictly worse."""
    for seed in range(64):
        q = _worst_query(seed, n_zero=64)
        w = A.with_zero_value(q, q)
        qh, _ = A.prep_qhat(q)
        if A.cosine(w[None], q)[0] - A.gemv_fast(w[None], qh, "fp32", image=True)[0] > 1e-3:
            break
    else:
        raise AssertionError("no seed gives an image score that underestimates the winner's cosine")
    decoys = A.decoy_rows(w, q, N_DECOYS)
    assert np.array_equal(A.bf16_exact(decoys[:, A.zero_positions(q)]), decoys[:, A.zero_positions(q)])
    rows = np.random.default_rng(7).standard_normal((N_ROWS, 1024)).astype(np.float32)
    rows[:N_DECOYS] = decoys
    rows[-1] = w
    ids = O.ids_arange(0, N_ROWS)
    want = O.topk_exact(rows, ids, q, max(KS), exhaustive=True)
    assert want[0][0, 1] == N_ROWS - 1
    return q, rows, ids, want


def _premise(scores, rows_n, want, k, width):
    w = rows_n - 1
    assert (scores[:N_DECOYS] == scores[w]).all(), "the decoys do not tie the winner's image score"
    assert int(np.sum(scores > scores[w]) + np.sum(scores[:w] == scores[w])) >= width
    assert w in want[0][:k, 1]
    if k > 1:
        assert 1.0 - want[1][k - 1] > float(scores[w])


@pytest.mark.parametrize("k", KS)
@pytest.mark.parametrize("form", ["single", "batch", "bitmap"])
def test_forced_inversion_on_the_image_falls_back_to_the_exact_answer(inversion, k, form):
    import outline_rag_b200 as orx
    if form == "batch" and k <= 64:
        pytest.skip("batches with k <= 64 run the tcgen05 scan")
    q, rows, ids, want = inversion
    allow = np.delete(ids, np.arange(1000, 1100), axis=0)
    with orx.Index("fp32", N_ROWS, 0) as ix:
        A.import_stored(ix, ids, rows)
        ix.set_option(_opt(), 0)
        _premise(ix.debug_image_scores(q[None]).cpu().numpy()[:, 0], N_ROWS, want, k, image_width(k))
        Q = np.stack([q] * (3 if form == "batch" else 1))
        st0 = ix.stats()
        got = ix.search_filtered(Q, k, allow) if form == "bitmap" else ix.search(Q, k)
        st1 = ix.stats()
    assert st1["last_path"] == 3
    assert st1["fallback_exhaustive"] - st0["fallback_exhaustive"] == len(Q)
    for i in range(len(Q)):
        assert got[2][i] == k
        assert np.array_equal(got[0][i], want[0][:k])
        assert np.array_equal(got[1][i].view(np.uint64), want[1][:k].view(np.uint64))


@pytest.mark.parametrize("k,nq", [(1, 1), (12, 1), (17, 1), (64, 1), (128, 1), (65, 3), (128, 3)])
def test_provable_tables_need_no_fallback_on_the_image(k, nq):
    import outline_rag_b200 as orx
    rng = np.random.default_rng(100 + k)
    q = rng.standard_normal(1024).astype(np.float32)
    u = q / np.linalg.norm(q)
    rows = rng.standard_normal((8192, 1024)).astype(np.float32)
    noise = rng.standard_normal((k, 1024)).astype(np.float32)
    noise -= np.outer(noise @ u, u)
    noise /= np.linalg.norm(noise, axis=1, keepdims=True)
    rows[:k] = 0.9 * u + np.sqrt(1 - 0.9 ** 2) * noise * rng.uniform(0.9, 1.1, (k, 1))
    ids = O.ids_arange(0, len(rows))
    cos = np.sort(A.cosine(rows, q))
    assert cos[-k] - cos[-k - 1] > 3 * EPS_GEMV_IMAGE
    want_ids, want_d = O.topk_exact(rows, ids, q, k, exhaustive=True)
    with orx.Index("fp32", len(rows), 0) as ix:
        ix.upsert(ids, rows)
        ix.set_option(_opt(), 0)
        st0 = ix.stats()
        got = ix.search(np.repeat(q[None], nq, axis=0), k)
        st1 = ix.stats()
    assert st1["last_path"] == 3
    assert st1["fallback_exhaustive"] == st0["fallback_exhaustive"]
    for i in range(nq):
        assert np.array_equal(got[0][i], want_ids) and np.array_equal(got[1][i].view(np.uint64), want_d.view(np.uint64))


def test_small_tables_get_no_image_until_a_search_needs_one():
    import outline_rag_b200 as orx
    X, Q = _random_rows(20_000, 4)
    ids = O.ids_arange(0, len(X))
    with orx.Index("fp32", len(X), 0) as ix:
        ix.upsert(ids, X)
        ix.search(Q[0], 12)
        assert ix.stats()["last_path"] == 1                # below 2^20 rows, no image was allocated
        _against_oracle(ix, X, ids, Q[:1], 12)             # lowering the option builds it from the rows
        image_in_step(ix, Q)
        ix.upsert(ids[:100], -X[:100])                     # and from then on writes keep it in step
        image_in_step(ix, Q)


# ------------------------------------------------------------ the re-scan of queries the tcgen05 pass could not prove
def test_tcgen05_unproven_batch_is_rescanned_over_the_fp32_rows_not_the_image():
    """200 rows at cosines 0.9, 0.9 - 1e-5, ... to the query: within the tensor pass's eps of the 12th, so its 64-key lists
    cannot prove a batch; 1e-5 apart, so the fp32 scan (eps 3e-6) proves every query -- the image's eps (3.92e-3) would
    not.  With the image enabled for this table, the level-1 re-scan must still settle the batch: fallback_gemv moves,
    fallback_exhaustive does not."""
    import outline_rag_b200 as orx
    rng = np.random.default_rng(21)
    q = rng.standard_normal(1024).astype(np.float32)
    u = q.astype(np.float64) / np.linalg.norm(q.astype(np.float64))
    rows = rng.standard_normal((49_664, 1024)).astype(np.float32)
    noise = rng.standard_normal((200, 1024))
    noise -= np.outer(noise @ u, u)
    noise /= np.linalg.norm(noise, axis=1, keepdims=True)
    c = 0.9 - 1e-5 * np.arange(200)
    rows[1000:1200] = (c[:, None] * u + np.sqrt(1 - c[:, None] ** 2) * noise).astype(np.float32)
    ids = O.ids_arange(0, len(rows))
    cos = np.sort(A.cosine(rows, q))[::-1]
    assert np.max(np.diff(cos[:40])) < -5e-6 and cos[11] - cos[63] < 2.5e-3     # proven by fp32, not by tcgen05
    want_ids, want_d = O.topk_exact(rows, ids, q, 12, exhaustive=True)
    Q = np.repeat(q[None], 4, axis=0)
    with orx.Index("fp32", len(rows), 0) as ix:
        ix.upsert(ids, rows)
        ix.set_option(_opt(), 0)
        ix.search(q[None], 12)
        assert ix.stats()["last_path"] == 3                # the image exists and single queries read it
        st0 = ix.stats()
        got = ix.search(Q, 12)
        st1 = ix.stats()
    assert st1["last_path"] == 2
    assert st1["fallback_gemv"] - st0["fallback_gemv"] == len(Q)
    assert st1["fallback_exhaustive"] == st0["fallback_exhaustive"]
    for i in range(len(Q)):
        assert np.array_equal(got[0][i], want_ids) and np.array_equal(got[1][i].view(np.uint64), want_d.view(np.uint64))
