"""The GEMV scans over the 8-bit image of a large fp32 table (DESIGN.md section 2, "8-bit image"): same answers as the
fp32 scans, bit for bit, on every path it serves and after every kind of write; its scores equal the CPU emulation of
tests/test_image8_scan.py bit for bit and stay within EPS_GEMV_IMAGE8 of the cosine; the full oracle at 2^22 rows with
no fallback; the completeness proof failing (and the fallback answering) when decoys outrank the winner on 8-bit
scores; rows over R8_CAP as always-candidates, and a table with too many of them back on the fp32 rows.

ORX_OPT_IMAGE8_MIN_ROWS = 0 gives small tables the 8-bit image; ORX_OPT_IMAGE_MIN_ROWS switches the same index between
scanning it (0, last_path 4) and scanning the fp32 rows (-1, last_path 1), so each comparison runs both on identical rows."""
import numpy as np
import pytest

from oracle import cosine_topk as O
from tests import adversarial as A
from tests.test_image8_scan import EPS_GEMV_IMAGE8, _adversarial_rows, image8_scores

pytestmark = pytest.mark.gpu
N = 200_000
NQ = 6
IMAGE_MIN_ROWS = 1 << 20
IMAGE8_MIN_ROWS = 1 << 22


def _lib():
    from outline_rag_b200 import _lib as L
    return L


def eight_bit(ix):
    """an index whose image is the 8-bit one whatever its capacity, scanned from the first row on"""
    L = _lib()
    ix.set_option(L.ORX_OPT_IMAGE8_MIN_ROWS, 0)
    ix.set_option(L.ORX_OPT_IMAGE_MIN_ROWS, 0)
    return ix


def both(ix, fn):
    """fn() over the 8-bit image and over the fp32 rows of the same index (the option left at 0)"""
    L = _lib()
    ix.set_option(L.ORX_OPT_IMAGE_MIN_ROWS, 0)
    a = fn()
    pa = ix.stats()["last_path"]
    ix.set_option(L.ORX_OPT_IMAGE_MIN_ROWS, -1)
    b = fn()
    pb = ix.stats()["last_path"]
    ix.set_option(L.ORX_OPT_IMAGE_MIN_ROWS, 0)
    return a, b, pa, pb


def same(a, b):
    return (np.array_equal(a[0], b[0]) and np.array_equal(a[1].view(np.uint64), b[1].view(np.uint64))
            and np.array_equal(a[2], b[2]))


def agree(ix, Q, k, filtered=None, want_paths=(4, 1), no_fallback=False):
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


def stored_rows(ix):
    n = len(ix)
    ids = np.zeros((n, 2), np.uint64)
    raw = np.zeros((n, 4096), np.uint8)
    ix.export_rows(0, n, ids, raw)
    return raw.view(np.float32)


def image8_in_step(ix, Q):
    """the 8-bit scores of every live row equal, bit for bit, the emulation over the fp32 rows now stored there"""
    got = ix.debug_image8_scores(Q).cpu().numpy()
    rows = stored_rows(ix)
    for j in range(len(Q)):
        want = image8_scores(rows, Q[j])
        fin = np.isfinite(want)
        assert np.array_equal(np.isfinite(got[:, j]), fin), j
        assert np.array_equal(got[fin, j].view(np.uint32), want[fin].view(np.uint32)), j


@pytest.fixture(scope="module")
def tab():
    import outline_rag_b200 as orx
    from orx_testkit.synth import Synth, default_centres
    syn = Synth(default_centres(N))
    X = syn.table(N)
    Q, anchors = syn.queries(NQ, N)
    ix = eight_bit(orx.Index("fp32", N + 4096, 0))
    ix.upsert(O.ids_arange(0, N), X)
    yield syn, ix, X, Q, anchors
    ix.close()


@pytest.mark.parametrize("k", [1, 5, 12])
def test_single_query_8bit_equals_fp32_scan(tab, k):
    _, ix, _, Q, _ = tab
    for i in range(NQ):
        agree(ix, Q[i], k, no_fallback=True)


@pytest.mark.parametrize("k", [13, 64, 97])
def test_wider_k_and_gemv_batches_read_the_fp32_rows(tab, k):
    _, ix, _, Q, _ = tab
    agree(ix, Q[0], k, want_paths=(1, 1))
    if k > 64:
        agree(ix, Q[:3], k, want_paths=(1, 1))


@pytest.mark.parametrize("k", [1, 12, 33])
def test_filtered_bitmap_and_filter_handle_8bit_equals_fp32_scan(tab, k):
    _, ix, _, Q, _ = tab
    allow = O.ids_arange(0, N)[::3]
    paths = (4, 1) if k <= 12 else (1, 1)
    agree(ix, Q[1:2], k, filtered=lambda q, kk: ix.search_filtered(q, kk, allow), want_paths=paths)
    with ix.make_filter(allow) as flt:
        agree(ix, Q[2:3], k, filtered=lambda q, kk: ix.search_filtered(q, kk, flt), want_paths=paths)


def test_8bit_scores_equal_the_emulation_and_the_oracle(tab):
    _, ix, X, Q, anchors = tab
    image8_in_step(ix, Q[:3])
    for i in range(NQ):
        got = agree(ix, Q[i], 12, no_fallback=True)
        w_ids, w_d = O.topk_exact(X, O.ids_arange(0, N), Q[i], 12)
        assert np.array_equal(got[0][0], w_ids) and np.array_equal(got[1][0].view(np.uint64), w_d.view(np.uint64))
        assert got[0][0, 0, 1] == anchors[i]


def test_in_place_upsert_and_delete_compaction_keep_the_8bit_image_in_step(tab):
    """Runs last on the module table (it mutates it)."""
    syn, ix, _, Q, _ = tab
    rng = np.random.default_rng(5)
    hits = ix.search(Q, 12)[0][:, :4, 1].reshape(-1)
    new = syn.rows(rng.integers(0, N, size=hits.size).astype(np.uint64))
    new[::2] = -syn.rows(hits[::2])
    ix.upsert(np.stack([np.zeros_like(hits), hits], 1), new)
    image8_in_step(ix, Q[:2])
    agree(ix, Q[0], 12, no_fallback=True)
    before = ix.stats()["rows_moved"]
    doomed = np.unique(np.concatenate([ix.search(Q, 12)[0][:, :3, 1].reshape(-1),
                                       rng.integers(0, N // 2, size=3000).astype(np.uint64)]))
    assert ix.delete(np.stack([np.zeros_like(doomed), doomed], 1)) == doomed.size
    assert ix.stats()["rows_moved"] > before
    image8_in_step(ix, Q[:2])
    for i in range(NQ):
        agree(ix, Q[i], 12, no_fallback=True)


# --------------------------------------------------------------------------------- growth, restore, load, shards
def _synth_rows(n, seed):
    from orx_testkit.synth import Synth
    syn = Synth(256, seed=seed)
    return syn.table(n), syn.queries(4, n)[0]


def _against_oracle(ix, rows, ids, Q, k, want_paths=(4, 1)):
    got = agree(ix, Q, k, want_paths=want_paths)
    for i in range(len(Q)):
        w_ids, w_d = O.topk_exact(rows, ids, Q[i], k)
        assert np.array_equal(got[0][i], w_ids) and np.array_equal(got[1][i].view(np.uint64), w_d.view(np.uint64))


def test_growth_across_image8_min_rows_replaces_the_bf16_image():
    import outline_rag_b200 as orx
    L = _lib()
    X, Q = _synth_rows(12_000, 1)
    ids = O.ids_arange(0, len(X))
    with orx.Index("fp32", 1024, 0) as ix:
        ix.set_option(L.ORX_OPT_IMAGE_MIN_ROWS, 0)
        ix.set_option(L.ORX_OPT_IMAGE8_MIN_ROWS, 4096)
        ix.upsert(ids[:2000], X[:2000])                  # capacity 2560: the bf16 image
        assert ix.capacity < 4096
        _against_oracle(ix, X[:2000], ids[:2000], Q[:1], 12, want_paths=(3, 1))
        for s in range(2000, len(X), 2500):              # growth past 4096 rows: an 8-bit image built from the rows
            ix.upsert(ids[s:s + 2500], X[s:s + 2500])
        assert ix.capacity >= len(X)
        image8_in_step(ix, Q[:2])
        with pytest.raises(Exception):
            ix.debug_image_scores(Q[:1])                 # one image per table
        for k in (1, 12):
            _against_oracle(ix, X, ids, Q[:1], k)


def test_snapshot_restore_and_copy_binary_load_build_the_8bit_image(tmp_path):
    import outline_rag_b200 as orx
    from oracle import pgvector_wire as W
    X, Q = _synth_rows(30_000, 2)
    ids = O.ids_arange(0, len(X))
    with orx.Index("fp32", len(X), 0) as ix:
        ix.upsert(ids, X)
        ix.save(str(tmp_path / "snap"))
    restored = orx.Index.load(str(tmp_path / "snap"), device=0, capacity=IMAGE8_MIN_ROWS)   # 8-bit image from the start
    with restored:
        restored.set_option(_lib().ORX_OPT_IMAGE_MIN_ROWS, 0)
        image8_in_step(restored, Q[:2])
        _against_oracle(restored, X, ids, Q[:1], 12)
    with orx.Index("fp32", IMAGE8_MIN_ROWS, 0) as ix:
        ix.set_option(_lib().ORX_OPT_IMAGE_MIN_ROWS, 0)
        stream = W.copy_binary_stream(ids, X)
        assert ix.load_pgcopy([stream]) == (len(X), 0)
        image8_in_step(ix, Q[:2])
        _against_oracle(ix, X, ids, Q[:1], 5)


def test_two_shard_handle_merges_8bit_scans():
    import outline_rag_b200 as orx
    X, Q = _synth_rows(30_000, 3)
    ids = O.ids_arange(0, len(X))
    with orx.Index("fp32", len(X), devices=[0, 0]) as ix:
        eight_bit(ix)
        ix.upsert(ids, X)
        for k in (1, 12):
            got = ix.search(Q[:1], k)
            w_ids, w_d = O.topk_exact(X, ids, Q[0], k)
            assert np.array_equal(got[0][0], w_ids) and np.array_equal(got[1][0].view(np.uint64), w_d.view(np.uint64))


# ---------------------------------------------------------------------------------------- the bound, the proof
def test_8bit_error_is_below_eps_on_adversarial_rows():
    import outline_rag_b200 as orx
    rng = np.random.default_rng(9)
    rows, names = _adversarial_rows(rng)
    Q = np.concatenate([rows[:2], rng.standard_normal((4, 1024)).astype(np.float32)])
    with orx.Index("fp32", len(rows), 0) as ix:
        eight_bit(ix)
        ix.upsert(O.ids_arange(0, len(rows)), rows)
        got = ix.debug_image8_scores(Q).cpu().numpy()
    err = 0.0
    for j in range(len(Q)):
        want = image8_scores(rows, Q[j])
        fin = np.isfinite(want)
        assert np.array_equal(np.isfinite(got[:, j]), fin)
        assert np.array_equal(got[fin, j].view(np.uint32), want[fin].view(np.uint32))
        err = max(err, float(np.abs(got[fin, j].astype(np.float64) - A.cosine(rows[fin], Q[j])).max()))
    print(f"\nmax |8-bit score - cosine| = {err:.4e} (EPS_GEMV_IMAGE8 {EPS_GEMV_IMAGE8:.3e})")
    assert 1e-4 < err <= EPS_GEMV_IMAGE8
    for n in ("one dominant", "half steps", "below the band", "above the band", "zero"):
        assert not np.isfinite(got[names.index(n)]).any(), n          # markers: always / never a candidate


def _decoy_table(n_decoys, seed):
    """A winner w whose elements are exact multiples of d = 2^-7 (so w is its own 8-bit image) and decoys w + eta with
    |eta_i| = d / 4 against the sign of w_i: the same int8 image, a smaller norm, so an 8-bit score ABOVE the winner's,
    and a cosine with q = w below 1.  With more decoys than a candidate list holds, the winner is not listed at all."""
    rng = np.random.default_rng(seed)
    Xw = rng.integers(-40, 41, 1024)
    Xw[0] = 127
    Xw[Xw == 0] = 1
    w = (Xw * 2.0 ** -7).astype(np.float32)
    dec = np.repeat(w[None], n_decoys, 0)
    for j in range(n_decoys):
        sel = rng.choice(np.arange(1, 1024), 64, replace=False)
        dec[j, sel] -= np.sign(w[sel]) * np.float32(2.0 ** -9)
    filler = rng.standard_normal((5000, 1024)).astype(np.float32) * np.float32(0.1)
    rows = np.concatenate([dec, filler, w[None]]).astype(np.float32)          # the winner is the LAST row
    return rows, w


@pytest.mark.parametrize("k", [1, 12])
def test_forced_inversion_on_the_8bit_image_falls_back_to_the_exact_answer(k):
    import outline_rag_b200 as orx
    rows, w = _decoy_table(200, k)
    s = image8_scores(rows, w)
    assert (s[:200] > s[-1]).all()                       # every decoy outranks the winner on the 8-bit score
    ids = O.ids_arange(0, len(rows))
    with orx.Index("fp32", len(rows), 0) as ix:
        eight_bit(ix)
        ix.upsert(ids, rows)
        st0 = ix.stats()
        got = ix.search(w, k)
        st1 = ix.stats()
    assert st1["last_path"] == 4
    assert st1["fallback_exhaustive"] + st1["fallback_gemv"] > st0["fallback_exhaustive"] + st0["fallback_gemv"]
    w_ids, w_d = O.topk_exact(rows, ids, w, k)
    assert np.array_equal(got[0][0], w_ids) and np.array_equal(got[1][0].view(np.uint64), w_d.view(np.uint64))
    assert got[0][0, 0, 1] == len(rows) - 1              # the winner


def test_rows_over_the_cap_are_always_candidates_and_too_many_return_to_the_fp32_rows():
    import outline_rag_b200 as orx
    X, Q = _synth_rows(20_000, 4)
    rng = np.random.default_rng(4)
    spiky = X[:40].copy()                                 # one outlier dimension: relative residual over 2^-6
    spiky[:, 7] = np.float32(50.0) * np.abs(spiky).max(1)
    assert not np.isfinite(image8_scores(spiky, Q[0])).any()
    ids = O.ids_arange(0, len(X))
    with orx.Index("fp32", len(X) + 64, 0) as ix:
        eight_bit(ix)
        ix.upsert(ids, X)
        agree(ix, Q[0], 12, no_fallback=True)
        cap_ids = O.ids_arange(0, 40)
        ix.upsert(cap_ids[:16], spiky[:16])               # 16 capped rows: still the 8-bit scan
        X[:16] = spiky[:16]
        got = agree(ix, Q[0], 12)
        ix.upsert(cap_ids[16:], spiky[16:])               # 40: the fp32 rows
        X[:40] = spiky
        agree(ix, Q[0], 12, want_paths=(1, 1))
        ix.delete(cap_ids[:30])                           # 10 left: the 8-bit scan again
        keep = np.ones(len(X), bool)
        keep[:30] = False
        got = agree(ix, Q[1], 12)
        w_ids, w_d = O.topk_exact(X[keep], ids[keep], Q[1], 12)
        assert np.array_equal(got[0][0], w_ids) and np.array_equal(got[1][0].view(np.uint64), w_d.view(np.uint64))
        q = spiky[35] + np.float32(0.01) * rng.standard_normal(1024).astype(np.float32)   # a capped row is found
        got = agree(ix, q, 1)
        assert got[0][0, 0, 1] == 35


# --------------------------------------------------------------------------------------- the full oracle at 2^22
def test_8bit_scan_equals_the_full_oracle_pass_at_2_22_rows_without_fallbacks():
    import outline_rag_b200 as orx
    from oracle.synth_host import FastSynth
    from orx_testkit.device import synth_rows_device
    from orx_testkit.synth import SEED_TABLE, default_centres
    n = IMAGE8_MIN_ROWS + 100_000
    syn = FastSynth(default_centres(n))
    Q, anchors = syn.queries(8, n)
    with orx.Index("fp32", n, 0) as ix:                   # defaults: an 8-bit image, scanned from 2^20 live rows
        chunk = 262_144
        for s in range(0, n, chunk):
            m = min(chunk, n - s)
            ix.upsert(O.ids_arange(s, s + m), synth_rows_device(0, SEED_TABLE, syn.n_centres, s, m))
        truth = O.StreamingTopK(Q, 12)
        for s in range(0, n, 131_072):
            m = min(131_072, n - s)
            truth.feed(syn.table(m, start=s), O.ids_arange(s, s + m))
        want = truth.result()
        st0 = ix.stats()
        for i in range(len(Q)):
            got = ix.search(Q[i], 12)
            assert ix.stats()["last_path"] == 4
            assert np.array_equal(got[0][0], want[i][0]), i
            assert np.array_equal(got[1][0].view(np.uint64), want[i][1].view(np.uint64)), i
            assert got[0][0, 0, 1] == anchors[i]
        st1 = ix.stats()
    assert st1["fallback_exhaustive"] == st0["fallback_exhaustive"]
    assert st1["fallback_gemv"] == st0["fallback_gemv"]
