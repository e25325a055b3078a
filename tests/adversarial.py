"""Adversarial inputs for the exactness argument of DESIGN.md section 2, and bit-exact CPU emulations of what the
scans compute from them.

The argument: a scan's fast (GEMV) or coarse (tcgen05) score s satisfies |s - cos| <= eps; finalize rescores the
candidates in binary64 and proves that no row outside the list sorts before the k-th.  Random data tests neither half
where it is thin, so this module builds

* queries whose normalised copy q^ keeps a chosen mantissa pattern bit for bit (24 "ballast" elements fix the norm),
  with the pattern the operand conversion of the tensor-core pass treats worst, and rows parallel, antiparallel and
  sign-balanced to them (`adversarial_query`, `adversarial_rows`);
* rank inversions: decoy rows whose fast AND coarse scores equal the winner's bit for bit (they differ from the winner
  only where q^ is exactly 0, so every product is the same) while their canonical distance is strictly worse (they
  differ exactly there, so |x|^2 is larger), placed at lower row indices so that they win every key tie
  (`decoy_rows`).

Everything but `import_stored` is NumPy; tests/test_adversarial.py pins it on the CPU, the *_gpu.py tests run it
through the device.
"""
import numpy as np

from oracle.cosine_topk import canon_distance, canon_sqnorm
from tests._helpers import bf16_rne, stored_bf16_rows

D = 1024
N_BALLAST = 24
AMP = np.float32(2.0 ** -5)          # pattern elements are +-pattern * 2^-5

# Mantissa patterns the operand conversion of the tensor-core pass handles worst (all just below a rounding boundary,
# so the converted operand loses the most it can):
PATTERNS = {
    # kind::tf32 dropping the low 13 mantissa bits: 1.0000000000 followed by 13 ones -> 1.0 (loses 2^-10 - 2^-23)
    "tf32_trunc": np.float32(1.0 + (2 ** 13 - 1) * 2.0 ** -23),
    # kind::tf32 rounding to nearest: just below the tf32 midpoint 1 + 2^-11 -> 1.0
    "tf32_rn": np.float32(1.0 + 2.0 ** -11 - 2.0 ** -23),
    # RNE to bf16 (the query operand of the bf16 pass): just below the midpoint 1 + 2^-9 -> 1.0
    "bf16": np.float32(1.0 + 2.0 ** -9 - 2.0 ** -23),
}
# The conversion kind::tf32 applies to fp32 operands on sm_100a, as measured by
# tests/test_epsilon_adversarial_gpu.py::test_operand_conversion_mode (and assumed by csrc/internal.h).
TF32_MODE = "trunc"
WORST = {"fp32": "tf32_" + TF32_MODE, "bf16": "bf16"}

# rank inversions: the winner carries ZV at the zero positions of the query, decoy j raises one of them by a multiple
# of STEP (bf16-exact: ZV + m * STEP for m < 128 has 8 significant bits)
ZV = np.float32(2.0 ** -16)
STEP = np.float32(2.0 ** -23)


# ------------------------------------------------------------------------------------------------ emulations
def prep_qhat(q):
    """Bit-exact emulation of prep_queries_kernel: canonical |q|^2, 1/sqrt in binary64, q * inv rounded to fp32 (RN),
    then RNE to bf16 for the bf16 pass.  Returns (qhat fp32, qhat16 as fp32 values)."""
    q = np.asarray(q, np.float32)
    n2 = canon_sqnorm(q.reshape(-1, D))
    inv = 1.0 / np.sqrt(n2)
    qh = (q.reshape(-1, D).astype(np.float64) * inv[:, None]).astype(np.float32).reshape(q.shape)
    return qh, bf16_rne(qh)


def tf32_trunc(x):
    return (np.ascontiguousarray(x, np.float32).view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)


def tf32_rn(x):
    """round to nearest, ties away from zero (cvt.rna.tf32.f32)"""
    u = np.ascontiguousarray(x, np.float32).view(np.uint32).astype(np.uint64)
    return (((u + np.uint64(0x1000)) & np.uint64(0xFFFFE000)).astype(np.uint32)).view(np.float32).reshape(np.shape(x))


def to_tf32(x, mode=TF32_MODE):
    return tf32_trunc(x) if mode == "trunc" else tf32_rn(x)


def row_scale(rows):
    """The per-row 1/|x| the table keeps (table_ops.cu scale_from_n2): NaN for a zero row, +inf outside
    |x| in [2^-40, 2^40], else fp32(1 / sqrt(canonical |x|^2))."""
    n2 = canon_sqnorm(np.asarray(rows, np.float32).reshape(-1, D))
    with np.errstate(divide="ignore"):
        s = (1.0 / np.sqrt(n2)).astype(np.float32)
    s = np.where(n2 > 0, s, np.float32(np.nan))
    return np.where((n2 > 0) & ((n2 < 2.0 ** -80) | (n2 > 2.0 ** 80)), np.float32(np.inf), s).astype(np.float32)


def _fma32(a, b, c):
    # a*b of two fp32 values is exact in binary64; rounding the binary64 sum to fp32 equals the fused rounding unless
    # that sum was itself rounded onto an fp32 rounding boundary (rare; the GPU tests compare this with the device)
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(np.float32)


def gemv_fast(rows, qhat, dtype, image=False):
    """Emulation of warp_row_dot (scan_common.cuh) times the row scale: lane l runs an fp32 FMA chain over its 32
    elements in load order, then the xor butterfly 16, 8, 4, 2, 1.  rows: stored values as fp32 [n, D].
    image=True: the scan over the bf16 image of fp32 rows -- the chain runs over RNE-bf16 of the rows (8 elements per
    vector), the scale is still the fp32 row's."""
    X = np.asarray(rows, np.float32).reshape(-1, D)
    qh = np.asarray(qhat, np.float32)
    scale = row_scale(X)
    if image:
        X, dtype = bf16_exact(X), "bf16"
    w = 4 if dtype == "fp32" else 8                      # elements per lane per 16-byte vector
    # element order of lane l: vectors v = l + 32 j, elements w*v .. w*v + w-1
    lanes = np.arange(32)[:, None, None]
    j = np.arange(32 // w)[None, :, None]
    t = np.arange(w)[None, None, :]
    order = (w * (lanes + 32 * j) + t).reshape(32, 32)  # [lane, step]
    acc = np.zeros((X.shape[0], 32), np.float32)
    for s in range(32):
        e = order[:, s]
        acc = _fma32(X[:, e], qh[e][None, :], acc)
    for d in (16, 8, 4, 2, 1):
        acc = (acc + acc[:, np.arange(32) ^ d]).astype(np.float32)
    with np.errstate(invalid="ignore", over="ignore"):
        return (acc[:, 0] * scale).astype(np.float32)


def coarse_conversion_only(rows, qhat, dtype, mode=TF32_MODE):
    """The tcgen05 pass's coarse score with exact accumulation: converted operands (tf32 for fp32 tables, the RNE-bf16
    q^ for bf16 tables, whose rows are exact bf16) summed in binary64, times the row scale.  What the hardware adds on
    top is its accumulation error."""
    X = np.asarray(rows, np.float32).reshape(-1, D)
    qh = np.asarray(qhat, np.float32)
    if dtype == "fp32":
        a, b = to_tf32(X, mode), to_tf32(qh, mode)
    else:
        a, b = X, bf16_rne(qh)
    return (a.astype(np.float64) @ b.astype(np.float64)) * row_scale(X).astype(np.float64)


def cosine(rows, q):
    return 1.0 - canon_distance(np.asarray(rows, np.float32).reshape(-1, D), np.asarray(q, np.float32))


def stored(rows, dtype):
    """What a table of `dtype` stores for input rows (fp32 verbatim; bf16: RNE of the normalised row)."""
    rows = np.asarray(rows, np.float32).reshape(-1, D)
    return rows if dtype == "fp32" else stored_bf16_rows(rows)


# ------------------------------------------------------------------------------------------ ε constructions
def adversarial_query(kind, seed=0, n_zero=0):
    """A unit query whose pattern elements are +-PATTERNS[kind] * 2^-5 and whose normalised copy keeps them bit for
    bit (prep_qhat(q) == q there); N_BALLAST elements make |q| = 1; the last `n_zero` elements are exactly 0.
    Returns (q, pattern element mask)."""
    rng = np.random.default_rng(seed)
    pat = PATTERNS[kind]
    n_pat = D - N_BALLAST - n_zero
    signs = rng.choice(np.array([-1.0, 1.0], np.float32), D)
    q = np.zeros(D, np.float32)
    q[:n_pat] = signs[:n_pat] * pat * AMP
    s = float(canon_sqnorm(q[None])[0])
    q[n_pat:n_pat + N_BALLAST] = signs[n_pat:n_pat + N_BALLAST] * np.float32(np.sqrt((1.0 - s) / N_BALLAST))
    mask = np.zeros(D, bool)
    mask[:n_pat] = True
    qh, _ = prep_qhat(q)
    assert np.array_equal(qh[mask].view(np.uint32), q[mask].view(np.uint32)), "normalisation moved the pattern"
    return q, mask


def balanced_signs(q, seed=0):
    """+-1 per element such that sum s_i q_i^2 is as close to 0 as a greedy split gets (q_i^2 sorted descending)."""
    rng = np.random.default_rng(seed)
    sq = q.astype(np.float64) ** 2
    s = np.ones(D, np.float32)
    acc = 0.0
    for i in np.argsort(-sq + rng.uniform(0, 1e-30, D)):
        s[i] = -1.0 if acc > 0 else 1.0
        acc += s[i] * sq[i]
    return s


def adversarial_rows(q, seed=0):
    """Input rows for the query q: parallel (the query itself: cos ~ 1, every product positive), antiparallel
    (cos ~ -1, every product negative) and balanced-sign (|x_i| = |q_i|, sum |x_i q^_i| = 1, cos ~ 0)."""
    return {"parallel": q.copy(), "antiparallel": -q, "balanced": q * balanced_signs(q, seed)}


def emulated_coarse_error(kind, dtype, seed=0, mode=TF32_MODE):
    """CPU-emulated |coarse - cos| of the parallel row for the construction `kind` on a `dtype` table (operand
    conversion only).  For the worst pattern of each conversion this is >= 1.9e-3."""
    q, _ = adversarial_query(kind, seed)
    qh, _ = prep_qhat(q)
    x = stored(q, dtype)
    return float(abs(coarse_conversion_only(x, qh, dtype, mode)[0] - cosine(x, q)[0]))


# ------------------------------------------------------------------------------------------- rank inversions
def zero_positions(q):
    return np.nonzero(np.asarray(q) == 0)[0]


def with_zero_value(w, q):
    """The winner as stored: its elements at the query's zero positions set to ZV (bf16-exact values elsewhere are
    the caller's business)."""
    w = np.asarray(w, np.float32).copy()
    w[zero_positions(q)] = ZV
    return w


def decoy_rows(w, q, n):
    """n decoys for winner w (stored values, w == ZV at the query's zero positions): decoy j raises zero position
    Z[j % |Z|] by (1 + j // |Z|) * STEP.  The products x_i q^_i are those of w, so every scan computes the same dot,
    and the decoys are kept only where the emulated row scale equals w's -- so fast and coarse scores equal w's bit
    for bit; |x|^2 is strictly larger, so the canonical distance is strictly worse (cos > 0 required)."""
    Z = zero_positions(q)
    assert len(Z) > 0 and np.all(w[Z] == ZV)
    sw = row_scale(w[None])[0]
    out = []
    j = 0
    while len(out) < n:
        m = 1 + j // len(Z)
        assert m < 128, "not enough decoys with the winner's scale"
        d = w.copy()
        d[Z[j % len(Z)]] = ZV + np.float32(m) * STEP
        if row_scale(d[None])[0] == sw:
            out.append(d)
        j += 1
    return np.stack(out)


def bf16_exact(x):
    """x rounded to bf16 (values as fp32), so that a row is stored verbatim by either table dtype."""
    return bf16_rne(np.asarray(x, np.float32))


def inversion_case(dtype, n_zero=64, seed=0):
    """(q, w) for a rank-inversion table on a `dtype` table: q the worst-conversion query of that dtype with `n_zero`
    exact zeros, w the parallel row (stored form, ZV at the zeros).  The coarse score of w underestimates its cosine by
    ~1.8e-3, and the seed is advanced until the emulated GEMV fast score also UNDERestimates it, so that a proof bound
    without its + eps would accept a decoy as the k-th on every scan."""
    for s in range(seed, seed + 64):
        q, _ = adversarial_query(WORST[dtype], s, n_zero)
        w = with_zero_value(stored(q, dtype)[0], q)
        if dtype == "bf16":
            w = bf16_exact(w)
        qh, _ = prep_qhat(q)
        if cosine(w[None], q)[0] - gemv_fast(w[None], qh, dtype)[0] > 1e-8:
            return q, w
    raise AssertionError("no seed gives an underestimating fast score")


def import_stored(ix, ids, rows):
    """Append rows to an index VERBATIM in its dtype (orx_import_rows: no re-normalisation), so that a test controls
    the stored bits; `rows` are the stored values as fp32 (bf16-exact for a bf16 index)."""
    import ctypes as C
    from outline_rag_b200 import _lib
    rows = np.ascontiguousarray(rows, np.float32).reshape(-1, D)
    if ix.dtype == "bf16":
        assert np.array_equal(bf16_exact(rows), rows)
        raw = np.ascontiguousarray((rows.view(np.uint32) >> 16).astype(np.uint16))
    else:
        raw = rows
    ids = np.ascontiguousarray(ids, np.uint64).reshape(-1, 2)
    assert ids.shape[0] == rows.shape[0]
    _lib.check(_lib.lib.orx_import_rows(ix._h, C.c_void_p(ids.ctypes.data), C.c_void_p(raw.ctypes.data), rows.shape[0]))


# ------------------------------------------------------------------- inversions that only the image's eps can catch
# The rank inversions above tie the winner's score bit for bit, so ANY positive eps fails their proof.  These make the
# proof depend on the size of eps: the winner w's image score lies `deficit` below its cosine; k "strong" decoys are
# exact in the image (score == cosine to ~1e-6) at cosines a little below w's; more fillers than a candidate list holds
# score just above w, so w is not listed.  finalize then proves the decoys with any eps below the path's own (a wrong
# answer) and fails with the path's eps (the exact fallback answers w first).
EPS_UMMA = 2.5e-3                     # csrc/internal.h EPS_UMMA_TF32 / EPS_UMMA_BF16: the next bound below EPS_GEMV_IMAGE


def proof_holds(scores, cos, k, K, eps):
    """finalize's completeness proof (finalize.cu, GEMV scan) on emulated fast scores and exact cosines of every row:
    the list is the K best scores; cut = s_k - 2 eps - 1e-6 drops listed rows from the rescore; the proof holds iff the
    k-th best rescored cosine exceeds max(s_K, cut) + eps.  Returns (holds, listed rows)."""
    s = np.asarray(scores, np.float32)
    order = np.lexsort((np.arange(len(s)), -s.astype(np.float64)))
    top = order[:K]
    cut = np.float32(s[top[k - 1]] - np.float32(2.0 * eps + 1e-6))
    resc = top[s[top] > cut]
    cos_k = np.sort(np.asarray(cos, np.float64)[resc])[::-1][k - 1]
    return bool(cos_k > max(float(s[top[-1]]), float(cut)) + eps), top


def _toward(qh, c, rng):
    """a random direction at cosine ~c to the unit vector qh (float64)"""
    n = rng.standard_normal(D)
    n -= (n @ qh) * qh
    return c * qh + np.sqrt(1.0 - c * c) * n / np.linalg.norm(n)


def _exact_rows(q, score, lo, hi, n, rng, make):
    """n rows `make(direction)` whose score (`score(rows)`) lies in [lo, hi]: drawn at the band's centre, kept if in"""
    qh = q.astype(np.float64) / np.linalg.norm(q.astype(np.float64))
    out = []
    for _ in range(200):
        cand = np.stack([make(_toward(qh, (lo + hi) / 2, rng)) for _ in range(4 * n)])
        s = score(cand)
        out += list(cand[(s >= lo) & (s <= hi)])
        if len(out) >= n:
            return np.stack(out[:n])
    raise AssertionError("band too narrow")


def image8_inversion(k, seed=0, n_fillers=200, n_bulk=5000):
    """(rows, q, w_row) for the 8-bit image: w = 2^-7 (X + f) with integer X (one element 127, the rest +-20..45) and
    |f_i| = 0.484375 (just under half a step, so X is its 8-bit image) -- a relative residual ~0.0150, just under R8_CAP;
    q = w^ + t f^ leans on that residual so that w's 8-bit score is ~1.25e-2 below its cosine.  Decoys and fillers are
    2^-7 times integer vectors with max 127: their own image."""
    from tests.test_image8_scan import image8_scores
    rng = np.random.default_rng(seed)
    X = rng.integers(20, 46, D) * rng.choice([-1, 1], D)
    X[0] = 127
    f = np.float32(0.5 - 2.0 ** -6) * rng.choice([-1.0, 1.0], D).astype(np.float32)
    f[0] = 0
    w = ((X + f) * 2.0 ** -7).astype(np.float32)
    wh = w.astype(np.float64) / np.linalg.norm(w.astype(np.float64))
    fh = f.astype(np.float64) / np.linalg.norm(f.astype(np.float64))
    q = (wh + 1.5 * fh).astype(np.float32)
    cw = float(cosine(w[None], q)[0])
    sw = float(image8_scores(w[None], q)[0])

    def exact(v):
        return (np.rint(v * (127 / np.abs(v).max())) * 2.0 ** -7).astype(np.float32)

    def score(rows):
        return image8_scores(rows, q)
    dec = _exact_rows(q, score, cw - 0.0045, cw - 0.0035, k, rng, exact)
    fil = _exact_rows(q, score, sw + 0.0003, sw + 0.0015, n_fillers, rng, exact)
    bulk = rng.standard_normal((n_bulk, D)).astype(np.float32)
    rows = np.concatenate([dec, fil, bulk, w[None]]).astype(np.float32)   # the winner is the LAST row
    return rows, q, w


def image_inversion(k, seed=0, n_fillers=100, n_bulk=5000):
    """(rows, q, w_row) for the bf16 image: every element of w is +-(1 + 2^-8) 2^e, the RNE tie that rounds down to the
    even neighbour, so w's image is w / (1 + 2^-8) and its image score ~3.7e-3 below a cosine of ~0.95; decoys and
    fillers are bf16-exact rows (their own image)."""
    rng = np.random.default_rng(seed)
    w = (np.float32(1 + 2.0 ** -8) * np.float32(2.0) ** rng.integers(-7, -3, D).astype(np.float32)
         * rng.choice([-1.0, 1.0], D).astype(np.float32)).astype(np.float32)
    wh = w.astype(np.float64) / np.linalg.norm(w.astype(np.float64))
    q = _toward(wh, 0.95, rng).astype(np.float32)
    qh, _ = prep_qhat(q)
    cw = float(cosine(w[None], q)[0])
    sw = float(gemv_fast(w[None], qh, "fp32", image=True)[0])

    def exact(v):
        return bf16_exact(v * (0.1 / np.abs(v).max()))

    def score(rows):
        return gemv_fast(rows, qh, "fp32", image=True)
    dec = _exact_rows(q, score, cw - 0.0006, cw - 0.0002, k, rng, exact)
    fil = _exact_rows(q, score, sw + 0.00005, sw + 0.0002, n_fillers, rng, exact)
    bulk = rng.standard_normal((n_bulk, D)).astype(np.float32)
    rows = np.concatenate([dec, fil, bulk, w[None]]).astype(np.float32)
    return rows, q, w
