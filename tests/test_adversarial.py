"""CPU pins of the adversarial constructions and emulations in tests/adversarial.py (the GPU tests that use them:
test_epsilon_adversarial_gpu.py, test_completeness_gpu.py)."""
import numpy as np
import pytest

from tests import adversarial as A


@pytest.mark.parametrize("kind", sorted(A.PATTERNS))
def test_normalised_query_keeps_the_pattern_bits(kind):
    for n_zero in (0, 64):
        q, mask = A.adversarial_query(kind, seed=3, n_zero=n_zero)
        qh, qh16 = A.prep_qhat(q)
        assert np.array_equal(qh[mask].view(np.uint32), q[mask].view(np.uint32))
        assert mask.sum() == A.D - A.N_BALLAST - n_zero
        assert (q[A.D - n_zero:] == 0).all() and (qh[A.D - n_zero:] == 0).all()
        assert abs(float(np.sum(qh.astype(np.float64) ** 2)) - 1.0) < 1e-6
        # the pattern sits just below a rounding boundary of its conversion: it loses the most it can
        p = A.PATTERNS[kind]
        img = {"tf32_trunc": A.tf32_trunc, "tf32_rn": A.tf32_rn, "bf16": A.bf16_rne}[kind](np.array([p], np.float32))
        assert img[0] == 1.0


def test_prep_qhat_rounds_like_the_kernel():
    rng = np.random.default_rng(0)
    q = (rng.standard_normal(1024) * 3).astype(np.float32)
    qh, qh16 = A.prep_qhat(q)
    inv = 1.0 / np.sqrt(np.sum(q.astype(np.float64) ** 2))
    assert np.max(np.abs(qh.astype(np.float64) - q * inv)) <= 2.0 ** -24 * np.max(np.abs(qh))
    assert np.array_equal(qh16, A.bf16_rne(qh))


@pytest.mark.parametrize("kind,dtype,mode,least", [
    ("tf32_trunc", "fp32", "trunc", 1.9e-3),     # both operands lose 2^-10
    ("bf16", "bf16", "trunc", 1.9e-3),           # the query operand loses 2^-9 (rows are exact bf16)
    ("tf32_rn", "fp32", "rn", 0.9e-3),           # rounding to nearest loses at most half as much
])
def test_emulated_worst_case_conversion_error(kind, dtype, mode, least):
    assert A.emulated_coarse_error(kind, dtype, mode=mode) >= least
    # the truncation pattern is harmless under rounding, and vice versa it is not the worst
    if kind == "tf32_trunc":
        assert A.emulated_coarse_error(kind, dtype, mode="rn") < 1e-5


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_antiparallel_and_balanced_rows(dtype):
    q, _ = A.adversarial_query(A.WORST[dtype], 1)
    qh, _ = A.prep_qhat(q)
    rows = A.adversarial_rows(q, 1)
    x = A.stored(np.stack([rows["parallel"], rows["antiparallel"], rows["balanced"]]), dtype)
    cos = A.cosine(x, q)
    assert cos[0] > 0.999 and cos[1] < -0.999 and abs(cos[2]) < 1e-3
    # sum |x_i q^_i| = 1 for the balanced row: maximal magnitude, (almost) no signal
    assert abs(float(np.sum(np.abs(rows["balanced"].astype(np.float64) * qh))) - 1.0) < 1e-6
    err = np.abs(A.coarse_conversion_only(x, qh, dtype) - cos)
    assert err[0] >= 1.9e-3 and err[1] >= 1.9e-3


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_gemv_emulation_is_within_epsilon(dtype):
    rng = np.random.default_rng(2)
    X = A.stored(rng.standard_normal((512, 1024)).astype(np.float32), dtype)
    q = rng.standard_normal(1024).astype(np.float32)
    qh, _ = A.prep_qhat(q)
    err = np.abs(A.gemv_fast(X, qh, dtype) - A.cosine(X, q))
    assert 0 < err.max() < 3e-6


def test_row_scale_band_and_markers():
    u = np.full((1, 1024), 1.0 / 32, np.float32)             # |u| = 1
    assert A.row_scale(u)[0] == 1.0
    assert A.row_scale(np.zeros((1, 1024), np.float32))[0] != A.row_scale(np.zeros((1, 1024), np.float32))[0]
    big_in, big_out = u * np.float32(2.0 ** 39.99), u * np.float32(2.0 ** 40.01)
    small_in, small_out = u * np.float32(2.0 ** -39.99), u * np.float32(2.0 ** -40.01)
    assert np.isfinite(A.row_scale(big_in)[0]) and np.isfinite(A.row_scale(small_in)[0])
    assert A.row_scale(big_out)[0] == np.inf and A.row_scale(small_out)[0] == np.inf


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_decoys_tie_the_winner_and_lose_canonically(dtype):
    q, w = A.inversion_case(dtype)
    qh, _ = A.prep_qhat(q)
    d = A.decoy_rows(w, q, 200)
    rows = np.vstack([w[None], d])
    if dtype == "bf16":
        assert np.array_equal(A.bf16_exact(rows), rows)       # stored verbatim by a bf16 table
    f = A.gemv_fast(rows, qh, dtype)
    c = A.coarse_conversion_only(rows, qh, dtype)
    assert (f == f[0]).all() and (c == c[0]).all() and (A.row_scale(rows) == A.row_scale(w[None])[0]).all()
    cos = A.cosine(rows, q)
    assert (cos[1:] < cos[0]).all()
    # the premise of the inversion tests: every decoy's cosine is above the (tied) scores, so only the + eps of the
    # proof bound keeps the proof from accepting a decoy list
    assert cos[1:].min() > f[0] and cos[1:].min() - c[0] > 1.5e-3
