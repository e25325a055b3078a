"""CPU side of the bf16 image of fp32 tables (DESIGN.md section 2, "bf16 image"): the rounding facts the error bound
EPS_GEMV_IMAGE rests on, checked exhaustively over fp32 significands; the worst-case construction of
tests/test_image_scan_gpu.py reaching the bound in emulation; the constants of csrc/internal.h, include/orx.h and the
Python binding agreeing with each other."""
import os
import re

import numpy as np

from tests._helpers import bf16_rne

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _read(rel):
    with open(os.path.join(ROOT, rel)) as f:
        return f.read()


def _constexpr(name):
    m = re.search(rf"constexpr\s+\w+\s+{name}\s*=\s*([^;]+);", _read("outline_rag_b200/csrc/internal.h"))
    assert m, name
    return eval(m.group(1).replace("ull", ""))          # literals only: 3.92e-3, 1ull << 20


def _bf16(x):
    return bf16_rne(np.asarray(x, np.float32)).astype(np.float64)


def test_rne_to_bf16_is_within_2_to_minus_8_relative_for_every_normal_significand():
    x = (np.arange(1 << 23, dtype=np.uint32) | np.uint32(127 << 23)).view(np.float32)     # [1, 2): every significand
    rel = np.abs(_bf16(x) - x.astype(np.float64)) / x.astype(np.float64)
    assert rel.max() < 2.0 ** -8
    worst = x[np.argmax(rel)]
    assert worst == np.float32(1 + 2.0 ** -8)               # the tie, rounded to even: the construction's element
    big = (np.arange(0, 1 << 23, 4099, dtype=np.uint32) | np.uint32(254 << 23)).view(np.float32)   # top binade
    assert np.isfinite(_bf16(big[big < np.float32(3.3e38)])).all()


def test_subnormal_elements_err_by_at_most_half_a_bf16_subnormal_ulp():
    x = np.arange(1, 1 << 23, 97, dtype=np.uint32).view(np.float32)                       # fp32 subnormals
    err = np.abs(_bf16(x) - x.astype(np.float64))
    assert err.max() <= 2.0 ** -134


def test_eps_covers_the_derivation_and_the_worst_case_comes_close():
    eps_img, eps_bf16 = _constexpr("EPS_GEMV_IMAGE"), _constexpr("EPS_GEMV_BF16")
    assert eps_img >= 2.0 ** -8 * (1 + 2.0 ** -20) + eps_bf16 * (1 + 2.0 ** -8)
    assert eps_img < 2.0 ** -8 * 1.01                                  # no accidental slack
    from tests import adversarial as A
    from tests.test_image_scan_gpu import EPS_GEMV_IMAGE, _worst_query
    assert EPS_GEMV_IMAGE == eps_img
    for seed in range(3):
        q = _worst_query(seed)
        qh, _ = A.prep_qhat(q)
        x = q.astype(np.float64)
        err = abs(float(qh.astype(np.float64) @ (_bf16(q) - x)) / np.linalg.norm(x))
        assert 0.95 * 2.0 ** -8 < err < 2.0 ** -8


def test_option_and_debug_hook_are_declared_and_bound():
    from outline_rag_b200 import _lib
    h = _read("include/orx.h")
    m = re.search(r"#define ORX_OPT_IMAGE_MIN_ROWS (\d+)", h)
    assert m and int(m.group(1)) == _lib.ORX_OPT_IMAGE_MIN_ROWS != _lib.ORX_OPT_SCAN_TIMING
    assert "int orx_debug_image_scores(" in h and "orx_debug_image_scores" in _lib.SIGNATURES
    assert _constexpr("IMAGE_MIN_ROWS") == 1 << 20


def test_eps_carries_the_answer_of_the_bf16_image_inversion():
    """The construction of tests/test_image_property_gpu.py (adversarial.image_inversion): finalize's proof over the
    emulated image scores must FAIL with EPS_GEMV_IMAGE and HOLD with the tensor pass's 2.5e-3 -- which would prove k
    decoys in place of the winner."""
    from tests import adversarial as A
    eps_img = _constexpr("EPS_GEMV_IMAGE")
    assert _constexpr("EPS_UMMA_TF32") == A.EPS_UMMA < eps_img
    for k in (1, 12):
        rows, q, w = A.image_inversion(k, seed=k)
        qh, _ = A.prep_qhat(q)
        s, cos = A.gemv_fast(rows, qh, "fp32", image=True), A.cosine(rows, q)
        n = len(rows)
        assert np.argmax(cos) == n - 1
        assert 3.5e-3 < cos[-1] - s[-1] < eps_img                       # the winner's score is far below its cosine
        assert np.abs(s[:k] - cos[:k]).max() < 1e-6                     # the decoys are their own image
        width = 32 * (2 if k <= 16 else 4)                              # image_slots_for_k
        assert np.sum(s > s[-1]) > width
        holds, top = A.proof_holds(s, cos, k, width, eps_img)
        assert not holds and n - 1 not in top
        holds, top = A.proof_holds(s, cos, k, width, A.EPS_UMMA)
        assert holds and set(range(k)) <= set(top.tolist())
