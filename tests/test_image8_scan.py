"""CPU side of the 8-bit image of large fp32 tables (DESIGN.md section 2, "8-bit image"): the rounding facts and the
integer range the error bound EPS_GEMV_IMAGE8 rests on, checked over every fp32 significand where it matters; the
bound against a float64 emulation of the scan's score on adversarial rows; the constants of csrc/internal.h, include/orx.h
and the Python binding agreeing with each other.

`quantise_rows` / `quantise_query` / `image8_scores` emulate the device code bit for bit (table_ops.cu quantise8_row,
finalize.cu prep_queries_kernel, scan_gemv.cu image8_dot): tests/test_image8_scan_gpu.py compares the device scores
against them."""
import os
import re

import numpy as np

from oracle import cosine_topk as O
from tests import adversarial as A

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _read(rel):
    with open(os.path.join(ROOT, rel)) as f:
        return f.read()


def _constexpr(name):
    m = re.search(rf"constexpr\s+\w+\s+{name}\s*=\s*([^;]+);", _read("outline_rag_b200/csrc/internal.h"))
    assert m, name
    return eval(m.group(1).replace("ull", ""))          # literals only: 1.662e-2, 1.0 / 64, 1ull << 22


R8_CAP = 1.0 / 64
EPS_GEMV_IMAGE8 = 1.662e-2
N2_LO, N2_HI = 8.271806125530277e-25, 1.2089258196146292e24       # the regular band of table_ops.cu scale_from_n2


def quantise_rows(rows):
    """(X int8 [n, 1024], scale8 fp32 [n], residual float64 [n]) as the commit kernel stores them"""
    x = np.asarray(rows, np.float32).reshape(-1, 1024)
    n2 = O.canon_sqnorm(x)
    regular = (n2 >= N2_LO) & (n2 <= N2_HI)
    d = (np.abs(x).max(1) / np.float32(127)).astype(np.float32)
    with np.errstate(divide="ignore", invalid="ignore"):
        X = np.where(regular[:, None], np.rint((x / d[:, None]).astype(np.float32)), 0).astype(np.int64)
    X8 = X.astype(np.int8)                                       # what the store keeps (no clamp: the residual sees it)
    e = x.astype(np.float64) - d[:, None].astype(np.float64) * X8.astype(np.float64)
    e2 = (e ** 2).sum(1)
    with np.errstate(divide="ignore", invalid="ignore"):
        resid = np.sqrt(e2 / n2)
        s8 = (d.astype(np.float64) / np.sqrt(n2)).astype(np.float32)
    capped = regular & ~(e2 * (1 + 2.0 ** -30) <= R8_CAP * R8_CAP * n2)
    s8 = np.where(capped, np.float32(np.inf), s8)
    s8 = np.where(~regular, np.where(n2 > 0, np.float32(np.inf), np.float32(np.nan)), s8).astype(np.float32)
    return X8, s8, resid


def quantise_query(q):
    """(Q int64 [1024], dq fp32, residual |qhat - dq Q| float64) as prep_queries_kernel makes them"""
    qh, _ = A.prep_qhat(np.asarray(q, np.float32))
    dq = np.float32(np.abs(qh).max() / np.float32(16383))
    Q = np.rint(qh.astype(np.float64) / np.float64(dq)).astype(np.int64) if dq > 0 else np.zeros(1024, np.int64)
    return Q, dq, float(np.sqrt(((qh.astype(np.float64) - np.float64(dq) * Q) ** 2).sum()))


def image8_scores(rows, q):
    """the 8-bit scan's score of every row: (float(D) * dq) * scale8, each product rounded to fp32"""
    X8, s8, _ = quantise_rows(rows)
    Q, dq, _ = quantise_query(q)
    h, l = Q >> 7, Q & 127
    D = 128 * (X8.astype(np.int64) @ h) + X8.astype(np.int64) @ l
    with np.errstate(invalid="ignore", over="ignore"):
        return ((D.astype(np.float32) * dq).astype(np.float32) * s8).astype(np.float32)


def test_row_quantiser_stays_within_int8_for_every_significand_of_the_largest_element():
    m = (np.arange(1 << 23, dtype=np.uint32) | np.uint32(127 << 23)).view(np.float32)     # [1, 2): every significand
    d = (m / np.float32(127)).astype(np.float32)
    X = np.rint((m / d).astype(np.float32))
    assert X.max() == 127 and X.min() == 127
    for e in (-45, 40):                                                                   # the regular band's edges
        me = (m * np.float32(2.0 ** e)).astype(np.float32)
        de = (me / np.float32(127)).astype(np.float32)
        assert np.isfinite(de).all() and (de > np.float32(1.2e-38)).all()                 # the step is a normal number
        assert np.rint((me / de).astype(np.float32)).max() == 127


def test_query_quantiser_split_and_integer_range():
    m = (np.arange(0, 1 << 23, 7, dtype=np.uint32) | np.uint32(122 << 23)).view(np.float32)   # max|qhat| in [2^-5, 2^-4)
    dq = (m / np.float32(16383)).astype(np.float32)
    assert np.rint(m.astype(np.float64) / dq.astype(np.float64)).max() == 16383
    Q = np.arange(-16383, 16384, dtype=np.int64)
    h, l = Q >> 7, Q & 127
    assert h.min() == -128 and h.max() == 127 and l.min() == 0 and l.max() == 127
    assert np.array_equal(128 * h + l, Q)
    assert 1024 * 128 * 16383 < 2 ** 31                    # |X| <= 128 even if a store wrapped: D never overflows
    for seed in range(8):
        q = np.random.default_rng(seed).standard_normal(1024).astype(np.float32)
        Qq, dq, rq = quantise_query(q)
        assert np.abs(Qq).max() == 16383
        assert rq <= 16 * float(dq) * (1 + 2.0 ** -30) <= 9.7662e-4


def test_eps_covers_the_derivation():
    eps, cap = _constexpr("EPS_GEMV_IMAGE8"), _constexpr("R8_CAP")
    assert (eps, cap) == (EPS_GEMV_IMAGE8, R8_CAP)
    rq_max = 16 / 16383 * (1 + 2.0 ** -22)                 # 16 dq, dq <= max|qhat| / 16383 (1 + 2^-24), |qhat| <= 1 + 2^-23
    rounding = (1 + cap) * (1 + rq_max) * 5 * 2.0 ** -24   # fp32 of D, two products, scale8 (+ its binary64 ops)
    assert eps >= cap + (1 + cap) * (rq_max + 6e-8) + rounding
    assert eps < cap + 1.1e-3                              # no accidental slack


def _adversarial_rows(rng):
    rows, names = [], []

    def add(name, r):
        rows.append(np.asarray(r, np.float32))
        names.append(name)
    base = rng.standard_normal((32, 1024)).astype(np.float32)
    for i, r in enumerate(base):
        add(f"gauss{i}", r)
    add("equal magnitudes", np.where(rng.random(1024) < 0.5, -1, 1).astype(np.float32) * np.float32(0.03125))
    dom = base[0] * np.float32(1e-3)                        # one dominant element: the rest rounds to 0 or +-1
    dom[17] = np.float32(1.0)
    add("one dominant", dom)
    half = np.full(1024, np.float32(0.5 / 127 * 1.0001))    # every element just above half a step of the max
    half[0] = np.float32(1.0)
    add("half steps", half)
    sub = rng.uniform(-1, 1, 1024).astype(np.float32) * np.float32(1e-39)   # subnormals beside one normal element
    sub[0] = np.float32(2.0 ** -30)
    add("subnormals", sub)
    unit = base[1] / np.float32(np.linalg.norm(base[1]))
    for s, name in ((2.0 ** -40 * 1.01, "low band edge"), (2.0 ** 40 * 0.99, "high band edge"),
                    (2.0 ** -40 * 0.99, "below the band"), (2.0 ** 40 * 1.01, "above the band")):
        add(name, unit * np.float32(s))
    add("zero", np.zeros(1024, np.float32))
    return np.stack(rows), names


def test_bound_holds_on_adversarial_rows_and_capped_rows_are_always_candidates():
    rng = np.random.default_rng(11)
    rows, names = _adversarial_rows(rng)
    X8, s8, resid = quantise_rows(rows)
    assert np.abs(X8.astype(np.int64)).max() <= 127
    idx = {n: i for i, n in enumerate(names)}
    assert resid[idx["equal magnitudes"]] < 2.0 ** -24         # every element is +-127 steps: only d rounds
    assert resid[idx["one dominant"]] > R8_CAP and s8[idx["one dominant"]] == np.inf      # capped: always a candidate
    assert resid[idx["half steps"]] > R8_CAP and s8[idx["half steps"]] == np.inf
    # subnormal elements lie below half a step: they round to 0 and their whole value is residual, which is negligible
    assert (X8[idx["subnormals"], 1:] == 0).all() and resid[idx["subnormals"]] < 2.0 ** -24 and np.isfinite(s8[idx["subnormals"]])
    for n in ("below the band", "above the band"):
        assert s8[idx[n]] == np.inf
    assert np.isnan(s8[idx["zero"]])
    ok = np.isfinite(s8)
    assert ok[idx["low band edge"]] and ok[idx["high band edge"]] and ok[idx["gauss0"]]
    assert (resid[ok] <= R8_CAP).all()
    worst = 0.0
    for seed in range(6):
        q = rng.standard_normal(1024).astype(np.float32)
        if seed == 0:
            q = rows[idx["gauss3"]].copy()                   # a query on a row: the largest cosine
        s = image8_scores(rows, q).astype(np.float64)
        cos = A.cosine(rows[ok], q)
        worst = max(worst, float(np.abs(s[ok] - cos).max()))
    assert worst <= EPS_GEMV_IMAGE8
    assert worst > 1e-4                                      # the emulation does quantise


def test_option_and_debug_hook_are_declared_and_bound():
    from outline_rag_b200 import _lib
    h = _read("include/orx.h")
    m = re.search(r"#define ORX_OPT_IMAGE8_MIN_ROWS (\d+)", h)
    assert m and int(m.group(1)) == _lib.ORX_OPT_IMAGE8_MIN_ROWS
    assert len({_lib.ORX_OPT_IMAGE8_MIN_ROWS, _lib.ORX_OPT_IMAGE_MIN_ROWS, _lib.ORX_OPT_SCAN_TIMING}) == 3
    assert "int orx_debug_image8_scores(" in h and "orx_debug_image8_scores" in _lib.SIGNATURES
    assert _constexpr("IMAGE8_MIN_ROWS") == 1 << 22
    assert _constexpr("IMAGE8_MAX_K") == 12 and _constexpr("IMAGE8_SLOTS") == 5
