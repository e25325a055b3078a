"""The premise of the completeness proof, |scan score - cosine| <= eps, measured where it is thin (DESIGN.md section 2).

* The operand conversion of the tensor-core pass is probed bit for bit (unit basis rows), so the worst case below is
  built for the conversion the hardware really applies.
* tcgen05 (both operand kinds, both kernels): queries whose normalised copy sits just below a rounding boundary of the
  conversion, rows parallel / antiparallel / sign-balanced to them, mixed into synthetic rows.  Asserted: max error <
  eps (what the proof needs) and >= 0.9 x the CPU-emulated conversion error (the construction really bites).
* GEMV (both table dtypes) through orx_debug_fast_scores, the exact value the GEMV scans key on: 1M synthetic rows and
  the adversarial rows, rows at the edges of the regular-norm band, one-dominant-element rows and queries with a large
  element dynamic range.  Asserted: 0 < max error < EPS_GEMV, and rows outside the band are never trusted (non-finite).
The maxima are printed and recorded in DESIGN.md section 2."""
import numpy as np
import pytest

from oracle import cosine_topk as O
from tests import adversarial as A

pytestmark = pytest.mark.gpu
EPS_UMMA = 2.5e-3            # csrc/internal.h EPS_UMMA_TF32 / EPS_UMMA_BF16
EPS_GEMV = 3.0e-6            # csrc/internal.h EPS_GEMV_F32 / EPS_GEMV_BF16


def _index(dtype, cap=0):
    import outline_rag_b200 as orx
    return orx.Index(dtype, cap, 0)


def _exported(ix, n):
    """The rows as stored, as float64 CUDA tensor [n, 1024], table order."""
    import torch
    rb = 4096 if ix.dtype == "fp32" else 2048
    ids = np.zeros((n, 2), np.uint64)
    raw = np.zeros((n, rb), np.uint8)
    ix.export_rows(0, n, ids, raw)
    if ix.dtype == "fp32":
        return torch.from_numpy(raw.view(np.float32)).cuda().double()
    return torch.from_numpy(raw.view(np.int16).astype(np.int32) << 16).cuda().view(torch.float32).double()


def _cos_ref(X64, Q):
    """plain float64 reference: [rows, nq] cosines"""
    import torch
    Q64 = torch.as_tensor(np.asarray(Q), dtype=torch.float64, device=X64.device)
    Q64 = Q64 / Q64.norm(dim=1, keepdim=True)
    return (X64 @ Q64.T) / X64.norm(dim=1, keepdim=True)


# ------------------------------------------------------------------------------------------ conversion probe
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_operand_conversion_mode(dtype):
    """Unit basis rows e_i: the fast score is q^_i itself (prep_qhat bit for bit) and the coarse score is the tensor
    core's image of q^_i -- truncation vs rounding of kind::tf32, RNE of the bf16 query."""
    Q = np.stack([A.adversarial_query(kind, 5)[0] for kind in sorted(A.PATTERNS)])
    qh, qh16 = A.prep_qhat(Q)
    E = np.eye(1024, dtype=np.float32)
    with _index(dtype) as ix:
        A.import_stored(ix, O.ids_arange(0, 1024), E)
        fast = ix.debug_fast_scores(Q).cpu().numpy()             # [row i, query] = q^_i
        coarse = ix.debug_coarse_scores(Q).cpu().numpy()
    assert np.array_equal(fast.T.view(np.uint32), qh.view(np.uint32)), "prep_qhat is not the kernel's q^"
    if dtype == "bf16":
        assert np.array_equal(coarse.T, qh16), "the bf16 query operand is not RNE of q^"
        return
    # exact ties of rounding (low 13 bits 0x1000) would not tell ties-away from ties-to-even: compare elsewhere
    no_tie = (qh.view(np.uint32) & 0x1FFF) != 0x1000
    trunc = np.array_equal(coarse.T[no_tie], A.tf32_trunc(qh)[no_tie])
    rn = np.array_equal(coarse.T[no_tie], A.tf32_rn(qh)[no_tie])
    mode = "trunc" if trunc else "rn" if rn else "neither"
    print(f"\nkind::tf32 query-operand conversion on this device: {mode}")
    assert mode == A.TF32_MODE, mode
    # the row operand: rows c * e_i with pattern values c, against q = (1/32, ..., 1/32) (q^ = 2^-5 exactly)
    c = np.concatenate([np.full(341, A.PATTERNS[k]) for k in sorted(A.PATTERNS)] + [np.ones(1)]).astype(np.float32)
    c *= np.random.default_rng(6).choice(np.array([-1.0, 1.0], np.float32), 1024)
    q = np.full((1, 1024), 1.0 / 32, np.float32)
    with _index(dtype) as ix:
        A.import_stored(ix, O.ids_arange(0, 1024), E * c[:, None])
        coarse = ix.debug_coarse_scores(q).cpu().numpy()[:, 0]
    sc = A.row_scale(E * c[:, None])
    want = {m: (A.to_tf32(c, m) * np.float32(1.0 / 32)).astype(np.float32) * sc for m in ("trunc", "rn")}
    row_mode = [m for m in ("trunc", "rn") if np.array_equal(coarse, want[m])]
    print(f"kind::tf32 row-operand conversion on this device: {row_mode}")
    assert row_mode == [A.TF32_MODE], row_mode


# ------------------------------------------------------------------------------------------ tcgen05 adversarial
N_SYN, NQ = 65_536, 256


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_adversarial_coarse_error_is_below_epsilon(dtype):
    import torch
    from orx_testkit.device import synth_rows_device
    from orx_testkit.synth import SEED_TABLE, default_centres
    Q = np.stack([A.adversarial_query(A.WORST[dtype], s)[0] for s in range(NQ)])
    adv = []
    for s in range(0, NQ, 8):                      # parallel / antiparallel / balanced rows of every 8th query
        r = A.adversarial_rows(Q[s], s)
        adv += [r["parallel"], r["antiparallel"], r["balanced"]]
    adv = np.stack(adv)
    emulated = max(A.emulated_coarse_error(A.WORST[dtype], dtype, s) for s in range(0, NQ, 8))
    n = N_SYN + len(adv)
    with _index(dtype, n) as ix:
        ix.upsert(O.ids_arange(0, N_SYN), synth_rows_device(0, SEED_TABLE, default_centres(N_SYN), 0, N_SYN))
        ix.upsert(O.ids_arange(N_SYN, n), adv)
        X64 = _exported(ix, n)
        cos = _cos_ref(X64, Q)
        worst = {}
        for pairs in (False, True):
            coarse = ix.debug_coarse_scores(torch.from_numpy(Q).cuda(), use_pairs=pairs).double()
            err = (coarse - cos).abs()
            worst["pairs" if pairs else "one_cta"] = (float(err[N_SYN:].max()), float(err[:N_SYN].max()))
    print(f"\nmax |coarse - cosine|, {dtype} table, {N_SYN} synthetic + {len(adv)} adversarial rows x {NQ} "
          f"worst-case queries ({A.WORST[dtype]}): (adversarial, synthetic) {worst}; emulated conversion "
          f"error {emulated:.3e}; eps {EPS_UMMA}")
    for adv_err, syn_err in worst.values():
        assert adv_err < EPS_UMMA and syn_err < EPS_UMMA
        assert adv_err >= 0.9 * emulated, "the worst case did not reach the device"


# ------------------------------------------------------------------------------------------------ GEMV
N_GEMV, NQ_GEMV = 1_000_000, 64


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_gemv_fast_error_on_a_million_rows(dtype):
    import torch
    from orx_testkit.device import synth_rows_device
    from orx_testkit.synth import SEED_TABLE, Synth, default_centres
    nc = default_centres(N_GEMV)
    Q = Synth(nc).queries(NQ_GEMV, N_GEMV)[0]
    with _index(dtype, N_GEMV) as ix:
        for s in range(0, N_GEMV, 262_144):
            m = min(262_144, N_GEMV - s)
            ix.upsert(O.ids_arange(s, s + m), synth_rows_device(0, SEED_TABLE, nc, s, m))
        fast = ix.debug_fast_scores(torch.from_numpy(Q).cuda())
        err = 0.0
        for s in range(0, N_GEMV, 131_072):
            m = min(131_072, N_GEMV - s)
            rb = 4096 if dtype == "fp32" else 2048
            ids = np.zeros((m, 2), np.uint64)
            raw = np.zeros((m, rb), np.uint8)
            ix.export_rows(s, m, ids, raw)
            X64 = (torch.from_numpy(raw.view(np.float32)).cuda().double() if dtype == "fp32" else
                   torch.from_numpy(raw.view(np.int16).astype(np.int32) << 16).cuda().view(torch.float32).double())
            err = max(err, float((fast[s:s + m].double() - _cos_ref(X64, Q)).abs().max()))
    print(f"\nmax |fast - cosine| over {N_GEMV} synthetic rows x {NQ_GEMV} queries, {dtype} table (GEMV): {err:.3e} "
          f"(eps {EPS_GEMV})")
    assert 0.0 < err < EPS_GEMV


def _gemv_adversarial_table(dtype):
    """(queries, stored rows, labels): worst-case-pattern and random unit queries, queries with elements over 2^-20 ..
    2^20; per query its own row, its negation and a sign-balanced row; one-dominant-element rows; rows at the edges of
    the regular band |x| in [2^-40, 2^40]."""
    rng = np.random.default_rng(11)
    Q = [A.adversarial_query(kind, s)[0] for kind in sorted(A.PATTERNS) for s in range(4)]
    Q += [rng.standard_normal(1024).astype(np.float32) for _ in range(8)]
    Q += [(rng.standard_normal(1024) * 2.0 ** rng.uniform(-20, 20, 1024)).astype(np.float32) for _ in range(8)]
    Q = np.stack(Q)
    rows, labels = [], []
    for i, q in enumerate(Q):
        for name, r in A.adversarial_rows(q, i).items():
            rows.append(A.stored(r, dtype)[0])
            labels.append(name)
    for i in range(32):                                      # one element carries almost all of the norm
        r = (rng.standard_normal(1024) * 1e-3).astype(np.float32)
        r[rng.integers(1024)] = np.float32(rng.choice([-1.0, 1.0]))
        rows.append(A.stored(r, dtype)[0])
        labels.append("dominant")
    u = np.where(rng.uniform(size=1024) < 0.5, -1.0, 1.0).astype(np.float32) / 32          # |u| = 1
    for c, name in ((2.0 ** 40 * (1 - 2.0 ** -8), "band_in"), (2.0 ** -40 * (1 + 2.0 ** -7), "band_in"),
                    (2.0 ** 40 * (1 + 2.0 ** -7), "band_out"), (2.0 ** -40 * (1 - 2.0 ** -8), "band_out")):
        rows.append((u * np.float32(c)).astype(np.float32))                                  # bf16-exact, stored as is
        labels.append(name)
    return Q, np.stack(rows), np.array(labels)


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_gemv_fast_error_on_adversarial_rows(dtype):
    Q, X, labels = _gemv_adversarial_table(dtype)
    with _index(dtype) as ix:
        A.import_stored(ix, O.ids_arange(0, len(X)), X)
        fast = ix.debug_fast_scores(Q).cpu().numpy().astype(np.float64)        # [rows, queries]
    cos = np.stack([A.cosine(X, q) for q in Q], axis=1)
    out = labels == "band_out"
    assert not np.isfinite(fast[out]).any(), "a row outside the regular band got a trusted score"
    assert np.isfinite(fast[~out]).all()
    # the emulation of the GEMV arithmetic agrees with the device where it is exact
    for j in range(4):
        qh, _ = A.prep_qhat(Q[j])
        assert np.array_equal(A.gemv_fast(X[~out], qh, dtype), fast[~out, j].astype(np.float32))
    err = np.abs(fast[~out] - cos[~out])
    per = {name: float(err[labels[~out] == name].max()) for name in sorted(set(labels[~out]))}
    print(f"\nmax |fast - cosine|, {dtype} table (GEMV), adversarial rows x {len(Q)} queries: {per} (eps {EPS_GEMV})")
    assert 0.0 < err.max() < EPS_GEMV, per
