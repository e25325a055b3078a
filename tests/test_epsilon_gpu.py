"""The completeness proof of the tcgen05 batch scan assumes |coarse score - cosine| <= eps for EVERY row
(csrc/internal.h: EPS_UMMA_TF32 = EPS_UMMA_BF16 = 2.5e-3).  This test MEASURES the left-hand side: the coarse scores of
all 1M rows x 256 queries come out of the very TMA / tcgen05.mma / TMEM pipeline the search runs
(`orx_debug_coarse_scores`: only the epilogue differs -- it writes instead of selecting), for both operand kinds (tf32
on fp32 tables, bf16 on bf16 tables) and both kernels (one CTA per tile, CTA pairs); the reference cosine is a plain
PyTorch float64 matmul on the rows as stored.  Asserted: max error < eps / 2.  The measured maxima are printed and
recorded in DESIGN.md section 2.  This is the benign corpus: the worst-case inputs of both scans, and the GEMV scan's
eps, are measured in tests/test_epsilon_adversarial_gpu.py."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
EPS_UMMA = 2.5e-3            # csrc/internal.h
N, NQ = 1_000_000, 256


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_measured_coarse_error_is_below_half_epsilon(dtype):
    import torch
    import outline_rag_b200 as orx
    from orx_testkit.device import synth_rows_device
    from orx_testkit.synth import SEED_TABLE, Synth, default_centres
    nc = default_centres(N)
    Q = torch.from_numpy(Synth(nc).queries(NQ, N)[0]).cuda()
    with orx.Index(dtype, N, 0) as ix:
        for s in range(0, N, 262_144):
            m = min(262_144, N - s)
            ids = np.zeros((m, 2), np.uint64)
            ids[:, 1] = np.arange(s, s + m, dtype=np.uint64)
            ix.upsert(ids, synth_rows_device(0, SEED_TABLE, nc, s, m))
        # the rows AS STORED (fp32 verbatim / bf16 of the normalised row), in table order
        rb = 4096 if dtype == "fp32" else 2048
        Q64 = Q.double()
        Q64 = Q64 / Q64.norm(dim=1, keepdim=True)
        worst = {}
        for pairs in (False, True):
            coarse = ix.debug_coarse_scores(Q, use_pairs=pairs)              # [N, NQ] fp32 on the device
            assert coarse.shape == (N, NQ)
            err = 0.0
            for s in range(0, N, 131_072):
                m = min(131_072, N - s)
                e_ids = np.zeros((m, 2), np.uint64)
                raw = np.zeros((m, rb), np.uint8)
                ix.export_rows(s, m, e_ids, raw)
                assert (e_ids[:, 1] == np.arange(s, s + m, dtype=np.uint64)).all()      # table order = insertion order
                if dtype == "fp32":
                    X = torch.from_numpy(raw.view(np.float32)).cuda().double()
                else:
                    X = torch.from_numpy(raw.view(np.int16).astype(np.int32) << 16).cuda().view(torch.float32).double()
                cos = (X @ Q64.T) / X.norm(dim=1, keepdim=True)             # plain float64 reference of the same op
                err = max(err, float((coarse[s:s + m].double() - cos).abs().max()))
            worst["pairs" if pairs else "one_cta"] = err
        print(f"\nmax |coarse - cosine| over {N} rows x {NQ} queries, {dtype} table "
              f"({'tf32' if dtype == 'fp32' else 'bf16'} operands): {worst}  (eps = {EPS_UMMA})")
        assert max(worst.values()) < EPS_UMMA / 2, worst
        assert min(worst.values()) > 0.0          # the dump is really the tensor-core result, not the reference
