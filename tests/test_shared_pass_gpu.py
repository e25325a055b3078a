"""Two single-query searches in flight over the 8-bit image share one pass (DESIGN.md section 4): whenever the second
joins the first's lap -- at once, mid-lap, after it or never -- each answer equals the same query searched alone and the
fp32-rows scan, bit for bit, with no fallback (a lap that missed a row would leave its query unproven); writes between
tickets keep their order; the adversarial 8-bit construction still returns the oracle's answer through a joined search."""
import time

import numpy as np
import pytest

from oracle import cosine_topk as O
from tests import adversarial as A

pytestmark = pytest.mark.gpu
N = 1 << 22
K = 12


def _lib():
    from outline_rag_b200 import _lib as L
    return L


@pytest.fixture(scope="module")
def big():
    import torch
    import outline_rag_b200 as orx
    from orx_testkit.device import synth_rows_device
    from orx_testkit.synth import SEED_TABLE, Synth, default_centres
    nc = default_centres(N)
    ix = orx.Index("fp32", N, 0)
    chunk = 1 << 18
    buf = torch.empty((chunk, 1024), dtype=torch.float32, device="cuda:0")
    for s in range(0, N, chunk):
        synth_rows_device(0, SEED_TABLE, nc, s, chunk, out=buf)
        ix.upsert(O.ids_arange(s, s + chunk), buf)
    torch.cuda.synchronize()
    del buf
    Q, _ = Synth(nc).queries(8, N)
    Qd = torch.from_numpy(Q).cuda()
    want = []
    for q in Q:
        got = ix.search(q[None], K)
        assert ix.stats()["last_path"] == 4
        want.append(got)
    ix.set_option(_lib().ORX_OPT_IMAGE_MIN_ROWS, -1)                    # the fp32 rows, same table
    for q, w in zip(Q, want):
        assert _same(ix.search(q[None], K), w)
    ix.set_option(_lib().ORX_OPT_IMAGE_MIN_ROWS, 1 << 20)
    yield ix, Qd, want
    ix.close()


def _same(a, b):
    return (np.array_equal(a[0], b[0]) and np.array_equal(a[1].view(np.uint64), b[1].view(np.uint64))
            and np.array_equal(a[2], b[2]))


def _out(k=K):
    import torch
    return (torch.empty((1, k, 2), dtype=torch.int64, device="cuda:0"),
            torch.empty((1, k), dtype=torch.float64, device="cuda:0"),
            torch.empty((1,), dtype=torch.int32, device="cuda:0"))


def _host(out):
    return out[0].cpu().numpy().view(np.uint64), out[1].cpu().numpy(), out[2].cpu().numpy()


@pytest.mark.parametrize("gap_s", [0.0, 0.0005, 0.05, None])
def test_pair_equals_each_query_alone(big, gap_s):
    """gap_s: seconds between the two submits -- 0 joins at once, 0.5 ms mid-lap, 50 ms after the lap; None waits for
    the first before submitting the second"""
    ix, Q, want = big
    st0 = ix.stats()
    for i in range(0, 8, 2):
        oa, ob = _out(), _out()
        ta = ix.search_submit(Q[i:i + 1], K, oa)
        if gap_s is None:
            ix.search_wait(ta)
        elif gap_s:
            time.sleep(gap_s)
        tb = ix.search_submit(Q[i + 1:i + 2], K, ob)
        if gap_s is not None:
            ix.search_wait(ta)
        ix.search_wait(tb)
        assert ix.stats()["last_path"] == 4
        assert _same(_host(oa), want[i]) and _same(_host(ob), want[i + 1]), (i, gap_s)
    st1 = ix.stats()
    assert st1["fallback_exhaustive"] == st0["fallback_exhaustive"]
    if gap_s == 0.0:
        assert st1["shared_scans"] > st0["shared_scans"]
    if gap_s is None:
        assert st1["shared_scans"] == st0["shared_scans"]


def test_pipeline_of_two_in_flight_shares_and_stays_exact(big):
    ix, Q, want = big
    st0 = ix.stats()
    outs = [_out() for _ in range(3)]
    tickets, order = [], []
    for step in range(24):
        i = step % 8
        tickets.append(ix.search_submit(Q[i:i + 1], K, outs[step % 3]))
        order.append(i)
        if len(tickets) == 2:
            ix.search_wait(tickets.pop(0))
            j = order.pop(0)
            assert _same(_host(outs[(step - 1) % 3]), want[j]), step
    ix.search_wait(tickets.pop(0))
    assert _same(_host(outs[23 % 3]), want[order.pop(0)])
    st1 = ix.stats()
    assert st1["shared_scans"] > st0["shared_scans"] and st1["shared_rows"] > st0["shared_rows"]
    assert st1["fallback_exhaustive"] == st0["fallback_exhaustive"]


def test_a_write_between_tickets_settles_both_in_order(big):
    """the upsert rewrites rows with their own values: every answer stays the same, and both tickets are complete
    before it touches the table"""
    import torch
    ix, Q, want = big
    ids = O.ids_arange(100, 104)
    rows = torch.from_numpy(ix.fetch(ids)[0]).cuda()
    oa, ob = _out(), _out()
    ta = ix.search_submit(Q[0:1], K, oa)
    tb = ix.search_submit(Q[1:2], K, ob)
    ix.upsert(ids, rows)
    ix.search_wait(ta)
    ix.search_wait(tb)
    assert _same(_host(oa), want[0]) and _same(_host(ob), want[1])
    oc = _out()
    tc = ix.search_submit(Q[2:3], K, oc)
    ix.search_wait(tc)
    assert _same(_host(oc), want[2])


def test_adversarial_inversion_through_a_joined_search():
    """adversarial.image8_inversion (the winner's 8-bit score ~1.2e-2 below its cosine) padded with 4M rows near -q, so
    that the lap lasts long enough to be joined; the second search is a different query (the strongest decoy's row).
    Both answers equal the oracle's on the construction, and the pad is shown unable to enter either top-k."""
    import torch
    import outline_rag_b200 as orx
    L = _lib()
    rows, q, _ = A.image8_inversion(K, seed=3)
    n = len(rows)
    ids = O.ids_arange(0, n)
    cos = A.cosine(rows, q)
    q2 = rows[np.argsort(-cos)[1]].astype(np.float32)                 # a decoy row, not the winner
    want = [O.topk_exact(rows, ids, qq, K) for qq in (q, q2)]
    pad_n, chunk = 1 << 22, 1 << 18
    gen = torch.Generator(device="cuda:0").manual_seed(7)
    qd = torch.from_numpy(np.ascontiguousarray(np.stack([q, q2]), dtype=np.float32)).cuda()
    qh = qd / qd.norm(dim=1, keepdim=True)
    with orx.Index("fp32", n + pad_n, 0) as ix:
        ix.set_option(L.ORX_OPT_IMAGE8_MIN_ROWS, 0)
        ix.set_option(L.ORX_OPT_IMAGE_MIN_ROWS, 0)
        ix.upsert(ids, rows)
        worst = torch.full((2,), -2.0, dtype=torch.float64, device="cuda:0")
        for s in range(0, pad_n, chunk):
            pad = -qh[0] + 0.5 * torch.randn((chunk, 1024), generator=gen, device="cuda:0") / 32
            c = (pad.double() @ qh.double().T) / pad.double().norm(dim=1, keepdim=True)
            worst = torch.maximum(worst, c.max(dim=0).values)
            ix.upsert(O.ids_arange(n + s, n + s + chunk), pad)
        for j in range(2):                                            # the pad sorts after every row of the answer
            assert worst[j].item() < 1.0 - want[j][1][-1] - 0.05, (j, worst[j].item())
        st0 = ix.stats()
        for _ in range(3):
            oa, ob = _out(), _out()
            ta = ix.search_submit(qd[0:1], K, oa)
            tb = ix.search_submit(qd[1:2], K, ob)
            ix.search_wait(ta)
            ix.search_wait(tb)
            assert ix.stats()["last_path"] == 4
            for o, w in zip((oa, ob), want):
                got = _host(o)
                assert np.array_equal(got[0][0], w[0])
                assert np.array_equal(got[1][0].view(np.uint64), w[1].view(np.uint64))
        st1 = ix.stats()
        assert st1["shared_scans"] > st0["shared_scans"] and st1["shared_rows"] > st0["shared_rows"]
