"""CPU oracle of exact maximal-marginal-relevance search (``orx_search_mmr*``) -- TEST INFRASTRUCTURE ONLY.

The rule (include/orx.h, DESIGN.md section 2 "MMR"), evaluated elementwise in binary64 in the order the CUDA kernel
uses, so positions and distances compare bit for bit:

* candidates: the exact top-``fetch_k`` (:func:`cosine_topk.topk_exact`) in contract order; position = tie-break;
* ``s_q[p] = 1 - d[p]``;
* ``s_dd(p, r) = clamp(canon_sum(x_p * x_r) / sqrt(n2_p * n2_r), -1, 1)`` on the rows as stored;
* first pick position 0, then the largest ``lam * s_q - (1 - lam) * max_r s_dd`` (NumPy never fuses the multiply
  into the subtraction), lowest position on ties, NaN scores only once no finite score is left, in position order.
"""
from __future__ import annotations

import numpy as np

from .cosine_topk import canon_sum, topk_exact


def mmr_select(dist, stored_rows, k: int, lam: float) -> list[int]:
    """Positions (selection order) of the min(k, m) picks among m candidates with canonical query distances `dist`
    [m] and stored rows `stored_rows` [m, 1024] (fp32, or the fp32 image of bf16 rows), in candidate order."""
    dist = np.asarray(dist, np.float64)
    m = dist.shape[0]
    n = min(int(k), m)
    if n <= 0:
        return []
    X = np.asarray(stored_rows, np.float32)[:m].astype(np.float64)
    n2 = canon_sum(X * X)
    s_q = 1.0 - dist
    lam = float(lam)
    one_minus_lam = 1.0 - lam
    red = np.full(m, -np.inf)
    avail = np.ones(m, bool)
    picks = [0]
    avail[0] = False
    while len(picks) < n:
        r = picks[-1]
        with np.errstate(invalid="ignore", divide="ignore"):
            s = canon_sum(X * X[r]) / np.sqrt(n2 * n2[r])
        s = np.where(s > 1.0, 1.0, s)
        s = np.where(s < -1.0, -1.0, s)
        red = np.maximum(red, s)                     # NaN propagates
        with np.errstate(invalid="ignore"):
            score = lam * s_q - one_minus_lam * red
        live = np.flatnonzero(avail & ~np.isnan(score))
        if live.size:
            p = int(live[np.argmax(score[live])])    # first maximum = lowest position
        else:
            p = int(np.flatnonzero(avail)[0])
        picks.append(p)
        avail[p] = False
    return picks


def mmr_exact(X_stored, ids, q, k: int, fetch_k: int, lam: float):
    """Exact MMR answer of one query over a table: ``(ids [n, 2] uint64, distance [n] float64)`` in selection order,
    n = min(k, rows).  `X_stored` are the rows as the table stores them (fp32 image)."""
    X_stored = np.asarray(X_stored, np.float32)
    ids = np.asarray(ids, np.uint64).reshape(-1, 2)
    c_ids, c_d = topk_exact(X_stored, ids, q, fetch_k)
    row_of = {(int(h), int(l)): i for i, (h, l) in enumerate(ids)}
    rows = X_stored[[row_of[(int(h), int(l))] for h, l in c_ids]] if len(c_ids) else np.zeros((0, X_stored.shape[1]), np.float32)
    picks = mmr_select(c_d, rows, k, lam)
    return c_ids[picks].copy(), c_d[picks].copy()
