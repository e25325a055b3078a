"""Exact MMR search (`orx_search_mmr`) against the plain exact search and against the host route langchain-postgres
takes (fetch fetch_k rows with their embeddings, then NumPy MMR), with sampled answers checked against oracle/mmr.py on
exported rows.  Prints one JSON line per measurement; the first line names the card and its power limit.

    python tools/bench_mmr.py [--rows 10000000] [--bf16-rows 2000000] [--iters 50] > profiles/rN_bench_mmr.jsonl
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True)
    name, power, clock = [s.strip() for s in out.stdout.splitlines()[0].split(",")]
    return {"card": name, "power_limit": power, "max_sm_clock": clock}


def timed(fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    ms = []
    for _ in range(iters):
        t0 = time.perf_counter()
        fn()                                  # every call returns with its results on the host (device synchronised)
        ms.append((time.perf_counter() - t0) * 1e3)
    return {"p50_ms": float(np.percentile(ms, 50)), "p99_ms": float(np.percentile(ms, 99))}


def host_mmr(ix, q, k, fetch_k, lam):
    """langchain-postgres' route: the exact top-fetch_k, their embeddings to the host, cosine Gram in NumPy."""
    from outline_rag_b200 import engine
    ids, dist, cnt = ix.search(q[None], fetch_k)
    rows, _ = ix.fetch(ids[0, :cnt[0]])
    Xn = rows / np.linalg.norm(rows, axis=1, keepdims=True)
    s_q = 1.0 - dist[0, :cnt[0]]
    picks, red = [0], np.full(cnt[0], -np.inf)
    while len(picks) < min(k, cnt[0]):
        red = np.maximum(red, Xn @ Xn[picks[-1]])
        score = lam * s_q - (1 - lam) * red
        score[picks] = -np.inf
        picks.append(int(np.argmax(score)))
    return engine.ids_to_ints(ids[0, picks])


def check(ix, Q, k, fetch_k, lam, which, dtype):
    """Sampled answers against the oracle, on the rows exported from the table (the candidates are the exact top)."""
    from oracle.cosine_topk import StreamingTopK
    from oracle.mmr import mmr_select
    g_ids, g_d, g_c = ix.search_mmr(Q[which], k, fetch_k, lam)
    st = StreamingTopK(Q[which], fetch_k)
    n, chunk = len(ix), 262_144
    ids_buf = np.empty((chunk, 2), np.uint64)
    rows_buf = np.empty((chunk, 1024 if dtype == "fp32" else 512), np.float32)
    for s in range(0, n, chunk):
        m = min(chunk, n - s)
        ix.export_rows(s, m, ids_buf, rows_buf)
        raw = rows_buf[:m] if dtype == "fp32" else rows_buf[:m].view(np.uint16)
        st.feed(raw, ids_buf[:m], rows_are_bf16=dtype == "bf16")
    for j, (c_ids, c_d) in enumerate(st.result()):
        rows = st._vec[j][[np.flatnonzero((st._ids[j] == i).all(axis=1))[0] for i in c_ids]]
        picks = mmr_select(c_d, rows, k, lam)
        assert g_c[j] == len(picks) and np.array_equal(g_ids[j, :len(picks)], c_ids[picks]), (j, "ids differ")
        assert np.array_equal(g_d[j, :len(picks)].view(np.uint64), c_d[picks].view(np.uint64)), (j, "distances differ")
    return len(which)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--bf16-rows", type=int, default=2_000_000)
    ap.add_argument("--iters", type=int, default=50)
    a = ap.parse_args()
    import torch
    import outline_rag_b200 as orx
    from bench import build_table
    from orx_testkit.synth import Synth, default_centres
    info = card()
    print(json.dumps(info), flush=True)

    syn = Synth(default_centres(a.rows))
    Q, _ = syn.queries(1024, min(a.rows, 100_000))
    with orx.Index("fp32", capacity=a.rows) as ix:
        build_table(ix.upsert, 0, a.rows, 0, 1)
        q = Q[0]
        res = {"rows": a.rows, "dtype": "fp32", "nq": 1, **info}
        res["search_k20"] = timed(lambda: ix.search(q[None], 20), a.iters)
        res["mmr_k4_fetch20"] = timed(lambda: ix.search_mmr(q[None], 4, 20, 0.5), a.iters)
        res["host_route_k4_fetch20"] = timed(lambda: host_mmr(ix, q, 4, 20, 0.5), a.iters)
        res["checked_queries"] = check(ix, Q, 4, 20, 0.5, [0, 1, 2], "fp32")
        got = orx.ids_to_ints(ix.search_mmr(q[None], 4, 20, 0.5)[0][0])
        res["host_route_same_ids"] = got == host_mmr(ix, q, 4, 20, 0.5)
        print(json.dumps(res), flush=True)

    with orx.Index("bf16", capacity=a.bf16_rows) as ix:
        build_table(ix.upsert, 0, a.bf16_rows, 0, 1)
        for nq in (256, 1024):
            for fetch_k in (20, 64, 128):
                res = {"rows": a.bf16_rows, "dtype": "bf16", "nq": nq, "k": 12, "fetch_k": fetch_k, "lambda": 0.5,
                       **info}
                it = max(3, a.iters // 10)
                res["search_fetch_k"] = timed(lambda: ix.search(Q[:nq], fetch_k), it)
                res["search_k12"] = timed(lambda: ix.search(Q[:nq], 12), it)
                res["mmr"] = timed(lambda: ix.search_mmr(Q[:nq], 12, fetch_k, 0.5), it)
                res["checked_queries"] = check(ix, Q[:nq], 12, fetch_k, 0.5, [0, nq - 1], "bf16")
                print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
