"""The single-query exact scan of a large fp32 table over its 8-bit image, over its bf16 image and over its fp32 rows, on
ONE index and one GPU.

    python tools/bench_image.py [--rows 10000000] [--steps 200] [--reps 3] [--k 12]

Builds rows x 1024 fp32 synthetic rows (bench.py's generator), then cycles `reps` times through three arms:
ORX_OPT_IMAGE8_MIN_ROWS 0 (the GEMV scans read the 8-bit image, last_path 4), ORX_OPT_IMAGE8_MIN_ROWS -1 (the bf16
image, last_path 3; a search rebuilds the image when the option changes its kind, outside the timed window) and
ORX_OPT_IMAGE_MIN_ROWS -1 (the fp32 rows, last_path 1).  Per arm: step time of a closed loop of batch-1 searches
(device queries and outputs, CUDA events), the scan kernel's own device time (the library's per-launch event pair), the
bytes one query actually streams (8-bit: 1 B/element + 4 B scale8; bf16: 2 B/element + 4 B scale; fp32: 4 B/element +
4 B scale) and the bandwidth that makes, the fallback counters, and how many rows a query's finalize rescores (rows
whose fast score is within 2 eps + 1e-6 of the k-th best fast score, at most the candidate list's width -- measured
with the debug hooks on a few queries).  All arms must return the same ids and distance bits.  The card's name, power
limit and clocks are read in the same run.  Prints one JSON line."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

EPS = {"image8": 1.662e-2, "image": 3.92e-3, "fp32": 3.0e-6}   # csrc/internal.h EPS_GEMV_IMAGE8 / _IMAGE / _F32
LIST = {"image8": 160, "image": 64, "fp32": 32}                 # candidate keys per query at k <= 12


def card(dev):
    q = "name,power.limit,power.default_limit,clocks.sm,clocks.max.sm,clocks.mem"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", str(dev)],
                             capture_output=True, text=True, timeout=20).stdout.strip()
        return dict(zip(q.split(","), [v.strip() for v in out.split(",")]))
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--k", type=int, default=12)
    ap.add_argument("--rescore-queries", type=int, default=4)
    a = ap.parse_args()

    import torch
    import outline_rag_b200 as orx
    from outline_rag_b200 import _lib
    from orx_testkit.device import synth_rows_device
    from orx_testkit.synth import SEED_TABLE, Synth, default_centres

    dev = torch.cuda.current_device()
    ix = orx.Index("fp32", a.rows + 65_536, dev)
    ix.use_torch_stream()
    nc = default_centres(a.rows)
    chunk = 262_144
    buf = torch.empty((chunk, 1024), dtype=torch.float32, device=f"cuda:{dev}")
    t0 = time.perf_counter()
    for s in range(0, a.rows, chunk):
        m = min(chunk, a.rows - s)
        synth_rows_device(dev, SEED_TABLE, nc, s, m, out=buf[:m])
        ids = np.zeros((m, 2), np.uint64)
        ids[:, 1] = np.arange(s, s + m, dtype=np.uint64)
        ix.upsert(ids, buf[:m])
    torch.cuda.synchronize()
    build_s = time.perf_counter() - t0
    del buf

    nq = 64
    Q = torch.from_numpy(Synth(nc).queries(nq, a.rows)[0]).cuda(dev)
    out = (torch.empty((1, a.k, 2), dtype=torch.int64, device=Q.device),
           torch.empty((1, a.k), dtype=torch.float64, device=Q.device),
           torch.empty((1,), dtype=torch.int32, device=Q.device))
    arms = {"image8": (0, 0), "image": (-1, 0), "fp32": (0, -1)}    # (IMAGE8_MIN_ROWS, IMAGE_MIN_ROWS)

    def arm(mode):
        ix.set_option(_lib.ORX_OPT_IMAGE8_MIN_ROWS, arms[mode][0])
        ix.set_option(_lib.ORX_OPT_IMAGE_MIN_ROWS, arms[mode][1])

    def answers(mode):
        arm(mode)
        got = [ix.search(Q[i:i + 1], a.k) for i in range(nq)]
        return (torch.cat([g[0] for g in got]).cpu().numpy(), torch.cat([g[1] for g in got]).cpu().numpy(),
                ix.stats()["last_path"])

    ans = {m: answers(m) for m in arms}
    same = all(bool(np.array_equal(ans[m][0], ans["fp32"][0]) and
                    np.array_equal(ans[m][1].view(np.uint64), ans["fp32"][1].view(np.uint64))) for m in arms)

    runs = {m: [] for m in arms}
    for _ in range(a.reps):
        for mode in arms:
            arm(mode)
            for i in range(a.warmup):
                ix.search(Q[i % nq:i % nq + 1], a.k, out=out)
            torch.cuda.synchronize()
            st0 = ix.stats()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(a.steps):
                ix.search(Q[i % nq:i % nq + 1], a.k, out=out)
            e1.record()
            torch.cuda.synchronize()
            st1 = ix.stats()
            launches = st1["scan_launches"] - st0["scan_launches"]
            runs[mode].append({"step_ms": e0.elapsed_time(e1) / a.steps,
                               "kernel_ms": (st1["scan_ms_total"] - st0["scan_ms_total"]) / max(launches, 1),
                               "last_path": st1["last_path"],
                               "fallback_gemv": st1["fallback_gemv"] - st0["fallback_gemv"],
                               "fallback_exhaustive": st1["fallback_exhaustive"] - st0["fallback_exhaustive"]})

    # rows finalize may rescore: fast score >= k-th best fast score - 2 eps - 1e-6 (finalize.cu, round 2 cut)
    rq = Q[:a.rescore_queries]
    rescore = {}
    for mode, fn in (("image8", ix.debug_image8_scores), ("image", ix.debug_image_scores), ("fp32", ix.debug_fast_scores)):
        arm(mode)
        ix.search(Q[0:1], a.k, out=out)                # the image this arm reads
        s = fn(rq)
        kth = torch.topk(s, a.k, dim=0).values[-1]
        rescore[mode] = [int(c) for c in (s >= kth - (2 * EPS[mode] + 1e-6)).sum(dim=0).tolist()]
        del s

    elems = a.rows * 1024
    bytes_q = {"image8": elems + a.rows * 4, "image": elems * 2 + a.rows * 4, "fp32": elems * 4 + a.rows * 4}
    res = {"what": "8-bit image vs bf16 image vs fp32 rows, single-query exact scan", "rows": a.rows, "k": a.k,
           "steps": a.steps, "reps": a.reps, "card": card(dev), "table_build_s": round(build_s, 2),
           "same_ids_and_distance_bits": same, "paths": {m: ans[m][2] for m in arms}, "arms": {}}
    for mode in arms:
        st = np.array([r["step_ms"] for r in runs[mode]])
        km = np.array([r["kernel_ms"] for r in runs[mode]])
        res["arms"][mode] = {
            "step_ms": [round(float(v), 4) for v in st], "kernel_ms": [round(float(v), 4) for v in km],
            "step_ms_median": round(float(np.median(st)), 4), "kernel_ms_median": round(float(np.median(km)), 4),
            "qps": round(1e3 / float(np.median(st)), 1),
            "bytes_per_query": bytes_q[mode],
            "TBps_kernel": round(bytes_q[mode] / (float(np.median(km)) * 1e-3) / 1e12, 3),
            "fallbacks": {"gemv": sum(r["fallback_gemv"] for r in runs[mode]),
                          "exhaustive": sum(r["fallback_exhaustive"] for r in runs[mode])},
            "rows_within_2eps_of_kth": rescore[mode],
            "rows_rescored": [min(c, LIST[mode]) for c in rescore[mode]]}
    for mode in ("image8", "image"):
        for what in ("step", "kernel"):
            res[f"speedup_{what}_{mode}_vs_fp32"] = round(res["arms"]["fp32"][f"{what}_ms_median"] /
                                                          res["arms"][mode][f"{what}_ms_median"], 3)
    res["speedup_step_image8_vs_image"] = round(res["arms"]["image"]["step_ms_median"] /
                                                res["arms"]["image8"]["step_ms_median"], 3)
    print(json.dumps(res), flush=True)
    ix.close()


if __name__ == "__main__":
    main()
