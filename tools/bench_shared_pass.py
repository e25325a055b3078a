"""Scan times of the single-query 8-bit scan alone and with a second query riding along (DESIGN.md section 4, "two
searches in flight"), on the bench table (10M x 1024 fp32 by default, 8-bit image).

    python tools/bench_shared_pass.py [--rows N] [--reps R] [--lib path/to/liborx.so]

- `one`: a closed loop of orx_search; scan kernel time per search from CUDA events (ORX_OPT_SCAN_TIMING);
- `two`: pairs submitted back to back (orx_search_submit x2, then both waits); the first search's scan time is its lap
  with the second query joined (a build without shared passes scans the two one after the other);
- `pipelined`: two searches in flight, as bench.py's `value` runs them: queries per second (CUDA events);
- the card's name, power limit and clocks from nvidia-smi, read in the same run.
One JSON line."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return dict(zip(q.split(","), [s.strip() for s in out.split(",")])) if out else {}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--lib", default=None, help="another build of liborx.so with this tree's C-ABI")
    a = ap.parse_args()
    if a.lib:                                   # as bench.py --lib: select the build before the package loads
        import types
        sys.modules["orx_lib_override"] = types.SimpleNamespace(LIB_PATH=os.path.abspath(a.lib))
    import numpy as np
    import torch
    import outline_rag_b200 as orx
    from bench import build_table
    from orx_testkit.synth import Synth, default_centres
    k = 12
    ix = orx.Index("fp32", a.rows, 0)
    ix.use_torch_stream()
    build_table(ix.upsert, 0, a.rows, 0, 1)
    Q, _ = Synth(default_centres(a.rows)).queries(16, a.rows)
    Qd = torch.from_numpy(Q).cuda()
    outs = [(torch.empty((1, k, 2), dtype=torch.int64, device="cuda:0"),
             torch.empty((1, k), dtype=torch.float64, device="cuda:0"),
             torch.empty((1,), dtype=torch.int32, device="cuda:0")) for _ in range(3)]

    for i in range(3):
        ix.search(Qd[i:i + 1], k, out=outs[0])
    one = []
    for i in range(a.reps):
        ix.search(Qd[i % 16:i % 16 + 1], k, out=outs[0])
        one.append(ix.stats()["last_scan_ms"])
    assert ix.stats()["last_path"] == 4

    two, second = [], []
    s0 = ix.stats()
    for i in range(a.reps):
        ta = ix.search_submit(Qd[i % 16:i % 16 + 1], k, outs[0])
        tb = ix.search_submit(Qd[(i + 1) % 16:(i + 1) % 16 + 1], k, outs[1])
        ix.search_wait(ta)
        two.append(ix.stats()["last_scan_ms"])
        ix.search_wait(tb)
        second.append(ix.stats()["last_scan_ms"])
    s1 = ix.stats()

    steps = 200
    from outline_rag_b200 import _lib
    ix.set_option(_lib.ORX_OPT_SCAN_TIMING, 0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    prev = None
    for i in range(steps):
        t = ix.search_submit(Qd[i % 16:i % 16 + 1], k, outs[i % 3])
        if prev is not None:
            ix.search_wait(prev)
        prev = t
    ix.search_wait(prev)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    p2 = ix.stats()
    print(json.dumps({
        "rows": a.rows, "lib": a.lib or "in-tree", "card": card(),
        "one_query_scan_ms": {"median": float(np.median(one)), "min": float(np.min(one)), "max": float(np.max(one))},
        "two_query_scan_ms": {"median": float(np.median(two)), "min": float(np.min(two)), "max": float(np.max(two))},
        "second_catch_up_ms": {"median": float(np.median(second)), "max": float(np.max(second))},
        "pairs_shared": s1.get("shared_scans", 0) - s0.get("shared_scans", 0), "pairs": a.reps,
        "pipelined_qps": steps / (ms * 1e-3),
        "pipelined_shared": p2.get("shared_scans", 0) - s1.get("shared_scans", 0),
        "pipelined_shared_rows": p2.get("shared_rows", 0) - s1.get("shared_rows", 0),
        "fallback_exhaustive": p2["fallback_exhaustive"],
        "time": time.strftime("%Y-%m-%dT%H:%M:%S"),
    }), flush=True)
    ix.close()


if __name__ == "__main__":
    main()
