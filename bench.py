#!/usr/bin/env python
"""bench.py -- the headline benchmark of BASELINE.json: exact cosine top-12 QPS / latency.

A "step" is ONE pass of the hot path over one batch of synthetic queries: one search of `--batch`
queries (default 1) against the device-resident table (default 10M x 1024 fp32, the configuration
BASELINE.json's metric is quoted on; 41 GB, fits one B200).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--rows R] [--batch B] [--dtype fp32|bf16]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...   (N > 1)
    python bench.py --impl reference ...      # the CPU arm (NumPy replica of the SQL ordering)
    python bench.py ... --dump-outputs DIR    # also write the last timed step's answer to DIR/*.npy (rank 0)

Output: ONE JSON line on rank 0.
  value      whole-job QPS over EXACTLY K steps, queries already in HBM, results left in HBM (CUDA events on the
             launching stream, barrier + synchronize on both sides, max over ranks), with TWO searches in flight
             (orx_search_submit / orx_search_wait: the throughput mode of the engine); `closed_loop` repeats the same K
             steps as a loop of dependent calls (each search complete before the next is issued)
  e2e        the same through the public host API on HOST buffers: per step the query batch goes host->device and
             ids / distances / counts come back device->host inside the timed region
  latency    closed-loop p50 / p99 over a separately timed run of >= 1 s (K may be too small for percentiles)
  roofline   the scan kernel: algorithmic bytes (rows x 1024 x sizeof(elem)) or flops (2 x rows x 1024 x batch) per
             launch / the kernel's own CUDA-event time (events recorded around the scan launch on its stream)
  verify     FULL-SCAN parity at the benchmarked size: every rank exports its live shard to the host, the oracle
             (oracle/cosine_topk.py StreamingTopK) scans all of it, rank 0 merges the shards' candidates; the
             engine's ids AND distance bits must equal the oracle's for every checked query
  configs    the other BASELINE.json configurations measured in the same run (each with its own roofline, clocks,
             fallbacks; bf16 tables with recall@12 against the fp32 table's answers)
  cpu_baseline  the NumPy replica of the SQL ordering timed on this box's host cores: 100k rows (BASELINE configs[0])
             and 1M rows MEASURED; the figure at the full row count is a linear extrapolation and says so
Multi-GPU: the table is row-sharded (mix64(id) mod N); per step every rank scans its shard and the k candidates per
query are exchanged over NVLink peer memory and merged on device -> "scaling": "strong" (total rows fixed).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
import types

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

K = 12
DIM = 1024
METRIC = "qps_exact_cosine_top12"
UNIT = "queries/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--batch", type=int, default=1)
    ap.add_argument("--dtype", default="fp32", choices=["fp32", "bf16"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--verify", type=int, default=4,
                    help="queries checked by the FULL-SCAN oracle pass over the exported table (0 = off)")
    ap.add_argument("--configs", default="auto", choices=["auto", "none", "all"],
                    help="extra BASELINE.json configurations measured in the same run (auto: on the default 1-GPU and "
                         "8-GPU runs)")
    ap.add_argument("--recall-queries", type=int, default=128)
    ap.add_argument("--latency-s", type=float, default=1.0, help="minimum duration of the separate p50/p99 run")
    ap.add_argument("--mixed", action="store_true",
                    help="config 5: REFRESH_BATCH_SIZE=50-doc delete+upsert between every 100 single-query searches")
    ap.add_argument("--mixed-rounds", type=int, default=20)
    ap.add_argument("--no-group-e2e", action="store_true",
                    help="N > 1: keep e2e on the rank-per-GPU path instead of the one-process multi-GPU index")
    ap.add_argument("--lib", default=None, help="A/B: load this build of liborx.so instead of the in-tree default")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the headline's last timed step returned (ids, distances, counts) to DIR/<name>.npy; "
                         "the inputs depend on the arguments only, so two builds can be compared output for output")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.mixed:
        ap.error("--dump-outputs is not available with --mixed")
    return a


def workload_name(rows, dtype, batch):
    return f"exact cosine top-{K}, {rows}x{DIM} {dtype}, query batch {batch}"


def config_of(rows, dtype, batch):
    """The SAME dict in both arms (the driver compares them)."""
    return {"workload": workload_name(rows, dtype, batch), "rows": rows, "dim": DIM, "k": K, "batch": batch,
            "table_dtype": dtype,
            "l2": "inputs larger than L2: the table (>= 20 GB) is streamed from HBM every step, no flush needed"
                  if rows * DIM * (4 if dtype == "fp32" else 2) > 512e6 else "table fits L2: numbers are L2-resident"}


# ------------------------------------------------------------------ clocks (B200_PROFILING.md)
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0])); smax.append(float(p[1])); power.append(float(p[2]))
            except ValueError:
                continue
            for nm, v in zip(names, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(smax)), "power_w_max": float(max(power)),
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return (float(d["hbm_gbs"]), float(d.get("bf16_tflops", 1590.0)), float(d.get("bf16_tflops_sustained", 1400.0)),
                "measured (MEASURED_PEAKS.json)")
    return 6650.0, 1590.0, 1400.0, "fallback (B200_PROFILING.md)"


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, ids, dist, counts) -> None:
    """`--dump-outputs`: one search answer as float64 .npy files -- `ids` [B, k, 2] (the hi and lo words of each 128-bit
    id; every id the bench generates is below 2**53, so the float64 values are exact), `distances` [B, k] and `counts`
    [B].  A batch whose answer exceeds 64 MB is cut to a fixed, seeded sample of its queries, whose positions in the
    batch go to `query_index.npy`."""
    ids = np.asarray(ids, np.uint64).reshape(len(dist), -1, 2)
    assert not (ids >> np.uint64(53)).any(), "ids of 2**53 and above have no exact float64 form"
    out = {"ids": ids.astype(np.float64), "distances": np.asarray(dist, np.float64),
           "counts": np.asarray(counts, np.float64)}
    per_query = sum(v[0].nbytes for v in out.values()) + 8
    if per_query * len(dist) > DUMP_LIMIT_BYTES:
        sel = np.sort(np.random.default_rng(0).choice(len(dist), DUMP_LIMIT_BYTES // per_query, replace=False))
        out = {name: v[sel] for name, v in out.items()}
        out["query_index"] = sel.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, v in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), v)


def traffic_from_profile(tag: str, rows: int):
    """DRAM bytes per launch from the committed ncu --set full capture (profiles/traffic.json holds
    bytes for the captured row count; the scan is linear in rows, so it is scaled to this launch)."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        with open(p) as f:
            e = json.load(f).get(tag)
        if isinstance(e, dict) and e.get("rows"):
            return e["bytes"] * rows / e["rows"]
    return None


# ------------------------------------------------------------------ CPU arm
# Nothing in this section imports outline_rag_b200: the reference arm's process loads oracle/ libraries only.
def _blas_threads(n):
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=n)
    except Exception:
        pass


def _time_queries(X, inv, ids, Q, n_warm, n_timed, budget_s):
    """Closed loop of single-query NumPy-replica searches; returns the per-query latencies (s) and the last answer."""
    from oracle import cosine_topk as O
    for i in range(n_warm):
        O.numpy_replica_topk(X, ids, Q[i % Q.shape[0]], K, row_inv_norm=inv)
    lat, t_end = [], time.perf_counter() + budget_s
    for i in range(n_timed):
        t0 = time.perf_counter()
        last = O.numpy_replica_topk(X, ids, Q[i % Q.shape[0]], K, row_inv_norm=inv)
        lat.append(time.perf_counter() - t0)
        if time.perf_counter() > t_end and len(lat) >= 3:
            break
    return np.asarray(lat), last


def time_cpu_arm(rows_full: int, batch: int, steps: int, warmup: int, budget_s: float = 25.0, exact_steps=False):
    """The reference's CPU path as north_star defines it when Postgres cannot be installed: the NumPy replica of
    the SQL ordering (OpenBLAS sgemv + argpartition + lexsort, row norms precomputed -- which favours the CPU),
    all host threads.  MEASURED on 100k rows (BASELINE.json configs[0], its own 1024-centre table) and on
    min(rows_full, 1M) rows of the benchmarked table; the figure at rows_full is a linear extrapolation of the
    latter (the scan is linear in rows) and is labelled as such."""
    from oracle import cosine_topk as O
    from oracle.synth_host import FastSynth
    from orx_testkit.synth import default_centres
    n_cores = len(os.sched_getaffinity(0))
    _blas_threads(n_cores)      # torchrun exports OMP_NUM_THREADS=1; the CPU arm is entitled to every host core
    out = {"unit": UNIT, "kind": "port", "host_cpus": os.cpu_count(), "measured": []}
    # -- BASELINE.json configs[0]: 100k rows, single query, measured as stated
    syn = FastSynth(default_centres(100_000))
    X = syn.table(100_000)
    Q, _ = syn.queries(64, 100_000)
    inv = 1.0 / np.sqrt(np.einsum("ij,ij->i", X, X).astype(np.float64))
    lat, _ = _time_queries(X, inv, O.ids_arange(0, 100_000), Q, 5, max(200, steps), budget_s * 0.2)
    out["measured"].append({"rows": 100_000, "config": "BASELINE.json configs[0]", "queries": int(lat.size),
                            "p50_ms": float(np.median(lat) * 1e3), "p99_ms": float(np.percentile(lat, 99) * 1e3),
                            "qps": float(1.0 / np.median(lat)), "extrapolated": False})
    # -- the benchmarked table, measured at up to 1M rows
    n_meas = min(rows_full, 1_000_000)
    syn = FastSynth(default_centres(rows_full))
    X = syn.table(n_meas)
    Q, _ = syn.queries(64, rows_full)
    inv = 1.0 / np.sqrt(np.einsum("ij,ij->i", X, X).astype(np.float64))
    ids = O.ids_arange(0, n_meas)
    lat, last = _time_queries(X, inv, ids, Q, max(warmup, 3), steps if exact_steps else max(60, steps),
                              1e9 if exact_steps else budget_s * 0.5)
    p50 = float(np.median(lat))
    out["measured"].append({"rows": n_meas, "config": "first rows of the benchmarked table", "queries": int(lat.size),
                            "p50_ms": p50 * 1e3, "p99_ms": float(np.percentile(lat, 99) * 1e3), "qps": 1.0 / p50,
                            "mean_ms": float(lat.mean() * 1e3), "extrapolated": False})
    scale = rows_full / n_meas
    try:
        out["pgvector_loop"] = time_pgvector_loop(X, Q, rows_full, n_cores)
    except Exception as e:      # noqa: BLE001 -- an optional extra must never cost the bench line
        out["pgvector_loop"] = {"unavailable": str(e)[:120]}
    # the arm's figure is the FASTER of the two CPU statements, both measured on the same n_meas rows
    best_s, which = p50, "NumPy replica (OpenBLAS sgemv+argpartition+lexsort, precomputed row norms)"
    par = out["pgvector_loop"].get("parallel_seq_scan")
    if par and par["p50_ms_measured"] * 1e-3 < best_s:
        best_s, which = par["p50_ms_measured"] * 1e-3, f"C restatement of pgvector's scan loop, {par['threads']} threads (parallel seq scan)"
    out["value"] = 1.0 / (best_s * scale)
    out["extrapolated"] = scale != 1.0
    out["extrapolated_from_rows"] = n_meas
    out["sample"] = (f"{which}: single queries MEASURED on the first {n_meas} rows (p50 {best_s * 1e3:.2f} ms; the NumPy "
                     f"replica ran {lat.size} queries, p50 {p50 * 1e3:.2f} ms)"
                     + (f"; value = the faster latency scaled x{scale:.0f} to {rows_full} rows (EXTRAPOLATED, the scan is "
                        f"linear in rows)" if scale != 1.0 else ""))
    try:
        from threadpoolctl import threadpool_info
        thr = max([p.get("num_threads", 1) for p in threadpool_info() if p.get("user_api") == "blas"] or [1])
    except Exception:
        thr = os.cpu_count() or 1
    out["cores"] = int(min(thr, n_cores))
    out["_lat_measured"] = lat
    out["_last_answer"] = last
    return out


def time_pgvector_loop(X, Q, rows_full: int, n_cores: int, reps: int = 3):
    """The C restatement of pgvector's own scan loop (oracle/pgv_cosine.c: per-row cosine_distance with float
    accumulators + bounded heap, compiled with pgvector's flags): one thread = one Postgres backend running
    the sequential scan, all threads = a parallel seq scan.  Measured on X, scaled to rows_full by rows.  Reported
    next to the NumPy arm, which is the faster of the two CPU statements and therefore the one compared against."""
    import ctypes
    path = os.path.join(ROOT, "oracle", "libpgv_cosine.so")
    if not os.path.exists(path):
        subprocess.run(["make", "-C", os.path.join(ROOT, "oracle")], check=True, capture_output=True)
    lib = ctypes.CDLL(path)
    lib.pgv_scan_topk_mt.restype = ctypes.c_int
    lib.pgv_scan_topk_mt.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_void_p, ctypes.c_int,
                                     ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
    n = X.shape[0]
    rows = np.zeros(K, np.int64)
    dist = np.zeros(K, np.float64)
    out = {"measured_rows": int(n)}
    for name, threads in (("one_backend", 1), ("parallel_seq_scan", n_cores)):
        lat = []
        for r in range(reps):
            q = np.ascontiguousarray(Q[r % Q.shape[0]], np.float32)
            t0 = time.perf_counter()
            lib.pgv_scan_topk_mt(X.ctypes.data, n, DIM, q.ctypes.data, K, threads, rows.ctypes.data, dist.ctypes.data)
            lat.append(time.perf_counter() - t0)
        s_full = float(np.median(lat)) * (rows_full / n)
        out[name] = {"threads": threads, "p50_ms_measured": float(np.median(lat)) * 1e3,
                     "queries_per_s_at_full_rows_extrapolated": 1.0 / s_full}
    return out


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cb = time_cpu_arm(a.rows, a.batch, a.steps, a.warmup, exact_steps=True)
    lat = cb.pop("_lat_measured")
    ids, dist = cb.pop("_last_answer")
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, ids[None], dist[None], [len(dist)])
    qps = cb["value"]
    line = {"impl": "reference", "metric": METRIC, "value": qps, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
            "warmup": max(a.warmup, 3), "ms_per_step": a.batch / qps * 1e3,
            "ms_per_step_measured_on_sample": float(lat.mean() * 1e3) * a.batch, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_of(a.rows, a.dtype, a.batch), "cpu_baseline": cb,
            "e2e": {"value": qps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------ GPU arm
def build_table(ix_upsert, device, rows, rank, world, chunk=262_144):
    """Generate the synthetic table in HBM chunk by chunk and upsert the rows this rank owns."""
    import torch
    from orx_testkit.device import synth_rows_device
    from outline_rag_b200.sharded import shard_of
    from orx_testkit.synth import SEED_TABLE, default_centres
    nc = default_centres(rows)
    buf = torch.empty((min(chunk, rows), DIM), dtype=torch.float32, device=f"cuda:{device}")
    owned = 0
    for s in range(0, rows, chunk):
        m = min(chunk, rows - s)
        synth_rows_device(device, SEED_TABLE, nc, s, m, out=buf[:m])
        ids = np.zeros((m, 2), np.uint64)
        ids[:, 1] = np.arange(s, s + m, dtype=np.uint64)
        if world > 1:
            sel = np.nonzero(shard_of(ids, world) == rank)[0]
            if sel.size == 0:
                continue
            ix_upsert(ids[sel], buf[:m].index_select(0, torch.from_numpy(sel).to(buf.device)))
            owned += sel.size
        else:
            ix_upsert(ids, buf[:m])
            owned += m
    torch.cuda.synchronize(device)
    del buf
    return owned


def step_out_to_host(out):
    ids, d, c = out
    if not isinstance(ids, np.ndarray):
        ids, d, c = ids.cpu().numpy().view(np.uint64), d.cpu().numpy(), c.cpu().numpy()
    return ids.copy(), d.copy(), c.copy()


class Bench:
    """One process = one rank = one GPU.  Holds the distributed context and the per-config measurement code."""

    def __init__(self, a):
        import torch
        import torch.distributed as dist
        self.a, self.torch, self.dist = a, torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            import datetime
            dist.init_process_group("nccl", device_id=torch.device(f"cuda:{self.local}"),
                                    timeout=datetime.timedelta(seconds=900))
            # a CPU-side group: ranks that wait for rank 0's one-process multi-GPU leg must not park a spinning NCCL
            # kernel on the GPUs that leg is measuring
            self.cpu_group = dist.new_group(backend="gloo", timeout=datetime.timedelta(seconds=900))
        self.hbm_peak, self.tensor_peak, self.tensor_sustained, self.peak_src = measured_peaks()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    # -------------------------------------------------------------- table
    def build(self, rows, dtype):
        from outline_rag_b200.sharded import ShardedIndex
        cap = rows // self.world + rows // (self.world * 8) + 4096 if self.world > 1 else rows + 65_536
        sh = ShardedIndex(dtype, cap, self.local)
        sh.local.use_torch_stream()
        t0 = time.perf_counter()
        owned = build_table(sh.local.upsert, self.local, rows, self.rank, self.world)
        assert len(sh.local) == owned
        return sh, owned, time.perf_counter() - t0

    def free(self, sh):
        self.barrier()              # every rank has finished its last search before any exchange buffer is unmapped
        sh.local.close()
        self.barrier()

    # -------------------------------------------------------------- one timed loop
    def timed(self, step_fn, steps, warmup):
        torch = self.torch
        for i in range(warmup):
            step_fn(i)
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        lat = np.empty(steps)
        e0.record()
        for i in range(steps):
            t = time.perf_counter()
            out = step_fn(warmup + i)
            lat[i] = time.perf_counter() - t
        e1.record()
        self.barrier()
        self.last_out = out
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(ms, op=self.dist.ReduceOp.MAX)
        return float(ms.item()), lat

    def timed_pipelined(self, sh, batches, steps, warmup):
        """EXACTLY `steps` searches with TWO in flight (`search_submit` / `search_wait`, device buffers): the host side
        and the first kernels of query i+1 overlap finalize / exchange / merge / completion of query i -- the engine's
        throughput mode.  Same bracketing as `timed` (barrier + synchronize on both sides, CUDA events, max over ranks)."""
        torch = self.torch
        n = len(batches)
        for i in range(warmup):
            sh.search(batches[i % n], K)
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        prev = None
        for i in range(steps):
            t, out = sh.search_submit(batches[(warmup + i) % n], K)
            if prev is not None:
                sh.search_wait(prev)
            prev = t
        sh.search_wait(prev)
        e1.record()
        self.barrier()
        self.last_out = out           # valid until the submit after next
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(ms, op=self.dist.ReduceOp.MAX)
        return float(ms.item())

    # -------------------------------------------------------------- e2e at N > 1: ONE process drives all the GPUs
    def group_e2e(self, rows, dtype, B, steps, warmup, check_queries, check_ids, check_dist):
        """The call a user of the drop-in makes on a multi-GPU box: `Index(devices=[0..N-1])` (what
        `GpuVectorStore.create(devices=...)` wraps; `orx_create_multi`) searched with HOST buffers -- the query batch
        goes host->device on every GPU, the k candidates per query meet on GPU 0 over NVLink peer memory, ids /
        distances / counts come back device->host, all inside the timed region.  Runs on rank 0 after the ranks have
        freed their tables; the other ranks wait on a CPU barrier."""
        import outline_rag_b200 as orx
        from orx_testkit.synth import Synth, default_centres
        torch = self.torch
        out = None
        if self.rank == 0:
            devs = list(range(self.world))
            t0 = time.perf_counter()
            ix = orx.Index(dtype, rows, devices=devs)
            build_table(ix.upsert, 0, rows, 0, 1)
            build_s = time.perf_counter() - t0
            assert len(ix) == rows
            n_batches = 8 if B * 8 <= 4096 else 1
            Qh, _ = Synth(default_centres(rows)).queries(max(B * n_batches, len(check_queries)), rows)
            Qpin = torch.from_numpy(Qh).pin_memory()
            host_batches = [Qpin[j * B:(j + 1) * B].numpy() for j in range(n_batches)]
            for i in range(max(warmup, 3)):
                ix.search(host_batches[i % n_batches], K)
            lat = np.empty(steps)
            t_all = time.perf_counter()
            for i in range(steps):
                t = time.perf_counter()
                ix.search(host_batches[i % n_batches], K)
                lat[i] = time.perf_counter() - t
            wall = time.perf_counter() - t_all
            same = True
            for j in range(len(check_queries)):
                g = ix.search(check_queries[j:j + 1], K)
                same &= bool(np.array_equal(g[0][0], np.asarray(check_ids[j], np.uint64).reshape(-1, 2)))
                same &= bool(np.array_equal(g[1][0].view(np.uint64), np.asarray(check_dist[j], np.float64).view(np.uint64)))
            st = ix.stats()
            ix.close()
            out = {"value": B * steps / wall, "unit": UNIT, "h2d_bytes_per_step": B * DIM * 4 * self.world,
                   "d2h_bytes_per_step": B * K * (16 + 8) + B * 4, "p50_ms": float(np.median(lat) * 1e3),
                   "p99_ms": float(np.percentile(lat, 99) * 1e3), "steps": steps,
                   "api": f"Index(devices={devs}).search on NumPy (host) buffers: one process, orx_create_multi, "
                          f"finalize -> peer stores into GPU 0 -> merge_wait -> mapped host memory",
                   "same_ids_and_distance_bits_as_the_rank_per_gpu_path": same, "table_build_s": round(build_s, 2),
                   "kernel_launches_total": int(st["kernel_launches"])}
        self.dist.barrier(group=self.cpu_group)
        return out

    # -------------------------------------------------------------- full-scan parity
    def full_scan_verify(self, sh, Qv, k, engine_ids, engine_dist, dtype):
        """Every rank exports its live shard (ids + rows verbatim in the table dtype) to the host in chunks and
        feeds the oracle's streaming full scan; rank 0 merges the shards' candidates with the ordering contract
        and compares ids AND distance bits with what the engine returned.  Outside every timed region."""
        from oracle import cosine_topk as O
        torch = self.torch
        t0 = time.perf_counter()
        _blas_threads(max(1, len(os.sched_getaffinity(0)) // max(1, min(self.world, 8))))
        ix = sh.local
        n = len(ix)
        chunk = 131_072
        rb = DIM * (4 if dtype == "fp32" else 2)
        pin_rows = torch.empty((chunk, rb), dtype=torch.uint8).pin_memory()
        pin_ids = torch.empty((chunk, 2), dtype=torch.int64).pin_memory()
        st = O.StreamingTopK(Qv, k)
        for s in range(0, n, chunk):
            m = min(chunk, n - s)
            ids_view = pin_ids.numpy()[:m].view(np.uint64)
            raw = pin_rows.numpy()[:m]
            ix.export_rows(s, m, ids_view, raw)
            if dtype == "fp32":
                st.feed(raw.view(np.float32), ids_view)
            else:
                st.feed(raw.view(np.uint16), ids_view, rows_are_bf16=True)
        mine = [st.candidates(j) for j in range(Qv.shape[0])]
        if self.world > 1:
            gathered = [None] * self.world
            self.dist.all_gather_object(gathered, mine)
        else:
            gathered = [mine]
        rows_total = torch.tensor([st.rows_seen], dtype=torch.int64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(rows_total)
        if self.rank != 0:
            return None
        ids_ok = bits_ok = True
        bad = []
        for j in range(Qv.shape[0]):
            w_ids, w_d = O.merge_shards([g[j] for g in gathered], k)
            g_ids = np.asarray(engine_ids[j], np.uint64).reshape(-1, 2)
            g_d = np.asarray(engine_dist[j], np.float64)
            i_ok = bool(np.array_equal(g_ids, w_ids))
            b_ok = bool(np.array_equal(g_d.view(np.uint64), w_d.view(np.uint64)))
            ids_ok &= i_ok
            bits_ok &= b_ok
            if not (i_ok and b_ok):
                bad.append(j)
        return {"full_scan_ids_match": ids_ok, "full_scan_distance_bits_match": bits_ok,
                "queries_checked": int(Qv.shape[0]), "rows_scanned_by_oracle": int(rows_total.item()),
                "shards": self.world, "mismatching_queries": bad, "seconds": round(time.perf_counter() - t0, 2),
                "how": "orx_export_rows of every live row -> oracle.StreamingTopK (fp32 BLAS shortlist, margin 2e-4, "
                       "canonical binary64 rescoring) -> merge_shards; compared with the engine's ids and float64 bits"}

    # -------------------------------------------------------------- one configuration
    def measure(self, sh, owned, rows, dtype, B, steps, warmup, verify_n, want_e2e=True, want_latency=True):
        torch, a = self.torch, self.a
        from orx_testkit.synth import Synth, default_centres
        ix = sh.local
        syn = Synth(default_centres(rows))
        n_batches = 8 if B * 8 <= 4096 else 1
        Qh, _ = syn.queries(max(B * n_batches, verify_n), rows)
        Qd = torch.from_numpy(Qh).cuda()
        Qpin = torch.from_numpy(Qh).pin_memory()
        dev_batches = [Qd[j * B:(j + 1) * B] for j in range(n_batches)]
        host_batches = [Qpin[j * B:(j + 1) * B].numpy() for j in range(n_batches)]

        def step_device(i):
            return sh.search(dev_batches[i % n_batches], K)

        def step_host(i):
            if self.world == 1 or sh.exchange == "p2p":
                return sh.search(host_batches[i % n_batches], K)      # host buffers straight through the C-ABI
            out = sh.search(Qpin[(i % n_batches) * B:(i % n_batches + 1) * B].cuda(non_blocking=True), K)
            return tuple(t.cpu() for t in out)

        warmup = max(warmup, 3)
        from outline_rag_b200._lib import ORX_OPT_SCAN_TIMING
        sampler = ClockSampler(self.local).start() if self.rank == 0 else None
        if want_latency:
            # (1) the headline region: EXACTLY `steps` steps, no instrumentation inside the library, two searches in
            #     flight (throughput); then the same `steps` steps as a closed loop of dependent calls (latency)
            ix.set_option(ORX_OPT_SCAN_TIMING, 0)
            pipelined = self.world == 1 or sh.exchange == "p2p"
            l0 = ix.stats()
            if pipelined:
                total_ms = self.timed_pipelined(sh, dev_batches, steps, warmup)
            else:
                total_ms, lat = self.timed(step_device, steps, warmup)
                closed_ms = total_ms
            l1 = ix.stats()
            if a.dump_outputs:          # before a later search can reuse the result buffers
                self.head_out = step_out_to_host(self.last_out)
            if pipelined:
                closed_ms, lat = self.timed(step_device, steps, warmup)
            # (2) the same loop again with a CUDA event pair recorded around every scan launch (on the stream the kernel
            #     runs on): the kernel's own duration for the roofline.  The two event records cost ~10 us per step, which
            #     is why they are not in region (1); this region's step time is reported beside the kernel time.
            ix.set_option(ORX_OPT_SCAN_TIMING, 1)
            s0 = ix.stats()
            ev_ms, _ = self.timed(step_device, steps, warmup)
            s1 = ix.stats()
            ix.set_option(ORX_OPT_SCAN_TIMING, 0)
        else:
            # the extra configurations (steps of >= 3 ms): ONE region with the event pair around every scan launch, so the
            # kernel time and the step time come from the same steps (the GPU's clocks wander under the power cap)
            ix.set_option(ORX_OPT_SCAN_TIMING, 1)
            l0 = s0 = ix.stats()
            total_ms, lat = self.timed(step_device, steps, warmup)
            l1 = s1 = ix.stats()
            ev_ms = closed_ms = total_ms
            pipelined = False
            ix.set_option(ORX_OPT_SCAN_TIMING, 0)
        lat_run = None
        if want_latency:
            est = max(total_ms / steps * 1e-3, 1e-5)
            n_lat = int(min(max(200, a.latency_s / est), 5000))
            _, lat_run = self.timed(step_device, n_lat, 3)
        clocks = sampler.stop() if sampler is not None else None
        e2e = None
        if want_e2e:
            e2e_ms, e2e_lat = self.timed(step_host, steps, warmup)
            e2e = {"value": B * steps / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": B * DIM * 4,
                   "d2h_bytes_per_step": B * K * (16 + 8) + B * 4, "p50_ms": float(np.median(e2e_lat) * 1e3),
                   "api": "Index.search / orx_search[_sharded] on NumPy (host) buffers"}

        # ---- full-scan parity (collective; outside the timed regions)
        verify = None
        if verify_n > 0:
            nv = verify_n
            e_ids, e_dist = [], []
            for b in range(0, nv, B):
                o = step_out_to_host(sh.search(Qd[b:b + B], K))
                e_ids += list(o[0])
                e_dist += list(o[1])
            verify = self.full_scan_verify(sh, Qh[:nv], K, e_ids[:nv], e_dist[:nv], dtype)
            self.last_check = (Qh[:nv].copy(), e_ids[:nv], e_dist[:nv])
        if self.rank != 0:
            return None

        scans = s1["scan_launches"] - s0["scan_launches"]
        scan_ms = (s1["scan_ms_total"] - s0["scan_ms_total"]) / max(scans, 1)
        elem = 4 if dtype == "fp32" else 2
        bytes_per_launch = owned * DIM * elem
        path = s1["last_path"]
        flops = 2.0 * owned * DIM * B
        tf32 = dtype == "fp32"
        t_hbm_ideal = bytes_per_launch / (self.hbm_peak * 1e9)
        t_tensor_ideal = flops / (self.tensor_peak * 1e12) * (2.0 if tf32 else 1.0)   # tf32 runs at half the bf16 rate
        kernel = "scan_umma" if path == 2 else "scan_gemv"
        if path == 2 and t_tensor_ideal > t_hbm_ideal:       # large batches: the tensor pipe bounds the scan
            ach = flops / (scan_ms * 1e-3) / 1e12
            peak = self.tensor_peak * (0.5 if tf32 else 1.0)
            roof = {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                    "frac_of_sustained_peak": ach / (self.tensor_sustained * (0.5 if tf32 else 1.0)),
                    "traffic": traffic_from_profile(f"{kernel}_{dtype}_b{B}", owned),
                    "traffic_source": "profiles/traffic.json (ncu --set full capture, scaled by rows)",
                    "peak_source": self.peak_src + (": cuBLAS bf16 burst; tf32 = half" if tf32 else ": cuBLAS bf16 burst"),
                    "kernel": kernel, "kernel_ms": scan_ms, "ms_per_step_in_the_event_timed_region": ev_ms / steps,
                    "hbm_gbs": bytes_per_launch / (scan_ms * 1e-3) / 1e9, "algorithmic_flops_per_launch": flops}
        else:
            ach = bytes_per_launch / (scan_ms * 1e-3) / 1e9
            roof = {"bound": "hbm", "achieved": ach, "peak": self.hbm_peak, "unit": "GB/s", "frac": ach / self.hbm_peak,
                    "traffic": traffic_from_profile(f"{kernel}_{dtype}", owned),
                    "traffic_source": "profiles/traffic.json (ncu --set full capture, scaled by rows)",
                    "peak_source": self.peak_src, "kernel": kernel,
                    "kernel_ms": scan_ms, "ms_per_step_in_the_event_timed_region": ev_ms / steps,
                    "algorithmic_bytes_per_launch": bytes_per_launch,
                    "frac_of_nominal_8TBs": ach / 8000.0, "tflops": flops / (scan_ms * 1e-3) / 1e12}
        res = {
            "config": config_of(rows, dtype, B), "value": B * steps / (total_ms * 1e-3), "unit": UNIT,
            "steps": steps, "warmup": warmup, "ms_per_step": total_ms / steps,
            "p50_ms": float(np.median(lat) * 1e3), "p99_ms": float(np.percentile(lat, 99) * 1e3),
            "gpu_launches": int(l1["kernel_launches"] - l0["kernel_launches"]),
            "roofline": roof, "clocks": clocks, "verify": verify,
            "fallbacks": {"gemv": int(s1["fallback_gemv"] - l0["fallback_gemv"]),
                          "exhaustive": int(s1["fallback_exhaustive"] - l0["fallback_exhaustive"])},
            "run": {"rows_per_gpu": owned, "parallelism": f"row-shard x{self.world}", "exchange": sh.exchange,
                    "searches_in_flight": 2 if pipelined else 1},
            "closed_loop": {"value": B * steps / (closed_ms * 1e-3), "unit": UNIT, "ms_per_step": closed_ms / steps,
                            "steps": steps, "how": "the same steps as a loop of dependent calls: each search is complete "
                                                   "before the next is issued (value: two searches in flight)"},
        }
        if lat_run is not None:
            res["latency"] = {"queries_per_step": B, "steps": int(lat_run.size), "seconds": float(lat_run.sum()),
                              "p50_ms": float(np.median(lat_run) * 1e3), "p99_ms": float(np.percentile(lat_run, 99) * 1e3),
                              "max_ms": float(lat_run.max() * 1e3), "how": "closed loop, wall clock per step on rank 0"}
        if e2e is not None:
            res["e2e"] = e2e
        return res


def run_ours(a):
    import torch
    import outline_rag_b200 as orx   # noqa: F401  (fails loudly when liborx.so is missing)
    bn = Bench(a)
    rank, world = bn.rank, bn.world
    default_headline = a.rows == 10_000_000 and a.batch == 1 and a.dtype == "fp32"
    extras_on = a.configs == "all" or (a.configs == "auto" and default_headline and world in (1, 8))

    sh, owned, build_s = bn.build(a.rows, a.dtype)
    head = bn.measure(sh, owned, a.rows, a.dtype, a.batch, a.steps, a.warmup, a.verify)
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, *bn.head_out)
    head_check = getattr(bn, "last_check", None) if a.verify > 0 else None       # (queries, ids, distances) the oracle confirmed
    extras = []

    def recall_vs(got_ids, want_ids, nrq, how):
        hits = sum(len(set(g.tolist()) & set(w.tolist())) for g, w in zip(got_ids, want_ids))
        return {"recall_at_12_vs_fp32": hits / (nrq * K), "queries": nrq, "how": how}

    def extra(sh_, owned_, rows, dtype, B, steps, verify_n=0):
        r = bn.measure(sh_, owned_, rows, dtype, B, steps, 3, verify_n, want_e2e=False, want_latency=False)
        if rank == 0:
            extras.append(r)
        return r

    sh_box = [sh]

    def run_extras():
        sh = sh_box[0]
        from orx_testkit.synth import Synth, default_centres
        nrq = a.recall_queries
        Qr = torch.from_numpy(Synth(default_centres(a.rows)).queries(nrq, a.rows)[0]).cuda()
        # ---- the fp32 table that is resident: batch 64 (tf32 tcgen05 scan, one table pass for 64 queries)
        extra(sh, owned, a.rows, "fp32", 64, 30, verify_n=4)
        recall_ref = step_out_to_host(sh.search(Qr, K))[0][:, :, 1].copy()        # fp32 answers for recall@12
        if world == 1:
            # ---- SURVEY.md 8f-4 (the rows marked "next"): a wide-k batch and a filtered batch on the same table
            for r in next_rows_on(sh.local, a.rows, "fp32"):
                r["run"] = {"rows_per_gpu": owned, "parallelism": "row-shard x1", "exchange": "none"}
                extras.append(r)
            # ---- BASELINE.json configs[4]: the refresh writer interleaved with single-query searches (mutates the table)
            r = mixed_on(sh.local, a.rows, "fp32", 6)
            r["run"] = {"rows_per_gpu": owned, "parallelism": "row-shard x1", "exchange": "none"}
            extras.append(r)
        bn.free(sh)
        sh_box[0] = None
        # ---- the same rows as a bf16 table
        shb, ownedb, _ = bn.build(a.rows, "bf16")
        for B, st, vn in ((1, 60, 0), (256, 20, 0), (1024, 12, 4)):
            r = extra(shb, ownedb, a.rows, "bf16", B, st, verify_n=vn)
            if B == 1024:
                got = step_out_to_host(shb.search(Qr, K))[0][:, :, 1]             # collective
                if rank == 0:
                    r["recall"] = recall_vs(got, recall_ref, nrq, "ids of the bf16 table vs ids of the fp32 table "
                                                                  "built from the same rows")
        bn.free(shb)
        if world == 8:
            # ---- BASELINE.json configs[3]: 100M x 1024 bf16 (25.6 GB / GPU), batch 1024, recall vs an fp32 twin
            big = 100_000_000
            Qb = torch.from_numpy(Synth(default_centres(big)).queries(nrq, big)[0]).cuda()
            shf, _, _ = bn.build(big, "fp32")
            ref = step_out_to_host(shf.search(Qb, K))[0][:, :, 1].copy()
            bn.free(shf)
            shb, ownedb, build_big = bn.build(big, "bf16")
            r = extra(shb, ownedb, big, "bf16", 1024, 8, verify_n=0)
            got = step_out_to_host(shb.search(Qb, K))[0][:, :, 1]
            if rank == 0:
                r["recall"] = recall_vs(got, ref, nrq, "ids of the bf16 table vs an fp32 twin of the same 100M rows")
                r["run"]["table_build_s"] = round(build_big, 2)
            bn.free(shb)
    # ---- the headline is complete once the one-process multi-GPU leg has run (the rank tables may stay resident:
    #      10M rows are 41 GB in total)
    group_e2e = None
    if world > 1 and not a.no_group_e2e:
        chk = head_check if head_check is not None else (np.zeros((0, DIM), np.float32), [], [])
        group_e2e = bn.group_e2e(a.rows, a.dtype, a.batch, a.steps, a.warmup, *chk)

    def headline_line():
        line = {"metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": a.steps,
                "warmup": head["warmup"], "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f32" if a.dtype == "fp32" else "bf16", "data": "synthetic",
                "config": head["config"], "run": dict(head["run"], table_build_s=round(build_s, 2)),
                "p50_ms": head["p50_ms"], "p99_ms": head["p99_ms"], "closed_loop": head.get("closed_loop"),
            "latency": head.get("latency"),
                "e2e": group_e2e if group_e2e is not None else head.get("e2e"),
                "gpu_launches": head["gpu_launches"], "roofline": head["roofline"], "clocks": head["clocks"],
                "verify": head["verify"], "fallbacks": head["fallbacks"]}
        if group_e2e is not None:
            line["e2e_rank_per_gpu"] = head.get("e2e")      # the same host-buffer step through orx_search_sharded on every rank
        return line

    # ---- the other BASELINE configurations.  They must never cost the headline line: a watchdog prints it and ends the
    #      process if they hang, an exception ends them early.
    printed = threading.Lock()

    def emit(line):
        if printed.acquire(blocking=False):
            if rank == 0:
                print(json.dumps(line), flush=True)
            return True
        return False

    def emergency(why):
        if rank == 0:
            line = headline_line()
            if extras:
                line["configs"] = list(extras)
            line["configs_error"] = why
            emit(line)
        sys.stdout.flush()
        os._exit(0)

    watchdog = None
    if extras_on and a.dtype == "fp32":
        watchdog = threading.Timer(600.0 if world > 1 else 400.0, emergency, args=("the extra configurations ran out of time",))
        watchdog.daemon = True
        watchdog.start()
        try:
            run_extras()
        except Exception as e:      # noqa: BLE001 -- whatever happened, the headline line is printed
            emergency(f"{type(e).__name__}: {str(e)[:300]}")
        watchdog.cancel()
    if sh_box[0] is not None:
        bn.free(sh_box[0])
    if world > 1:
        bn.dist.barrier()
        bn.dist.destroy_process_group()
    if rank != 0:
        return
    line = headline_line()
    if extras:
        line["configs"] = extras
    if not a.no_cpu_baseline and world == 1:
        cb = time_cpu_arm(a.rows, a.batch, 20, 3)
        cb.pop("_lat_measured", None)
        cb.pop("_last_answer", None)
        line["cpu_baseline"] = cb
    emit(line)


def next_rows_on(ix, rows, dtype):
    """SURVEY.md 8f-4 on the resident table, through the C-ABI with host buffers (wall clock per call): a batch of 64
    queries with k = 64 (the wider reranker feed; tcgen05 scan with 160-key candidate lists) and a batch of 64 queries under
    one prepared filter that admits every second row (one tcgen05 pass with the predicate folded into the row scale).
    Each batch answer is compared, ids and distance bits, with the same query run alone through the single-query scan
    (fp32 GEMV / bitmap GEMV): two independent device paths that must agree exactly."""
    from orx_testkit.synth import Synth, default_centres
    Qh, _ = Synth(default_centres(rows)).queries(64, rows)
    out = []

    def timed(fn, iters=10):
        ms = []
        for it in range(iters + 2):
            t0 = time.perf_counter()
            r = fn()
            if it >= 2:
                ms.append((time.perf_counter() - t0) * 1e3)
        return r, float(np.median(ms))

    def same(batch, single, i):
        return bool(np.array_equal(batch[0][i], single[0][0]) and
                    np.array_equal(batch[1][i].view(np.uint64), single[1][0].view(np.uint64)))

    def entry(what, k, extra_cfg, r, ms, s0, s1, ok):
        return {"config": dict({"workload": f"{what}, {rows}x{DIM} {dtype}", "rows": rows, "dim": DIM, "k": k, "batch": 64,
                                "table_dtype": dtype}, **extra_cfg),
                "value": 64 / ms * 1e3, "unit": UNIT, "steps": 10, "ms_per_step": ms,
                "path": "tcgen05" if s1["last_path"] == 2 else "gemv",
                "fallbacks": {"gemv": int(s1["fallback_gemv"] - s0["fallback_gemv"]),
                              "exhaustive": int(s1["fallback_exhaustive"] - s0["fallback_exhaustive"])},
                "h2d_bytes_per_step": 64 * DIM * 4, "d2h_bytes_per_step": 64 * (k * 24 + 4),
                "verify": {"batch_equals_single_query_scan_ids_and_distance_bits": ok, "queries_checked": 3}}

    s0 = ix.stats()
    r, ms = timed(lambda: ix.search(Qh, 64))
    s1 = ix.stats()
    ok = all(same(r, ix.search(Qh[i:i + 1], 64), i) for i in (0, 31, 63))
    out.append(entry("batch of 64 queries, k = 64", 64, {}, r, ms, s0, s1, ok))

    allow = np.zeros((rows // 2, 2), np.uint64)
    allow[:, 1] = np.arange(0, rows, 2, dtype=np.uint64)[:rows // 2]
    t0 = time.perf_counter()
    with ix.make_filter(allow) as flt:
        prepare_ms = (time.perf_counter() - t0) * 1e3
        s0 = ix.stats()
        r, ms = timed(lambda: ix.search_filtered(Qh, K, flt))
        s1 = ix.stats()
        ok = all(same(r, ix.search_filtered(Qh[i:i + 1], K, flt), i) for i in (0, 31, 63))
        single, single_ms = timed(lambda: ix.search_filtered(Qh[:1], K, flt), 5)
    e = entry("batch of 64 queries under one prepared filter (every second row eligible)", K,
              {"eligible_rows": rows // 2}, r, ms, s0, s1, ok)
    e["filter_prepare_ms"] = prepare_ms
    e["single_filtered_query_ms"] = single_ms
    out.append(e)
    return out


def mixed_on(ix, rows, dtype, rounds):
    """BASELINE.json configs[4] on a table that is already built: the webhook refresh (reference app/rag.py:216-235:
    look up the old chunk ids of REFRESH_BATCH_SIZE=50 docs, `adelete` them, `aadd_documents` the re-chunked rows)
    interleaved with top-12 queries.  One round = delete(~1000 ids) + upsert(~1000 rows, host buffers) + 100 searches
    (host buffers through the C-ABI).  Returns the result dict; the table keeps its size (old chunks out, new in)."""
    import torch
    import outline_rag_b200 as orx
    from orx_testkit.synth import Synth, default_centres, doc_chunk_counts
    syn = Synth(default_centres(rows))
    Qh, _ = syn.queries(128, rows)
    # documents = consecutive runs of 8..40 chunk ids (mean ~20) over the initial table
    counts = doc_chunk_counts(rows // 16)
    starts = np.concatenate([[0], np.cumsum(counts)])
    n_docs = int(np.searchsorted(starts, rows, side="right") - 1)
    rng = np.random.default_rng(20261020)
    order = rng.permutation(n_docs)
    docs_per_batch, searches_per_round = orx.REFRESH_BATCH_SIZE, 100
    next_id = rows + 1_000_000_000
    plan = []
    for r in range(rounds + 2):
        docs = order[r * docs_per_batch:(r + 1) * docs_per_batch]
        old_ids = np.concatenate([np.arange(starts[d], starts[d + 1]) for d in docs]).astype(np.uint64)
        n_new = int(counts[docs].sum())                       # re-chunked: same sizes, new uuids, new embeddings
        new_ids = np.arange(next_id, next_id + n_new, dtype=np.uint64)
        new_vecs = syn.rows(new_ids)                          # stands in for the remote embedding service
        next_id += n_new
        plan.append((old_ids, new_ids, new_vecs))

    def search_loop(n, lat):
        for i in range(n):
            t = time.perf_counter()
            ix.search(Qh[i % 128:i % 128 + 1], K)
            lat.append(time.perf_counter() - t)

    n0 = len(ix)
    lat_idle = []
    search_loop(50, [])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    search_loop(rounds * searches_per_round, lat_idle)
    idle_s = time.perf_counter() - t0

    lat_mixed, t_del, t_up = [], [], []
    for old_ids, new_ids, new_vecs in plan[:2]:               # warm-up rounds (buffers, maps)
        ix.delete(old_ids); ix.upsert(new_ids, new_vecs); search_loop(10, [])
    torch.cuda.synchronize()
    s0 = ix.stats()
    t0 = time.perf_counter()
    n_rows_written = 0
    for old_ids, new_ids, new_vecs in plan[2:]:
        t = time.perf_counter(); removed = ix.delete(old_ids); t_del.append(time.perf_counter() - t)
        assert removed == len(old_ids)
        t = time.perf_counter(); ix.upsert(new_ids, new_vecs); t_up.append(time.perf_counter() - t)
        n_rows_written += len(new_ids)
        search_loop(searches_per_round, lat_mixed)
    torch.cuda.synchronize()
    mixed_s = time.perf_counter() - t0
    s1 = ix.stats()
    assert len(ix) == n0
    # deleted chunks never come back, new ones are searchable
    got = ix.search(plan[-1][2][:4], 1)[0][:, 0, 1]
    ok = bool((got == plan[-1][1][:4]).all())
    gone = ix.search(syn.rows(plan[-1][0][:4]), 1)[0][:, 0, 1]
    ok &= bool((gone != plan[-1][0][:4]).all())
    n_search = rounds * searches_per_round
    return {"config": {"workload": f"mixed: per round delete+upsert of {docs_per_batch} docs (~{n_rows_written // rounds} rows) "
                                   f"then {searches_per_round} single-query top-{K} searches, {rows}x{DIM} {dtype}",
                       "rows": rows, "dim": DIM, "k": K, "batch": 1, "table_dtype": dtype, "rounds": rounds},
            "value": n_search / mixed_s, "unit": UNIT, "steps": n_search, "ms_per_step": mixed_s / n_search * 1e3,
            "search_only": {"qps": n_search / idle_s, "p50_ms": float(np.median(lat_idle) * 1e3),
                            "p99_ms": float(np.percentile(lat_idle, 99) * 1e3)},
            "with_writer": {"qps": n_search / mixed_s, "p50_ms": float(np.median(lat_mixed) * 1e3),
                            "p99_ms": float(np.percentile(lat_mixed, 99) * 1e3), "max_ms": float(np.max(lat_mixed) * 1e3),
                            "delete_ms_p50": float(np.median(t_del) * 1e3), "upsert_ms_p50": float(np.median(t_up) * 1e3),
                            "delete_ms_mean": float(np.mean(t_del) * 1e3), "upsert_ms_mean": float(np.mean(t_up) * 1e3),
                            "rows_moved_by_compaction": int(s1["rows_moved"] - s0["rows_moved"])},
            "fallbacks": {"gemv": int(s1["fallback_gemv"] - s0["fallback_gemv"]),
                          "exhaustive": int(s1["fallback_exhaustive"] - s0["fallback_exhaustive"])},
            "gpu_launches": int(s1["kernel_launches"] - s0["kernel_launches"]),
            "h2d_bytes_per_step": DIM * 4 + n_rows_written * DIM * 4 // n_search, "d2h_bytes_per_step": K * 24 + 4,
            "verify": {"new_rows_searchable_deleted_rows_gone_table_size_constant": ok}}


def run_mixed(a):
    import torch
    import outline_rag_b200 as orx
    torch.cuda.set_device(0)
    ix = orx.Index(a.dtype, a.rows + 200_000, 0)
    ix.use_torch_stream()
    build_table(ix.upsert, 0, a.rows, 0, 1)
    r = mixed_on(ix, a.rows, a.dtype, a.mixed_rounds)
    line = {"metric": METRIC + "_mixed", "value": r["value"], "unit": UNIT, "n_gpus": 1, "steps": r["steps"], "warmup": 70,
            "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32" if a.dtype == "fp32" else "bf16", "data": "synthetic", "config": r["config"],
            "search_only": r["search_only"], "with_writer": r["with_writer"], "fallbacks": r["fallbacks"],
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": r["h2d_bytes_per_step"],
                    "d2h_bytes_per_step": r["d2h_bytes_per_step"]},
            "gpu_launches": r["gpu_launches"], "verify": r["verify"]}
    print(json.dumps(line), flush=True)
    ix.close()


def main():
    a = parse_args()
    if a.lib:
        sys.modules["orx_lib_override"] = types.SimpleNamespace(LIB_PATH=os.path.abspath(a.lib))
    if a.impl == "reference":
        run_reference(a)
    elif a.mixed:
        run_mixed(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
