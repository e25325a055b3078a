"""bench.py's CPU arm (`--impl reference`: the NumPy replica of the SQL ordering, timed on host cores)
must run without a GPU and print the contract's JSON line."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--rows", "50000",
                          "--steps", "3", "--warmup", "1"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "qps_exact_cosine_top12" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["gpu_launches"] == 0
    assert "50000x1024" in line["config"]["workload"]
    cb = line["cpu_baseline"]
    pgv = cb["pgvector_loop"]                                    # the C restatement of pgvector's scan loop, timed too
    assert pgv["one_backend"]["threads"] == 1 and pgv["one_backend"]["p50_ms_measured"] > 0
    assert pgv["parallel_seq_scan"]["queries_per_s_at_full_rows_extrapolated"] > 0
    # BASELINE.json configs[0] (100k rows) is measured as stated; 50k rows <= 1M are measured, not extrapolated
    assert cb["measured"][0]["rows"] == 100_000 and cb["measured"][0]["extrapolated"] is False
    assert cb["measured"][1]["rows"] == 50_000 and cb["extrapolated"] is False
    assert line["config"]["rows"] == 50_000 and line["config"]["batch"] == 1


def test_reference_arm_loads_no_product_library():
    """The CPU arm's process must not map liborx.so (VERDICT r1: it did, through the package __init__)."""
    code = ("import sys, types; sys.argv=['bench.py','--impl','reference','--rows','20000','--steps','2','--warmup','1'];"
            "import runpy; runpy.run_path('bench.py', run_name='__main__');"
            "maps=open('/proc/self/maps').read(); assert 'liborx' not in maps, 'product library mapped';"
            "assert 'outline_rag_b200' not in sys.modules; print('CLEAN')")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0 and "CLEAN" in out.stdout, out.stderr[-2000:]


def test_non_zero_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_dump_outputs_writes_the_last_timed_answer_the_same_on_every_run(tmp_path):
    """`--dump-outputs DIR`: the answer of the last of exactly `--steps` timed queries, as float64 arrays; the same
    arguments give the same inputs, so two runs write the same files."""
    dumps = []
    for run in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--rows", "20000",
                              "--steps", "5", "--warmup", "1", "--dump-outputs", str(tmp_path / run)],
                             capture_output=True, text=True, timeout=300, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        line = json.loads(out.stdout.strip().splitlines()[-1])
        assert line["steps"] == 5 and line["cpu_baseline"]["measured"][1]["queries"] == 5
        assert sorted(os.listdir(tmp_path / run)) == ["counts.npy", "distances.npy", "ids.npy"]
        dumps.append({n: np.load(tmp_path / run / f"{n}.npy") for n in ("ids", "distances", "counts")})
    a, b = dumps
    assert a["ids"].shape == (1, 12, 2) and a["distances"].shape == (1, 12) and a["counts"].tolist() == [12.0]
    assert all(v.dtype == np.float64 for v in a.values())
    assert (a["ids"][..., 0] == 0).all() and ((a["ids"][..., 1] >= 0) & (a["ids"][..., 1] < 20000)).all()
    assert (np.diff(a["distances"][0]) >= 0).all()
    for n in a:
        assert np.array_equal(a[n], b[n]), n


def test_dump_outputs_samples_an_answer_above_the_size_limit(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 10_000)
    B, k = 100, 12
    ids = np.zeros((B, k, 2), np.uint64)
    ids[:, :, 1] = np.arange(B * k, dtype=np.uint64).reshape(B, k) + np.uint64(2**53 - 1 - B * k)
    dist = np.random.default_rng(1).random((B, k))
    counts = np.full(B, k, np.int32)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), ids, dist, counts)
    got = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in ("ids", "distances", "counts", "query_index")}
    assert sum(v.nbytes for v in got.values()) <= 10_000
    sel = got["query_index"].astype(np.int64)
    assert len(sel) > 0 and (np.diff(sel) > 0).all() and sel[-1] < B
    assert np.array_equal(got["ids"], ids[sel].astype(np.float64))
    assert np.array_equal(got["ids"].astype(np.uint64), ids[sel])                  # exact below 2**53
    assert np.array_equal(got["distances"], dist[sel]) and (got["counts"] == k).all()
    assert np.array_equal(np.load(tmp_path / "b" / "query_index.npy"), got["query_index"])   # a fixed sample
