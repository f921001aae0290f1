"""bench.py contract: the reference arm prints one JSON line with the agreed keys (CPU); --dump-outputs writes the
per-pod outputs of the last timed step exactly (encoding on CPU, the timed path on the GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--cfg", "1",
                        "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["unit"] == "decisions/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["vs_baseline"] is None
    assert "workload" in line["config"]


def test_ncu_traffic_summary_is_readable():
    sys.path.insert(0, ROOT)
    import importlib
    bench = importlib.import_module("bench")
    t, src = bench.ncu_traffic()
    assert t is None or (t > 2.0e8 and t < 3.2e8), (t, src)   # ~276 MB per 4M-node launch vs 280 MB algorithmic


def test_reference_arm_under_torchrun_prints_once():
    """The driver launches the reference arm like the GPU arm (torchrun, N ranks): rank 0 alone measures and prints,
    the other ranks exit 0 without work."""
    port = 29900 + os.getpid() % 500
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "bench.py"),
                        "--impl", "reference", "--gpus", "2", "--cfg", "1", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [json.loads(x) for x in r.stdout.splitlines() if x.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    assert lines[0]["impl"] == "reference" and lines[0]["n_gpus"] == 2 and lines[0]["value"] > 0


def test_steps_below_one_is_rejected():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                       timeout=120)
    assert r.returncode == 2 and "--steps" in r.stderr, r.stderr[-2000:]


def _read_dump(d):
    got = {f: np.load(os.path.join(d, f + ".npy")) for f in ("node", "status", "alloc_mask", "fit_count")}
    for f in ("fit_digest", "score_digest"):
        a = np.load(os.path.join(d, f + ".npy"))
        assert a.dtype == np.float64 and a.shape[1] == 2
        got[f] = a[:, 0].astype(np.uint64) | (a[:, 1].astype(np.uint64) << np.uint64(32))
    return got


def test_write_outputs_round_trips_exactly(tmp_path):
    import bench
    rng = np.random.default_rng(7)
    P = 1000
    out = dict(node=rng.integers(-1, 100000, P, dtype=np.int32), status=rng.integers(0, 4, P, dtype=np.int32),
               alloc_mask=rng.integers(0, 256, (P, 4), dtype=np.uint8), fit_count=rng.integers(0, 100000, P, dtype=np.int32),
               fit_digest=rng.integers(0, 2**64, P, dtype=np.uint64), score_digest=rng.integers(0, 2**64, P, dtype=np.uint64))
    out["fit_digest"][:2] = [0, 2**64 - 1]
    bench.write_outputs(str(tmp_path), out)
    assert sorted(os.listdir(tmp_path)) == sorted(f + ".npy" for f in bench.FIELDS)
    got = _read_dump(str(tmp_path))
    for f in bench.FIELDS:
        assert np.array_equal(got[f], out[f].astype(got[f].dtype)), f
        assert np.load(os.path.join(tmp_path, f + ".npy")).dtype in (np.float32, np.float64)


@pytest.mark.gpu
def test_dump_outputs_are_the_timed_step_and_match_the_oracle(tmp_path):
    """The dumped arrays are the driver rule's per-pod answers for the benchmark batch (config 4, a pod prefix)."""
    import bench
    import egs_b200
    P = 2000
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--pods", str(P), "--steps", "2", "--warmup", "1",
                        "--no-cpu", "--no-roofline", "--no-configs", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    got = _read_dump(str(tmp_path))
    w = egs_b200.workloads.config(4).prefix(P)
    ref = bench.oracle_for(w).schedule_batch(w.c_off, w.units64(), threads=4)
    for f in bench.FIELDS:
        assert got[f].shape == ref[f].shape, f
        assert np.array_equal(got[f], ref[f].astype(got[f].dtype)), f
