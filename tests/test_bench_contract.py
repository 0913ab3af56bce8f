"""bench.py's contract, as far as a machine without a GPU can check it: the reference arm (which times the oracle on the
host cores and needs no device) prints one JSON line with the keys the driver reads, and its `config` equals the one
the B200 arm would print for the same command line (the driver compares the two arms on `config`)."""
import json
import os
import subprocess
import sys
from types import SimpleNamespace

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_reference_arm_prints_the_contract_line():
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "3", "--warmup", "1", "--repeats", "2", "--prime", "4"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1  # ONE JSON line
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 1 and d["steps"] == 3 and d["warmup"] == 1
    assert d["metric"].startswith("scans/sec") and d["unit"] == "scans/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["data"] == "synthetic" and d["vs_baseline"] is None
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and isinstance(cb["sample"], str)
    assert d["e2e"] == {"value": d["value"], "unit": "scans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["windows"]["scans"] == [2, 1] and len(d["windows"]["ms"]) == 2  # --steps 3 timed scans in --repeats 2 windows
    # the same command line gives the same `config` in both arms
    import bench
    args = SimpleNamespace(gpus=1, steps=3, warmup=1, repeats=2, prime=4, workload="kitti", impl="b200", cpu_sample=60, streams=4,
                           no_nn=False, no_cpu=False, no_extra=False, no_clocks=False)
    assert bench.common_config(args, 1) == d["config"]
    assert "workload" in d["config"] and "model" not in d["config"]


def test_steps_set_the_number_of_timed_scans():
    import bench
    for steps, repeats, sizes in ((20, None, [20]), (50, None, [25, 25]), (7, 3, [3, 2, 2]), (2, 5, [1, 1]), (180, 9, [20] * 9)):
        assert bench.window_sizes(SimpleNamespace(steps=steps, repeats=repeats)) == sizes


@pytest.mark.gpu
def test_dump_outputs_are_what_the_last_timed_scan_returned(tmp_path):
    """bench.py --dump-outputs against the same stream registered one blocking call at a time"""
    import numpy as np
    import kiss_icp_b200 as K
    from kiss_icp_b200 import synthetic
    prime, warmup, steps = 4, 1, 3
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup),
           "--prime", str(prime), "--no-nn", "--no-cpu", "--no-extra", "--no-clocks", "--streams", "0", "--dump-outputs", str(tmp_path)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    dumped = {n: np.load(tmp_path / f"{n}.npy") for n in ("pose", "preprocessed", "source")}
    assert all(a.dtype == np.float64 for a in dumped.values())
    lidar = synthetic.kitti_shape(seed=0, device="cuda")
    icp = K.KissICP(K.load_config())
    for k in range(prime + warmup + steps):
        pre, src = icp.register_frame(*lidar.scan(k))
    assert np.array_equal(dumped["preprocessed"], pre) and np.array_equal(dumped["source"], src)
    assert np.abs(dumped["pose"] - icp.last_pose).max() < 1e-9


def test_profiled_traffic_reads_the_committed_ncu_summaries():
    import bench
    for tag in ("r2_register_frame", "r1_nn_query", "r2_nn_query"):
        traffic, src = bench.profiled_traffic(tag)
        assert traffic is not None and traffic > 1e6 and tag in src and src.startswith("static")
    assert bench.profiled_traffic("r9_nothing") == (None, None)
