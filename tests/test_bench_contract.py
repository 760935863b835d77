"""bench.py prints exactly one JSON line with the keys the driver's contract names.  The reference arm runs on
the CPU (here, small workload); the GPU arm is checked on the GPU box."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "cpu_baseline"}


def run_bench(*args, timeout=600):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=timeout, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    return json.loads(lines[0])


def test_reference_arm_line():
    d = run_bench("--impl", "reference", "--workload", "cfg1", "--steps", "1", "--warmup", "1")
    assert BASE_KEYS <= set(d) and d["impl"] == "reference" and d["steps"] == 1
    assert d["metric"] == "scan2map_registrations_per_sec" and d["unit"] == "registrations/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["vs_baseline"] is None and d["data"] == "synthetic" and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


@pytest.mark.gpu
def test_gpu_arm_line():
    d = run_bench("--workload", "cfg1", "--steps", "5", "--warmup", "3", "--cpu-steps", "3", "--seq-scans", "12")
    assert BASE_KEYS | {"roofline", "clocks", "cfg1", "cfg4", "cfg5", "lm_loop_ab", "like_for_like"} <= set(d)
    assert d["cfg4"]["bit_equal_to_1gpu"] is True and d["cfg4"]["n_points"] > 4_000_000
    assert d["cfg5"]["total_scans"] == 8 * 12 and d["cfg5"]["value"] > 0 and d["cfg5"]["scaling"] == "strong"
    assert d["cfg5"]["max_position_error_vs_ground_truth_m"] < 0.15
    assert d["lm_loop_ab"]["fused_one_launch"]["poses_bit_equal_to_two_kernel"] in (True, False)
    assert set(d["cpu_baseline"]["by_number_of_cores"]) >= {"4"}
    assert d["n_gpus"] == 1 and d["steps"] == 5 and d["warmup"] >= 3 and d["scaling"] == "weak" and d["dtype"] == "f32"
    assert d["value"] > 0 and d["gpu_launches"] > 0
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and "traffic" in r
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["value"] != d["value"]
    cb = d["cpu_baseline"]
    assert cb["value"] > 0 and cb["cores"] >= 1 and cb["kind"] == "port"
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}


@pytest.mark.gpu
def test_gpu_arm_dump_outputs(tmp_path):
    """--dump-outputs writes what the last timed registration returned: the same bytes from run to run, and the same
    bytes as one registration of that sweep outside the bench"""
    from bench import MAX_ITER, WORKLOADS, make_workload
    from lio_slam_b200.liogpu import LioGpu, default_params
    runs = []
    for k in range(2):
        out = tmp_path / f"run{k}"
        d = run_bench("--workload", "cfg1", "--steps", "3", "--warmup", "1", "--no-extras", "--no-cpu-baseline",
                      "--dump-outputs", str(out))
        assert d["steps"] == 3
        runs.append({f[:-4]: np.load(out / f) for f in os.listdir(out)})
    a, b = runs
    assert set(a) == {"pose", "matP", "status", "n_query", "iterations", "converged", "n_sel", "is_degenerate",
                      "tie_queries", "delta_r", "delta_t", "JtJ", "Jtr", "pose_hist", "nsel_hist"}
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    for name, v in a.items():
        assert v.dtype in (np.float32, np.float64), name
        assert v.dtype == b[name].dtype and v.shape == b[name].shape and v.tobytes() == b[name].tobytes(), name
    w = WORKLOADS["cfg1"]
    map4, scans, guesses = make_workload("cfg1", 0)
    g = LioGpu(default_params(n_scan=w["beams"], horizon_scan=w["cols"], surrounding_keyframe_map_leaf_size=w["map_leaf"]))
    g.set_local_map(map4)
    pose, P, info = g.scan2map(scans[2], guesses[2], max_iter=MAX_ITER)   # step 2 of 3 registers sweep 2
    g.close()
    assert np.array_equal(pose.view(np.uint32), a["pose"].view(np.uint32)) and np.array_equal(P, a["matP"])
    assert a["iterations"].tolist() == [info["iterations"]] and np.array_equal(a["pose_hist"], info["pose_hist"])
