#!/usr/bin/env python
"""Loop-closure detection (SURVEY §8 f3, detection half): the online liogpu_sc_detect_loop at 10^3 / 10^4 / 10^5 stored
descriptors (snapshot rebuilt and not), one liogpu_sc_detect_loops call for a whole sequence (a call per keyframe) of
10^4 and 10^5 keyframes, and the radius detector liogpu_detect_loop_distance at 10^3 / 10^4 / 10^5 key poses.  Every
GPU result is compared with the CPU oracle first.

The CPU arm is the oracle's EXHAUSTIVE restatement (ring-key kNN by full scan of the snapshot), not the reference's
nanoflann tree, which is not part of this project; the reference's own comment puts its tree rebuild at "~5-50 ms wrt N"
(a comment in Scancontext.cpp, not a measurement).  The online records' `oracle_exhaustive_ms_1_thread` times a fresh
oracle manager that stores all n descriptors and then makes the one call, so it is not the cost of a call alone.

Descriptors: 500 Scan Context descriptors of seeded 32-beam sweeps along the synthetic path, made on the device, then
repeated with seeded multiplicative noise (1 +- 5 %) on the occupied bins to fill 10^5 distinct entries.  Timings do not
depend on the content except through the candidates' occupied columns.

    python tests/perf/bench_loop_detection.py [--out profiles/r03_loop_detection.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from lio_slam_b200 import synth  # noqa: E402
from lio_slam_b200.liogpu import LioGpu  # noqa: E402
from oracle.loop_oracle import LoopOracle  # noqa: E402

WARMUP, SAMPLES = 3, 20


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def make_descs(n, seed=1):
    import torch
    from lio_slam_b200 import synth_torch
    world = synth.make_world(1234)
    w = synth_torch.TorchWorld(world, torch.device("cuda", 0))
    g = LioGpu()
    base = []
    for j in range(500):
        rec = synth_torch.make_scan_records(w, synth.path_pose(0.37 * j), 32, seed=5000 + j, cols=900)
        base.append(g.make_scancontext((rec.data_ptr(), rec.shape[0], 32))[0])
    g.close()
    base = np.array(base)
    rng = np.random.default_rng(seed)
    out = np.empty((n, 20, 60))
    for a in range(0, n, 10000):
        b = min(n, a + 10000)
        out[a:b] = base[np.arange(a, b) % 500] * rng.uniform(0.95, 1.05, (b - a, 20, 60))
    out[:500] = base[: min(500, n)]
    return out


def stats(x):
    x = np.asarray(x, np.float64)
    return dict(median=float(np.median(x)), p10=float(np.percentile(x, 10)), p90=float(np.percentile(x, 90)), n=int(x.size))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_loop_detection.jsonl"))
    args = ap.parse_args()
    o = LoopOracle()
    threads = o.max_threads()
    gpu = card()
    recs = []

    def emit(**kw):
        kw = dict(gpu=gpu, **kw)
        print(json.dumps(kw), flush=True)
        recs.append(kw)

    descs = make_descs(100000)
    # ---- online call ------------------------------------------------------------------------------------------------
    for n in (1000, 10000, 100000):
        g = LioGpu()
        g.sc_add(descs[:n])
        want = o.sc_detect_loops(descs[:n], [n], threads=threads)[0]
        for rebuilt, period in (("rebuilt", 1), ("not_rebuilt", 1000000)):
            g.sc_clear()
            g.sc_add(descs[:n])
            wall, dev = [], []
            for it in range(WARMUP + SAMPLES):
                t0 = time.perf_counter()
                lid, yaw, info = g.sc_detect_loop(tree_making_period=period)
                t1 = time.perf_counter()
                if it == 0:
                    assert lid == want["loop_id"] and info["min_dist"] == want["min_dist"] and \
                        list(info["candidates"]) == list(want["candidates"]), (info, want)
                assert info["tree_rebuilt"] == (1 if (period == 1 or it == 0) else 0)
                if it >= WARMUP:
                    wall.append(1e3 * (t1 - t0))
                    dev.append(info["gpu_ms"])
            t0 = time.perf_counter()
            o.sc_detect_loops(descs[:n], [n], threads=1)
            cpu1 = 1e3 * (time.perf_counter() - t0)
            emit(stage="sc_detect_loop online", n_stored=n, snapshot=rebuilt, wall_ms=stats(wall), device_ms=stats(dev),
                 oracle_exhaustive_ms_1_thread=cpu1, parity="loop id, min_dist, candidates equal")
        g.close()
    # ---- whole sequence ---------------------------------------------------------------------------------------------
    for n in (10000, 100000):
        g = LioGpu()
        g.sc_add(descs[:n])
        sizes = np.arange(1, n + 1)
        g.sc_detect_loops(sizes[: min(n, 2000)])  # warm-up
        wall, dev = [], []
        for _ in range(3 if n == 100000 else 10):
            t0 = time.perf_counter()
            ids, yaw, md = g.sc_detect_loops(sizes)
            wall.append(1e3 * (time.perf_counter() - t0))
            dev.append(g.last_gpu_ms())
        t0 = time.perf_counter()
        want = o.sc_detect_loops(descs[:n], sizes, threads=threads)
        cpu_all = 1e3 * (time.perf_counter() - t0)
        assert np.array_equal(ids, [r["loop_id"] for r in want])
        assert np.array_equal(md.view(np.uint64), np.array([r["min_dist"] for r in want]).view(np.uint64))
        cpu1 = None
        if n <= 10000:
            t0 = time.perf_counter()
            o.sc_detect_loops(descs[:n], sizes, threads=1)
            cpu1 = 1e3 * (time.perf_counter() - t0)
        emit(stage="sc_detect_loops whole sequence", n_keyframes=n, n_calls=n, loops=int((ids >= 0).sum()),
             wall_ms=stats(wall), device_ms=stats(dev), oracle_exhaustive_ms_all_threads=cpu_all, oracle_threads=threads,
             oracle_exhaustive_ms_1_thread=cpu1 if cpu1 is not None else "not measured (too slow on one core)",
             parity="loop ids and min_dist bits equal on every call")
        g.close()
    # ---- radius detector --------------------------------------------------------------------------------------------
    g = LioGpu()
    rng = np.random.default_rng(4)
    for n in (1000, 10000, 100000):
        arc = 0.35 * np.arange(n)
        th = arc / 8.0
        key = np.c_[8 * np.cos(th), 8 * np.sin(th), 0.02 * np.sin(th) + rng.normal(0, 0.05, n), np.arange(n)].astype(np.float32)
        t = 0.1 * np.arange(n, dtype=np.float64)
        want = o.detect_loop_distance(key, t, t[-1], 10.0, 30.0)
        wall, dev = [], []
        for it in range(WARMUP + SAMPLES):
            t0 = time.perf_counter()
            got = g.detect_loop_distance(key, t, t[-1], 10.0, 30.0)
            t1 = time.perf_counter()
            assert got == want
            if it >= WARMUP:
                wall.append(1e3 * (t1 - t0))
                dev.append(g.last_gpu_ms())
        cpu = []
        for _ in range(5):
            t0 = time.perf_counter()
            o.detect_loop_distance(key, t, t[-1], 10.0, 30.0)
            cpu.append(1e3 * (time.perf_counter() - t0))
        emit(stage="detect_loop_distance", n_key_poses=n, wall_ms=stats(wall), device_ms=stats(dev),
             oracle_ms_1_thread=stats(cpu), parity="same loop_key_pre")
    g.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for r in recs:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
