#!/usr/bin/env python
"""Whole-sequence radius loop detection (detectLoopClosureDistance with a call per keyframe) and the host mirror's
offline loop-closure pass.

Radius detection at 10^3 .. 10^6 key poses, radius 10 m, time_diff 30 s, call j on the first j + 1 key poses at that
pose's time + 0.05 s.  Two shapes:
  path        a drive on a street grid (blocks of 100 m, keyframes 1 m and 0.1 s apart, a random turn at every
              intersection) in a square that grows with the sequence (200 m at 10^3 .. 2 km at 10^6): revisits from
              the second pass over a street on;
  stationary  every key pose within 0.2 m of the origin: every pose is within the radius of every query and the grid is
              one cell, so every arm is O(n^2).  Run up to 10^5 (10^6 would be 5 * 10^11 pair tests in every arm).
Arms:
  per_call   liogpu_detect_loop_distance on each call's prefix (uploads the prefix every call);
  host_1t    the mirror's host loop (map_optimization_gpu.cpp detectLoopClosureDistance) on one thread;
  host_all   the same loop with the calls spread over every core (OpenMP, one call per iteration);
  batch      one liogpu_detect_loops_distance call.
The batch arm answers every call; its median over REPS runs after a warm-up is reported with the spread.  The other
arms run a strided sample of the calls when the whole sequence would take too long (`calls_timed` < `calls`): their
whole-sequence time is the sample's time scaled by calls / calls_timed (`extrapolated`).  Parity is asserted in the
run: the batch answers equal per_call's and the host loop's on every timed call.

Offline loop closure at 10^4 keyframes: tests/loop_offline_mirror.cpp runs the loop thread per tick (performRSLoopClosure
+ performSCLoopClosure) and performLoopClosuresOffline over the same ticks, and checks every tick equal.

    python tests/perf/bench_loop_distance_batch.py [--out profiles/r05_loop_distance_batch.jsonl]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
from bench_loop_icp import card, stats  # noqa: E402
from lio_slam_b200.liogpu import LioGpu  # noqa: E402

RADIUS, TIME_DIFF, REPS = 10.0, 30.0, 5
SAMPLE = {1000: 1000, 10000: 10000, 100000: 1000, 1000000: 200}  # per-call arms: calls timed per size

HOST_LOOP = r'''
// detectLoopClosureDistance's host loop of map_optimization_gpu.cpp, for many calls (each call reads a prefix)
#include <cmath>
#include <omp.h>
extern "C" int n_procs() { return omp_get_num_procs(); }
extern "C" void run(const float* key, const double* t, const int* at, const double* tc, int n_calls, float radius,
                    float time_diff, int threads, int* out) {
  const float r2 = (float)((double)radius * (double)radius);
#pragma omp parallel for schedule(dynamic, 16) num_threads(threads)
  for (int j = 0; j < n_calls; ++j) {
    const int n = at[j];
    const float* last = key + 4 * (n - 1);
    int pre = -1;
    float best = 0.f;
    for (int i = 0; i < n; ++i) {
      const float* p = key + 4 * i;
      float d2 = 0.f, d = last[0] - p[0];
      d2 += d * d; d = last[1] - p[1];
      d2 += d * d; d = last[2] - p[2];
      d2 += d * d;
      if (!(d2 < r2) || !(std::fabs(t[i] - tc[j]) > (double)time_diff)) continue;
      if (pre < 0 || d2 < best) { pre = i; best = d2; }
    }
    out[j] = pre == n - 1 ? -1 : pre;
  }
}
'''


def host_lib(tmp):
    src = os.path.join(tmp, "host_loop.cpp")
    so = os.path.join(tmp, "host_loop.so")
    with open(src, "w") as f:
        f.write(HOST_LOOP)
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++14", "-fPIC", "-shared", "-fopenmp", "-ffp-contract=off",
                           src, "-o", so])
    lib = C.CDLL(so)
    lib.run.argtypes = [C.c_void_p] * 4 + [C.c_int, C.c_float, C.c_float, C.c_int, C.c_void_p]
    return lib


def street_path(n, seed=1):
    rng = np.random.default_rng(seed)
    side = int(np.clip(2 * np.sqrt(n) // 100 * 100, 200, 2000))
    pos, d = np.array([0.0, 0.0]), np.array([1.0, 0.0])
    pts = []
    while len(pts) < n:
        for _ in range(100):
            pos = pos + d
            pts.append(pos.copy())
        turns = [t for t in (d, d[::-1] * [1, -1], d[::-1] * [-1, 1]) if 0 <= (pos + 100 * t)[0] <= side and
                 0 <= (pos + 100 * t)[1] <= side]
        d = turns[rng.integers(len(turns))] if turns else -d
    xy = np.array(pts[:n]) + rng.normal(0.0, 0.3, (n, 2))
    z = rng.normal(0.0, 0.05, (n, 1))
    return np.c_[xy, z, np.arange(n)].astype(np.float32), np.arange(n) * 0.1


def stationary(n, seed=2):
    rng = np.random.default_rng(seed)
    return np.c_[rng.normal(0.0, 0.1, (n, 3)).clip(-0.2, 0.2), np.arange(n)].astype(np.float32), np.arange(n) * 0.1


def timed(fn, reps):
    fn()  # warm-up
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return ts


def radius_records(g, hl, n, shape, meta):
    key, t = (street_path if shape == "path" else stationary)(n)
    at = np.arange(1, n + 1, dtype=np.int32)
    tc = t + 0.05
    rec = dict(meta, bench="loop_distance_batch", shape=shape, n_key=n, calls=n, radius=RADIUS, time_diff=TIME_DIFF)
    got = g.detect_loops_distance(key, t, at, tc, RADIUS, TIME_DIFF)
    gpu_ms = []

    def batch():
        g.detect_loops_distance(key, t, at, tc, RADIUS, TIME_DIFF)
        gpu_ms.append(g.last_gpu_ms())
    out = [dict(rec, arm="batch", calls_timed=n, extrapolated=False, wall_s=stats(timed(batch, REPS)),
                device_ms=stats(gpu_ms[1:]), hits=int((got >= 0).sum()))]
    k = SAMPLE[n] if shape == "path" or n <= 10000 else max(SAMPLE[n] // 10, 50)
    idx = np.unique(np.linspace(0, n - 1, min(k, n)).round().astype(np.int64))
    s_at, s_tc = np.ascontiguousarray(at[idx]), np.ascontiguousarray(tc[idx])
    scale = n / idx.size
    res = {}

    def per_call():
        res["per_call"] = np.array([g.detect_loop_distance(key[:m], t[:m], c, RADIUS, TIME_DIFF) for m, c in zip(s_at, s_tc)])
    ts = timed(per_call, REPS)
    out.append(dict(rec, arm="per_call", calls_timed=int(idx.size), extrapolated=bool(idx.size < n),
                    wall_s=stats(np.array(ts) * scale)))
    threads = {"host_1t": 1, "host_all": int(hl.n_procs())}
    for arm, th in threads.items():
        o = np.zeros(idx.size, np.int32)

        def host():
            hl.run(key.ctypes.data, t.ctypes.data, s_at.ctypes.data, s_tc.ctypes.data, idx.size, C.c_float(RADIUS),
                   C.c_float(TIME_DIFF), th, o.ctypes.data)
        ts = timed(host, REPS)
        res[arm] = o.copy()
        out.append(dict(rec, arm=arm, threads=th, calls_timed=int(idx.size), extrapolated=bool(idx.size < n),
                        wall_s=stats(np.array(ts) * scale)))
    for arm in ("per_call", "host_1t", "host_all"):
        assert np.array_equal(res[arm], got[idx]), (shape, n, arm)
    for r in out:
        r["parity"] = "batch == per_call == host loop on every timed call"
    return out


def mirror_record(meta, n_target):
    import test_gpu_loop_distance_batch as T
    from lio_slam_b200 import synth
    laps = max(2, n_target // T.N_POOL)
    case = T.mirror_case(synth.make_world(1234), laps=laps, search_num=25, exclude=30, cols=120, tick_stride=10 ** 9)
    with tempfile.TemporaryDirectory() as tmp:
        exe = T.build_mirror(tmp)
        blob = os.path.join(tmp, "case.bin")
        T.write_mirror_case(blob, case)
        r, s = T.run_mirror(exe, blob)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    return dict(meta, bench="loop_closure_offline", n_key=int(case["poses"].shape[0]), ticks=int(s["ticks"]),
                search_num=25, num_exclude_recent=30, online_ms=s["online_ms"], offline_ms=s["offline_ms"],
                online_icp=int(s["online_icp"]), offline_icp=int(s["offline_icp"]),
                rs_detected=int(s["rs_detected"]), rs_accepted=int(s["rs_accepted"]),
                sc_detected=int(s["sc_detected"]), sc_accepted=int(s["sc_accepted"]),
                parity="every tick's pairs, acceptances, correction bytes and noise scores equal")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_loop_distance_batch.jsonl"))
    ap.add_argument("--sizes", default="1000,10000,100000,1000000")
    ap.add_argument("--mirror-keyframes", type=int, default=10000)
    a = ap.parse_args()
    c = [x.strip() for x in card().split(",")]
    meta = dict(card=c[0], power_limit=c[1] if len(c) > 1 else None, max_sm_clock=c[2] if len(c) > 2 else None,
                host_cores=os.cpu_count())
    g = LioGpu()
    records = []
    with tempfile.TemporaryDirectory() as tmp:
        hl = host_lib(tmp)
        for n in [int(x) for x in a.sizes.split(",")]:
            for shape in ("path", "stationary"):
                if shape == "stationary" and n > 100000:
                    continue
                for r in radius_records(g, hl, n, shape, meta):
                    print(json.dumps(r), flush=True)
                    records.append(r)
    g.close()
    if a.mirror_keyframes > 0:
        r = mirror_record(meta, a.mirror_keyframes)
        print(json.dumps(r), flush=True)
        records.append(r)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for r in records:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
