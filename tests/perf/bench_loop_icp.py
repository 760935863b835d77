#!/usr/bin/env python
"""Loop-closure ICP for many candidate pairs (liogpu_loop_closure_icp_batch) against the path it replaces.

Keyframes: 64-beam sweeps (900 columns, kitti.yaml's downsampleRate 2 of 1800) voxelised at 0.4 m (its
mappingSurfLeafSize), every 0.65 m along two laps of synth.path_pose; the second lap's key poses drift so that ICP has
work.  Pairs (lap-2 keyframe, the lap-1 keyframe at the same place), historyKeyframeSearchNum 25, leaf 0.3 (utility.h
defaults).  Three arms, warmed up, median of >= 10 repetitions:
  (a) the mirror's old loopClosureICP: merge_keyframes of both windows fetched to the host, then icp_align, per pair;
  (b) liogpu_loop_closure_icp_batch with one pair per call;
  (c) one liogpu_loop_closure_icp_batch call for all B pairs.
Every run checks that (c) is bit-equal to (a).  Device split of (c): submap assembly = the device time of the same
merge_keyframes calls in (a) (same code), ICP = the rest of (c)'s device time.

    python tests/perf/bench_loop_icp.py [--out profiles/r04_loop_icp_batch.jsonl]
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

SEARCH_NUM, LEAF, REPS, WARMUP = 25, 0.3, 10, 2


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def keyframes(g, n_key):
    import torch
    from lio_slam_b200 import synth_torch
    w = synth_torch.TorchWorld(synth.make_world(1234), torch.device("cuda", 0))
    lap = n_key // 2
    poses = []
    for j in range(n_key):
        s = 0.65 * j
        rec = synth_torch.make_scan_records(w, synth.path_pose(s), 64, seed=7000 + j, cols=900)
        ds, _ = g.voxel_downsample((rec.data_ptr(), rec.shape[0], 32), 0.4)
        g.keyframe_put(j, ds)
        p = synth.path_pose(s).astype(np.float32)
        if j >= lap:
            f = (j - lap + 1) / lap
            p[3] += 0.8 * f
            p[4] -= 0.5 * f
            p[2] += 0.03 * f
        poses.append(p)
    return np.array(poses, np.float32)


def window(key, s, n_key):
    return list(range(max(key - s, 0), min(key + s, n_key - 1) + 1))


def stats(x):
    x = np.asarray(x, np.float64)
    return dict(median=float(np.median(x)), p10=float(np.percentile(x, 10)), p90=float(np.percentile(x, 90)), n=int(x.size))


def arm_a(g, pairs, poses):
    """merge both windows to the host, then icp_align: (T, infos, submap device ms, icp device ms, launches, bytes)"""
    n_key = poses.shape[0]
    Ts, infos, sub_ms, icp_ms, nbytes = [], [], 0.0, 0.0, 0
    l0 = g.launch_count()
    for c, p in pairs:
        src, _ = g.merge_keyframes([c], poses[[c]], LEAF)
        sub_ms += g.last_gpu_ms()
        w = window(p, SEARCH_NUM, n_key)
        tgt, _ = g.merge_keyframes(w, poses[w], LEAF)
        sub_ms += g.last_gpu_ms()
        nbytes += 2 * 16 * (src.shape[0] + tgt.shape[0])           # down to the host and back up
        T, info = g.icp_align(src, tgt)
        icp_ms += info["gpu_ms"]
        Ts.append(T)
        infos.append(info)
    return np.array(Ts), infos, sub_ms, icp_ms, g.launch_count() - l0, nbytes


def timed(fn, reps=REPS, warmup=WARMUP):
    out, wall = None, []
    for it in range(warmup + reps):
        t0 = time.perf_counter()
        out = fn()
        t1 = time.perf_counter()
        if it >= warmup:
            wall.append(1e3 * (t1 - t0))
    return out, wall


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_loop_icp_batch.jsonl"))
    ap.add_argument("--keyframes", type=int, default=160)
    args = ap.parse_args()
    gpu = card()
    g = LioGpu()
    poses = keyframes(g, args.keyframes)
    lap = args.keyframes // 2
    pool = [(j, j - lap) for j in range(lap, args.keyframes)]
    recs = []
    for b in (1, 8, 64, 256):
        pairs = [pool[(7 * j) % len(pool)] for j in range(b)]
        cur = np.array([c for c, _ in pairs], np.int32)
        pre = np.array([p for _, p in pairs], np.int32)
        (Ta, ia, sub_ms, icp_ms, la, bytes_a), wall_a = timed(lambda: arm_a(g, pairs, poses))

        def arm_b():
            l0, dev = g.launch_count(), 0.0
            for c, p in pairs:
                g.loop_closure_icp_batch([c], [p], poses, search_num=SEARCH_NUM, icp_leaf=LEAF)
                dev += g.last_gpu_ms()
            return dev, g.launch_count() - l0
        (dev_b, lb), wall_b = timed(arm_b)

        def arm_c():
            l0 = g.launch_count()
            T, res = g.loop_closure_icp_batch(cur, pre, poses, search_num=SEARCH_NUM, icp_leaf=LEAF)
            return T, res, g.last_gpu_ms(), g.launch_count() - l0
        (Tc, rc, dev_c, lc), wall_c = timed(arm_c)
        assert np.array_equal(Tc.view(np.uint32), Ta.view(np.uint32)), "batched T differs from the two-call path"
        for r, i in zip(rc, ia):
            for k in ("iterations", "convergence_state", "converged", "n_correspondences", "fitness_score", "last_mse"):
                assert r[k] == i[k], (k, r[k], i[k])
        ns = [r["n_source"] for r in rc]
        nt = [r["n_target"] for r in rc]
        # host <-> device traffic of (c): per window the keyframe table (poses, offsets, pointers) and the results
        n_win = sum(1 + len(window(p, SEARCH_NUM, args.keyframes)) for _, p in pairs)
        bytes_c = n_win * (6 * 4 + 4 + 8) + b * 160
        med = {k: float(np.median(v)) for k, v in (("a", wall_a), ("b", wall_b), ("c", wall_c))}
        rec = dict(gpu=gpu, stage="loop-closure ICP batch", pairs=b, n_key=args.keyframes, search_num=SEARCH_NUM, leaf=LEAF,
                   n_source_median=float(np.median(ns)), n_target_median=float(np.median(nt)),
                   iterations_max=int(max(r["iterations"] for r in rc)), converged=int(sum(r["converged"] for r in rc)),
                   wall_ms=dict(a_two_calls=stats(wall_a), b_one_pair_per_call=stats(wall_b), c_batched=stats(wall_c)),
                   pairs_per_s=dict(a_two_calls=1e3 * b / med["a"], b_one_pair_per_call=1e3 * b / med["b"],
                                    c_batched=1e3 * b / med["c"]),
                   device_ms=dict(a_submaps=sub_ms, a_icp=icp_ms, b_total=dev_b, c_total=dev_c,
                                  c_icp_estimate=dev_c - sub_ms),
                   launches=dict(a_two_calls=int(la), b_one_pair_per_call=int(lb), c_batched=int(lc)),
                   pcie_bytes=dict(a_two_calls=int(bytes_a), c_batched=int(bytes_c)),
                   c_faster_per_pair_than_b=bool(med["c"] < med["b"]),
                   parity="(c) bit-equal to (a): T, iterations, state, correspondences, fitness, last MSE")
        print(json.dumps(rec), flush=True)
        recs.append(rec)
    g.close()
    with open(args.out, "w") as f:
        for r in recs:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
