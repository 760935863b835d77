#!/usr/bin/env python
"""Loop-closure submaps built many windows at a time (liogpu_merge_keyframes_batch) against one window per call
(liogpu_merge_keyframes).

Keyframes, pairs and windows are those of bench_loop_icp.py: 64-beam sweeps voxelised at 0.4 m every 0.65 m along two
laps, pairs (lap-2 keyframe, the lap-1 keyframe at the same place), historyKeyframeSearchNum 25, leaf 0.3.  For B = 1,
8, 64 and 256 pairs the 2B windows (each pair's source keyframe and its target window) are built
  (a) by 2B liogpu_merge_keyframes calls,
  (b) by one liogpu_merge_keyframes_batch call,
both writing to device memory (nothing is fetched to the host), warmed up, median of >= 10 repetitions.  Every run
checks that each window of (b) is byte-equal to (a).  Host round trips, counted from the code: two per window for (a)
(the VoxelGrid's voxel count, then the copy out), two per pass of at most 2^25 input points plus the copy out for (b).

    python tests/perf/bench_merge_batch.py [--out profiles/r04_merge_batch.jsonl]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bench_loop_icp import LEAF, SEARCH_NUM, card, keyframes, stats, timed, window  # noqa: E402
from lio_slam_b200.liogpu import LioGpu  # noqa: E402

PASS_POINTS = 1 << 25


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_merge_batch.jsonl"))
    ap.add_argument("--keyframes", type=int, default=160)
    args = ap.parse_args()
    gpu = card()
    g = LioGpu()
    poses = keyframes(g, args.keyframes)
    sizes = [g.merge_keyframes([j], poses[[j]], 0.0)[0].shape[0] for j in range(args.keyframes)]
    lap = args.keyframes // 2
    pool = [(j, j - lap) for j in range(lap, args.keyframes)]
    out_single = torch.empty((1 << 22, 4), dtype=torch.float32, device="cuda")
    recs = []
    for b in (1, 8, 64, 256):
        pairs = [pool[(7 * j) % len(pool)] for j in range(b)]
        windows = []
        for c, p in pairs:
            for w in ([c], window(p, SEARCH_NUM, args.keyframes)):
                windows.append((np.asarray(w, np.int32), np.ascontiguousarray(poses[w], np.float32)))

        def arm_single():
            l0, dev, n_out = g.launch_count(), 0.0, []
            for w, pw in windows:
                n = C.c_int(0)
                st = g.lib.liogpu_merge_keyframes(g.h, w.ctypes.data, pw.ctypes.data, len(w), C.c_float(LEAF),
                                                  out_single.data_ptr(), 16, out_single.shape[0], C.byref(n))
                assert st >= 0, st
                dev += g.last_gpu_ms()
                n_out.append(n.value)
            return dev, g.launch_count() - l0, n_out
        (dev_a, la, n_a), wall_a = timed(arm_single)

        flat_ids = np.concatenate([w for w, _ in windows])
        flat_poses = np.ascontiguousarray(np.concatenate([pw for _, pw in windows]), np.float32)
        win_off = np.r_[0, np.cumsum([len(w) for w, _ in windows])].astype(np.int32)
        out_off = np.zeros(len(windows) + 1, np.int32)
        out_batch = torch.empty((max(sum(n_a), 1), 4), dtype=torch.float32, device="cuda")

        def arm_batch():
            l0 = g.launch_count()
            st = g.lib.liogpu_merge_keyframes_batch(g.h, flat_ids.ctypes.data, flat_poses.ctypes.data,
                                                    win_off.ctypes.data, len(windows), C.c_float(LEAF),
                                                    out_batch.data_ptr(), 16, out_batch.shape[0], out_off.ctypes.data,
                                                    None)
            assert st >= 0, st
            return g.last_gpu_ms(), g.launch_count() - l0, np.diff(out_off).tolist()
        (dev_b, lb, n_b), wall_b = timed(arm_batch)

        assert n_b == n_a, "merge_keyframes_batch sizes differ from merge_keyframes"
        clouds, _, _ = g.merge_keyframes_batch(windows, LEAF)
        for (w, pw), cl in zip(windows, clouds):
            ref, _ = g.merge_keyframes(w, pw, LEAF)
            assert ref.tobytes() == cl.tobytes(), "merge_keyframes_batch differs from merge_keyframes"
        n_in = [sum(sizes[i] for i in w) for w, _ in windows]
        passes, acc = 1, n_in[0]
        for m in n_in[1:]:
            if acc + m > PASS_POINTS:
                passes, acc = passes + 1, m
            else:
                acc += m
        med_a, med_b = float(np.median(wall_a)), float(np.median(wall_b))
        rec = dict(gpu=gpu, stage="loop-closure submaps, many windows per call", pairs=b, windows=len(windows),
                   n_key=args.keyframes, search_num=SEARCH_NUM, leaf=LEAF, input_points=int(sum(n_in)),
                   output_points=int(sum(n_a)), passes=passes,
                   wall_ms=dict(a_merge_keyframes=stats(wall_a), b_merge_keyframes_batch=stats(wall_b)),
                   device_ms=dict(a_merge_keyframes=dev_a, b_merge_keyframes_batch=dev_b),
                   launches=dict(a_merge_keyframes=int(la), b_merge_keyframes_batch=int(lb)),
                   host_round_trips=dict(a_merge_keyframes=2 * len(windows), b_merge_keyframes_batch=2 * passes + 1),
                   speedup_wall=med_a / med_b,
                   parity="every window of (b) byte-equal to merge_keyframes")
        print(json.dumps(rec), flush=True)
        recs.append(rec)
    g.close()
    with open(args.out, "w") as f:
        for r in recs:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
