#!/usr/bin/env python
"""Scan Context descriptor store filled from resident keyframes: one liogpu_sc_add_keyframes call against the
per-keyframe path (liogpu_make_scancontext + liogpu_sc_add for every keyframe), and the offline loop-closure chain on
the device (descriptors, detection, ICP).

Keyframes: P = 200 distinct 64-beam sweeps (900 columns) taken every 0.65 m along synth.path_pose, voxelised at 0.2 m
(the default mappingSurfLeafSize of liogpu_default_params), repeated in turn to fill 10^3, 10^4 and 10^5 keyframe ids
(each id is a keyframe of its own in HBM).  The second and later laps' key poses drift, as in bench_loop_icp.py.

  (a) per-keyframe: for every keyframe, make_scancontext of its cloud (a device copy: no host-to-device upload of the
      cloud) and sc_add of the descriptor, through ctypes with preallocated buffers: 2 host round trips per keyframe;
  (b) batch: one sc_add_keyframes call over all ids (descriptors stay on the device); one host round trip per pass of
      at most 2^31 - 1 points.
Warmed up once, then REPS repetitions on a cleared store, median and spread.  Wall = host clock around the arm (the
calls end with a stream sync); device = the sum of liogpu_last_gpu_ms over the arm's calls.  Every size checks the
batch descriptors (written to device memory) byte-equal to (a), and at 10^3 and 10^4 the two stores give byte-equal
sc_detect_loops results over every store size.

Chain at 10^4 keyframes (and detection at 10^5): sc_add_keyframes, sc_detect_loops with a call per keyframe, then
loop_closure_icp_batch (historyKeyframeSearchNum 25, leaf 0.3) on every detected pair.

    python tests/perf/bench_sc_batch.py [--out profiles/r04_sc_batch.jsonl]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bench_loop_icp import card, stats  # noqa: E402
from lio_slam_b200 import synth  # noqa: E402
from lio_slam_b200.liogpu import LioGpu  # noqa: E402

P, STEP, LEAF, REPS = 200, 0.65, 0.2, 5
PASS_POINTS = (1 << 31) - 1   # a pass of liogpu_sc_add_keyframes: at most this many points, one sync each
SEARCH_NUM, ICP_LEAF = 25, 0.3


def base_keyframes(g):
    """P voxelised 64-beam keyframes as device tensors, and their key poses"""
    import torch
    from lio_slam_b200 import synth_torch
    w = synth_torch.TorchWorld(synth.make_world(1234), torch.device("cuda", 0))
    lap = int(round(2 * np.pi * 8.0 / STEP))
    clouds, poses = [], []
    for j in range(P):
        s = STEP * j
        rec = synth_torch.make_scan_records(w, synth.path_pose(s), 64, seed=9000 + j, cols=900)
        ds, _ = g.voxel_downsample((rec.data_ptr(), rec.shape[0], 32), LEAF)
        clouds.append(torch.from_numpy(ds).cuda())
        p = synth.path_pose(s).astype(np.float32)
        f = j / lap
        p[3] += 0.3 * f
        p[4] -= 0.2 * f
        poses.append(p)
    return clouds, np.array(poses, np.float32)


def put(g, clouds, n):
    g.keyframe_clear()
    for j in range(n):
        c = clouds[j % P]
        g.keyframe_put(j, (c.data_ptr(), c.shape[0], 16))


def arm_single(g, clouds, n, desc, rk, sk):
    lib, h = g.lib, g.h
    ptrs = [(c.data_ptr(), c.shape[0]) for c in clouds]
    dp, rp, sp = desc.ctypes.data, rk.ctypes.data, sk.ctypes.data
    dev = 0.0
    t0 = time.perf_counter()
    for j in range(n):
        p, m = ptrs[j % P]
        assert lib.liogpu_make_scancontext(h, p, m, 16, 2.0, 80.0, dp, rp, sp) == 0
        dev += lib.liogpu_last_gpu_ms(h)
        assert lib.liogpu_sc_add(h, dp, 1) == 0
        dev += lib.liogpu_last_gpu_ms(h)
    return 1e3 * (time.perf_counter() - t0), dev


def arm_batch(g, ids, out_ptr=None):
    t0 = time.perf_counter()
    assert g.lib.liogpu_sc_add_keyframes(g.h, ids.ctypes.data, ids.shape[0], 2.0, 80.0, out_ptr) == 0
    return 1e3 * (time.perf_counter() - t0), g.last_gpu_ms()


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_sc_batch.jsonl"))
    args = ap.parse_args()
    gpu = card()
    ga, gb = LioGpu(), LioGpu()
    clouds, poses = base_keyframes(gb)
    pts = [int(c.shape[0]) for c in clouds]
    desc, rk, sk = np.zeros(1200), np.zeros(20), np.zeros(60)
    ref = torch.from_numpy(np.array([ga.make_scancontext(c.cpu().numpy())[0] for c in clouds])).cuda()
    recs = []

    def emit(**kw):
        kw = dict(gpu=gpu, **kw)
        print(json.dumps(kw), flush=True)
        recs.append(kw)

    for n in (1000, 10000, 100000):
        put(gb, clouds, n)
        ids = np.arange(n, dtype=np.int32)
        wall_a, dev_a, wall_b, dev_b = [], [], [], []
        l0 = ga.launch_count()
        for it in range(REPS + 1):
            ga.sc_clear()
            w, d = arm_single(ga, clouds, n, desc, rk, sk)
            if it == 0:
                la = ga.launch_count() - l0
            else:
                wall_a.append(w)
                dev_a.append(d)
        for it in range(REPS + 1):
            gb.sc_clear()
            l0 = gb.launch_count()
            w, d = arm_batch(gb, ids)
            if it == 0:
                lb = gb.launch_count() - l0
            else:
                wall_b.append(w)
                dev_b.append(d)
        out = torch.empty((n, 20, 60), dtype=torch.float64, device="cuda")
        gb.sc_clear()
        arm_batch(gb, ids, out.data_ptr())
        idx = torch.arange(n, device="cuda") % P
        assert torch.equal(out.view(torch.int64), ref[idx].view(torch.int64)), "batch descriptors differ"
        parity = "descriptors byte-equal to make_scancontext"
        if n <= 10000:
            sizes = np.arange(1, n + 1)
            ia, ya, ma = ga.sc_detect_loops(sizes)
            ib, yb, mb = gb.sc_detect_loops(sizes)
            assert np.array_equal(ia, ib) and np.array_equal(ma.view(np.uint64), mb.view(np.uint64))
            assert np.array_equal(ya.view(np.uint32), yb.view(np.uint32))
            parity += "; sc_detect_loops over every store size byte-equal between the two stores"
        del out
        passes, acc = 1, 0
        for j in range(n):
            if j > 0 and acc + pts[j % P] > PASS_POINTS:
                passes, acc = passes + 1, 0
            acc += pts[j % P]
        ma_, mb_ = float(np.median(wall_a)), float(np.median(wall_b))
        emit(stage="descriptor store from resident keyframes", n_keyframes=n, distinct_clouds=P,
             points_per_keyframe=dict(mean=float(np.mean(pts)), min=min(pts), max=max(pts)),
             keyframe="64-beam, 900 columns, voxelised at 0.2 m", total_points=int(sum(pts[j % P] for j in range(n))),
             wall_ms=dict(a_make_scancontext_sc_add=stats(wall_a), b_sc_add_keyframes=stats(wall_b)),
             device_ms=dict(a_make_scancontext_sc_add=stats(dev_a), b_sc_add_keyframes=stats(dev_b)),
             launches=dict(a_make_scancontext_sc_add=int(la), b_sc_add_keyframes=int(lb)),
             passes=passes, host_round_trips=dict(a_make_scancontext_sc_add=2 * n, b_sc_add_keyframes=passes),
             speedup_wall=ma_ / mb_, parity=parity, reps=REPS, warmup=1)
        if n == 100000:   # detection over the whole sequence, for the 10^5 comparison
            sizes = np.arange(1, n + 1)
            gb.sc_detect_loops(sizes[:2000])
            wall = []
            for _ in range(3):
                t0 = time.perf_counter()
                gb.sc_detect_loops(sizes)
                wall.append(1e3 * (time.perf_counter() - t0))
            emit(stage="sc_detect_loops whole sequence", n_keyframes=n, n_calls=n, wall_ms=stats(wall),
                 descriptor_build_wall_ms=mb_, reps=3, warmup=1)
    # ---- chain at 10^4 ----------------------------------------------------------------------------------------------
    n = 10000
    put(gb, clouds, n)
    ids = np.arange(n, dtype=np.int32)
    key_poses = poses[ids % P]
    sizes = np.arange(1, n + 1)
    t_desc, t_det, t_icp, n_pairs = [], [], [], None
    for it in range(4):
        gb.sc_clear()
        t0 = time.perf_counter()
        gb.sc_add_keyframes(ids)
        t1 = time.perf_counter()
        loops, _, _ = gb.sc_detect_loops(sizes)
        t2 = time.perf_counter()
        cur = np.nonzero(loops >= 0)[0].astype(np.int32)
        pre = loops[cur].astype(np.int32)
        T, res = gb.loop_closure_icp_batch(cur, pre, key_poses, search_num=SEARCH_NUM, icp_leaf=ICP_LEAF)
        t3 = time.perf_counter()
        if it == 0:
            n_pairs = int(cur.shape[0])
            n_icp = int(sum(1 for r in res if not r["rejected_by_size"]))
            n_conv = int(sum(1 for r in res if r["converged"]))
        else:
            t_desc.append(1e3 * (t1 - t0))
            t_det.append(1e3 * (t2 - t1))
            t_icp.append(1e3 * (t3 - t2))
    emit(stage="offline loop-closure chain on the device", n_keyframes=n, distinct_clouds=P, detected_pairs=n_pairs,
         icp_run=n_icp, icp_converged=n_conv, search_num=SEARCH_NUM, icp_leaf=ICP_LEAF,
         wall_ms=dict(sc_add_keyframes=stats(t_desc), sc_detect_loops=stats(t_det), loop_closure_icp_batch=stats(t_icp)),
         reps=3, warmup=1)
    ga.close()
    gb.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for r in recs:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
