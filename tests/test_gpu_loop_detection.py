"""GPU parity of loop-closure detection (liogpu_sc_add / liogpu_sc_detect_loop / liogpu_sc_detect_loops /
liogpu_detect_loop_distance) against the oracle's restatement of SCManager::detectLoopClosureID and
detectLoopClosureDistance: every call bit-equal (loop id, yaw, best candidate and shift, min_dist bits, candidates with
their ring-key distances, distances and shifts, snapshot size, rebuild flag), and the replay of a multi-lap drive with
both detectors on gives the same registration as with them off."""
import numpy as np
import pytest

from lio_slam_b200 import synth

pytestmark = pytest.mark.gpu

LAP = 2 * np.pi * 8.0   # synth.path_pose: a circle of radius 8 m


@pytest.fixture(scope="module")
def g():
    """a context of its own: the descriptor store lives in the context"""
    from lio_slam_b200.liogpu import LioGpu
    ctx = LioGpu()
    yield ctx
    ctx.close()

@pytest.fixture(scope="module")
def loop_oracle():
    """the oracle's restatement of loop-closure detection (oracle/liorf_oracle_loop.h)"""
    from oracle.loop_oracle import LoopOracle
    return LoopOracle()



@pytest.fixture(scope="module")
def two_laps(g, world):
    """keyframe sweeps every 1 m along two laps of the circle (32 beams), their descriptors made on the device"""
    s = np.arange(0, 101) * 1.0
    descs = []
    for j, sj in enumerate(s):
        scan = synth.to_packed(synth.make_scan(world, synth.path_pose(sj), 32, seed=900 + j, cols=900))
        descs.append(g.make_scancontext(scan)[0])
    return dict(s=s, descs=np.array(descs), poses=np.array([synth.path_pose(v) for v in s]))


def same(got, want, where=""):
    """one online call (loop_id, yaw, info) against one oracle call"""
    loop_id, yaw, info = got
    assert loop_id == want["loop_id"], where
    assert np.float32(yaw).view(np.uint32) == np.float32(want["yaw"]).view(np.uint32), where
    for k in ("n_stored", "n_searchable", "tree_rebuilt", "n_candidates", "nn_idx", "nn_align", "knn_ties"):
        assert info[k] == want[k], (where, k, info[k], want[k])
    assert np.float64(info["min_dist"]).view(np.uint64) == np.float64(want["min_dist"]).view(np.uint64), where
    assert np.array_equal(info["candidates"], want["candidates"]), where
    assert np.array_equal(info["candidate_key_d2"].view(np.uint32), want["candidate_key_d2"].view(np.uint32)), where
    assert np.array_equal(info["candidate_dist"].view(np.uint64), want["candidate_dist"].view(np.uint64)), where
    assert np.array_equal(info["candidate_shift"], want["candidate_shift"]), where


def run_online(g, loop_oracle, descs, sizes=None, **prm):
    """fresh store; add descriptors and detect after each size in `sizes` (default: after every descriptor)"""
    sizes = list(range(1, len(descs) + 1)) if sizes is None else list(sizes)
    want = loop_oracle.sc_detect_loops(descs, sizes, threads=8, **prm)
    g.sc_clear()
    got, n = [], 0
    for j, size in enumerate(sizes):
        if size > n:
            g.sc_add(descs[n:size])
            n = size
        r = g.sc_detect_loop(**prm)
        same(r, want[j], f"call {j} size {size} {prm}")
        got.append(r)
    return got, want


def test_two_laps_online_bit_equal(g, loop_oracle, two_laps):
    got, want = run_online(g, loop_oracle, two_laps["descs"])
    s, poses = two_laps["s"], two_laps["poses"]
    loops = [(j, r[0]) for j, r in enumerate(got) if r[0] >= 0]
    # expectations set from the oracle (deterministic): lap 2 closes loops onto lap 1
    lap2 = [(j, i) for j, i in loops if s[j] >= LAP]
    assert len(lap2) >= 30, loops
    d = [np.linalg.norm(poses[j, 3:5] - poses[i, 3:5]) for j, i in loops]
    assert max(d) < 11.0, d                                   # a few places ~10.7 m apart on the small circle look alike
    assert sum(x < 2.0 for x in d) >= 30, d
    assert all(r[2]["knn_ties"] == 0 for r in got)


PARAM_GRID = [dict(num_exclude_recent=ne, num_candidates=k, tree_making_period=p, search_ratio=sr, sc_dist_thres=th)
              for ne, k, p, sr, th in [(0, 1, 1, 0.05, 0.2), (1, 3, 7, 0.1, 10.0), (30, 10, 30, 0.5, -1.0),
                                       (1, 32, 1, 1.0, 0.2), (30, 32, 7, 0.1, 10.0), (0, 10, 30, 1.0, -1.0),
                                       (30, 1, 1, 0.5, 0.3), (1, 3, 30, 0.05, 0.2)]]


@pytest.mark.parametrize("prm", PARAM_GRID)
def test_parameter_grid_online_bit_equal(g, loop_oracle, two_laps, prm):
    got, _ = run_online(g, loop_oracle, two_laps["descs"], **prm)
    if prm["sc_dist_thres"] == 10.0:   # accepts everything that was scored
        assert all(r[0] >= 0 for r in got if r[2]["n_candidates"] > 0)
    if prm["sc_dist_thres"] == -1.0:   # accepts nothing
        assert all(r[0] == -1 for r in got)


def test_batch_equals_online_and_irregular_sizes(g, loop_oracle, two_laps):
    descs = two_laps["descs"]
    rng = np.random.default_rng(3)
    irregular = np.sort(np.r_[rng.integers(1, 102, 60), [1, 31, 31, 31, 101, 101]])   # repeats, gaps of a 1 Hz thread
    for sizes, prm in ((np.arange(1, 102), {}), (irregular, dict(num_exclude_recent=5, tree_making_period=4)),
                       (irregular, dict(num_exclude_recent=0, num_candidates=32, tree_making_period=1, search_ratio=1.0))):
        got, want = run_online(g, loop_oracle, descs, sizes, **prm)
        g.sc_clear()
        g.sc_add(descs)
        ids, yaw, md = g.sc_detect_loops(sizes, **prm)
        assert np.array_equal(ids, [r[0] for r in got])
        assert np.array_equal(yaw.view(np.uint32), np.array([r[1] for r in got], np.float32).view(np.uint32))
        assert np.array_equal(md.view(np.uint64), np.array([w["min_dist"] for w in want]).view(np.uint64))
        # the batch call does not touch the online counter
        before = g.sc_detect_loop(**prm)
        g.sc_detect_loops(sizes, **prm)
        after = g.sc_detect_loop(**prm)
        assert before[2]["tree_rebuilt"] == 1 and after[2]["tree_rebuilt"] == (1 if prm.get("tree_making_period", 30) == 1 else 0)


def test_large_store_batch_against_oracle(loop_oracle, world):
    """>= 20,000 descriptors made on the device from seeded sweeps, a detectLoopClosureID call per keyframe"""
    import torch
    from lio_slam_b200 import synth_torch
    from lio_slam_b200.liogpu import LioGpu
    dev = torch.device("cuda", 0)
    w = synth_torch.TorchWorld(world, dev)
    n = 20000
    g2 = LioGpu()
    try:
        descs = np.empty((n, 20, 60))
        for j in range(n):
            rec = synth_torch.make_scan_records(w, synth.path_pose(0.37 * j), 16, seed=7000 + j, cols=120)
            descs[j] = g2.make_scancontext((rec.data_ptr(), rec.shape[0], 32))[0]
        g2.sc_add(descs)
        sizes = np.arange(1, n + 1)
        ids, yaw, md = g2.sc_detect_loops(sizes)
        want = loop_oracle.sc_detect_loops(descs, sizes, threads=loop_oracle.max_threads())
        assert np.array_equal(ids, [r["loop_id"] for r in want])
        assert np.array_equal(yaw.view(np.uint32), np.array([r["yaw"] for r in want], np.float32).view(np.uint32))
        assert np.array_equal(md.view(np.uint64), np.array([r["min_dist"] for r in want]).view(np.uint64))
        assert (ids >= 0).sum() > 100
        # the online call at the full store (snapshot of 19,971 keys over 20 chunks) agrees as well
        g2.sc_clear()
        g2.sc_add(descs)
        same(g2.sc_detect_loop(), loop_oracle.sc_detect_loops(descs, [n])[0])
    finally:
        g2.close()


def test_edges(g, loop_oracle, two_laps):
    d = two_laps["descs"]
    z = np.zeros((20, 60))
    e = d[7].copy()
    e[:, 10:25] = 0.0
    dup = d[11]
    cases = [
        (d[:5], dict(num_exclude_recent=30)),                                   # store < NE + 1 throughout
        (d[:40], dict(num_exclude_recent=30, num_candidates=32)),               # snapshot smaller than k
        (np.array([z, z, z, d[3], z]), dict(num_exclude_recent=1, num_candidates=3, tree_making_period=1)),
        (np.array([d[3], e, d[9], np.roll(e, 3, axis=1), z, e]), dict(num_exclude_recent=1, num_candidates=4,
                                                                     tree_making_period=1, search_ratio=0.2)),
        (np.array([d[0], dup, d[30], dup, dup, d[2], dup]), dict(num_exclude_recent=1, num_candidates=2, tree_making_period=1)),
    ]
    for descs, prm in cases:
        got, want = run_online(g, loop_oracle, descs, **prm)
    loop_id, yaw, info = got[-1]                                                # duplicates: ties logged, lower index
    assert list(info["candidates"]) == [1, 3] and info["knn_ties"] >= 2 and loop_id == 1 and info["min_dist"] == 0.0
    # store < NE + 1: -1, counter not advanced (the next call that passes the guard rebuilds)
    g.sc_clear()
    g.sc_add(d[:3])
    r = g.sc_detect_loop(num_exclude_recent=3, tree_making_period=5)
    assert r[0] == -1 and r[1] == 0 and r[2]["tree_rebuilt"] == 0 and r[2]["n_candidates"] == 0
    g.sc_add(d[3:4])
    assert g.sc_detect_loop(num_exclude_recent=3, tree_making_period=5)[2]["tree_rebuilt"] == 1
    # circshifted copies: distance 0 at the planted shift
    for s in (1, 17, 59):
        g.sc_clear()
        g.sc_add(np.array([d[0], d[5], d[20], np.roll(d[5], s, axis=1)]))
        loop_id, yaw, info = g.sc_detect_loop(num_exclude_recent=1, tree_making_period=1)
        assert loop_id == 1 and info["nn_align"] == s and info["min_dist"] < 1e-12


def test_state_and_bad_arguments(g, loop_oracle, two_laps, small_case):
    from lio_slam_b200 import liogpu
    d = two_laps["descs"]
    g.sc_clear()
    g.sc_add(d[:60])
    first = g.sc_detect_loop()
    # keyframe_clear leaves the store alone
    g.keyframe_put(0, small_case["map4"][:1000])
    g.keyframe_clear()
    assert g.sc_detect_loop()[2]["n_stored"] == 60
    # sc_clear resets the store and the counter
    g.sc_clear()
    g.sc_add(d[:60])
    same(g.sc_detect_loop(), loop_oracle.sc_detect_loops(d, [60])[0])
    assert first[2]["tree_rebuilt"] == 1
    # bad arguments: E_INVALID, nothing changes
    lib, h = g.lib, g.h
    import ctypes as C
    p = liogpu.sc_params()
    lid, yaw, info = C.c_int(5), C.c_float(1), liogpu.ScInfo()
    buf = np.zeros((2, 1200))
    assert lib.liogpu_sc_add(h, None, 1) == liogpu.E_INVALID
    assert lib.liogpu_sc_add(h, buf.ctypes.data, 0) == liogpu.E_INVALID
    for bad in (dict(num_exclude_recent=-1), dict(num_candidates_from_tree=0), dict(num_candidates_from_tree=33),
                dict(tree_making_period=0), dict(search_ratio=0.0), dict(search_ratio=1.5), dict(sc_dist_thres=float("nan"))):
        q = liogpu.sc_params(**bad)
        assert lib.liogpu_sc_detect_loop(h, C.byref(q), C.byref(lid), C.byref(yaw), C.byref(info)) == liogpu.E_INVALID, bad
    assert lib.liogpu_sc_detect_loop(h, C.byref(p), None, C.byref(yaw), None) == liogpu.E_INVALID
    out = np.zeros(4, np.int32)
    for sizes in ([3, 2], [61], [-1]):
        s = np.array(sizes, np.int32)
        assert lib.liogpu_sc_detect_loops(h, C.byref(p), s.ctypes.data, len(sizes), out.ctypes.data, None, None) == liogpu.E_INVALID
    s = np.array([60], np.int32)
    assert lib.liogpu_sc_detect_loops(h, C.byref(p), s.ctypes.data, 0, out.ctypes.data, None, None) == liogpu.E_INVALID
    key = np.zeros((3, 4), np.float32)
    t = np.zeros(3)
    assert lib.liogpu_detect_loop_distance(h, key.ctypes.data, 0, 16, t.ctypes.data, 8, 0.0, C.c_float(1), C.c_float(1),
                                           C.byref(lid)) == liogpu.E_INVALID
    assert lib.liogpu_detect_loop_distance(h, key.ctypes.data, 3, 16, t.ctypes.data, 8, 0.0, C.c_float(0), C.c_float(1),
                                           C.byref(lid)) == liogpu.E_INVALID
    # ... and the state is what it was: the next call is the second call of this store
    want = loop_oracle.sc_detect_loops(d, [60, 60])[1]
    same(g.sc_detect_loop(), want)


def test_detection_leaves_the_registration_untouched(g, small_case):
    g.set_local_map(small_case["map4"])
    ds = g.voxel_downsample(small_case["scan4"], 0.4)[0]
    before = g.surf_optimization(ds, small_case["guess"])
    g.sc_add(np.random.default_rng(1).uniform(0, 5, (40, 20, 60)))
    g.sc_detect_loop(num_exclude_recent=3)
    g.sc_detect_loops(np.arange(1, 41), num_exclude_recent=3)
    key = np.c_[np.random.default_rng(2).uniform(-9, 9, (500, 3)), np.arange(500)].astype(np.float32)
    g.detect_loop_distance(key, np.arange(500) * 0.5, 250.0)
    after = g.surf_optimization(ds, small_case["guess"])
    for k in before:
        assert np.array_equal(before[k].view(np.uint8), after[k].view(np.uint8)), k


@pytest.mark.parametrize("n", [1, 2, 7, 400, 5000, 60000])
def test_radius_detector_against_oracle(g, loop_oracle, n):
    rng = np.random.default_rng(n)
    key = np.c_[rng.uniform(-30, 30, (n, 2)), rng.uniform(-1, 1, (n, 1)), np.arange(n)].astype(np.float32)
    if n > 2:
        key[rng.random(n) < 0.1, :3] = key[-1, :3] + np.float32(rng.choice([0.0, 3.0]))   # equal distances
        key[1, :3] = key[-1, :3] + np.float32([6.0, 8.0, 0.0])                            # exactly on the radius
    t = np.sort(rng.uniform(0, 0.01 * n + 100, n))
    t_cur = t[-1] + 0.05
    if n > 2:
        t[1] = t_cur - 30.0                                                               # exactly time_diff old
    for radius, tdiff in ((10.0, 30.0), (3.0, 0.0), (25.0, 100.0), (10.0, 1e9)):
        assert g.detect_loop_distance(key, t, t_cur, radius, tdiff) == loop_oracle.detect_loop_distance(key, t, t_cur, radius, tdiff)


def test_replay_with_loop_detection(world):
    """loop_detection_every = 10 leaves the registration bit-identical and finds loops; the sequence covers 4 laps so
    that revisits are older than historyKeyframeSearchTimeDiff (30 s) for the radius detector"""
    import torch
    from lio_slam_b200 import replay, synth_torch
    n = 600
    times = 0.1 * np.arange(n)
    arc = 0.35 * np.arange(n)
    assert arc[-1] > 4 * LAP and times[int(np.ceil(LAP / 0.35))] < 30.0   # one lap is ~14 s of sweeps
    seq = synth_torch.make_sequence(world, 64, n, seed=13, device=torch.device("cuda", 0), step=0.35, cols=900)
    prm = replay.kitti_params()
    a = replay.replay_sequence(prm, seq)
    b = replay.replay_sequence(prm, seq, loop_detection_every=10)
    assert np.array_equal(a[0].view(np.uint32), b[0].view(np.uint32))
    assert np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])
    assert a[3]["loops_sc"] == 0 and a[3]["loops_rs"] == 0
    assert b[3]["loops_sc"] > 0 and b[3]["loops_rs"] > 0, b[3]
    # cut before the first revisit (< 31 keyframes, < 30 s): nothing to find
    c = replay.replay_sequence(prm, seq, count=80, loop_detection_every=10)
    assert c[3]["keyframes"] < 31 and c[3]["loops_sc"] == 0 and c[3]["loops_rs"] == 0
