"""liogpu_detect_loops_distance: detectLoopClosureDistance for many calls of the loop thread in one call, answered
against one sorted-grid index of all key poses.  Every answer must equal liogpu_detect_loop_distance on the call's
prefix and the oracle's restatement of the reference loop.  Also mapOptimization::performLoopClosuresOffline, the loop
thread's work for every tick of a sequence, against the online performRSLoopClosure + performSCLoopClosure per tick."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from lio_slam_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32_MAX = float(np.finfo(np.float32).max)


@pytest.fixture(scope="module")
def g():
    from lio_slam_b200.liogpu import LioGpu
    ctx = LioGpu()
    yield ctx
    ctx.close()


@pytest.fixture(scope="module")
def loop_oracle():
    from oracle.loop_oracle import LoopOracle
    return LoopOracle()


def walk(n, seed, laps=4, r=40.0):
    """n key poses over `laps` laps of a circle with a random-walk drift; times 0.5 s apart"""
    rng = np.random.default_rng(seed)
    th = np.linspace(0.0, 2 * np.pi * laps, n)
    drift = np.cumsum(rng.normal(0.0, 0.05, (n, 3)), 0)
    drift -= np.linspace(0.0, 1.0, n)[:, None] * drift[-1]
    xyz = np.c_[r * np.cos(th), r * np.sin(th), 0.3 * np.sin(3 * th)] + drift * [1.0, 1.0, 0.1]
    return np.c_[xyz, np.arange(n)].astype(np.float32), np.arange(n) * 0.5


def per_call(g, lo, key, t, at, tc, r, td):
    """liogpu_detect_loop_distance and the oracle on every call's prefix (they must agree)"""
    dev = np.array([g.detect_loop_distance(key[:m], t[:m], c, r, td) for m, c in zip(at, tc)], np.int32)
    k4 = np.ascontiguousarray(key[:, :4])
    ref = np.array([lo.detect_loop_distance(k4[:m], t[:m], c, r, td) for m, c in zip(at, tc)], np.int32)
    bad = np.nonzero(dev != ref)[0]
    assert bad.size == 0, (bad[:10], dev[bad[:10]], ref[bad[:10]])
    return dev


def check(g, lo, key, t, at, tc, r=10.0, td=30.0):
    at = np.asarray(at, np.int32)
    tc = np.asarray(tc, np.float64)
    got = g.detect_loops_distance(key, t, at, tc, r, td)
    want = per_call(g, lo, key, t, at, tc, r, td)
    bad = np.nonzero(got != want)[0]
    assert bad.size == 0, (r, td, bad[:10], at[bad[:10]], got[bad[:10]], want[bad[:10]])
    return got


def every_keyframe(t, seed=0):
    n = t.shape[0]
    return np.arange(1, n + 1), t + np.random.default_rng(seed).uniform(0.0, 0.4, n)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1000, 10000])
def test_multi_lap_walk_call_per_keyframe(g, loop_oracle, n):
    key, t = walk(n, n)
    at, tc = every_keyframe(t, n)
    got = check(g, loop_oracle, key, t, at, tc)
    assert (got >= 0).sum() > n // 4  # revisits on laps 2-4


@pytest.mark.gpu
def test_shuffled_repeated_and_single_pose_calls(g, loop_oracle):
    n = 3000
    key, t = walk(n, 7, laps=3)
    rng = np.random.default_rng(7)
    at = np.concatenate([rng.permutation(np.arange(1, n + 1)), rng.integers(1, n + 1, 500), np.ones(20, np.int64),
                         np.full(30, n)])
    tc = t[at - 1] + rng.choice([0.0, 0.2, 31.0, -40.0], at.shape[0])
    got = check(g, loop_oracle, key, t, at, tc)
    assert (got[at == 1] == -1).all() and (got >= 0).any()


def cloud_for(kind, seed):
    rng = np.random.default_rng(seed)
    if kind == "spread":  # 10 km cube at a 0.5 m radius: 2e13 cells, the cap doubles the cell many times
        base = rng.uniform(-5000.0, 5000.0, (1500, 3))
        near = base[rng.integers(0, 1500, 1500)] + rng.normal(0.0, 0.2, (1500, 3))
        xyz = np.vstack([base, near])[rng.permutation(3000)]
        return np.c_[xyz, np.arange(3000)].astype(np.float32), np.arange(3000) * 0.5
    key, t = walk(2000, seed, laps=3)
    if kind == "tiny":  # exact repeats of earlier poses (d2 = 0) and near repeats
        src = rng.integers(0, 1000, 400)
        dst = rng.integers(1000, 2000, 400)
        key[dst, :3] = key[src, :3]
        key[dst[:100], 0] += np.float32(5e-4)
    return key, t


@pytest.mark.gpu
@pytest.mark.parametrize("kind,radius", [
    ("tiny", 1e-3),
    ("walk", 10.1),          # 10.1 * 10.1 rounds when narrowed to f32
    ("walk", 1000.0),        # every pose in one cell
    ("spread", 0.5),
    ("walk", 1e30),          # r * r overflows f32: every finite pose is within the radius
    ("walk", F32_MAX),
    ("walk", float("inf")),
])
def test_radii(g, loop_oracle, kind, radius):
    key, t = cloud_for(kind, 11)
    n = key.shape[0]
    rng = np.random.default_rng(3)
    at = np.r_[np.arange(1, n + 1, 3 if n > 2500 else 1), n]
    tc = t[at - 1] + rng.uniform(0.0, 0.3, at.shape[0])
    got = check(g, loop_oracle, key, t, at, tc, r=radius)
    assert (got >= 0).any()


@pytest.mark.gpu
def test_time_filter_edges(g, loop_oracle):
    key, t = walk(2000, 5, laps=3)
    rng = np.random.default_rng(5)
    dup = rng.integers(1000, 2000, 200)
    key[dup, :3] = key[dup - 700, :3]  # d2 == 0 between poses 350 s apart
    at = np.arange(1, 2001)
    for tc in (t.copy(), t + 0.5, t + 30.0):  # times on a 0.5 s grid: |dt| hits time_diff exactly
        for td in (-1.0, 0.0, 30.0, 350.0):
            check(g, loop_oracle, key, t, at, tc, r=10.0, td=td)


@pytest.mark.gpu
@pytest.mark.parametrize("radius", [2.0, 3.0, float(np.sqrt(np.float32(5.0)))])
def test_lattice_ties_and_exact_radius(g, loop_oracle, radius):
    """integer lattice, every coordinate twice, indices shuffled: many equal d2 (lower index must win) and poses at
    exactly d2 == r2 (not within the radius)"""
    rng = np.random.default_rng(9)
    grid = np.stack(np.meshgrid(np.arange(8), np.arange(8), np.arange(4), indexing="ij"), -1).reshape(-1, 3)
    xyz = np.vstack([grid, grid])[rng.permutation(2 * grid.shape[0])]
    n = xyz.shape[0]
    key = np.c_[xyz, np.arange(n)].astype(np.float32)
    t = np.arange(n) * 100.0
    at = np.arange(1, n + 1)
    got = check(g, loop_oracle, key, t, at, t[at - 1], r=radius)
    assert (got >= 0).sum() > n // 2


@pytest.mark.gpu
def test_non_finite_poses(g, loop_oracle):
    key, t = walk(3000, 13, laps=3)
    rng = np.random.default_rng(13)
    idx = rng.choice(3000, 300, replace=False)
    for j, i in enumerate(idx):
        key[i, j % 3] = [np.nan, np.inf, -np.inf][j % 3]
    key[[0, 1, 2999], 0] = np.nan  # the first poses and the last query
    at = np.r_[np.arange(1, 3001), idx + 1]
    tc = t[at - 1] + 0.1
    got = check(g, loop_oracle, key, t, at, tc)
    assert (got[np.isin(at - 1, idx)] == -1).all() and (got >= 0).any()


@pytest.mark.gpu
def test_record_layouts(g, loop_oracle):
    """key poses as 32-byte PointType records, times as the `time` field of 48-byte PointTypePose records"""
    n = 2500
    key, t = walk(n, 17)
    rng = np.random.default_rng(17)
    key32 = np.c_[key, rng.uniform(-1, 1, (n, 4))].astype(np.float32)  # x y z intensity + 4 junk floats
    at, tc = every_keyframe(t, 17)
    want = check(g, loop_oracle, key, t, at, tc)
    assert np.array_equal(check(g, loop_oracle, key32, t, at, tc), want)
    rec = np.zeros(n, np.dtype({"names": ["f", "time"], "formats": [("f4", 7), "f8"], "offsets": [0, 32],
                                "itemsize": 48}))
    rec["f"] = rng.uniform(-1, 1, (n, 7))
    rec["time"] = t
    m = np.ascontiguousarray(at, np.int32)
    out = np.full(n, -7, np.int32)
    for k, stride in ((key, 16), (key32, 32)):
        k = np.ascontiguousarray(k)
        g._check(g.lib.liogpu_detect_loops_distance(g.h, k.ctypes.data, n, stride, rec.ctypes.data + 32, 48, m.ctypes.data,
                                                    tc.ctypes.data, n, C.c_float(10.0), C.c_float(30.0), out.ctypes.data))
        assert np.array_equal(out, want)


@pytest.mark.gpu
def test_bad_arguments_are_refused_before_any_launch(g):
    from lio_slam_b200.liogpu import E_INVALID
    n = 100
    key, t = walk(n, 1)
    m = np.arange(1, n + 1, dtype=np.int32)
    tc = t + 0.1
    out = np.zeros(n, np.int32)
    lib, h = g.lib, g.h
    ok = dict(k=key.ctypes.data, n=n, s=16, t=t.ctypes.data, ts=8, m=m.ctypes.data, tc=tc.ctypes.data, nc=n, r=10.0,
              td=30.0, o=out.ctypes.data)
    zero_m = np.r_[m[:-1], 0].astype(np.int32)
    big_m = np.r_[m[:-1], n + 1].astype(np.int32)
    bad = [dict(k=None), dict(n=0), dict(n=-1), dict(s=20), dict(s=8), dict(t=None), dict(ts=4), dict(m=None),
           dict(tc=None), dict(nc=0), dict(nc=-3), dict(r=0.0), dict(r=-1.0), dict(r=float("nan")),
           dict(td=float("nan")), dict(o=None), dict(m=zero_m.ctypes.data), dict(m=big_m.ctypes.data), dict(k=1), dict(k=2)]
    for over in bad:
        a = dict(ok, **over)
        before = g.launch_count()
        st = lib.liogpu_detect_loops_distance(h, a["k"], a["n"], a["s"], a["t"], a["ts"], a["m"], a["tc"], a["nc"],
                                              C.c_float(a["r"]), C.c_float(a["td"]), a["o"])
        assert st == E_INVALID and g.launch_count() == before, over
    a = ok
    assert lib.liogpu_detect_loops_distance(h, a["k"], a["n"], a["s"], a["t"], a["ts"], a["m"], a["tc"], a["nc"],
                                            C.c_float(a["r"]), C.c_float(a["td"]), a["o"]) == 0


@pytest.mark.gpu
def test_launches_do_not_depend_on_the_number_of_calls(g):
    key, t = walk(20000, 2)
    counts = []
    for at in (np.array([20000]), np.arange(1, 20001), np.r_[np.arange(1, 20001), np.arange(1, 20001)]):
        before = g.launch_count()
        g.detect_loops_distance(key, t, at, t[at - 1] + 0.1)
        counts.append(g.launch_count() - before)
    assert counts[0] == counts[1] == counts[2] and counts[0] > 0, counts


@pytest.mark.gpu
def test_registration_and_resident_cloud_untouched(g, small_case):
    g.set_local_map(small_case["map4"])
    p0, P0, i0 = g.scan2map(small_case["scan4"], small_case["guess"])
    n_res, _ = g.voxel_downsample(small_case["scan4"], 0.4, keep_on_device=True)
    q0, _, _ = g.scan2map("resident", small_case["guess"])
    n_map = g.local_map_size()
    key, t = walk(5000, 4)
    g.detect_loops_distance(key, t, np.arange(1, 5001), t + 0.1)
    assert g.resident_size() == n_res and g.local_map_size() == n_map
    q1, _, _ = g.scan2map("resident", small_case["guess"])
    assert np.array_equal(q0.view(np.uint32), q1.view(np.uint32))
    p1, P1, i1 = g.scan2map(small_case["scan4"], small_case["guess"])
    assert np.array_equal(p0.view(np.uint32), p1.view(np.uint32)) and np.array_equal(P0.view(np.uint32), P1.view(np.uint32))
    assert i0["iterations"] == i1["iterations"] and i0["n_sel"] == i1["n_sel"]


def test_export_argtypes_and_abi_version():
    from lio_slam_b200 import liogpu
    assert "liogpu_detect_loops_distance" in liogpu.EXPORTS
    lib = liogpu.load_library()
    assert lib.liogpu_abi_version() == 2
    assert lib.liogpu_detect_loops_distance.argtypes == [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                                         C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_float,
                                                         C.c_void_p]
    assert hasattr(liogpu.LioGpu, "detect_loops_distance")


# ---- the host mirror's offline pass ----

N_POOL = 32      # keyframe positions per lap of synth.path_pose's 50.3 m circle (1.6 m apart)


def mirror_case(world, laps, search_num, exclude, cols=900, tick_stride=7):
    """Keyframes on `laps` laps (sensor-frame sweeps from one pool, so revisits see the same cloud); lap 1 drifts,
    the others do not.  Ticks: two empty ones, then one per keyframe with every tick_stride-th repeated (no new
    keyframe)."""
    pool = [synth.to_packed(synth.make_scan(world, synth.path_pose(1.6 * j), 16, seed=4000 + j, cols=cols))
            for j in range(N_POOL)]
    n_key = laps * N_POOL
    poses = []
    for k in range(n_key):
        p = synth.path_pose(1.6 * (k % N_POOL)).astype(np.float32)
        if k // N_POOL == 1:
            f = (k % N_POOL + 1) / N_POOL
            p[3] += 0.8 * f
            p[4] -= 0.5 * f
            p[2] += 0.03 * f
        poses.append(p)
    times = np.arange(n_key) * 2.0
    ticks = [(0, 0.0), (0, 0.5)]
    for k in range(1, n_key + 1):
        ticks.append((k, times[k - 1] + 0.1))
        if k % tick_stride == 0:
            ticks.append((k, times[k - 1] + 0.7))
    return dict(pool=pool, which=np.arange(n_key) % N_POOL, poses=np.array(poses, np.float32), times=times, ticks=ticks,
                search_num=search_num, exclude=exclude)


def write_mirror_case(path, case, radius=10.0, time_diff=30.0):
    with open(path, "wb") as f:
        n_key = case["poses"].shape[0]
        f.write(np.array([n_key, len(case["pool"]), case["search_num"], case["exclude"]], np.int32).tobytes())
        f.write(np.array([radius, time_diff], np.float32).tobytes())
        for c in case["pool"]:
            f.write(np.int32(c.shape[0]).tobytes())
            f.write(np.ascontiguousarray(c, np.float32).tobytes())
        f.write(np.asarray(case["which"], np.int32).tobytes())
        f.write(case["poses"].astype(np.float32).tobytes())
        f.write(np.asarray(case["times"], np.float64).tobytes())
        f.write(np.int32(len(case["ticks"])).tobytes())
        for n, tc in case["ticks"]:
            f.write(np.int32(n).tobytes())
            f.write(np.float64(tc).tobytes())


def build_mirror(out_dir):
    host = os.path.join(ROOT, "lio_slam_b200", "host")
    exe = os.path.join(str(out_dir), "loop_offline_mirror")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++14", "-I", host, os.path.join(ROOT, "tests", "loop_offline_mirror.cpp"),
                           os.path.join(host, "map_optimization_gpu.cpp"), "-L", os.path.join(ROOT, "lio_slam_b200"),
                           "-lliogpu", "-Wl,-rpath," + os.path.join(ROOT, "lio_slam_b200"), "-o", exe])
    return exe


def run_mirror(exe, blob):
    r = subprocess.run([exe, str(blob)], capture_output=True, text=True, timeout=1200)
    words = r.stdout.split()
    stats = {words[i]: float(words[i + 1]) for i in range(0, len(words) - 1, 2)} if words[:1] == ["mismatched"] else {}
    return r, stats


@pytest.mark.gpu
def test_offline_pass_equals_the_loop_thread_tick_by_tick(tmp_path, world):
    """three laps, historyKeyframeSearchNum 40 (RS and SC windows clamped by the tick's n_key), NUM_EXCLUDE_RECENT 10"""
    exe = build_mirror(tmp_path)
    case = mirror_case(world, laps=3, search_num=40, exclude=10)
    blob = tmp_path / "case.bin"
    write_mirror_case(blob, case)
    r, s = run_mirror(exe, blob)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert s["mismatched"] == 0
    assert s["rs_accepted"] >= 1 and s["sc_accepted"] >= 1 and s["rs_detected"] > s["rs_accepted"] - 1, r.stdout
    assert s["rs_clamped"] >= 1 and s["rs_detected"] > s["rs_clamped"], r.stdout   # both kinds of RS pairs
    assert s["sc_clamped"] >= 1, r.stdout
    assert s["repeated_ticks"] >= 1 and s["rs_suppressed"] >= 1 and s["rs_suppressed_after_sc"] >= 1, r.stdout
    assert s["below_exclude"] >= 1, r.stdout
    assert 0 < s["offline_icp"] <= s["online_icp"], r.stdout
