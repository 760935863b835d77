"""liogpu_merge_keyframes_batch: many keyframe windows merged and voxelised in one call.  Every window's cloud must be
byte-equal to liogpu_merge_keyframes of that window on the same context, with the same overflow flag, whatever windows
surround it, however the call splits the windows into passes and whatever order the windows come in.  The loop-closure
ICP batch builds its submaps with the same code and must stay bit-equal to merge + icp_align."""
import ctypes as C

import numpy as np
import pytest

from lio_slam_b200 import synth

N_LAP = 48         # sweeps every 1.6 m along two laps of synth.path_pose's circle; the second lap's poses drift
LEAF = 0.3


def lattice(step, nx, ny, nz, x0=0.0, y0=0.0):
    g = np.stack(np.meshgrid(np.arange(nx) * step + x0, np.arange(ny) * step + y0, np.arange(nz) * step,
                             indexing="ij"), -1).reshape(-1, 3)
    return np.c_[g, np.zeros(len(g))].astype(np.float32)


def key_space_cloud(seed):
    """a few hundred points spanning 1999.95 x 999.95 x 0.85 m: about 1.8e9 cells at leaf 0.1, below the guard"""
    r = np.random.default_rng(seed)
    p = r.uniform([0, 0, 0], [1999.95, 999.95, 0.85], (200, 3))
    p = np.vstack([p, p + r.uniform(0, 0.01, p.shape), [[0, 0, 0], [1999.95, 999.95, 0.85]]])
    return np.c_[p, r.uniform(0, 100, len(p))].astype(np.float32)


@pytest.fixture(scope="module")
def g():
    from lio_slam_b200.liogpu import LioGpu
    ctx = LioGpu()
    yield ctx
    ctx.close()


@pytest.fixture(scope="module")
def kf(g, world):
    g.keyframe_clear()
    clouds, poses = [], []
    for j in range(N_LAP):
        s = 1.6 * j
        clouds.append(synth.to_packed(synth.make_scan(world, synth.path_pose(s), 16, seed=5000 + j, cols=900)))
        p = synth.path_pose(s).astype(np.float32)
        if j >= N_LAP // 2:
            f = (j - N_LAP // 2 + 1) / (N_LAP // 2)
            p[3] += 0.9 * f
            p[4] -= 0.6 * f
            p[2] += 0.04 * f
        poses.append(p)
    named = {}

    def add(name, cloud, pose):
        named[name] = len(clouds)
        clouds.append(np.ascontiguousarray(cloud, np.float32))
        poses.append(np.asarray(pose, np.float32))

    zero = np.zeros(6, np.float32)
    add("lattice", lattice(1.0, 41, 41, 3, -20.0, -20.0), zero)
    far = poses[5].copy()
    far[3] += 500.0
    add("far", clouds[5], far)
    add("tiny", clouds[7][:100], poses[7])
    add("small", clouds[9][:2000], poses[9])           # at most 2048 points: the single path's one-block kernel
    nf = clouds[11].copy()
    nf[::97, 0] = np.nan
    nf[5::89, 1] = np.inf
    nf[7::83, 2] = -np.inf
    add("nonfinite", nf, poses[11])
    add("allnan", np.full((50, 4), np.nan, np.float32), poses[3])
    ovf = np.array([[0, 0, 0, 1], [3000, 3000, 3000, 2], [np.nan, 0, 0, 3], [1, 2, 3, 4]], np.float32)
    add("overflow", ovf, zero)                          # VoxelGrid guard (q4) at any leaf up to a few metres
    big_ovf = np.vstack([clouds[13], [[4000, 4000, 4000, 9]]]).astype(np.float32)
    add("overflow_big", big_ovf, poses[13])
    for q in range(3):
        t = np.zeros(6, np.float32)
        t[3:] = (100.0 * q, -50.0 * q, 3.0 * q)
        add(f"keyspace{q}", key_space_cloud(q), t)
    for k, c in enumerate(clouds):
        g.keyframe_put(k, c)
    return dict(clouds=clouds, poses=np.array(poses, np.float32), **named)


def win(kf, ids):
    ids = list(ids)
    return ids, kf["poses"][ids] if ids else np.zeros((0, 6), np.float32)


def mixed_windows(kf):
    n = N_LAP
    w = [
        [0],
        [(i * 5) % n for i in range(51)],             # 51 keyframes, repeated ids inside the window
        list(range(10, 15)),
        [kf["lattice"]],
        [],
        [kf["small"]],
        list(range(20, 45)),
        [kf["tiny"]],
        [kf["far"], 6],
        [kf["overflow"]],                             # overflow window between normal ones
        [2, 2, 2],
        [kf["allnan"]],
        [kf["allnan"], kf["allnan"]],
        [kf["nonfinite"], 12],
        [kf["small"], kf["tiny"]],
        [kf["overflow_big"], 14],
        [],
        [0],                                          # repeated across windows
        list(range(n)),
        [kf["lattice"], kf["lattice"], kf["tiny"]],
    ]
    return [win(kf, ids) for ids in w]


def reference(g, windows, leaf):
    out = []
    for ids, poses in windows:
        cloud, st = g.merge_keyframes(ids, poses, leaf)
        out.append((cloud, st))
    return out


def check(clouds, ovf, st, ref, where):
    assert len(clouds) == len(ref)
    for w, (c, (r, rst)) in enumerate(zip(clouds, ref)):
        assert c.shape == r.shape, (where, w, c.shape, r.shape)
        assert c.tobytes() == r.tobytes(), (where, w)
        assert bool(ovf[w]) == (rst == 1), (where, w)
    assert st == (1 if any(s == 1 for _, s in ref) else 0), where


@pytest.mark.gpu
@pytest.mark.parametrize("leaf", [LEAF, 0.4, 0.0])
def test_windows_byte_equal_to_merge_keyframes(g, kf, leaf, monkeypatch):
    windows = mixed_windows(kf)
    ref = reference(g, windows, leaf)
    if leaf > 0:
        assert any(s == 1 for _, s in ref) and any(len(r) == 0 for r, _ in ref)
    clouds, ovf, st = g.merge_keyframes_batch(windows, leaf)
    check(clouds, ovf, st, ref, "default pass")
    # the partition into passes does not matter: one window per pass, a few windows, and a pass smaller than a window
    for cap in ("1", "40000", "300000"):
        monkeypatch.setenv("LIOGPU_MERGE_PASS_POINTS", cap)
        clouds, ovf, st = g.merge_keyframes_batch(windows, leaf)
        check(clouds, ovf, st, ref, f"pass cap {cap}")


@pytest.mark.gpu
def test_leaf_nan_means_no_voxel_grid(g, kf):
    windows = mixed_windows(kf)[:6]
    ref = reference(g, windows, float("nan"))
    clouds, ovf, st = g.merge_keyframes_batch(windows, float("nan"))
    check(clouds, ovf, st, ref, "nan leaf")
    assert sum(len(c) for c in clouds) == sum(kf["clouds"][i].shape[0] for ids, _ in windows for i in ids)


@pytest.mark.gpu
def test_permutation_only_permutes_results(g, kf):
    windows = mixed_windows(kf)
    base, ovf0, st0 = g.merge_keyframes_batch(windows, LEAF)
    perm = np.random.default_rng(3).permutation(len(windows))
    clouds, ovf, st = g.merge_keyframes_batch([windows[i] for i in perm], LEAF)
    assert st == st0
    for j, i in enumerate(perm):
        assert clouds[j].tobytes() == base[i].tobytes() and ovf[j] == ovf0[i], (j, i)


@pytest.mark.gpu
def test_key_space_split(g, kf):
    """three windows of about 1.8e9 cells each cannot share the 32-bit key space: the call splits it"""
    names = [kf[f"keyspace{q}"] for q in range(3)]
    windows = [win(kf, [i]) for i in names] + [win(kf, [names[0], names[0]]), win(kf, [0])]
    ref = reference(g, windows, 0.1)
    assert not any(s == 1 for _, s in ref) and all(len(r) > 150 for r, _ in ref[:3])
    clouds, ovf, st = g.merge_keyframes_batch(windows, 0.1)
    check(clouds, ovf, st, ref, "key space")


@pytest.mark.gpu
def test_capacity_then_fetch(g, kf):
    from lio_slam_b200.liogpu import E_CAPACITY, W_LEAF_OVERFLOW
    windows = mixed_windows(kf)
    want, _, want_st = g.merge_keyframes_batch(windows, LEAF)
    ids = np.concatenate([np.asarray(i, np.int32) for i, _ in windows])
    poses = np.concatenate([p for _, p in windows]).astype(np.float32)
    win_off = np.r_[0, np.cumsum([len(i) for i, _ in windows])].astype(np.int32)
    out_off = np.zeros(len(windows) + 1, np.int32)
    buf = np.empty((1, 4), np.float32)
    st = g.lib.liogpu_merge_keyframes_batch(g.h, ids.ctypes.data, poses.ctypes.data, win_off.ctypes.data, len(windows),
                                            C.c_float(LEAF), buf.ctypes.data, 16, 0, out_off.ctypes.data, None)
    assert st == E_CAPACITY and want_st == W_LEAF_OVERFLOW
    assert np.array_equal(np.diff(out_off), [len(c) for c in want])
    out = np.empty((int(out_off[-1]), 4), np.float32)
    n = C.c_int(0)
    st = g.lib.liogpu_fetch_result(g.h, out.ctypes.data, 16, out.shape[0], C.byref(n))
    assert st == W_LEAF_OVERFLOW and n.value == out.shape[0]
    assert out.tobytes() == np.concatenate(want).tobytes()


@pytest.mark.gpu
def test_bad_arguments_refused_before_any_launch(g, kf):
    from lio_slam_b200.liogpu import E_INVALID, E_NO_KEYFRAME
    lib, h = g.lib, g.h
    ids = np.array([0, 1, 2], np.int32)
    poses = kf["poses"][:3].copy()
    out = np.empty((10, 4), np.float32)
    out_off = np.zeros(4, np.int32)
    big = kf["lattice"]  # 5,043 points: 425,900 repeats pass INT32_MAX
    many = np.full(425900, big, np.int32)
    many_poses = np.zeros((many.shape[0], 6), np.float32)

    def call(i, p, off, n, stride=16, o=out, oo=out_off):
        off = np.asarray(off, np.int32)
        return lib.liogpu_merge_keyframes_batch(h, i.ctypes.data if i is not None else None,
                                                p.ctypes.data if p is not None else None,
                                                off.ctypes.data if off.size else None, n, C.c_float(LEAF),
                                                o.ctypes.data, stride, o.shape[0],
                                                oo.ctypes.data if oo is not None else None, None)
    cases = [
        ((ids, poses, [0, 1, 3], -1), E_INVALID),             # negative window count
        ((ids, poses, [1, 2, 3], 2), E_INVALID),              # win_off not from 0
        ((ids, poses, [0, 2, 1, 3], 3), E_INVALID),           # decreasing
        ((None, poses, [0, 1, 3], 2), E_INVALID),             # null ids
        ((ids, None, [0, 1, 3], 2), E_INVALID),               # null poses
        ((ids, poses, [], 2), E_INVALID),                     # null win_off
        ((ids, poses, [0, 1, 3], 2, 20), E_INVALID),          # record stride outside the ABI
        ((np.array([0, 10 ** 6], np.int32), poses, [0, 1, 2], 2), E_NO_KEYFRAME),
        ((many, many_poses, [0, many.shape[0]], 1), E_INVALID),  # more than INT32_MAX input points
    ]
    for args, status in cases:
        before = g.launch_count()
        assert call(*args) == status, args
        assert g.launch_count() == before, args
    one = np.array([0, 3], np.int32)
    before = g.launch_count()
    assert lib.liogpu_merge_keyframes_batch(h, ids.ctypes.data, poses.ctypes.data, one.ctypes.data, 1, C.c_float(LEAF),
                                            out.ctypes.data, 16, 10, None, None) == E_INVALID  # null out_off
    assert g.launch_count() == before
    clouds, ovf, st = g.merge_keyframes_batch([], LEAF)
    assert clouds == [] and ovf.shape == (0,) and st == 0


@pytest.mark.gpu
def test_keeps_registration_and_resident_cloud(g, kf, small_case):
    g.set_local_map(small_case["map4"])
    p0, _, i0 = g.scan2map(small_case["scan4"], small_case["guess"])
    n_res, _ = g.voxel_downsample(small_case["scan4"], 0.4, keep_on_device=True)
    q0, _, _ = g.scan2map("resident", small_case["guess"])
    g.merge_keyframes_batch(mixed_windows(kf), LEAF)
    g.merge_keyframes_batch(mixed_windows(kf)[:4], 0.0)
    assert g.resident_size() == n_res
    q1, _, _ = g.scan2map("resident", small_case["guess"])
    assert np.array_equal(q0.view(np.uint32), q1.view(np.uint32))
    p1, _, i1 = g.scan2map(small_case["scan4"], small_case["guess"])
    assert np.array_equal(p0.view(np.uint32), p1.view(np.uint32)) and i0["iterations"] == i1["iterations"]


@pytest.mark.gpu
def test_launches_fixed_per_pass(g, kf):
    """one pass costs the same launches whether it holds 2, 16 or 64 windows, and far fewer than one call per window
    (the lattice windows keep the sort at three 8-bit digits and the scan at one level for every count)"""
    lat = win(kf, [kf["lattice"]])
    before = g.launch_count()
    g.merge_keyframes(*lat, LEAF)
    single = g.launch_count() - before
    per = {}
    for n in (2, 16, 64):
        before = g.launch_count()
        g.merge_keyframes_batch([lat] * n, LEAF)
        per[n] = g.launch_count() - before
    assert per[2] == per[16] == per[64], per
    assert per[64] < 64 * single, (per, single)


# ---- the loop-closure ICP batch builds its submaps with the segmented pass

def window(key, s, n_key):
    return list(range(max(key - s, 0), min(key + s, n_key - 1) + 1))


@pytest.mark.gpu
@pytest.mark.parametrize("env", [{}, {"LIOGPU_MERGE_PASS_POINTS": "200000"}, {"LIOGPU_MERGE_PASS_POINTS": "1",
                                                                             "LIOGPU_LOOP_ICP_GROUP": "3"}])
def test_loop_icp_batch_bit_equal_to_two_calls(g, kf, env, monkeypatch):
    poses = kf["poses"][:N_LAP]
    half = N_LAP // 2
    pairs = [(j, j - half) for j in range(half, N_LAP, 3)] + [(N_LAP - 1, 0), (half, half - 1), (30, 6), (30, 6)]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    T, res = g.loop_closure_icp_batch([c for c, _ in pairs], [p for _, p in pairs], poses, search_num=25, icp_leaf=LEAF)
    for k in env:
        monkeypatch.delenv(k)
    assert sum(not r["rejected_by_size"] for r in res) >= len(pairs) - 2
    for j, (c, p) in enumerate(pairs):
        src, st_s = g.merge_keyframes([c], poses[[c]], LEAF)
        w = window(p, 25, N_LAP)
        tgt, st_t = g.merge_keyframes(w, poses[w], LEAF)
        r = res[j]
        assert (r["n_source"], r["n_target"]) == (src.shape[0], tgt.shape[0]), j
        assert (r["source_overflow"], r["target_overflow"]) == (int(st_s == 1), int(st_t == 1)), j
        if src.shape[0] < 300 or tgt.shape[0] < 1000:
            assert r["rejected_by_size"] == 1 and np.array_equal(T[j], np.eye(4, dtype=np.float32)), j
            continue
        Tr, info = g.icp_align(src, tgt)
        assert np.array_equal(T[j].view(np.uint32), Tr.view(np.uint32)), (j, T[j], Tr)
        for k in ("iterations", "convergence_state", "converged", "n_correspondences"):
            assert r[k] == info[k], (j, k)
        for k in ("fitness_score", "last_mse"):
            assert np.float64(r[k]).view(np.uint64) == np.float64(info[k]).view(np.uint64), (j, k)
