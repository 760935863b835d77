"""liogpu_sc_add_keyframes: Scan Context descriptors of many resident keyframes appended to the descriptor store in one
call.  Every descriptor must be byte-equal to liogpu_make_scancontext (and the oracle) of the same cloud whatever the
batch around it, and the store must behave exactly as the per-keyframe path make_scancontext + sc_add built it: the
same offline and online detection results, with the online tree counter untouched by the batch call."""
import ctypes as C

import numpy as np
import pytest

from lio_slam_b200 import synth

N_BASE = 60   # distinct 16-beam keyframes along two laps; the sequence test jitters them into 300 distinct clouds


def same_bytes(a, b):
    return np.array_equal(np.asarray(a).view(np.uint64), np.asarray(b).view(np.uint64))


def test_sc_add_keyframes_exported():
    from lio_slam_b200 import liogpu
    lib = liogpu.load_library()
    assert "liogpu_sc_add_keyframes" in liogpu.EXPORTS
    assert lib.liogpu_sc_add_keyframes.argtypes == [C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_void_p]
    assert lib.liogpu_abi_version() == 2


def ctx():
    from lio_slam_b200.liogpu import LioGpu
    return LioGpu()


@pytest.fixture(scope="module")
def g():
    c = ctx()
    yield c
    c.close()


@pytest.fixture(scope="module")
def base(g, world):
    """N_BASE 16-beam sweeps (900 columns) every 1.7 m along synth.path_pose, voxelised at 0.2 as keyframes"""
    out = []
    for j in range(N_BASE):
        scan = synth.to_packed(synth.make_scan(world, synth.path_pose(1.7 * j), 16, seed=8100 + j, cols=900))
        out.append(g.voxel_downsample(scan, 0.2)[0])
    return out


def sequence(base, n, seed=3):
    """n distinct keyframe clouds: base clouds in turn, each with seeded centimetre jitter"""
    rng = np.random.default_rng(seed)
    out = []
    for j in range(n):
        c = base[j % len(base)].copy()
        c[:, :3] += rng.normal(0, 0.01, (c.shape[0], 3)).astype(np.float32)
        out.append(c)
    return out


def put_all(c, clouds, id0=0):
    c.keyframe_clear()
    for j, cl in enumerate(clouds):
        c.keyframe_put(id0 + j, cl)


def edge_cloud():
    """the bin-edge and degenerate points of test_scancontext_bin_edges_and_degenerate_points"""
    ang = np.deg2rad(np.arange(0, 360, 6.0))
    r = np.arange(4.0, 84.0, 4.0)
    pts = [[rr * np.cos(a), rr * np.sin(a), 0.3 * k] for k, rr in enumerate(r) for a in ang]
    pts += [[0, 0, 1], [0, 5, 1], [5, 0, 1], [-5, 0, 1], [0, -5, 1], [80.0, 0, 3], [80.0001, 0, 9], [56.57, 56.57, 4],
            [1, 1, -1500.0], [2, 2, -1002.0], [3, 3, np.nan], [np.inf, 1, 1], [1e-30, -1e-30, 0.5]]
    return np.c_[np.array(pts, np.float64), np.zeros(len(pts))].astype(np.float32)


@pytest.mark.gpu
def test_descriptors_match_single_cloud_path(g, oracle, world):
    """16-, 64- and 128-beam sweeps voxelised as keyframes: one batch call, every descriptor byte-equal to
    make_scancontext and to the oracle"""
    clouds = []
    for beams, seed in ((16, 1), (64, 2), (128, 3), (64, 4), (16, 5)):
        scan = synth.to_packed(synth.make_scan(world, synth.path_pose(0.9 * seed), beams, seed=60 + seed))
        clouds.append(g.voxel_downsample(scan, 0.2)[0])
    clouds.append(synth.to_packed(synth.make_scan(world, synth.path_pose(2.0), 128, seed=70)))  # raw 128-beam sweep
    assert max(c.shape[0] for c in clouds) > 100000
    put_all(g, clouds)
    g.sc_clear()
    descs = g.sc_add_keyframes(range(len(clouds)), return_descs=True)
    assert descs.shape == (len(clouds), 20, 60) and descs.dtype == np.float64
    for j, cl in enumerate(clouds):
        assert same_bytes(descs[j], g.make_scancontext(cl)[0]), j
        assert same_bytes(descs[j], oracle.make_scancontext(cl)[0]), j
        assert (descs[j] != 0).sum() > 100


def detect_all(c, n):
    return c.sc_detect_loops(np.arange(1, n + 1))


def same_detection(a, b, n):
    ia, ya, ma = detect_all(a, n)
    ib, yb, mb = detect_all(b, n)
    assert np.array_equal(ia, ib)
    assert np.array_equal(ya.view(np.uint32), yb.view(np.uint32))
    assert np.array_equal(ma.view(np.uint64), mb.view(np.uint64))
    return ia


@pytest.mark.gpu
def test_store_matches_per_keyframe_path(base):
    """context A: make_scancontext + sc_add per keyframe; context B: sc_add_keyframes in chunks of 1, 7 and the rest,
    one external descriptor sc_add-ed at the same position in both.  Offline detection over every store size and a run
    of online calls (which also sees the tree counter) must agree bit for bit."""
    clouds = sequence(base, 340)
    ext = np.random.default_rng(9).uniform(0, 5, (20, 60))
    a, b = ctx(), ctx()
    try:
        put_all(a, clouds)
        put_all(b, clouds)
        want = []
        for j in range(300):
            if j == 8:
                a.sc_add(ext)
            d = a.make_scancontext(clouds[j])[0]
            a.sc_add(d)
            want.append(d)
        got = [b.sc_add_keyframes([0], return_descs=True), b.sc_add_keyframes(range(1, 8), return_descs=True)]
        b.sc_add(ext)
        got.append(b.sc_add_keyframes(range(8, 300), return_descs=True))
        assert same_bytes(np.concatenate(got), np.array(want))
        loops = same_detection(a, b, 301)
        assert (loops >= 0).sum() > 50, loops
        for j in range(300, 340):   # online: add one keyframe, detect
            a.sc_add(a.make_scancontext(clouds[j])[0])
            b.sc_add_keyframes([j])
            ra, rb = a.sc_detect_loop(), b.sc_detect_loop()
            assert ra[0] == rb[0] and np.float32(ra[1]).view(np.uint32) == np.float32(rb[1]).view(np.uint32), j
            for k in ("n_stored", "n_searchable", "tree_rebuilt", "n_candidates", "nn_idx", "nn_align", "knn_ties"):
                assert ra[2][k] == rb[2][k], (j, k)
            assert np.float64(ra[2]["min_dist"]).view(np.uint64) == np.float64(rb[2]["min_dist"]).view(np.uint64)
            assert np.array_equal(ra[2]["candidates"], rb[2]["candidates"])
            assert np.array_equal(ra[2]["candidate_key_d2"].view(np.uint32), rb[2]["candidate_key_d2"].view(np.uint32))
            assert np.array_equal(ra[2]["candidate_dist"].view(np.uint64), rb[2]["candidate_dist"].view(np.uint64))
            assert np.array_equal(ra[2]["candidate_shift"], rb[2]["candidate_shift"])
        assert a.sc_detect_loop()[2]["n_stored"] == 341
    finally:
        a.close()
        b.close()


@pytest.mark.gpu
def test_edge_clouds(g, oracle):
    """points on ring and sector boundaries, NaN / inf / huge negative z, an empty keyframe; default constants and
    lidar_height 0, max_radius 40"""
    e = edge_cloud()
    clouds = [e, np.zeros((0, 4), np.float32), e[::-1].copy(), e[:7].copy(), np.zeros((0, 4), np.float32)]
    put_all(g, clouds)
    for kw in ({}, dict(lidar_height=0.0, max_radius=40.0)):
        g.sc_clear()
        descs = g.sc_add_keyframes([0, 1, 2, 3, 4], return_descs=True, **kw)
        for j, cl in enumerate(clouds):
            assert same_bytes(descs[j], g.make_scancontext(cl, **kw)[0]), (j, kw)
            assert same_bytes(descs[j], oracle.make_scancontext(cl, **kw)[0]), (j, kw)
        assert not descs[1].any() and not descs[4].any() and descs[0].any()


@pytest.mark.gpu
def test_repeats_overwrite_and_skew(g, base):
    """repeated ids, an id put again (its new cloud is used), and one 300k-point keyframe among 500 small ones"""
    rng = np.random.default_rng(4)
    big = np.c_[rng.uniform(-90, 90, (300000, 2)), rng.normal(0, 2, (300000, 1)), np.zeros((300000, 1))].astype(np.float32)
    small = [base[j % N_BASE][rng.integers(0, base[j % N_BASE].shape[0], int(rng.integers(1, 700)))] for j in range(500)]
    clouds = small[:250] + [big] + small[250:]
    put_all(g, clouds)
    ids = np.r_[np.arange(len(clouds)), [250, 3, 3, 250, 0]]
    g.sc_clear()
    d1 = g.sc_add_keyframes(ids, return_descs=True)
    ref = {}
    for k in set(ids.tolist()):
        ref[k] = g.make_scancontext(clouds[k])[0]
    for j, k in enumerate(ids):
        assert same_bytes(d1[j], ref[k]), (j, k)
    new3 = base[7]
    g.keyframe_put(3, new3)
    d2 = g.sc_add_keyframes([3, 250, 3], return_descs=True)
    assert same_bytes(d2[0], g.make_scancontext(new3)[0]) and same_bytes(d2[2], d2[0])
    assert not same_bytes(d2[0], ref[3]) and same_bytes(d2[1], ref[250])
    assert g.sc_detect_loop()[2]["n_stored"] == len(ids) + 3


@pytest.mark.gpu
def test_store_growth(base):
    """100 entries stored, then 3,000 small keyframes in one call: the store grows past its first capacity (1024)
    and every entry, old and new, behaves as in a store filled by sc_add"""
    rng = np.random.default_rng(6)
    clouds = [base[j % N_BASE][rng.integers(0, base[j % N_BASE].shape[0], int(rng.integers(50, 400)))] for j in range(3100)]
    a, b = ctx(), ctx()
    try:
        put_all(b, clouds)
        want = np.array([a.make_scancontext(cl)[0] for cl in clouds])
        a.sc_add(want)
        b.sc_add_keyframes(range(100))
        got = b.sc_add_keyframes(range(100, 3100), return_descs=True)
        assert same_bytes(got, want[100:])
        same_detection(a, b, 3100)
    finally:
        a.close()
        b.close()


@pytest.mark.gpu
def test_forced_passes(g, base, monkeypatch):
    """the call works in passes of at most 2^31 - 1 points (the staged tables' 32-bit offsets); LIOGPU_SC_PASS_POINTS
    lowers the cap: one keyframe per pass, a few per pass, a pass smaller than a keyframe.  Results are unchanged and
    every pass costs two launches (one if it holds no point), plus one store launch per call."""
    clouds = sequence(base, 80, seed=11)
    clouds[17] = np.zeros((0, 4), np.float32)
    put_all(g, clouds)
    g.sc_clear()
    ids = np.r_[np.arange(80), [5, 17, 5]]
    ref = g.sc_add_keyframes(ids, return_descs=True)
    want = detect_all(g, len(ids))
    sizes = [c.shape[0] for c in clouds]
    for cap in (1, 100000, 1000000):
        monkeypatch.setenv("LIOGPU_SC_PASS_POINTS", str(cap))
        passes = [[]]
        for k in ids:
            if passes[-1] and sum(sizes[i] for i in passes[-1]) + sizes[k] > cap:
                passes.append([])
            passes[-1].append(k)
        launches = sum(1 + (sum(sizes[i] for i in p) > 0) for p in passes) + 1   # slot init, binning; store
        g.sc_clear()
        l0 = g.launch_count()
        got = g.sc_add_keyframes(ids, return_descs=True)
        assert g.launch_count() - l0 == launches, (cap, len(passes))
        assert same_bytes(got, ref), cap
        for a, b in zip(detect_all(g, len(ids)), want):
            assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), cap
    monkeypatch.delenv("LIOGPU_SC_PASS_POINTS")


@pytest.mark.gpu
def test_refusals_leave_store_and_launches_alone(base):
    from lio_slam_b200.liogpu import E_INVALID, E_NO_KEYFRAME, LioGpuError
    c = ctx()
    try:
        put_all(c, base[:10])
        c.sc_add_keyframes(range(10))
        ids = np.array([0, 1, 2, 77, 3], np.int32)
        out = np.zeros((5, 1200))
        cases = [(ids, 5, 80.0, E_NO_KEYFRAME), (ids, 0, 80.0, E_INVALID), (ids, -1, 80.0, E_INVALID),
                 (None, 3, 80.0, E_INVALID), (ids[:3], 3, 0.0, E_INVALID), (ids[:3], 3, float("nan"), E_INVALID),
                 (ids[:3], 3, -1.0, E_INVALID)]
        for arr, n, r, st in cases:
            l0 = c.launch_count()
            got = c.lib.liogpu_sc_add_keyframes(c.h, None if arr is None else arr.ctypes.data, n, 2.0, r, out.ctypes.data)
            assert got == st, (arr, n, r, got)
            assert c.launch_count() == l0
            assert not out.any()
        c.sc_detect_loops([10])
        with pytest.raises(LioGpuError) as e:
            c.sc_detect_loops([11])
        assert e.value.status == E_INVALID
        assert c.sc_detect_loop()[2]["n_stored"] == 10
    finally:
        c.close()


@pytest.mark.gpu
def test_store_survives_keyframe_clear(base):
    """the descriptors live in the store, not in the keyframes: keyframe_clear leaves detection as it was"""
    clouds = sequence(base, 120, seed=8)
    a, b = ctx(), ctx()
    try:
        put_all(b, clouds)
        for cl in clouds:
            a.sc_add(a.make_scancontext(cl)[0])
        b.sc_add_keyframes(range(120))
        b.keyframe_clear()
        assert b.keyframe_count() == 0
        same_detection(a, b, 120)
        ra, rb = a.sc_detect_loop(), b.sc_detect_loop()
        assert ra[0] == rb[0] and ra[2]["nn_idx"] == rb[2]["nn_idx"] and ra[2]["n_stored"] == rb[2]["n_stored"] == 120
        assert np.float64(ra[2]["min_dist"]).view(np.uint64) == np.float64(rb[2]["min_dist"]).view(np.uint64)
    finally:
        a.close()
        b.close()
