"""GPU parity of liogpu_publish_local_map against the oracle's restatement of publishLocalMap
(mapOptmization.cpp:2442-2541, SURVEY §8 row f2).  Bit-exact: cropped cloud, kept set, mean distances (through
the kept set and the statistics), VoxelGrid output.  The statistics (mean / stddev / threshold) are f64 sums whose
order differs (sequential in PCL and the oracle, tree-wise on the GPU): compared to 1e-12 relative, and a kept-set
comparison is only meaningful when no point sits within 1e-9 of the threshold (info.sor_borderline == 0)."""
import numpy as np
import pytest

from lio_slam_b200 import synth

pytestmark = pytest.mark.gpu


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def assert_biteq(a, b, what=""):
    assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
    if not np.array_equal(bits(a), bits(b)):
        bad = np.nonzero((bits(a) != bits(b)).any(axis=1))[0]
        raise AssertionError(f"{what}: {bad.size} rows differ, first {bad[0]}: {a[bad[0]]} vs {b[bad[0]]}")


def keyframes(world, oracle, n_kf, beams=16, cols=450, step=1.0, leaf=0.4, seed0=300):
    clouds, poses = [], []
    for k in range(n_kf):
        p = synth.path_pose(step * k)
        sc = synth.make_scan(world, p, beams, seed=seed0 + k, cols=cols)
        ds, _ = oracle.voxel_grid(synth.to_packed(sc), leaf)
        clouds.append(ds)
        poses.append(p.astype(np.float32))
    return clouds, np.array(poses, np.float32)


def put(gpu, clouds, base=500):
    gpu.keyframe_clear()
    for k, c in enumerate(clouds):
        gpu.keyframe_put(base + k, c)
    return [base + k for k in range(len(clouds))]


def check(gpu, oracle, clouds, poses, pose_now, ids=None, brute=False, **kw):
    okw = dict(left=kw.get("local_map_left", 40.0), right=kw.get("local_map_right", 40.0),
               front=kw.get("local_map_front", 70.0), back=kw.get("local_map_back", 20.0),
               use_removing_outliers=bool(kw.get("use_removing_outliers", 1)), mean_k=kw.get("mean_k", 10),
               stddev_threshold=kw.get("stddev_threshold", 1.0), use_down_sampling=bool(kw.get("use_down_sampling", 1)),
               leaf=kw.get("local_mapping_surf_leaf_size", 0.01))
    want, winfo, _ = oracle.publish_local_map(clouds, poses, pose_now, brute=brute, threads=8, **okw)
    if ids is None:
        ids = put(gpu, clouds)
    got, info, st = gpu.publish_local_map(ids, poses, pose_now, **kw)
    for key in ("n_concat", "n_cropped"):
        assert info[key] == winfo[key], (key, info[key], winfo[key])
    if okw["use_removing_outliers"] and winfo["n_cropped"] > okw["mean_k"]:
        for key in ("sor_mean", "sor_stddev", "sor_threshold"):
            assert info[key] == pytest.approx(winfo[key], rel=1e-12), key
        assert info["sor_borderline"] == 0
    assert info["n_after_sor"] == winfo["n_after_sor"]
    assert info["leaf_overflow"] == winfo["leaf_overflow"]
    assert st == (1 if winfo["leaf_overflow"] else 0)
    assert_biteq(got, want, "tempCloud")
    assert info["n_out"] == want.shape[0]
    return got, info, winfo


def test_publish_local_map_defaults(gpu, oracle, world):
    """utility.h defaults: crop, outlier filter (meanK 10, 1 sigma), leaf 0.01 -> the overflow guard fires (q4)."""
    clouds, poses = keyframes(world, oracle, 8)
    pose_now = synth.perturbed_guess(poses[-1], 3).astype(np.float32)
    got, info, winfo = check(gpu, oracle, clouds, poses, pose_now)
    assert info["leaf_overflow"] == 1 and info["n_out"] == info["n_after_sor"]
    assert 0 < info["n_after_sor"] < info["n_cropped"] < info["n_concat"]


@pytest.mark.parametrize("mean_k,std,leaf", [(10, 1.0, 0.2), (5, 0.5, 0.4), (15, 2.0, 0.2), (31, 1.0, 0.5), (1, 1.0, 0.3)])
def test_publish_local_map_outlier_filter_variants(gpu, oracle, world, mean_k, std, leaf):
    clouds, poses = keyframes(world, oracle, 6, seed0=340)
    pose_now = poses[-1].copy()
    pose_now[2] += 0.3
    got, info, _ = check(gpu, oracle, clouds, poses, pose_now, mean_k=mean_k, stddev_threshold=std,
                         local_mapping_surf_leaf_size=leaf)
    assert info["leaf_overflow"] == 0 and info["n_out"] < info["n_after_sor"]


def test_publish_local_map_matches_bruteforce_knn(gpu, oracle, world):
    """the oracle's exhaustive (meanK+1)-NN, independent of any tree or grid"""
    clouds, poses = keyframes(world, oracle, 3, cols=300, seed0=360)
    check(gpu, oracle, clouds, poses, poses[1], brute=True, local_mapping_surf_leaf_size=0.2)


def test_publish_local_map_shipped_yaml(gpu, oracle, world):
    """config/jeep.yaml: outlier filter off, leaf 0.2; 6t.yaml: leaf 0.01 (guard)"""
    clouds, poses = keyframes(world, oracle, 10, seed0=380)
    ids = put(gpu, clouds)
    now = poses[-1]
    check(gpu, oracle, clouds, poses, now, ids=ids, use_removing_outliers=0, local_mapping_surf_leaf_size=0.2)
    check(gpu, oracle, clouds, poses, now, ids=ids, use_removing_outliers=0, local_mapping_surf_leaf_size=0.01)
    check(gpu, oracle, clouds, poses, now, ids=ids, use_removing_outliers=0, use_down_sampling=0)
    # the last localMapKeyFramesNumber keyframes only (mapOptmization.cpp:2462)
    check(gpu, oracle, clouds[-4:], poses[-4:], now, ids=ids[-4:], local_mapping_surf_leaf_size=0.2)


@pytest.mark.parametrize("yaw", [0.0, 1.0, -2.5, 3.1])
def test_publish_local_map_yaw_frame(gpu, oracle, world, yaw):
    """Eigen's angle-axis matrix has zz = (1 - c) + c: the z coordinate is scaled by a value that is not always 1"""
    clouds, poses = keyframes(world, oracle, 3, cols=300, seed0=400)
    now = np.array([0.01, -0.02, yaw, 3.0, -2.0, 0.4], np.float32)
    m = oracle.yaw_frame_T(now)
    assert m[10] == np.float32(np.float32(1.0) - m[0]) + m[0]
    check(gpu, oracle, clouds, poses, now, use_removing_outliers=0, use_down_sampling=0)


def test_publish_local_map_isolated_points_and_cell_size(gpu, oracle, world):
    """sparse cloud with far-away stragglers: the wide search (many shells, then exhaustive) must agree, and the
    tuning knob must not change anything"""
    rng = np.random.default_rng(5)
    base = np.c_[rng.uniform(-30, 30, (4000, 2)), rng.normal(0, 0.05, (4000, 1)), rng.uniform(0, 100, (4000, 1))]
    lone = np.c_[rng.uniform(-39, 39, (40, 2)), rng.uniform(5, 60, (40, 1)), rng.uniform(0, 100, (40, 1))]
    cluster = np.c_[rng.normal(20, 0.02, (60, 3)), rng.uniform(0, 100, (60, 1))]
    clouds = [base.astype(np.float32), np.vstack([lone, cluster]).astype(np.float32)]
    poses = np.zeros((2, 6), np.float32)
    now = np.zeros(6, np.float32)
    ids = put(gpu, clouds)
    ref = None
    for cell in (0.0, 0.15, 1.0, 5.0):
        got, info, _ = check(gpu, oracle, clouds, poses, now, ids=ids, brute=True, sor_cell_size=cell,
                             local_mapping_surf_leaf_size=0.3, local_map_back=40.0, local_map_front=40.0)
        if cell == 0.0:
            assert info["sor_leftover"] > 0 and info["sor_exhaustive"] > 0
        if ref is None:
            ref = got
        assert_biteq(got, ref, f"cell {cell}")


def test_publish_local_map_duplicates(gpu, oracle):
    """coincident points: zero distances, (meanK+1)-th neighbour tied many times"""
    rng = np.random.default_rng(9)
    pts = np.c_[rng.integers(-20, 20, (3000, 2)) * 0.5, np.zeros((3000, 1)), rng.uniform(0, 100, (3000, 1))].astype(np.float32)
    clouds = [pts, pts[:1000].copy()]
    poses = np.zeros((2, 6), np.float32)
    check(gpu, oracle, clouds, poses, np.zeros(6, np.float32), brute=True, local_mapping_surf_leaf_size=0.3)


def test_publish_local_map_small_and_empty(gpu, oracle):
    from lio_slam_b200.liogpu import LioGpuError, W_NO_KEYFRAMES
    rng = np.random.default_rng(2)
    # fewer points than meanK + 1: PCL's search comes back short, nothing is removed
    few = np.c_[rng.uniform(-5, 5, (7, 3)), rng.uniform(0, 100, (7, 1))].astype(np.float32)
    poses = np.zeros((1, 6), np.float32)
    got, info, _ = check(gpu, oracle, [few], poses, np.zeros(6, np.float32), local_mapping_surf_leaf_size=0.2)
    assert info["n_after_sor"] == 7
    # exactly meanK + 1 points
    eleven = np.c_[rng.uniform(-5, 5, (11, 3)), rng.uniform(0, 100, (11, 1))].astype(np.float32)
    check(gpu, oracle, [eleven], poses, np.zeros(6, np.float32), local_mapping_surf_leaf_size=0.2)
    # everything cropped away
    far = few.copy()
    far[:, 0] += 500.0
    got, info, _ = check(gpu, oracle, [far], poses, np.zeros(6, np.float32))
    assert got.shape[0] == 0 and info["n_cropped"] == 0
    # non-finite points are dropped by PassThrough
    bad = eleven.copy()
    bad[3, 1] = np.nan
    bad[5, 2] = np.inf
    got, info, _ = check(gpu, oracle, [bad], poses, np.zeros(6, np.float32), use_removing_outliers=0, use_down_sampling=0)
    assert info["n_cropped"] == 9
    # no keyframes: publishLocalMap returns at once (mapOptmization.cpp:2444)
    got, info, st = gpu.publish_local_map(np.zeros(0, np.int32), np.zeros((0, 6), np.float32), np.zeros(6, np.float32))
    assert st == W_NO_KEYFRAMES and got.shape[0] == 0
    with pytest.raises(LioGpuError):
        gpu.publish_local_map([12345], poses, np.zeros(6, np.float32))
    with pytest.raises(LioGpuError):
        gpu.publish_local_map(put(gpu, [few]), poses, np.zeros(6, np.float32), mean_k=40)


def test_publish_local_map_keeps_registration_index(gpu, oracle, small_case):
    """publishLocalMap runs between registrations (mapOptmization.cpp:504): it must not disturb the local-map index"""
    gpu.set_local_map(small_case["map4"])
    p0, _, i0 = gpu.scan2map(small_case["scan4"], small_case["guess"])
    clouds = [small_case["scan4"], small_case["map4"][:5000]]
    poses = np.array([small_case["pose_gt"], np.zeros(6)], np.float32)
    put(gpu, clouds)
    gpu.publish_local_map([500, 501], poses, small_case["pose_gt"].astype(np.float32), local_mapping_surf_leaf_size=0.2)
    p1, _, i1 = gpu.scan2map(small_case["scan4"], small_case["guess"])
    assert np.array_equal(bits(p0), bits(p1)) and i0["iterations"] == i1["iterations"]


def test_publish_local_map_realistic_size(gpu, oracle, world):
    """50 keyframes (6t.yaml localMapKeyFramesNumber) of a 32-beam sweep against the nanoflann-backed oracle when it is
    built, else against the oracle's own KD-tree.  The outlier filter reads only the k nearest distances, which every
    exact k-NN search returns alike, and the own tree is held to exhaustive search bit for bit
    (tests/test_oracle_core.py::test_knn_kdtree_equals_bruteforce, test_oracle_sor_knn_providers_agree and
    test_publish_local_map_matches_bruteforce_knn above)"""
    from oracle.oracle import Oracle
    ref = Oracle("nanoflann") if Oracle.available("nanoflann") else oracle
    clouds, poses = keyframes(world, ref, 50, beams=32, cols=900, step=0.5, seed0=700)
    got, info, _ = check(gpu, ref, clouds, poses, poses[-1], local_mapping_surf_leaf_size=0.2)
    assert info["n_concat"] > 300000


def test_merge_keyframes_global_map_and_save_map(gpu, oracle, world, small_case):
    """saveMapService (mapOptmization.cpp:936-950) / publishGlobalMap (:1031-1039) cloud assembly: transform +
    concatenate (+ VoxelGrid), bit-exact, without touching the registration's local map"""
    from lio_slam_b200.liogpu import LioGpuError
    gpu.set_local_map(small_case["map4"])
    p0, _, i0 = gpu.scan2map(small_case["scan4"], small_case["guess"])
    clouds, poses = keyframes(world, oracle, 7, seed0=420)
    ids = put(gpu, clouds)
    raw = np.concatenate([oracle.transform_cloud(c, p) for c, p in zip(clouds, poses)])
    got, st = gpu.merge_keyframes(ids, poses, 0.0)              # req.resolution == 0: the raw concatenation
    assert st == 0
    assert_biteq(got, raw, "globalSurfCloud")
    for leaf in (0.4, 1.0):                                     # globalMapVisualizationLeafSize / req.resolution
        want, ov = oracle.build_local_map(clouds, poses, leaf, threads=4)
        got, st = gpu.merge_keyframes(ids, poses, leaf)
        assert st == 0 and not ov
        assert_biteq(got, want, f"leaf {leaf}")
    sel = [5, 1, 3]                                             # the host's choice and order of key poses
    want, _ = oracle.build_local_map([clouds[j] for j in sel], poses[sel], 0.4)
    got, _ = gpu.merge_keyframes([ids[j] for j in sel], poses[sel], 0.4)
    assert_biteq(got, want, "subset")
    got, st = gpu.merge_keyframes(ids, poses, 0.001)            # overflow guard: input returned unchanged (q4)
    assert st == 1
    assert_biteq(got, raw, "guard")
    got, st = gpu.merge_keyframes(np.zeros(0, np.int32), np.zeros((0, 6), np.float32), 0.4)
    assert got.shape[0] == 0 and st == 0
    with pytest.raises(LioGpuError):
        gpu.merge_keyframes([4242], poses[:1], 0.4)
    assert gpu.local_map_size() == small_case["map4"].shape[0]
    p1, _, i1 = gpu.scan2map(small_case["scan4"], small_case["guess"])
    assert np.array_equal(bits(p0), bits(p1)) and i0["iterations"] == i1["iterations"]
