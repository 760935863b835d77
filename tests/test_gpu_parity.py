"""GPU parity tests: the CUDA path, called through the C ABI (libliogpu.so), against the CPU oracle on
identical seeded inputs.  Bars (BASELINE.json north_star): voxel outputs and neighbour sets bit-exact
(modulo logged equidistant ties), poses within 1e-4 m / 1e-5 rad, JtJ within 1e-5 relative."""
import numpy as np
import pytest

from lio_slam_b200 import synth

pytestmark = pytest.mark.gpu

POS_TOL = 1e-4   # metres
ROT_TOL = 1e-5   # radians
JTJ_RTOL = 1e-5


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def assert_biteq(a, b, what=""):
    a = np.ascontiguousarray(a, np.float32); b = np.ascontiguousarray(b, np.float32)
    assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
    ne = bits(a) != bits(b)
    assert not ne.any(), f"{what}: {int(ne.sum())} of {ne.size} words differ; first at {np.argwhere(ne)[:3].tolist()}"


# ---------------------------------------------------------------- a2 transformPointCloud
def test_transform_cloud_bitexact(gpu, oracle, small_case):
    pose = np.array([0.03, -0.02, 1.2, 10.5, -3.25, 0.7], np.float32)
    got = gpu.transform_cloud(small_case["scan4"], pose)
    assert_biteq(got, oracle.transform_cloud(small_case["scan4"], pose), "transform")
    # 32-byte PointXYZI records in, packed out
    got32 = gpu.transform_cloud(synth.xyzirt_to_xyzi(small_case["scan"]), pose)
    assert_biteq(got32, got, "transform stride 32")


# ---------------------------------------------------------------- a3 / a4 VoxelGrid
@pytest.mark.parametrize("leaf", [0.1, 0.2, 0.4, 0.5, 1.0, 2.0])
def test_voxel_scan_bitexact(gpu, oracle, small_case, leaf):
    want, ov = oracle.voxel_grid(small_case["scan4"], leaf)
    got, st = gpu.voxel_downsample(small_case["scan4"], leaf)
    assert not ov and st == 0
    assert_biteq(got, want, f"voxel leaf {leaf}")


@pytest.mark.parametrize("n,scale,leaf,seed", [(1, 1.0, 0.2, 0), (2, 1.0, 0.2, 1), (31, 5.0, 0.5, 2), (2048, 30.0, 0.3, 3),
                                                (2049, 30.0, 0.3, 4), (100000, 60.0, 0.4, 5), (300001, 100.0, 0.2, 6),
                                                (50000, 0.05, 1.0, 7)])
def test_voxel_random_bitexact(gpu, oracle, n, scale, leaf, seed):
    rng = np.random.default_rng(seed)
    cloud = np.column_stack([rng.normal(0, scale, n), rng.normal(0, scale, n), rng.normal(0, scale / 10, n),
                             rng.uniform(0, 100, n)]).astype(np.float32)
    want, ov = oracle.voxel_grid(cloud, leaf)
    got, st = gpu.voxel_downsample(cloud, leaf)
    assert (st == 1) == ov
    assert_biteq(got, want, f"voxel random n={n}")


def test_voxel_overflow_guard_returns_input(gpu, oracle, small_case):
    # 6t.yaml's mappingSurfLeafSize 0.01 over a 100 m sweep: PCL's index would overflow -> input returned (q4)
    want, ov = oracle.voxel_grid(small_case["scan4"], 0.001)
    got, st = gpu.voxel_downsample(small_case["scan4"], 0.001)
    assert ov and st == 1
    assert_biteq(got, small_case["scan4"], "overflow passthrough")
    assert_biteq(got, want)


def test_voxel_nonfinite_and_empty(gpu, oracle):
    rng = np.random.default_rng(9)
    cloud = rng.normal(0, 10, (5000, 4)).astype(np.float32)
    cloud[::7, 0] = np.nan
    cloud[3::11, 2] = np.inf
    want, _ = oracle.voxel_grid(cloud, 0.5)
    got, st = gpu.voxel_downsample(cloud, 0.5)
    assert_biteq(got, want, "voxel with non-finite points")
    got, st = gpu.voxel_downsample(np.zeros((0, 4), np.float32), 0.5)
    assert got.shape[0] == 0 and st == 0


def test_voxel_stride32_roundtrip(gpu, oracle, small_case):
    recs = synth.xyzirt_to_xyzi(small_case["scan"])
    want, _ = oracle.voxel_grid(small_case["scan4"], 0.4)
    got, st = gpu.voxel_downsample(recs, 0.4, out_stride=32)
    assert got.shape[1] == 8
    assert_biteq(got[:, [0, 1, 2, 4]], want, "voxel 32-byte records")
    assert (got[:, 3] == 1.0).all()  # PCL keeps data[3] = 1


# ---------------------------------------------------------------- a5 / a7 k-NN + plane fit
def test_knn_bitexact_vs_bruteforce(gpu, oracle, small_case):
    map4 = small_case["map4"]
    ds, _ = oracle.voxel_grid(small_case["scan4"], 0.4)
    T = oracle.pose_to_T(small_case["guess"])
    ref = oracle.surf_optimization(map4, ds, T12=T, threads=8)           # brute force k-NN
    gpu.set_local_map(map4)
    got = gpu.surf_optimization(ds, T12=T)
    gate = ref["nn_d2"][:, 4] < 1.0                                       # MO:1641: others are discarded
    assert gate.sum() > 1000
    notie = gate & (ref["tie"] == 0)
    assert np.array_equal(got["nn_idx"][notie], ref["nn_idx"][notie]), "neighbour sets differ outside ties"
    assert_biteq(got["nn_d2"][gate], ref["nn_d2"][gate], "pointSearchSqDis")
    assert np.array_equal(got["tie"][gate], ref["tie"][gate]), "tie log differs"
    # with the canonical tie-break (lower map index) even tied queries must agree
    assert np.array_equal(got["nn_idx"][gate], ref["nn_idx"][gate])
    # queries outside the gate must be reported as such
    assert (got["nn_d2"][~gate, 4] >= 1.0).all()
    assert np.array_equal(got["flag"], ref["flag"])
    assert_biteq(got["coeff"], ref["coeff"], "coeffSel")
    print(f"queries={ds.shape[0]} gated={int(gate.sum())} accepted={int(ref['flag'].sum())} ties={int(ref['tie'].sum())}")


def test_knn_ties_are_logged_and_canonical(gpu, oracle):
    # a lattice map makes equidistant neighbours the rule, not the exception
    g = np.arange(-3, 3.01, 0.25, dtype=np.float32)
    X, Y, Z = np.meshgrid(g, g, np.array([0.0, 0.25], np.float32), indexing="ij")
    map4 = np.column_stack([X.ravel(), Y.ravel(), Z.ravel(), np.zeros(X.size)]).astype(np.float32)
    rng = np.random.default_rng(3)
    q = np.column_stack([rng.choice(g, 4000), rng.choice(g, 4000), rng.uniform(0, 0.25, 4000), np.ones(4000)]).astype(np.float32)
    T = np.array([1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0], np.float32)
    ref = oracle.surf_optimization(map4, q, T12=T, threads=8)
    gpu.set_local_map(map4)
    got = gpu.surf_optimization(q, T12=T)
    assert ref["tie"].sum() > 1000
    assert np.array_equal(got["tie"], ref["tie"])
    assert np.array_equal(got["nn_idx"], ref["nn_idx"])
    assert_biteq(got["nn_d2"], ref["nn_d2"])


@pytest.mark.parametrize("cell,r1", [(0.25, 0.0), (0.5, -1.0), (1.0, 0.3), (2.0, 0.6), (0.0, 0.45), (0.3, 0.79)])
def test_knn_independent_of_cell_size(oracle, small_case, cell, r1):
    # cell edge and phase-1 radius are tuning knobs: results must not depend on them
    from lio_slam_b200.liogpu import LioGpu
    g = LioGpu(knn_cell_size=cell, knn_phase1_radius=r1)
    try:
        ds, _ = oracle.voxel_grid(small_case["scan4"], 0.8)
        T = oracle.pose_to_T(small_case["guess"])
        ref = oracle.surf_optimization(small_case["map4"], ds, T12=T, threads=8)
        g.set_local_map(small_case["map4"])
        got = g.surf_optimization(ds, T12=T)
        gate = ref["nn_d2"][:, 4] < 1.0
        assert np.array_equal(got["nn_idx"][gate], ref["nn_idx"][gate])
        assert_biteq(got["nn_d2"][gate], ref["nn_d2"][gate])
        assert np.array_equal(got["tie"][gate], ref["tie"][gate])
        assert np.array_equal(got["flag"], ref["flag"])
        assert_biteq(got["coeff"], ref["coeff"])
    finally:
        g.close()


def test_knn_map_far_from_origin(gpu, oracle, small_case):
    # large coordinates stress the positional slack of the grid pruning
    off = np.array([4000.0, -7000.0, 300.0, 0.0], np.float32)
    map4 = (small_case["map4"] + off).astype(np.float32)
    ds, _ = oracle.voxel_grid(small_case["scan4"], 0.6)
    pose = small_case["guess"].copy(); pose[3:] += off[:3]
    T = oracle.pose_to_T(pose)
    ref = oracle.surf_optimization(map4, ds, T12=T, threads=8)
    gpu.set_local_map(map4)
    got = gpu.surf_optimization(ds, T12=T)
    gate = ref["nn_d2"][:, 4] < 1.0
    assert gate.sum() > 500
    assert np.array_equal(got["nn_idx"][gate], ref["nn_idx"][gate])
    assert_biteq(got["nn_d2"][gate], ref["nn_d2"][gate])
    assert np.array_equal(got["flag"], ref["flag"])


# ---------------------------------------------------------------- a8 / a9 / a10 the LM loop
def check_s2m(got_pose, got_info, ref_pose, ref_info):
    assert got_info["iterations"] == ref_info["iterations"]
    assert got_info["converged"] == ref_info["converged"]
    assert np.array_equal(got_info["nsel_hist"], ref_info["nsel_hist"])
    assert np.abs(got_pose[:3] - ref_pose[:3]).max() <= ROT_TOL
    assert np.abs(got_pose[3:] - ref_pose[3:]).max() <= POS_TOL
    scale = np.abs(ref_info["JtJ"]).max()
    assert np.abs(got_info["JtJ"] - ref_info["JtJ"]).max() <= JTJ_RTOL * scale
    assert np.abs(got_info["Jtr"] - ref_info["Jtr"]).max() <= JTJ_RTOL * max(np.abs(ref_info["Jtr"]).max(), 1e-12) + 1e-9
    assert got_info["is_degenerate"] == ref_info["is_degenerate"]
    assert got_info["tie_queries"] == ref_info["tie_queries"]


@pytest.mark.parametrize("max_iter", [1, 2, 30])
def test_scan2map_pose_parity(gpu, oracle, small_case, max_iter):
    ds, _ = oracle.voxel_grid(small_case["scan4"], 0.4)
    ref_pose, ref_P, ref_info = oracle.scan2map(small_case["map4"], ds, small_case["guess"], max_iter=max_iter, threads=8)
    gpu.set_local_map(small_case["map4"])
    pose, P, info = gpu.scan2map(ds, small_case["guess"], max_iter=max_iter)
    check_s2m(pose, info, ref_pose, ref_info)
    assert np.abs(info["pose_hist"] - ref_info["pose_hist"]).max() <= POS_TOL
    assert np.abs(P - ref_P).max() <= 1e-5
    # the registration must actually move toward ground truth
    if max_iter == 30:
        gt = small_case["pose_gt"].astype(np.float32)
        assert np.abs(pose[3:] - gt[3:]).max() < 0.05 and np.abs(pose[:3] - gt[:3]).max() < 0.01
        assert info["converged"]
    print(f"iters={info['iterations']} nsel={info['n_sel']} gpu_ms={info['gpu_ms']:.3f} bit_equal_pose={np.array_equal(pose, ref_pose)}")


def test_scan2map_degenerate_direction(gpu, oracle):
    # a single ground plane constrains only z, roll, pitch: eigenvalues of AtA below 100 must be
    # projected out through matP (MO:1786-1815)
    rng = np.random.default_rng(4)
    gx, gy = np.meshgrid(np.arange(-20, 20, 0.4), np.arange(-20, 20, 0.4), indexing="ij")
    map4 = np.column_stack([gx.ravel(), gy.ravel(), rng.normal(0, 0.005, gx.size), np.zeros(gx.size)]).astype(np.float32)
    q = np.column_stack([rng.uniform(-15, 15, 3000), rng.uniform(-15, 15, 3000), np.full(3000, -1.5), np.ones(3000)]).astype(np.float32)
    guess = np.array([0.01, -0.01, 0.3, 0.2, -0.1, 1.55], np.float32)
    ref_pose, ref_P, ref_info = oracle.scan2map(map4, q, guess, threads=8)
    gpu.set_local_map(map4)
    pose, P, info = gpu.scan2map(q, guess)
    assert ref_info["is_degenerate"] == 1
    check_s2m(pose, info, ref_pose, ref_info)
    assert np.abs(P - ref_P).max() <= 1e-5


def test_scan2map_guards(gpu, oracle, small_case):
    from lio_slam_b200 import liogpu as L
    gpu.set_local_map(small_case["map4"])
    few = small_case["scan4"][:30]
    pose, P, info = gpu.scan2map(few, small_case["guess"])
    assert info["status"] == L.W_FEW_FEATURES and np.array_equal(pose, small_case["guess"])
    # < 50 accepted correspondences: LMOptimization returns false, pose untouched, 30 iterations (q2)
    far = small_case["scan4"][:200].copy(); far[:, :3] += 500.0
    ref_pose, _, ref_info = oracle.scan2map(small_case["map4"], far, small_case["guess"], threads=4)
    pose, P, info = gpu.scan2map(far, small_case["guess"])
    assert info["iterations"] == ref_info["iterations"] == 30 and not info["converged"]
    assert np.array_equal(pose, small_case["guess"]) and np.array_equal(ref_pose, small_case["guess"])
    # matP / isDegenerate persist when iteration 0 bails out (q3)
    P0 = np.eye(6, dtype=np.float32) * 0.5
    pose, P, info = gpu.scan2map(far, small_case["guess"], matP=P0, degenerate=1)
    assert np.array_equal(P, P0) and info["is_degenerate"] == 1
    gpu.set_local_map(np.zeros((0, 4), np.float32))
    pose, P, info = gpu.scan2map(small_case["scan4"], small_case["guess"])
    assert info["status"] == L.W_NO_KEYFRAMES


def test_downsample_scan2map_fused(gpu, oracle, small_case):
    from lio_slam_b200.liogpu import LioGpu
    g = LioGpu(mapping_surf_leaf_size=0.4)
    try:
        ds, _ = oracle.voxel_grid(small_case["scan4"], 0.4)
        ref_pose, ref_P, ref_info = oracle.scan2map(small_case["map4"], ds, small_case["guess"], threads=8)
        g.set_local_map(small_case["map4"])
        pose, P, info = g.downsample_scan2map(synth.xyzirt_to_xyzi(small_case["scan"]), small_case["guess"], fetch_ds=True)
        assert info["n_ds"] == ds.shape[0]
        assert_biteq(info["scan_ds"], ds, "laserCloudSurfLastDS")
        check_s2m(pose, info, ref_pose, ref_info)
    finally:
        g.close()


# ---------------------------------------------------------------- a2 + a3: extractCloud
def test_build_local_map_bitexact(gpu, oracle, world):
    clouds, poses = [], []
    for k in range(6):
        p = synth.path_pose(-0.7 * k)
        sc = synth.make_scan(world, p, 16, seed=100 + k, cols=450)
        ds, _ = oracle.voxel_grid(synth.to_packed(sc), 0.4)
        clouds.append(ds); poses.append(p.astype(np.float32))
    want, ov = oracle.build_local_map(clouds, np.array(poses), 0.5, threads=4)
    gpu.keyframe_clear()
    for k, c in enumerate(clouds):
        gpu.keyframe_put(10 + k, c)
    assert gpu.keyframe_count() == 6
    got, st = gpu.build_local_map([10 + k for k in range(6)], np.array(poses), 0.5)
    assert st == 0 and not ov
    assert_biteq(got, want, "laserCloudSurfFromMapDS")
    assert gpu.local_map_size() == want.shape[0]
    # and the installed index answers queries like the oracle on that map
    q = clouds[0]
    T = oracle.pose_to_T(poses[0])
    ref = oracle.surf_optimization(want, q, T12=T, threads=8)
    res = gpu.surf_optimization(q, T12=T)
    gate = ref["nn_d2"][:, 4] < 1.0
    assert np.array_equal(res["nn_idx"][gate], ref["nn_idx"][gate])
    # subset + different order = different concatenation order
    got2, _ = gpu.build_local_map([13, 10, 15], np.array(poses)[[3, 0, 5]], 0.5)
    want2, _ = oracle.build_local_map([clouds[3], clouds[0], clouds[5]], np.array(poses)[[3, 0, 5]], 0.5)
    assert_biteq(got2, want2)
    from lio_slam_b200.liogpu import LioGpuError
    with pytest.raises(LioGpuError):
        gpu.build_local_map([99], np.array(poses)[:1], 0.5)


def test_keyframe_slabs_are_reused_after_clear(oracle, world):
    """liogpu_keyframe_clear keeps the device slabs (no cudaFree / cudaMalloc between sequences): keyframes put after a
    clear land in the old slabs — several slabs' worth, other sizes, other ids — and the map built from them is the oracle's."""
    from lio_slam_b200.liogpu import LioGpu, LioGpuError
    g = LioGpu()
    try:
        rng = np.random.default_rng(5)
        big = (rng.standard_normal((1_200_000, 4)) * np.array([30, 30, 3, 1])).astype(np.float32)   # 19 MB each: 2 per slab at most
        for k in range(4):                       # generation 1: fills three 32 MiB slabs
            g.keyframe_put(k, big[: 1_200_000 - 1000 * k])
        assert g.keyframe_count() == 4
        g.keyframe_clear()
        assert g.keyframe_count() == 0
        with pytest.raises(LioGpuError):         # nothing of generation 1 is reachable any more
            g.build_local_map([0], np.zeros((1, 6), np.float32), 0.5)
        clouds, poses = [], []
        for k in range(5):                       # generation 2: small clouds first, then a large one crossing into the next slab
            p = synth.path_pose(-0.5 * k)
            sc = synth.make_scan(world, p, 16, seed=300 + k, cols=450)
            clouds.append(oracle.voxel_grid(synth.to_packed(sc), 0.4)[0]); poses.append(p.astype(np.float32))
        for k, c in enumerate(clouds):
            g.keyframe_put(100 + k, c)
        g.keyframe_put(200, big)                 # does not fit behind the small ones in slab 0 -> slab 1 (kept from generation 1)
        g.keyframe_put(100, clouds[0])           # overwrite in place
        want, _ = oracle.build_local_map(clouds, np.array(poses), 0.5, threads=4)
        got, st = g.build_local_map([100 + k for k in range(5)], np.array(poses), 0.5)
        assert st == 0
        assert_biteq(got, want, "map from keyframes stored in reused slabs")
        g.keyframe_clear()
        g.keyframe_put(7, clouds[2])             # generation 3 starts at the first slab again
        got3, _ = g.build_local_map([7], np.array(poses)[2:3], 0.5)
        want3, _ = oracle.build_local_map([clouds[2]], np.array(poses)[2:3], 0.5, threads=2)
        assert_biteq(got3, want3)
    finally:
        g.close()


# ---------------------------------------------------------------- a1 deskew
@pytest.mark.parametrize("cfg", [dict(), dict(downsample_rate=2, point_filter_num=3), dict(point_filter_num=5, lidar_max_range=40.0)])
def test_deskew_parity(oracle, world, cfg):
    from lio_slam_b200.liogpu import LioGpu
    from oracle.oracle import DeskewParams
    kw = dict(n_scan=32, downsample_rate=1, point_filter_num=1, lidar_min_front=2.0, lidar_min_back=10.0,
              lidar_min_left=2.0, lidar_min_right=2.0, lidar_max_range=100.0, lidar_max_intensity=90.0)
    kw.update(cfg)
    g = LioGpu(**kw)
    try:
        scan = synth.make_scan(world, synth.path_pose(1.0), 32, seed=77, cols=600)
        t0 = 1700000000.25
        imu_t, rx, ry, rz = synth.make_imu_table(t0, seed=8)
        dp = DeskewParams(kw["n_scan"], kw["downsample_rate"], kw["point_filter_num"], kw["lidar_min_front"],
                          kw["lidar_min_back"], kw["lidar_min_left"], kw["lidar_min_right"], kw["lidar_max_range"],
                          kw["lidar_max_intensity"])
        want = oracle.deskew(scan, dp, t0, imu_t, rx, ry, rz, True)
        got, st = g.deskew(scan, t0, imu_t, rx, ry, rz, True)
        assert want.shape[0] > 1000
        assert_biteq(got, want, "deskew")
        # deskewFlag == -1 / no IMU: crop + decimation only, points unchanged
        want0 = oracle.deskew(scan, dp, t0, imu_t, rx, ry, rz, False)
        got0, _ = g.deskew(scan, t0, imu_t, rx, ry, rz, False)
        assert_biteq(got0, want0, "passthrough")
    finally:
        g.close()


@pytest.mark.parametrize("beams", [64, 128])
def test_deskew_full_sweep_parity(oracle, world, beams):
    """a whole 1800-column sweep (115,200 / 230,400 points, 450 / 900 blocks of the flag and apply kernels)"""
    from lio_slam_b200.liogpu import LioGpu
    from oracle.oracle import DeskewParams
    kw = dict(n_scan=beams, downsample_rate=1, point_filter_num=1, lidar_min_front=2.0, lidar_min_back=10.0,
              lidar_min_left=2.0, lidar_min_right=2.0, lidar_max_range=100.0, lidar_max_intensity=90.0)
    g = LioGpu(**kw)
    try:
        scan = synth.make_scan(world, synth.path_pose(3.0), beams, seed=78, cols=1800)
        assert scan.shape[0] == beams * 1800
        t0 = 1700000000.75
        imu = synth.make_imu_table(t0, seed=9)
        want = oracle.deskew(scan, DeskewParams(*kw.values()), t0, *imu, True)
        got, st = g.deskew(scan, t0, *imu, True)
        assert st == 0 and want.shape[0] > scan.shape[0] // 2
        assert_biteq(got, want, f"deskew {beams}-beam sweep")
    finally:
        g.close()


# ---------------------------------------------------------------- committed golden case + tiled rebuild
def test_gpu_matches_committed_golden(gpu):
    import os
    G = np.load(os.path.join(os.path.dirname(__file__), "golden", "path_small.npz"))
    ds, st = gpu.voxel_downsample(G["scan4"], 0.4)
    assert_biteq(ds, G["ds"], "golden VoxelGrid")
    gpu.set_local_map(G["map4"])
    got = gpu.surf_optimization(ds, pose6=G["guess"])
    gate = G["nn_d2"][:, 4] < 1.0
    assert np.array_equal(got["nn_idx"][gate], G["nn_idx"][gate])
    assert_biteq(got["nn_d2"][gate], G["nn_d2"][gate])
    assert np.array_equal(got["flag"], G["flag"])
    assert_biteq(got["coeff"], G["coeff"])
    pose, P, info = gpu.scan2map(ds, G["guess"])
    assert info["iterations"] == int(G["iterations"]) and np.array_equal(info["nsel_hist"], G["nsel_hist"])
    assert np.abs(pose[:3] - G["pose"][:3]).max() <= ROT_TOL and np.abs(pose[3:] - G["pose"][3:]).max() <= POS_TOL
    assert np.abs(info["JtJ"] - G["JtJ"]).max() <= JTJ_RTOL * np.abs(G["JtJ"]).max()


@pytest.mark.parametrize("tiles", [2, 4, 8])
def test_tiled_voxel_rebuild_on_gpu(gpu, oracle, world, tiles):
    # BASELINE configs[3]: the full-map VoxelGrid sharded by spatial tile; tile outputs concatenated in tile
    # order must reproduce the single-shot output bit for bit (here all tiles run on the one GPU present)
    from lio_slam_b200 import sharding
    clouds = []
    for i in range(8):
        p = synth.path_pose(-0.8 * i)
        clouds.append(synth.transform_packed(synth.to_packed(synth.make_scan(world, p, 32, seed=500 + i, cols=600)), p))
    cloud = np.concatenate(clouds)
    want, _ = oracle.voxel_grid(cloud, 0.5)
    single, st = gpu.voxel_downsample(cloud, 0.5)
    assert_biteq(single, want)
    got, ov = sharding.voxel_downsample_sharded(cloud, 0.5, tiles, lambda pts, leaf: gpu.voxel_downsample(pts, leaf))
    assert not ov
    assert_biteq(got, want, f"{tiles} tiles")


@pytest.mark.parametrize("tiles", [1, 2, 3, 4, 8])
def test_device_planned_tiles_equal_build_local_map(gpu, oracle, world, tiles):
    # liogpu_voxel_tile: the tile plan (coarse histogram of the voxel-row index) is made on the device; the tiles'
    # outputs concatenated in tile order must equal extractCloud's single-GPU output and the oracle's, bit for bit
    clouds, poses = [], []
    for k in range(8):
        p = synth.path_pose(-0.8 * k)
        clouds.append(synth.to_packed(synth.make_scan(world, p, 32, seed=500 + k, cols=600)))
        poses.append(p.astype(np.float32))
    poses = np.array(poses)
    want, ov = oracle.build_local_map(clouds, poses, 0.5, threads=8)
    assert not ov
    gpu.keyframe_clear()
    for k, c in enumerate(clouds):
        gpu.keyframe_put(k, c)
    ids = np.arange(8)
    single, st = gpu.build_local_map(ids, poses, 0.5, fetch=True, cap=want.shape[0])
    assert_biteq(single, want, "single GPU")
    from lio_slam_b200 import sharding
    raw = np.concatenate([oracle.transform_cloud(c, p) for c, p in zip(clouds, poses)])
    host_tile, host_bounds = sharding.plan_voxel_tiles(raw, 0.5, tiles)   # numpy restatement of the device plan
    parts, npts = [], 0
    for t in range(tiles):
        out, info, st = gpu.voxel_tile(ids, poses, 0.5, t, tiles)
        assert st == 0 and info["n_points"] == sum(c.shape[0] for c in clouds)
        assert (info["bin_lo"], info["bin_hi"]) == (host_bounds[t], host_bounds[t + 1]), "device plan != host restatement"
        assert info["n_tile_points"] == int((host_tile == t).sum())
        npts += info["n_tile_points"]
        parts.append(out)
    assert npts == sum(c.shape[0] for c in clouds)                    # every point belongs to exactly one tile
    sizes = [p.shape[0] for p in parts]
    assert_biteq(np.concatenate(parts), want, f"{tiles} device-planned tiles")
    if tiles > 1:
        assert max(sizes) < 0.8 * want.shape[0]                       # the plan actually splits the work
    # the installed local map of the registration is untouched by the tile calls
    assert gpu.local_map_size() == want.shape[0]
    print(f"tiles={tiles} voxels per tile={sizes}")


def test_device_planned_tiles_overflow_guard(gpu, oracle, small_case):
    # leaf 0.01 over a 100 m sweep: the guard of the WHOLE cloud fires (q4) -> the concatenated tiles are the input
    gpu.keyframe_clear()
    gpu.keyframe_put(0, small_case["scan4"])
    pose = np.zeros((1, 6), np.float32)
    want, ov = oracle.build_local_map([small_case["scan4"]], pose, 0.01, threads=2)
    assert ov
    parts = []
    for t in range(3):
        out, info, st = gpu.voxel_tile([0], pose, 0.01, t, 3)
        assert st == 1 and info["leaf_overflow"] == 1
        parts.append(out)
    assert_biteq(np.concatenate(parts), want, "overflow guard")


def test_scan2map_full_size_properties(gpu):
    # BASELINE-size property checks that need no oracle run: a 64-beam sweep registered against a map built
    # from the same world converges toward ground truth from different perturbations, and re-running is
    # bit-reproducible (fixed summation order)
    world = synth.make_world(1234)
    pose_gt = synth.path_pose(0.2)
    scan4 = synth.to_packed(synth.make_scan(world, pose_gt, 64, seed=31))
    map4 = synth.make_local_map(world, 64, 120000, 0.3, seed=9, s0=-0.3, max_poses=16)
    gpu.set_local_map(map4)
    ds, _ = gpu.voxel_downsample(scan4, 0.4)
    poses = []
    for s in (1, 2, 3):
        pose, P, info = gpu.scan2map(ds, synth.perturbed_guess(pose_gt, s))
        assert info["converged"] and info["n_sel"] > 0.5 * ds.shape[0]
        poses.append(pose)
    poses = np.array(poses)
    assert np.abs(poses[:, 3:] - pose_gt[3:]).max() < 0.05 and np.abs(poses[:, :3] - pose_gt[:3]).max() < 0.01
    assert np.abs(poses - poses[0]).max() < 5e-3
    a = gpu.scan2map(ds, synth.perturbed_guess(pose_gt, 1))
    b = gpu.scan2map(ds, synth.perturbed_guess(pose_gt, 1))
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[2]["JtJ"], b[2]["JtJ"])


def test_gpu_matches_committed_golden_rows_f(gpu):
    """the widened rows against the committed fixture (tests/golden/rows_f_small.npz) — no oracle involved at run time"""
    import os
    G = np.load(os.path.join(os.path.dirname(__file__), "golden", "rows_f_small.npz"))
    offs = G["offsets"]
    clouds = [np.ascontiguousarray(G["clouds"][offs[k]:offs[k + 1]]) for k in range(len(offs) - 1)]
    gpu.keyframe_clear()
    for k, c in enumerate(clouds):
        gpu.keyframe_put(k, c)
    ids = list(range(len(clouds)))
    lm, info, st = gpu.publish_local_map(ids, G["poses"], G["pose_now"], local_mapping_surf_leaf_size=0.3)
    assert_biteq(lm, G["local_map"], "golden publishLocalMap")
    assert [info["n_concat"], info["n_cropped"], info["n_after_sor"], info["n_out"]] == G["local_map_counts"].tolist()
    merged, _ = gpu.merge_keyframes(ids, G["poses"], 0.4)
    assert_biteq(merged, G["merged"], "golden merged keyframes")
    T, ii = gpu.icp_align(G["icp_source"], merged)
    assert [ii["iterations"], ii["converged"], ii["convergence_state"], ii["n_correspondences"]] == G["icp_ints"].tolist()
    assert np.abs(T - G["icp_T"]).max() <= 1e-5 and ii["fitness_score"] == pytest.approx(float(G["icp_fitness"]), rel=1e-6)
    sc, rk, sk = gpu.make_scancontext(clouds[0])
    assert np.array_equal(sc, G["sc_desc"]) and np.array_equal(rk, G["sc_ringkey"]) and np.array_equal(sk, G["sc_sectorkey"])
    got, _ = gpu.extract_nearby(G["key3d"], G["key_time"], float(G["key_time"][-1]) + 0.1, 30.0, 2.0)
    assert np.array_equal(got, G["nearby_ids"])


def test_replay_driver_tracks_ground_truth(world, tmp_path):
    # the C++ host mirror (lio_slam_b200/host) driving the C ABI over a short sequence: keyframes are
    # added by the reference's saveFrame rule, the local map is rebuilt from device-resident keyframes,
    # and every registered pose stays near ground truth
    import json
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "lio_slam_b200", "replay_driver")
    if not os.path.exists(exe):
        pytest.skip("replay_driver not built")
    seq = str(tmp_path / "seq.bin")
    out = str(tmp_path / "poses.txt")
    gts = synth.write_sequence(seq, world, 16, 14, seed=3)
    r = subprocess.run([exe, seq, out, "0", "0.4", "0.5"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    summary = json.loads(r.stdout.strip().splitlines()[-1])
    rows = np.loadtxt(out)
    assert rows.shape[0] == 14 and summary["keyframes"] >= 3 and summary["registered"] == 13
    poses = rows[:, 1:7]
    assert np.abs(poses[:, 3:] - gts[:, 3:]).max() < 0.08 and np.abs(poses[:, :3] - gts[:, :3]).max() < 0.01
    assert (rows[1:, 7] >= 1).all() and (rows[1:, 8] > 500).all()
    print(summary)
    # the same replay with publishLocalMap after every scan (mapOptmization.cpp:504): poses unchanged, a cloud published
    out2 = str(tmp_path / "poses2.txt")
    r = subprocess.run([exe, seq, out2, "0", "0.4", "0.5", "1"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    s2 = json.loads(r.stdout.strip().splitlines()[-1])
    assert np.array_equal(np.loadtxt(out2), rows) and s2["local_map_points"] > 1000 and s2["local_map_gpu_ms_per_scan"] > 0
    # and with the key poses selected on the device (liogpu_extract_nearby): the same keyframes, the same poses
    out3 = str(tmp_path / "poses3.txt")
    r = subprocess.run([exe, seq, out3, "0", "0.4", "0.5", "0", "1"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    assert np.array_equal(np.loadtxt(out3), rows)


def test_device_resident_pipeline_config2(oracle, world):
    # BASELINE configs[1]: 32-beam sweep with 200 Hz IMU deskew + scan-to-map, the sweep crossing PCIe once:
    # deskew (kept in HBM) -> VoxelGrid + registration on the resident cloud -> keyframe from the resident
    # downsampled sweep.  Every stage must equal the oracle pipeline run stage by stage on the host.
    from lio_slam_b200.liogpu import LioGpu, RESIDENT
    from oracle.oracle import DeskewParams
    kw = dict(n_scan=32, downsample_rate=1, point_filter_num=1, lidar_min_front=2.0, lidar_min_back=10.0,
              lidar_min_left=2.0, lidar_min_right=2.0, lidar_max_range=100.0, lidar_max_intensity=100.0,
              mapping_surf_leaf_size=0.4, surrounding_keyframe_map_leaf_size=0.5)
    g = LioGpu(**kw)
    try:
        pose_gt = synth.path_pose(0.5)
        scan = synth.make_scan(world, pose_gt, 32, seed=91, cols=900)
        t0 = 1700000100.0
        imu_t, rx, ry, rz = synth.make_imu_table(t0, seed=12)
        map4 = synth.make_local_map(world, 32, 30000, 0.5, seed=6, s0=0.0, cols=900, max_poses=32)
        guess = synth.perturbed_guess(pose_gt, 33)
        dp = DeskewParams(32, 1, 1, 2.0, 10.0, 2.0, 2.0, 100.0, 100.0)
        dsk = oracle.deskew(scan, dp, t0, imu_t, rx, ry, rz, True)
        ds, _ = oracle.voxel_grid(dsk, 0.4)
        ref_pose, ref_P, ref_info = oracle.scan2map(map4, ds, guess, threads=8)
        g.set_local_map(map4)
        n_dsk, st = g.deskew(scan, t0, imu_t, rx, ry, rz, True, keep_on_device=True)
        assert n_dsk == dsk.shape[0] == g.resident_size()
        pose, P, info = g.downsample_scan2map(RESIDENT, guess, keep_ds_on_device=True)
        assert info["n_ds"] == ds.shape[0] == g.resident_size()
        check_s2m(pose, info, ref_pose, ref_info)
        # the resident downsampled sweep becomes a keyframe without leaving the GPU; rebuilding the local
        # map from it must equal the oracle's extractCloud on the same cloud and pose
        g.keyframe_clear()
        g.keyframe_put(0, RESIDENT)
        got, _ = g.build_local_map([0], pose.reshape(1, 6), 0.5)
        want, _ = oracle.build_local_map([ds], pose.reshape(1, 6), 0.5)
        assert_biteq(got, want, "keyframe from resident cloud")
        # and the resident cloud can be voxelised / inspected again
        again, _ = g.voxel_downsample(RESIDENT, 0.8)
        want2, _ = oracle.voxel_grid(ds, 0.8)
        assert_biteq(again, want2)
    finally:
        g.close()
