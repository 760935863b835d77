"""GPU edge cases and randomized property checks (through the C ABI, against the oracle): tiny and empty maps,
duplicate points and exact ties, coincident query/map points, huge sparse extents (grid cell doubling), voxel
boundary values, deskew corner cases, repeated use of one context."""
import numpy as np
import pytest

from lio_slam_b200 import synth

pytestmark = pytest.mark.gpu
I12 = np.array([1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0], np.float32)


def biteq(a, b):
    a = np.ascontiguousarray(a, np.float32); b = np.ascontiguousarray(b, np.float32)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def compare_surf(gpu, oracle, map4, q4, T=I12, threads=8):
    ref = oracle.surf_optimization(map4, q4, T12=T, threads=threads)
    gpu.set_local_map(map4)
    got = gpu.surf_optimization(q4, T12=T)
    gate = ref["nn_d2"][:, 4] < 1.0
    assert np.array_equal(got["nn_idx"][gate], ref["nn_idx"][gate])
    assert biteq(got["nn_d2"][gate], ref["nn_d2"][gate])
    assert np.array_equal(got["tie"][gate], ref["tie"][gate])
    assert (got["nn_d2"][~gate, 4] >= 1.0).all()
    assert np.array_equal(got["flag"], ref["flag"])
    assert biteq(got["coeff"], ref["coeff"])
    return ref, gate


@pytest.mark.parametrize("nm", [0, 1, 4, 5, 6, 17])
def test_tiny_maps(gpu, oracle, nm):
    rng = np.random.default_rng(nm)
    map4 = (rng.normal(0, 0.2, (nm, 4)) + [3, 1, 0, 0]).astype(np.float32)
    q = (rng.normal(0, 0.3, (200, 4)) + [3, 1, 0, 0]).astype(np.float32)
    if nm < 5:   # fewer than 5 map points: no correspondences at all (SURVEY A.2)
        gpu.set_local_map(map4)
        got = gpu.surf_optimization(q, T12=I12)
        assert not got["flag"].any() and (got["nn_idx"] == -1).all()
    else:
        compare_surf(gpu, oracle, map4, q)


def test_duplicates_and_coincident_points(gpu, oracle):
    rng = np.random.default_rng(11)
    base = rng.uniform(-4, 4, (3000, 4)).astype(np.float32)
    base[:, 2] *= 0.05
    map4 = np.concatenate([base, base[:1500], base[:700]])          # exact duplicates -> equidistant ties
    map4 = map4[rng.permutation(map4.shape[0])]
    q = np.concatenate([base[:2000], rng.uniform(-4, 4, (2000, 4)).astype(np.float32)])   # queries ON map points (d = 0)
    q[2000:, 2] *= 0.05
    ref, gate = compare_surf(gpu, oracle, map4, q)
    assert ref["tie"].sum() > 500 and (ref["nn_d2"][:2000, 0] == 0).all()


def test_huge_sparse_extent_forces_cell_doubling(gpu, oracle):
    # clusters spread over 6 km x 6 km x 400 m: a 0.4 m grid would need 5e10 cells, so the cell edge doubles
    # until the table fits; results must not change
    rng = np.random.default_rng(5)
    centres = np.column_stack([rng.uniform(-3000, 3000, 40), rng.uniform(-3000, 3000, 40), rng.uniform(-200, 200, 40)])
    pts = []
    for c in centres:
        p = rng.normal(0, 1.0, (400, 3)); p[:, 2] *= 0.02
        pts.append(p + c)
    map4 = np.column_stack([np.concatenate(pts), np.zeros(16000)]).astype(np.float32)
    q = map4[rng.choice(16000, 3000, replace=False)].copy()
    q[:, :3] += rng.normal(0, 0.05, (3000, 3)).astype(np.float32)
    ref, gate = compare_surf(gpu, oracle, map4, q)
    assert gate.sum() > 2000


@pytest.mark.parametrize("seed", range(6))
def test_random_planar_scenes(gpu, oracle, seed):
    rng = np.random.default_rng(100 + seed)
    n_planes = rng.integers(1, 6)
    pts = []
    for _ in range(n_planes):
        R = synth.rpy_to_R(*rng.uniform(-1.5, 1.5, 3))
        p = np.column_stack([rng.uniform(-6, 6, 4000), rng.uniform(-6, 6, 4000), rng.normal(0, 0.01, 4000)])
        pts.append(p @ R.T + rng.uniform(-3, 3, 3))
    allp = np.concatenate(pts)
    leaf = float(rng.choice([0.15, 0.2, 0.3, 0.5]))
    map4, _ = oracle.voxel_grid(np.column_stack([allp, np.zeros(allp.shape[0])]).astype(np.float32), leaf)
    got, _ = gpu.voxel_downsample(np.column_stack([allp, np.zeros(allp.shape[0])]).astype(np.float32), leaf)
    assert biteq(got, map4)
    q = allp[rng.choice(allp.shape[0], 3000, replace=False)] + rng.normal(0, 0.03, (3000, 3))
    q4 = np.column_stack([q, np.ones(3000)]).astype(np.float32)
    pose = np.concatenate([rng.uniform(-0.02, 0.02, 3), rng.uniform(-0.05, 0.05, 3)]).astype(np.float32)
    T = oracle.pose_to_T(pose)
    compare_surf(gpu, oracle, map4, q4, T)
    # and the full loop from that pose
    ref_pose, ref_P, ref_info = oracle.scan2map(map4, q4, pose, threads=8)
    pose_g, P_g, info = gpu.scan2map(q4, pose)
    assert info["iterations"] == ref_info["iterations"] and np.array_equal(info["nsel_hist"], ref_info["nsel_hist"])
    assert np.abs(pose_g[:3] - ref_pose[:3]).max() <= 1e-5 and np.abs(pose_g[3:] - ref_pose[3:]).max() <= 1e-4
    assert info["is_degenerate"] == ref_info["is_degenerate"]
    assert np.abs(P_g - ref_P).max() <= 1e-5


def test_voxel_boundary_values(gpu, oracle):
    # coordinates exactly on voxel faces, negative zero, negative coordinates, leaf not representable in binary
    g = np.arange(-8, 8.01, 0.5, dtype=np.float32)
    X, Y, Z = np.meshgrid(g, g, np.array([-0.5, -0.0, 0.0, 0.3], np.float32), indexing="ij")
    cloud = np.column_stack([X.ravel(), Y.ravel(), Z.ravel(), np.arange(X.size) % 97]).astype(np.float32)
    cloud = np.concatenate([cloud, cloud[::3] + np.float32(1e-7)])
    for leaf in (0.5, 0.3, 0.25, 1.0, 0.1):
        want, ov = oracle.voxel_grid(cloud, leaf)
        got, st = gpu.voxel_downsample(cloud, leaf)
        assert biteq(got, want), leaf


def test_voxel_heavy_voxels(gpu, oracle):
    # a few voxels with tens of thousands of members (the warp-per-voxel path) next to many singletons
    rng = np.random.default_rng(8)
    heavy = np.concatenate([rng.normal(c, 0.03, (40000, 3)) for c in ([0.25, 0.25, 0.25], [5.25, -3.25, 1.25], [-7.75, 2.25, 0.25])])
    light = rng.uniform(-20, 20, (60000, 3))
    xyz = np.concatenate([heavy, light])[rng.permutation(180000)]
    cloud = np.column_stack([xyz, rng.uniform(0, 255, 180000)]).astype(np.float32)
    want, _ = oracle.voxel_grid(cloud, 0.5)
    got, _ = gpu.voxel_downsample(cloud, 0.5)
    assert biteq(got, want)


def test_deskew_corner_cases(oracle, world):
    from lio_slam_b200.liogpu import LioGpu
    from oracle.oracle import DeskewParams
    scan = synth.make_scan(world, synth.path_pose(2.0), 16, seed=5, cols=200)
    t0 = 50.0
    imu_t, rx, ry, rz = synth.make_imu_table(t0, seed=2)
    base = dict(n_scan=16, downsample_rate=1, point_filter_num=1, lidar_min_front=1.0, lidar_min_back=5.0, lidar_min_left=2.0,
                lidar_min_right=2.0, lidar_max_range=1000.0, lidar_max_intensity=100.0)

    def run(kw, imu, enabled=True, sc=scan, t_scan=t0):
        g = LioGpu(**kw)
        try:
            dp = DeskewParams(kw["n_scan"], kw["downsample_rate"], kw["point_filter_num"], kw["lidar_min_front"], kw["lidar_min_back"],
                              kw["lidar_min_left"], kw["lidar_min_right"], kw["lidar_max_range"], kw["lidar_max_intensity"])
            want = oracle.deskew(sc, dp, t_scan, *imu, enabled)
            got, st = g.deskew(sc, t_scan, *imu, enabled)
            assert biteq(got, want)
            return want.shape[0]
        finally:
            g.close()
    assert run(base, (imu_t, rx, ry, rz)) > 0
    # a single IMU row: imuAvailable is false in the reference (IP:413) -> points pass through unchanged
    assert run(base, (imu_t[:1], rx[:1], ry[:1], rz[:1])) > 0
    # every point filtered out (range gate) -> empty cloud
    assert run(dict(base, lidar_max_range=0.1), (imu_t, rx, ry, rz)) == 0
    # ring bound: only rings < 4 survive; decimation by raw index
    assert run(dict(base, n_scan=4, point_filter_num=7), (imu_t, rx, ry, rz)) > 0
    # sweep starting after the last IMU sample / before the first one (findRotation's two clamps, IP:514)
    assert run(base, (imu_t, rx, ry, rz), t_scan=t0 + 10.0) > 0
    assert run(base, (imu_t, rx, ry, rz), t_scan=t0 - 10.0) > 0
    # empty input
    assert run(base, (imu_t, rx, ry, rz), sc=scan[:0]) == 0


DESKEW_BASE = dict(n_scan=32, downsample_rate=1, point_filter_num=1, lidar_min_front=2.0, lidar_min_back=10.0,
                   lidar_min_left=2.0, lidar_min_right=2.0, lidar_max_range=100.0, lidar_max_intensity=90.0)


def deskew_vs_oracle(oracle, scan, t_scan, imu, enabled=True, **over):
    """liogpu_deskew on a fresh context and oracle.deskew with the same parameters -> (gpu, oracle); bit-equal"""
    from lio_slam_b200.liogpu import LioGpu
    from oracle.oracle import DeskewParams
    kw = dict(DESKEW_BASE, **over)
    g = LioGpu(**kw)
    try:
        want = oracle.deskew(scan, DeskewParams(*kw.values()), t_scan, *imu, enabled)
        got, st = g.deskew(scan, t_scan, *imu, enabled)
    finally:
        g.close()
    assert st == 0 and biteq(got, want)
    return got, want


def test_deskew_first_survivor_in_a_later_block(oracle, world):
    """the first surviving point fixes transStartInverse for the whole sweep; the flag kernel finds it with atomicMin.
    Here points 0..4999 fail the range gate or the crop box, so it sits in block 19 (5,001 with point_filter_num 3)"""
    scan = synth.make_scan(world, synth.path_pose(2.5), 32, seed=41, cols=900).copy()
    for f in ("x", "y", "z"):
        scan[f][:2500] *= np.float32(1000.0)    # beyond lidarMaxRange
        scan[f][2500:5000] *= np.float32(1e-3)  # inside the vehicle's crop box
    t0 = 300.0
    imu = synth.make_imu_table(t0, seed=4)
    got, want = deskew_vs_oracle(oracle, scan, t0, imu, point_filter_num=3)
    p = synth.to_packed(scan)
    rng_ok = np.sqrt((p[:, :3].astype(np.float64) ** 2).sum(axis=1)) <= 100.0
    x, y = p[:, 0], p[:, 1]
    crop = (y < 2.0) & (-10.0 < y) & (x < 2.0) & (-2.0 < x)
    survives = rng_ok & ~crop & (p[:, 3] <= 90.0) & (np.arange(p.shape[0]) % 3 == 0)
    first = int(np.argmax(survives))
    assert first >= 19 * 256 and want.shape[0] > 1000
    # the first survivor is deskewed by its own rotation and transStartInverse: the identity up to rounding
    assert np.abs(want[0, :3] - p[first, :3]).max() <= 1e-5 * np.abs(p[first, :3]).max()


def test_deskew_permuted_sweep(oracle, world):
    """point order that is not column-major: the first survivor and every point's IMU row come from arbitrary places"""
    scan = synth.make_scan(world, synth.path_pose(4.0), 32, seed=42, cols=900)
    scan = scan[np.random.default_rng(6).permutation(scan.shape[0])]
    t0 = 301.0
    got, want = deskew_vs_oracle(oracle, scan, t0, synth.make_imu_table(t0, seed=5), point_filter_num=2)
    assert want.shape[0] > 5000


def test_deskew_imu_table_at_its_limit(oracle, world):
    """2,000 IMU rows (imuQueLength), the sweep over the last ten, so findRotation scans about 1,990 rows per point;
    2,001 rows are refused"""
    from lio_slam_b200.liogpu import E_INVALID, LioGpu, LioGpuError
    rng = np.random.default_rng(12)
    dt, t0 = 0.01, 500.0
    t = t0 - 1990 * dt + dt * np.arange(2000)                 # the last row at t0 + 0.09, inside the 0.1 s sweep
    rates = np.c_[0.2 * np.sin(2 * np.pi * 0.3 * t), 0.2 * np.cos(2 * np.pi * 0.2 * t), 0.6 + rng.normal(0, 1e-3, 2000)]
    rot = np.vstack([np.zeros(3), np.cumsum(rates[1:] * dt, axis=0)])
    imu = (t, rot[:, 0].copy(), rot[:, 1].copy(), rot[:, 2].copy())
    scan = synth.make_scan(world, synth.path_pose(5.0), 32, seed=43, cols=900)
    got, want = deskew_vs_oracle(oracle, scan, t0, imu)
    assert want.shape[0] > 5000
    longer = tuple(np.r_[a[:1] - (dt if k == 0 else 0.0), a] for k, a in enumerate(imu))
    assert longer[0].shape[0] == 2001
    g = LioGpu(**DESKEW_BASE)
    try:
        with pytest.raises(LioGpuError) as e:
            g.deskew(scan, t0, *longer, True)
        assert e.value.status == E_INVALID
    finally:
        g.close()


def test_deskew_enabled_without_imu_rows(oracle, world):
    """n_imu == 0 with deskew on: imuAvailable is false, so the points pass through the crop and decimation unchanged"""
    scan = synth.make_scan(world, synth.path_pose(6.0), 32, seed=44, cols=600)
    empty = tuple(np.zeros(0, np.float64) for _ in range(4))
    got, want = deskew_vs_oracle(oracle, scan, 700.0, empty, point_filter_num=2)
    off, _ = deskew_vs_oracle(oracle, scan, 700.0, synth.make_imu_table(700.0, seed=1), enabled=False, point_filter_num=2)
    assert want.shape[0] > 1000 and biteq(got, off)


def test_context_reuse_and_errors(gpu, oracle, small_case):
    from lio_slam_b200 import liogpu as L
    # shrinking and growing inputs on one context (buffers are reused)
    for n in (5000, 100, 20000, 31, 12000):
        want, _ = oracle.voxel_grid(small_case["scan4"][:n], 0.4)
        got, _ = gpu.voxel_downsample(small_case["scan4"][:n], 0.4)
        assert biteq(got, want)
    with pytest.raises(L.LioGpuError):          # leaf must be positive
        gpu.voxel_downsample(small_case["scan4"], 0.0)
    with pytest.raises(L.LioGpuError):          # max_iter out of range
        gpu.set_local_map(small_case["map4"]); gpu.scan2map(small_case["scan4"], small_case["guess"], max_iter=31)
    with pytest.raises(L.LioGpuError):          # no resident cloud yet on a fresh context
        g2 = L.LioGpu()
        try:
            g2.set_local_map(small_case["map4"]); g2.scan2map(L.RESIDENT, small_case["guess"])
        finally:
            g2.close()
    g3 = L.LioGpu()
    try:
        with pytest.raises(L.LioGpuError) as e:  # registration before any map
            g3.scan2map(small_case["scan4"], small_case["guess"])
        assert e.value.status == L.E_NO_MAP
    finally:
        g3.close()


def test_sparse_map_single_phase_and_seeds(oracle, world):
    # leaf-0.5 map (no phase-1 gate: every point goes through the warp-cooperative kernel on iteration 0, the
    # seeded main kernel from iteration 1) with a large initial error so that several iterations run
    from lio_slam_b200.liogpu import LioGpu
    g = LioGpu(surrounding_keyframe_map_leaf_size=0.5)
    try:
        pose_gt = synth.path_pose(0.1)
        scan4 = synth.to_packed(synth.make_scan(world, pose_gt, 16, seed=17, cols=900))
        map4 = synth.make_local_map(world, 16, 20000, 0.5, seed=4, s0=-0.4, cols=900, max_poses=32)
        ds, _ = oracle.voxel_grid(scan4, 0.4)
        guess = synth.perturbed_guess(pose_gt, 3, rot_deg=(1.0, 1.0, 2.5), trans=(0.3, 0.3, 0.1))
        ref_pose, ref_P, ref_info = oracle.scan2map(map4, ds, guess, threads=8)
        g.set_local_map(map4)
        pose, P, info = g.scan2map(ds, guess)
        assert ref_info["iterations"] >= 4
        assert info["iterations"] == ref_info["iterations"] and np.array_equal(info["nsel_hist"], ref_info["nsel_hist"])
        assert np.abs(pose[:3] - ref_pose[:3]).max() <= 1e-5 and np.abs(pose[3:] - ref_pose[3:]).max() <= 1e-4
        assert np.abs(info["pose_hist"] - ref_info["pose_hist"]).max() <= 1e-4
        assert info["seeded"] > 0.5 * ds.shape[0]
    finally:
        g.close()


def test_pinned_host_sweep_identical(oracle, world):
    # a sweep in PINNED host memory (liogpu_host_alloc), as 32-byte records and as packed float4, must give
    # the same bits as the pageable path
    import ctypes as C
    from lio_slam_b200.liogpu import LioGpu, load_library
    lib = load_library()
    g = LioGpu(surrounding_keyframe_map_leaf_size=0.2)
    try:
        pose_gt = synth.path_pose(0.1)
        scan = synth.xyzirt_to_xyzi(synth.make_scan(world, pose_gt, 64, seed=41))          # 115,200 records of 32 B
        n = scan.shape[0]
        assert n >= 65536
        map4 = synth.make_local_map(world, 64, 150000, 0.2, seed=2, s0=-0.4, max_poses=8)
        guess = synth.perturbed_guess(pose_gt, 9)
        g.set_local_map(map4)
        pose_a, P_a, info_a = g.scan2map(scan, guess)                                        # pageable numpy buffer
        ptr = lib.liogpu_host_alloc(C.c_ulonglong(n * 32))
        assert ptr
        try:
            C.memmove(ptr, scan.ctypes.data, n * 32)
            pose_b, P_b, info_b = g.scan2map((ptr, n, 32), guess)                             # pinned 32-byte records
            packed = synth.to_packed(scan)
            C.memmove(ptr, packed.ctypes.data, n * 16)
            pose_c, P_c, info_c = g.scan2map((ptr, n, 16), guess)                             # pinned, packed float4
        finally:
            lib.liogpu_host_free(C.c_void_p(ptr))
        for pose_x, info_x in ((pose_b, info_b), (pose_c, info_c)):
            assert np.array_equal(pose_a, pose_x) and info_a["iterations"] == info_x["iterations"]
            assert np.array_equal(info_a["JtJ"], info_x["JtJ"]) and np.array_equal(info_a["nsel_hist"], info_x["nsel_hist"])
        ref_pose, _, ref_info = oracle.scan2map(map4, synth.to_packed(scan), guess, threads=8)
        assert ref_info["iterations"] == info_a["iterations"]
        assert np.abs(pose_a[:3] - ref_pose[:3]).max() <= 1e-5 and np.abs(pose_a[3:] - ref_pose[3:]).max() <= 1e-4
    finally:
        g.close()


def test_full_size_config3_parity(oracle):
    # BASELINE configs[2] at full size: 128-beam sweep (230,400 points) vs a 500,000-point map, against the
    # oracle with its exact KD-tree (brute force would take minutes).  Per-point results on one
    # surfOptimization pass, then the whole loop.
    import bench
    from lio_slam_b200.liogpu import LioGpu
    map4, scans, guesses = bench.make_workload("cfg3", 0, 1)
    assert scans[0].shape[0] == 230400 and map4.shape[0] == 500000
    g = LioGpu(n_scan=128, surrounding_keyframe_map_leaf_size=0.2)
    try:
        h = oracle.index_build(map4)
        ref = oracle.surf_optimization(map4, scans[0], pose6=guesses[0], handle=h, threads=16)
        g.set_local_map(map4)
        got = g.surf_optimization(scans[0], pose6=guesses[0])
        gate = ref["nn_d2"][:, 4] < 1.0
        assert gate.mean() > 0.99
        assert np.array_equal(got["nn_idx"][gate], ref["nn_idx"][gate])
        assert biteq(got["nn_d2"][gate], ref["nn_d2"][gate])
        assert np.array_equal(got["flag"], ref["flag"]) and biteq(got["coeff"], ref["coeff"])
        assert np.array_equal(got["tie"][gate], ref["tie"][gate])
        ref_pose, ref_P, ref_info = oracle.scan2map(map4, scans[0], guesses[0], threads=16, handle=h)
        oracle.index_free(h)
        pose, P, info = g.scan2map(scans[0], guesses[0])
        assert info["iterations"] == ref_info["iterations"] and np.array_equal(info["nsel_hist"], ref_info["nsel_hist"])
        assert np.abs(pose[:3] - ref_pose[:3]).max() <= 1e-5 and np.abs(pose[3:] - ref_pose[3:]).max() <= 1e-4
        assert np.abs(info["JtJ"] - ref_info["JtJ"]).max() <= 1e-5 * np.abs(ref_info["JtJ"]).max()
        assert info["tie_queries"] == ref_info["tie_queries"] and info["is_degenerate"] == ref_info["is_degenerate"]
        print("cfg3 full size: iterations", info["iterations"], "n_sel", info["n_sel"], "pose bit-equal",
              np.array_equal(pose, ref_pose), "JtJ max rel", float(np.abs(info["JtJ"] - ref_info["JtJ"]).max() / np.abs(ref_info["JtJ"]).max()))
    finally:
        g.close()


def test_full_size_config4_voxel_5M(gpu, oracle):
    # BASELINE configs[3] size: 5,000,000 points (walls + ground layout, heavy overlap), leaf 0.5 and 0.2
    rng = np.random.default_rng(44)
    n = 5_000_000
    xy = rng.uniform(-60, 60, (n, 2))
    z = np.where(rng.uniform(size=n) < 0.6, rng.normal(0, 0.02, n), rng.uniform(0, 12, n))
    near = rng.uniform(size=n) < 0.3                       # a dense blob near the sensor: voxels with 1e4+ members
    xy[near] = rng.normal(0, 3.0, (int(near.sum()), 2))
    cloud = np.column_stack([xy, z, rng.uniform(0, 100, n)]).astype(np.float32)
    for leaf in (0.5, 0.2):
        want, ov = oracle.voxel_grid(cloud, leaf)
        got, st = gpu.voxel_downsample(cloud, leaf)
        assert not ov and biteq(got, want), leaf
    print("5M voxel: device ms", gpu.last_gpu_ms(), "voxels", want.shape[0])


def test_large_scale_1p2M_queries_1p4M_map(oracle):
    # 1.2 M points = 4,688 main-kernel blocks: the leftover kernel derives the segment offsets in shared memory
    large_scale_registration(oracle, 1_200_000)


def test_large_scale_2p4M_queries_1p4M_map(oracle):
    # above 2,096,896 points (more than LEFT_OFF_CAP - 1 = 8191 main-kernel blocks of 256) the leftover kernel's
    # segment-offset table no longer fits its shared memory: the main kernel's last block scans the offsets into global
    # memory and the leftover kernel reads them there
    large_scale_registration(oracle, 2_400_000)


def large_scale_registration(oracle, n_q):
    # beyond BASELINE sizes: n_q sweep points against a 1.4 M-point map; spot-checked against the oracle
    from lio_slam_b200.liogpu import LioGpu
    rng = np.random.default_rng(77)

    def surfaces(n, noise):
        k = n // 3
        g = np.column_stack([rng.uniform(-80, 80, k), rng.uniform(-80, 80, k), rng.normal(0, noise, k)])
        w1 = np.column_stack([rng.uniform(-80, 80, k), np.full(k, 35.0) + rng.normal(0, noise, k), rng.uniform(0, 15, k)])
        w2 = np.column_stack([np.full(n - 2 * k, -40.0) + rng.normal(0, noise, n - 2 * k), rng.uniform(-80, 80, n - 2 * k), rng.uniform(0, 15, n - 2 * k)])
        return np.concatenate([g, w1, w2])
    raw = np.column_stack([surfaces(12_000_000, 0.01), np.zeros(12_000_000)]).astype(np.float32)
    g = LioGpu(surrounding_keyframe_map_leaf_size=0.2)
    try:
        map4, _ = g.voxel_downsample(raw, 0.2)
        assert map4.shape[0] > 1_000_000
        q = np.column_stack([surfaces(n_q, 0.02), np.ones(n_q)]).astype(np.float32)
        q = q[rng.permutation(q.shape[0])]
        pose = np.array([0.002, -0.003, 0.004, 0.05, -0.04, 0.02], np.float32)
        g.set_local_map(map4)
        got = g.surf_optimization(q, pose6=pose)
        sub = rng.choice(q.shape[0], 20000, replace=False)
        h = oracle.index_build(map4)
        ref = oracle.surf_optimization(map4, q[sub], pose6=pose, handle=h, threads=16)
        gate = ref["nn_d2"][:, 4] < 1.0
        assert gate.mean() > 0.9
        assert np.array_equal(got["nn_idx"][sub][gate], ref["nn_idx"][gate])
        assert biteq(got["nn_d2"][sub][gate], ref["nn_d2"][gate])
        assert np.array_equal(got["flag"][sub], ref["flag"]) and biteq(got["coeff"][sub], ref["coeff"])
        ref_pose, _, ref_info = oracle.scan2map(map4, q, pose, threads=16, handle=h)
        oracle.index_free(h)
        pose_g, _, info = g.scan2map(q, pose)
        assert info["iterations"] == ref_info["iterations"] and np.array_equal(info["nsel_hist"], ref_info["nsel_hist"])
        assert np.abs(pose_g[:3] - ref_pose[:3]).max() <= 1e-5 and np.abs(pose_g[3:] - ref_pose[3:]).max() <= 1e-4
        print(n_q, "x", map4.shape[0], "iterations", info["iterations"], "gpu loop ms", info["gpu_ms"], "bit-equal pose", np.array_equal(pose_g, ref_pose),
              "leftovers per iteration", info["leftover_hist"].tolist())
    finally:
        g.close()


def test_resident_cloud_is_invalidated_when_clobbered(oracle, small_case):
    # a call that reuses the buffer holding the resident cloud must invalidate it (never serve stale data)
    from lio_slam_b200 import liogpu as L
    g = L.LioGpu(mapping_surf_leaf_size=0.4)
    try:
        g.set_local_map(small_case["map4"])
        n_ds, _ = g.voxel_downsample(small_case["scan4"], 0.4, keep_on_device=True)
        assert g.resident_size() == n_ds > 0
        want, _ = oracle.voxel_grid(small_case["scan4"], 0.4)
        got = g.surf_optimization(L.RESIDENT, pose6=small_case["guess"])            # consuming it keeps it
        assert got["flag"].shape[0] == want.shape[0] and g.resident_size() == n_ds
        g.voxel_downsample(small_case["scan4"][:1000], 0.4)                           # reuses the same scratch
        assert g.resident_size() == 0
        with pytest.raises(L.LioGpuError):
            g.scan2map(L.RESIDENT, small_case["guess"])
    finally:
        g.close()


@pytest.mark.parametrize("n", [1, 2, 3, 31, 32, 33, 100, 1023, 1024, 1025, 2047, 2048, 2049, 4100])
def test_voxel_small_cloud_path_matches_pipeline(gpu, oracle, n):
    """clouds of <= 2048 points (the key-pose filter, mapOptmization.cpp:1535-1536) take a single-block kernel;
    sizes straddling the switch must all equal the oracle, including duplicates, non-finite points and the guard"""
    rng = np.random.default_rng(n)
    pts = np.c_[rng.uniform(-60, 60, (n, 2)), rng.uniform(-2, 6, (n, 1)), np.arange(n)].astype(np.float32)
    pts[n // 3] = pts[0]                      # duplicate point
    for leaf in (2.0, 0.3, 25.0):
        want, ov = oracle.voxel_grid(pts, leaf)
        got, st = gpu.voxel_downsample(pts, leaf)
        assert st == (1 if ov else 0)
        assert got.shape == want.shape and np.array_equal(got.view(np.uint32), want.view(np.uint32)), (n, leaf)
    bad = pts.copy()
    bad[::7, 1] = np.nan
    bad[n // 2, 0] = np.inf
    want, ov = oracle.voxel_grid(bad, 2.0)
    got, st = gpu.voxel_downsample(bad, 2.0)
    assert got.shape == want.shape and np.array_equal(got.view(np.uint32), want.view(np.uint32))
    want, ov = oracle.voxel_grid(pts, 1e-4)   # overflow guard -> input unchanged (for n >= 2 spread over 120 m)
    got, st = gpu.voxel_downsample(pts, 1e-4)
    assert st == (1 if ov else 0) and np.array_equal(got.view(np.uint32), want.view(np.uint32))
    allbad = np.full((min(n, 50), 4), np.nan, np.float32)
    got, st = gpu.voxel_downsample(allbad, 2.0)
    assert got.shape[0] == 0


# ---------------------------------------------------------------- round 2: ABI additions and advisor findings
def test_upload_scan_async_equals_direct_call(small_case, oracle):
    """liogpu_upload_scan_async + LIOGPU_UPLOADED_SCAN: same registration as handing the host buffer to the call itself"""
    from lio_slam_b200.liogpu import LioGpu, UPLOADED, LioGpuError
    g = LioGpu()
    try:
        g.set_local_map(small_case["map4"])
        ds, _ = oracle.voxel_grid(small_case["scan4"], 0.4)
        rec = synth.from_packed(ds)                      # 32-byte PointXYZI records
        want_pose, _, want = g.scan2map(rec, small_case["guess"])
        with pytest.raises(LioGpuError):                 # nothing uploaded yet
            g.scan2map(UPLOADED, small_case["guess"])
        g.upload_scan_async(rec)
        got_pose, _, got = g.scan2map(UPLOADED, small_case["guess"])
        assert got["iterations"] == want["iterations"] and np.array_equal(got_pose.view(np.uint32), want_pose.view(np.uint32))
        # two sweeps in flight are consumed first in, first out; a third is refused; packed stride works too
        half = np.ascontiguousarray(ds[: ds.shape[0] // 2])
        g.upload_scan_async(ds)
        g.upload_scan_async(half)
        with pytest.raises(LioGpuError):
            g.upload_scan_async(ds)
        n_a, st = g.voxel_downsample(UPLOADED, 0.8, keep_on_device=True)
        n_b, st = g.voxel_downsample(UPLOADED, 0.8, keep_on_device=True)
        assert n_a == oracle.voxel_grid(ds, 0.8)[0].shape[0] and n_b == oracle.voxel_grid(half, 0.8)[0].shape[0]
    finally:
        g.close()


def test_merge_more_keyframes_than_the_old_pose_table_held(oracle):
    """saveMapService merges EVERY keyframe (mapOptmization.cpp:936-941); round 1 capped a call at 1365 (ADVICE.md)"""
    from lio_slam_b200.liogpu import LioGpu
    rng = np.random.default_rng(3)
    k = 1500
    clouds = [rng.normal(0, 5, (7 + (i % 5), 4)).astype(np.float32) for i in range(k)]
    poses = np.column_stack([rng.uniform(-0.1, 0.1, (k, 2)), rng.uniform(-3, 3, k), rng.uniform(-200, 200, (k, 2)),
                             rng.uniform(-2, 2, k)]).astype(np.float32)
    g = LioGpu()
    try:
        for i, c in enumerate(clouds):
            g.keyframe_put(i, c)
        got, st = g.merge_keyframes(np.arange(k), poses, 0.0)
        want = np.concatenate([oracle.transform_cloud(c, p) for c, p in zip(clouds, poses)])
        assert st == 0 and np.array_equal(got.view(np.uint32), want.view(np.uint32))
        got2, st2 = g.merge_keyframes(np.arange(k), poses, 2.0)
        want2, _ = oracle.voxel_grid(want, 2.0)
        assert np.array_equal(got2.view(np.uint32), want2.view(np.uint32))
    finally:
        g.close()


def test_failed_keyframe_overwrite_keeps_the_old_keyframe(small_case):
    """ADVICE.md: a failed liogpu_keyframe_put must neither leak nor delete the keyframe that was there"""
    import ctypes as C
    from lio_slam_b200.liogpu import LioGpu, E_INVALID
    g = LioGpu()
    try:
        cloud = small_case["scan4"][:500]
        g.keyframe_put(7, cloud)
        pose = np.zeros((1, 6), np.float32)
        before, _ = g.merge_keyframes([7], pose, 0.0)
        st = g.lib.liogpu_keyframe_put(g.h, 7, cloud.ctypes.data, 500, 20)     # bad stride
        assert st == E_INVALID
        st = g.lib.liogpu_keyframe_put(g.h, 7, None, 500, 16)                   # null cloud
        assert st == E_INVALID
        after, _ = g.merge_keyframes([7], pose, 0.0)
        assert g.keyframe_count() == 1 and np.array_equal(before.view(np.uint32), after.view(np.uint32))
        g.keyframe_put(7, cloud[:100])                                          # a real overwrite still works, in place
        again, _ = g.merge_keyframes([7], pose, 0.0)
        assert again.shape[0] == 100
    finally:
        g.close()


def test_fetch_result_serves_only_the_call_before_it(small_case):
    import ctypes as C
    from lio_slam_b200.liogpu import LioGpu, E_CAPACITY, E_INVALID
    g = LioGpu()
    try:
        g.keyframe_put(0, small_case["scan4"])
        pose = np.zeros((1, 6), np.float32)
        ids = np.zeros(1, np.int32)
        n = C.c_int(0)
        tiny = np.empty((1, 4), np.float32)
        st = g.lib.liogpu_merge_keyframes(g.h, ids.ctypes.data, pose.ctypes.data, 1, C.c_float(0.5), tiny.ctypes.data, 16, 1, C.byref(n))
        assert st == E_CAPACITY and n.value > 1
        out = np.empty((n.value, 4), np.float32)
        assert g.lib.liogpu_fetch_result(g.h, out.ctypes.data, 16, n.value, C.byref(n)) == 0
        want, _ = g.merge_keyframes([0], pose, 0.5)        # (this wrapper fetches too)
        assert np.array_equal(out.view(np.uint32), want.view(np.uint32))
        g.keyframe_count()
        g.voxel_downsample(small_case["scan4"], 1.0)       # any other call invalidates the pending result
        assert g.lib.liogpu_fetch_result(g.h, out.ctypes.data, 16, n.value, C.byref(n)) == E_INVALID
    finally:
        g.close()
