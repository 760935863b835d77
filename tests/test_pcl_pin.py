"""Pins the CPU oracle against the REAL PCL / FLANN / Eigen / OpenCV outputs produced by tests/golden/pcl_pin/pcl_pin.cpp
on a ROS Noetic machine (README there).  The fixture cannot be produced in the build container (none of the libraries is
installed, no network): while tests/golden/pcl_pin/out/pcl_pin_outputs.lpin is absent these tests SKIP with the reason
"unpinned", which is also what DESIGN.md §2 and the oracle header say.  Once the fixture is committed they run in the
CPU suite and every call site that compares equal is pinned."""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
KIT = os.path.join(HERE, "golden", "pcl_pin")
sys.path.insert(0, KIT)
import lpin  # noqa: E402

OUT = os.environ.get("PCL_PIN_OUT") or os.path.join(KIT, "out", "pcl_pin_outputs.lpin")   # env: the kit's selfcheck.py
INP = os.path.join(KIT, "pin_inputs.lpin")
pinned = pytest.mark.skipif(not os.path.exists(OUT), reason="unpinned: tests/golden/pcl_pin/out/pcl_pin_outputs.lpin absent "
                            "(produce it with the kit's README recipe on a ROS Noetic image)")


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def ulp_diff(a, b):
    ia = bits(a).astype(np.int64); ib = bits(b).astype(np.int64)
    ia = np.where(ia < 0x80000000, ia, 0x80000000 - ia); ib = np.where(ib < 0x80000000, ib, 0x80000000 - ib)
    return np.abs(ia - ib)


def test_kit_inputs_are_committed_and_reproducible():
    """the inputs the kit feeds to the real libraries are in the tree and match their generator (seeded)"""
    assert os.path.exists(INP)
    rec = lpin.read(INP)
    assert set(rec) >= {"cloud_a", "cloud_b", "pose_guess", "icp_source", "lm_A", "lm_b", "pose_now"}
    from lio_slam_b200 import synth
    world = synth.make_world(1234)
    a = synth.to_packed(synth.make_scan(world, synth.path_pose(0.0), 16, seed=11, cols=450))
    assert np.array_equal(bits(rec["cloud_a"]), bits(a))
    for f in ("CMakeLists.txt", "pcl_pin.cpp", "README.md"):
        assert os.path.exists(os.path.join(KIT, f))


@pytest.fixture(scope="module")
def pin():
    return lpin.read(INP), lpin.read(OUT)


@pinned
@pytest.mark.parametrize("rec,src,leaf", [("vox_a_04", "cloud_a", 0.4), ("vox_b_05", "cloud_b", 0.5), ("vox_a_20", "cloud_a", 2.0)])
def test_voxelgrid_matches_pcl(oracle, pin, rec, src, leaf):
    inp, out = pin
    got, ov = oracle.voxel_grid(inp[src], leaf)
    want = out[rec]
    assert not ov and got.shape == want.shape, "voxel count / membership differs from pcl::VoxelGrid"
    # PCL's within-voxel order is an unstable-sort artefact: centroids of <= 2-point voxels are bit-equal, the others
    # agree within the reordering error of an n-term f32 sum
    exact = (bits(got) == bits(want)).all(axis=1)
    assert np.abs(got - want).max() <= 2e-5 * max(1.0, float(np.abs(want[:, :3]).max()))
    print(f"{rec}: {int(exact.sum())} of {want.shape[0]} voxels bit-equal")


@pinned
def test_voxelgrid_overflow_guard_matches_pcl(oracle, pin):
    inp, out = pin
    got, ov = oracle.voxel_grid(inp["cloud_a"], 0.001)
    assert ov and int(out["vox_guard_n"][0]) == int(out["vox_guard_n"][1]) == got.shape[0]


@pinned
def test_transform_and_knn_and_plane_fit_match_pcl_flann_eigen(oracle, pin):
    inp, out = pin
    T = oracle.pose_to_T(inp["pose_guess"])
    # canonical trig (f64 sin/cos rounded to f32) vs glibc sinf/cosf: <= 1 ulp per entry, not bit-equal by design
    assert np.abs(T.reshape(3, 4) - out["T_pose"][:3]).max() <= 2e-7 * max(1.0, float(np.abs(out["T_pose"]).max()))
    a04, _ = oracle.voxel_grid(inp["cloud_a"], 0.4)
    b05, _ = oracle.voxel_grid(inp["cloud_b"], 0.5)
    # feed the REAL transform so that the k-NN inputs are the same bytes on both sides
    res = oracle.surf_optimization(b05, a04, T12=out["T_pose"][:3].reshape(12), threads=4)
    d2, idx = out["knn_d2"], out["knn_idx"]
    assert np.array_equal(bits(res["nn_d2"]), bits(d2)), "pointSearchSqDis differs from FLANN L2_Simple"
    ties = res["tie"].astype(bool) | (d2[:, 3] == d2[:, 4])
    same = (res["nn_idx"] == idx).all(axis=1)
    assert same[~ties].all(), "neighbour indices differ outside logged equidistant ties"
    print(f"kNN: {int(same.sum())} of {idx.shape[0]} rows index-equal, {int(ties.sum())} logged ties")
    x = np.array([oracle.qr53_solve(b05[idx[i], :3], -np.ones(5, np.float32)) for i in range(0, idx.shape[0], 7)])
    assert ulp_diff(x, out["qr_x"][::7]).max() <= 4, "colPivHouseholderQr().solve differs from Eigen by more than 4 ulp"


@pinned
def test_local_map_chain_matches_pcl(oracle, pin):
    inp, out = pin
    kf = [inp["cloud_b"]]
    poses = np.zeros((1, 6), np.float32)
    lm, info, _ = oracle.publish_local_map(kf, poses, inp["pose_now"], use_removing_outliers=True, mean_k=10,
                                           stddev_threshold=1.0, use_down_sampling=False, threads=4)
    assert lm.shape == out["sor_out"].shape and np.array_equal(bits(lm), bits(out["sor_out"])), \
        "transformPointCloud + PassThrough + StatisticalOutlierRemoval differ from PCL"


@pinned
def test_icp_matches_pcl(oracle, pin):
    inp, out = pin
    b05, _ = oracle.voxel_grid(inp["cloud_b"], 0.5)
    r = oracle.icp_align(inp["icp_source"], b05, threads=4)
    assert bool(r["converged"]) == bool(out["icp_meta"][0])
    assert np.abs(r["T"] - out["icp_T"]).max() <= 1e-4
    assert abs(r["fitness_score"] - out["icp_meta"][1]) <= 1e-6 * max(1.0, out["icp_meta"][1])


def test_opencv_6x6_pieces_match_opencv_cpp(oracle):
    """the kit's fixture when it is present, else OpenCV's outputs for the same system stored by
    tests/golden/make_golden.py (Python cv2 calls the same cv::gemm / cv::solve / cv::eigen / cv::invert)"""
    inp = lpin.read(INP)
    if os.path.exists(OUT):
        out = lpin.read(OUT)
    else:
        G = np.load(os.path.join(HERE, "golden", "cv2_live.npz"))
        out = {"cv_AtA": G["pin_AtA"], "cv_x": G["pin_X"], "cv_E": G["pin_E"], "cv_V": G["pin_V"], "cv_Vinv": G["pin_Vi"]}
    A, b = inp["lm_A"], inp["lm_b"]
    AtA = (A.astype(np.float64).T @ A.astype(np.float64)).astype(np.float32)   # what oracle::normal_equations computes
    assert np.array_equal(bits(AtA), bits(out["cv_AtA"])), "AtA differs from cv::gemm (f64 accumulation rounded once)"
    Atb = (A.astype(np.float64).T @ b.astype(np.float64)).astype(np.float32)
    ok, x = oracle.cv_solve6_qr(out["cv_AtA"], Atb)
    assert ok and np.array_equal(bits(x), bits(out["cv_x"].reshape(6))), "cv::solve(DECOMP_QR) differs"
    E, V = oracle.cv_eigen6(out["cv_AtA"])
    assert np.array_equal(bits(E), bits(out["cv_E"].reshape(6))) and np.array_equal(bits(V), bits(out["cv_V"]))
    ok, Vi = oracle.cv_inv6(out["cv_V"])
    assert ok and np.array_equal(bits(Vi), bits(out["cv_Vinv"]))
