"""CPU checks of the oracle's loop-closure ICP restatement (pcl::IterativeClosestPoint as configured at
mapOptmization.cpp:1111-1123; SURVEY §8 row f3): nearest-neighbour providers agree, a known rigid motion is
recovered, and one ICP step equals an independent numpy Kabsch/Umeyama step.  (PARITY UNPINNED: no PCL here.)"""
import numpy as np
import pytest

from lio_slam_b200 import synth


def rigid(rx, ry, rz, t):
    T = np.eye(4)
    T[:3, :3] = synth.rpy_to_R(rx, ry, rz)
    T[:3, 3] = t
    return T


def apply(T, c):
    out = c.copy()
    out[:, :3] = (c[:, :3].astype(np.float64) @ T[:3, :3].T + T[:3, 3]).astype(np.float32)
    return out


@pytest.fixture(scope="module")
def clouds(world, oracle):
    p = synth.path_pose(2.0)
    tgt, _ = oracle.voxel_grid(synth.transform_packed(synth.to_packed(synth.make_scan(world, p, 32, seed=41, cols=600)), p), 0.4)
    return tgt


def test_oracle_icp_recovers_known_motion(oracle, clouds):
    tgt = clouds
    Tm = rigid(0.004, -0.003, 0.02, [0.35, -0.25, 0.05])
    src = apply(np.linalg.inv(Tm), tgt[::2])                   # moving src by Tm lands exactly on target points
    r = oracle.icp_align(src, tgt, threads=4)
    assert r["converged"] == 1 and r["state"] in (2, 3, 4) and r["iterations"] < 60
    assert np.abs(r["T"].astype(np.float64) - Tm).max() < 2e-3 and r["fitness_score"] < 1e-4
    assert r["n_correspondences"] == src.shape[0]


def test_oracle_icp_nn_providers_agree(oracle, clouds):
    from oracle.oracle import Oracle
    tgt = clouds
    src = apply(rigid(0.0, 0.0, 0.03, [0.6, 0.4, 0.0]), tgt[::5])
    a = oracle.icp_align(src, tgt, brute=True, threads=4)
    b = oracle.icp_align(src, tgt, brute=False, threads=4)
    c = oracle.icp_align(src, tgt, brute=False, threads=1)
    for other in (b, c):
        assert np.array_equal(a["T"], other["T"]) and a["iterations"] == other["iterations"]
        assert a["fitness_score"] == other["fitness_score"]
    if Oracle.available("nanoflann"):
        d = Oracle("nanoflann").icp_align(src, tgt, threads=4)
        assert np.array_equal(a["T"], d["T"]) and a["iterations"] == d["iterations"]


def test_oracle_icp_single_step_equals_numpy_umeyama(oracle, clouds):
    tgt = clouds
    src = apply(rigid(0.01, 0.0, -0.02, [0.2, 0.1, -0.05]), tgt[::4])
    r = oracle.icp_align(src, tgt, max_iterations=1, brute=True, threads=4)
    assert r["iterations"] == 1 and r["state"] == 1 and r["converged"] == 1       # iteration limit counts as converged
    # independent step: exhaustive nearest neighbours in f32, Kabsch in f64
    d = src[:, None, :3] - tgt[None, :, :3]
    d2 = (d[:, :, 0] * d[:, :, 0] + d[:, :, 1] * d[:, :, 1]) + d[:, :, 2] * d[:, :, 2]
    j = d2.argmin(axis=1)
    S, D = src[:, :3].astype(np.float64), tgt[j, :3].astype(np.float64)
    ms, md = S.mean(0), D.mean(0)
    sigma = (D - md).T @ (S - ms) / S.shape[0]
    U, sv, Vt = np.linalg.svd(sigma)
    dd = np.ones(3)
    if np.linalg.det(U) * np.linalg.det(Vt) < 0:
        dd[2] = -1
    R = U @ np.diag(dd) @ Vt
    t = md - R @ ms
    assert np.abs(r["T"][:3, :3] - R).max() < 2e-6 and np.abs(r["T"][:3, 3] - t).max() < 2e-4
    assert r["last_mse"] == pytest.approx(float(d2.min(axis=1).astype(np.float64).mean()), rel=1e-9)


def test_oracle_icp_max_distance_and_no_correspondences(oracle, clouds):
    tgt = clouds
    src = apply(rigid(0, 0, 0, [300.0, 0, 0]), tgt[::10])
    r = oracle.icp_align(src, tgt, max_correspondence_distance=5.0, threads=4)
    assert r["state"] == 5 and r["converged"] == 0 and r["iterations"] == 0
    assert np.array_equal(r["T"], np.eye(4, dtype=np.float32))


def _kabsch(sigma):
    """R = U diag(1, 1, d) V^T of sigma = U S V^T in f64 (the rotation Eigen::umeyama returns)"""
    U, _, Vt = np.linalg.svd(np.asarray(sigma, np.float64))
    d = np.sign(np.linalg.det(U) * np.linalg.det(Vt))
    return U @ np.diag([1.0, 1.0, d]) @ Vt


def test_oracle_umeyama_rotation_equals_numpy_kabsch(oracle):
    """the exported rotation tail of Eigen::umeyama against an f64 Kabsch solution, on cross-covariances with a
    unique answer: proper rotations (up to 180 degrees), reflections (det < 0 -> the nearest rotation) and coplanar
    (rank 2) clouds; 2e-6 covers the f32 input and output roundings"""
    rng = np.random.default_rng(5)
    worst = 0.0
    for t in range(400):
        q = rng.normal(size=4)
        if t % 50 == 0:
            q[0] = 0.0  # 180 degrees
        q /= np.linalg.norm(q)
        w, x, y, z = q
        R = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                      [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                      [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])
        src = rng.normal(size=(50, 3)) * rng.uniform(0.5, 5.0, size=3)
        if t % 4 == 1:
            src[:, 2] = 0.0                      # coplanar source: sigma has rank 2
        dst = src @ R.T
        if t % 4 == 2:
            dst[:, 0] = -dst[:, 0]               # a reflection: det(U) det(V) < 0
        sc, dc = src - src.mean(0), dst - dst.mean(0)
        sigma = (dc.T @ sc / len(src)).astype(np.float32)
        want = _kabsch(sigma)
        got = oracle.umeyama_rotation(sigma)
        assert abs(np.linalg.det(got.astype(np.float64)) - 1.0) < 1e-5
        if t % 4 != 2:
            assert np.abs(want - R).max() < 1e-5, t
        worst = max(worst, float(np.abs(got - want).max()))
        assert np.abs(got - want).max() <= 2e-6, (t, got, want)
    print(f"umeyama_rotation vs f64 Kabsch: max |dR| = {worst:.3g} over 400 cross-covariances")


def test_oracle_plane_residual_export(oracle):
    """the exported per-point plane fit: its plane is qr53_solve's, the points' residuals decide the flag, and a
    neighbour set farther than 1 m (d2_4 >= 1) is rejected before any fit"""
    rng = np.random.default_rng(9)
    for t in range(200):
        n = rng.normal(size=3); n /= np.linalg.norm(n)
        d = rng.uniform(0.5, 20.0)
        pts = rng.normal(size=(5, 3)) * 0.3
        pts -= np.outer(pts @ n, n)
        pts += (d * n) + rng.normal(size=(5, 3)) * (0.001 if t % 2 else 0.3)
        nbr = np.concatenate([pts, np.zeros((5, 1))], 1).astype(np.float32)
        sel = np.array([*(d * n + rng.normal(size=3) * 0.05), 0], np.float32)
        ori = np.array([*rng.normal(size=3) * 10, 0], np.float32)
        ok, coeff = oracle.plane_residual(ori, sel, nbr)
        x = oracle.qr53_solve(nbr[:, :3], -np.ones(5, np.float32))
        pn = x / np.float32(np.sqrt(np.float32(x @ x)))
        r = np.abs(nbr[:, :3].astype(np.float64) @ pn.astype(np.float64) + 1.0 / np.linalg.norm(x.astype(np.float64)))
        if r.max() > 0.2 + 1e-4:
            assert not ok
        if ok:
            assert np.allclose(coeff[:3] / np.linalg.norm(coeff[:3]), pn, atol=1e-5)
        far_ok, far_coeff = oracle.plane_residual(ori, sel, nbr, d2_4=1.0)
        assert not far_ok and not far_coeff.any()
