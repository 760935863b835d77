"""Generates tests/golden/*.npz — run in the build container:  python tests/golden/make_golden.py

1. cv2_6x6.npz  : inputs and outputs of the REAL OpenCV (Python cv2, the version is stored in the file) for
   the 6x6 pieces of LMOptimization (mapOptmization.cpp:1781-1814): At*A / At*b (cv::gemm), cv::solve(QR),
   cv::eigen, Mat::inv (LU), V.inv()*V2.  These pin the oracle's restatement of OpenCV to the library itself.
2. path_small.npz : a small end-to-end case (scan, map, guess) with the oracle's outputs (VoxelGrid, one
   surfOptimization pass, the full scan2map loop).  These are ORACLE outputs, not reference outputs — the
   reference cannot be built here (parity unpinned); they guard the oracle and the CUDA path against drift.
2b. cv2_live.npz : OpenCV's outputs (cv2) for the seeded random systems of tests/test_oracle_cv2.py
   (test_live_cv2_random, test_normal_equations_match_cv_gemm) and for the 6x6 system of the PCL pinning kit's
   inputs (tests/test_pcl_pin.py, pin_*), so that those comparisons run without cv2.
3. rows_f_small.npz : the same for the widened rows (publishLocalMap, keyframe merging, loop-closure ICP, Scan
   Context, key-pose selection), again ORACLE outputs.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)


def make_cv2():
    import cv2
    rng = np.random.default_rng(20261018)
    cases = []
    for t in range(24):
        n = int(rng.integers(60, 800))
        A = (rng.normal(size=(n, 6)) * rng.uniform(0.1, 10, size=6)).astype(np.float32)
        if t % 4 == 1:
            A[:, 3] *= 1e-3           # nearly rank deficient -> eigenvalue below 100
        if t % 4 == 2:
            A[:, 0] = A[:, 1] * 0.5   # exactly dependent columns
        b = rng.normal(size=(n, 1)).astype(np.float32)
        At = np.ascontiguousarray(A.T)
        AtA = cv2.gemm(At, A, 1.0, None, 0.0)
        Atb = cv2.gemm(At, b, 1.0, None, 0.0)
        ok, X = cv2.solve(AtA, Atb, flags=cv2.DECOMP_QR)
        _, E, V = cv2.eigen(AtA)
        V2 = V.copy()
        for i in range(5, -1, -1):
            if E[i, 0] < 100:
                V2[i, :] = 0
            else:
                break
        rc, Vi = cv2.invert(V, flags=cv2.DECOMP_LU)
        P = cv2.gemm(Vi, V2, 1.0, None, 0.0)
        cases.append(dict(A=A, b=b[:, 0], AtA=AtA, Atb=Atb[:, 0], X=X[:, 0], ok=ok, E=E[:, 0], V=V, Vi=Vi, P=P))
    out = {"cv2_version": np.array(cv2.__version__), "n_cases": np.array(len(cases))}
    for k, c in enumerate(cases):
        for name, v in c.items():
            out[f"{name}_{k}"] = np.asarray(v)
    np.savez_compressed(os.path.join(HERE, "cv2_6x6.npz"), **out)
    print("cv2_6x6.npz:", len(cases), "cases, cv2", cv2.__version__)


def make_cv2_live():
    import cv2
    sys.path.insert(0, os.path.dirname(HERE))
    from test_oracle_cv2 import cv2_live_outputs, live_cases
    from oracle.oracle import Oracle
    out = {"cv2_version": np.array(cv2.__version__)}
    for t, (A, b) in enumerate(live_cases()):
        for name, v in cv2_live_outputs(cv2, A, b).items():
            out[f"{name}_{t}"] = np.asarray(v)
    rng = np.random.default_rng(1)          # the normal equations of test_normal_equations_match_cv_gemm
    n = 5000
    scan = rng.normal(0, 20, (n, 4)).astype(np.float32)
    coeff = rng.normal(0, 1, (n, 4)).astype(np.float32)
    flag = (rng.uniform(size=n) < 0.8).astype(np.uint8)
    _, JtJ, Jtr = Oracle("port").normal_equations(scan, coeff, flag, np.array([0.01, -0.02, 0.5, 1, 2, 3], np.float32))
    ok, X = cv2.solve(JtJ.astype(np.float32), Jtr.astype(np.float32).reshape(6, 1), flags=cv2.DECOMP_QR)
    out.update(ne_JtJ=JtJ, ne_Jtr=Jtr, ne_ok=np.array(ok), ne_X=X[:, 0])
    sys.path.insert(0, os.path.join(HERE, "pcl_pin"))
    import lpin
    inp = lpin.read(os.path.join(HERE, "pcl_pin", "pin_inputs.lpin"))
    for name, v in cv2_live_outputs(cv2, inp["lm_A"], inp["lm_b"].reshape(-1, 1)).items():
        out[f"pin_{name}"] = np.asarray(v)
    np.savez_compressed(os.path.join(HERE, "cv2_live.npz"), **out)
    print("cv2_live.npz: 60 systems, the normal equations and the pin kit's system, cv2", cv2.__version__)


def make_path():
    from lio_slam_b200 import synth
    from oracle.oracle import Oracle
    o = Oracle("port")
    world = synth.make_world(1234)
    pose_gt = synth.path_pose(0.0)
    scan4 = synth.to_packed(synth.make_scan(world, pose_gt, 16, seed=11, cols=300))
    map4 = synth.make_local_map(world, 16, 4000, 0.5, seed=5, s0=-0.5, cols=300, max_poses=32)
    guess = synth.perturbed_guess(pose_gt, 21)
    ds, _ = o.voxel_grid(scan4, 0.4)
    surf = o.surf_optimization(map4, ds, pose6=guess, threads=4)
    pose, P, info = o.scan2map(map4, ds, guess, threads=4)
    np.savez_compressed(os.path.join(HERE, "path_small.npz"), scan4=scan4, map4=map4, guess=guess, ds=ds,
                        nn_idx=surf["nn_idx"], nn_d2=surf["nn_d2"], coeff=surf["coeff"], flag=surf["flag"],
                        tie=surf["tie"], pose=pose, matP=P, iterations=np.array(info["iterations"]),
                        nsel_hist=info["nsel_hist"], pose_hist=info["pose_hist"], JtJ=info["JtJ"], Jtr=info["Jtr"])
    print("path_small.npz: scan", scan4.shape, "ds", ds.shape, "map", map4.shape, "iters", info["iterations"])


def make_rows_f():
    """rows_f_small.npz: small cases of the widened rows (SURVEY §8 f2-f4) with the oracle's outputs."""
    from lio_slam_b200 import synth
    from oracle.oracle import Oracle
    o = Oracle("port")
    world = synth.make_world(1234)
    clouds, poses = [], []
    for k in range(4):
        p = synth.path_pose(1.0 * k)
        ds, _ = o.voxel_grid(synth.to_packed(synth.make_scan(world, p, 16, seed=40 + k, cols=200)), 0.4)
        clouds.append(ds)
        poses.append(p.astype(np.float32))
    poses = np.array(poses, np.float32)
    offs = np.zeros(5, np.int32)
    offs[1:] = np.cumsum([c.shape[0] for c in clouds])
    now = np.array([0.01, -0.02, 2.0, 7.5, 1.0, 1.8], np.float32)
    lm, lm_info, md = o.publish_local_map(clouds, poses, now, leaf=0.3, threads=4)
    merged, _ = o.build_local_map(clouds, poses, 0.4, threads=4)
    wrong = poses[2].copy()
    wrong[3] += 0.5
    wrong[4] -= 0.3
    wrong[2] += 0.02
    src = o.transform_cloud(clouds[2], wrong)
    icp = o.icp_align(src, merged, threads=4)
    sc, rk, sk = o.make_scancontext(clouds[0])
    n = 120
    xyz = np.array([synth.path_pose(0.7 * k)[3:6] for k in range(n)])
    key3d = np.c_[xyz, np.arange(n)].astype(np.float32)
    key_t = 0.5 * np.arange(n)
    ids = o.extract_nearby(key3d, key_t, key_t[-1] + 0.1, 30.0, 2.0)
    np.savez_compressed(os.path.join(HERE, "rows_f_small.npz"), clouds=np.concatenate(clouds), offsets=offs, poses=poses,
                        pose_now=now, local_map=lm, local_map_counts=np.array([lm_info["n_concat"], lm_info["n_cropped"],
                                                                               lm_info["n_after_sor"], lm_info["n_out"]]),
                        mean_distances=md, merged=merged, icp_source=src, icp_T=icp["T"],
                        icp_ints=np.array([icp["iterations"], icp["converged"], icp["state"], icp["n_correspondences"]]),
                        icp_fitness=np.array(icp["fitness_score"]), sc_desc=sc, sc_ringkey=rk, sc_sectorkey=sk,
                        key3d=key3d, key_time=key_t, nearby_ids=ids)
    print("rows_f_small.npz: local map", lm.shape, "icp iters", icp["iterations"], "nearby ids", ids.shape)


if __name__ == "__main__":
    make_cv2()
    make_path()
    make_rows_f()
