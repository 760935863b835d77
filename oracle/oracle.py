"""ctypes binding of the CPU oracle (oracle/liboracle.so, oracle/_ref/liboracle_nf.so).

TEST INFRASTRUCTURE — imported only by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs.  PARITY UNPINNED (see oracle/liorf_oracle_core.h).  Clouds are (n,4) float32
arrays (x, y, z, intensity).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))


class S2MResult(C.Structure):
    _fields_ = [("iterations", C.c_int), ("converged", C.c_int), ("n_sel", C.c_int), ("is_degenerate", C.c_int),
                ("tie_queries", C.c_int), ("delta_r", C.c_float), ("delta_t", C.c_float),
                ("JtJ", C.c_double * 36), ("Jtr", C.c_double * 6), ("pose_hist", (C.c_float * 6) * 30),
                ("nsel_hist", C.c_int * 30), ("ms_build", C.c_double), ("ms_loop", C.c_double)]


class DeskewParams(C.Structure):
    _fields_ = [("n_scan", C.c_int), ("downsample_rate", C.c_int), ("point_filter_num", C.c_int),
                ("min_front", C.c_float), ("min_back", C.c_float), ("min_left", C.c_float), ("min_right", C.c_float),
                ("max_range", C.c_float), ("max_intensity", C.c_float)]


class LocalMapParams(C.Structure):
    _fields_ = [("left", C.c_float), ("right", C.c_float), ("front", C.c_float), ("back", C.c_float),
                ("use_removing_outliers", C.c_int), ("mean_k", C.c_int), ("stddev_threshold", C.c_float),
                ("use_down_sampling", C.c_int), ("leaf", C.c_float)]


class LocalMapInfo(C.Structure):
    _fields_ = [("n_concat", C.c_int), ("n_cropped", C.c_int), ("n_after_sor", C.c_int), ("n_out", C.c_int),
                ("leaf_overflow", C.c_int), ("pad", C.c_int), ("sor_mean", C.c_double), ("sor_stddev", C.c_double),
                ("sor_threshold", C.c_double)]


class IcpParams(C.Structure):
    _fields_ = [("max_correspondence_distance", C.c_double), ("max_iterations", C.c_int),
                ("transformation_epsilon", C.c_double), ("euclidean_fitness_epsilon", C.c_double)]


class IcpResult(C.Structure):
    _fields_ = [("final_transformation", C.c_float * 16), ("iterations", C.c_int), ("converged", C.c_int),
                ("state", C.c_int), ("n_correspondences", C.c_int), ("fitness_score", C.c_double),
                ("last_mse", C.c_double)]


def build(force: bool = False) -> None:
    """Compile the oracle (and oracle/_ref when the reference tree is present)."""
    if force or not os.path.exists(os.path.join(_HERE, "liboracle.so")):
        subprocess.check_call(["make", "-C", _HERE, "all"], stdout=subprocess.DEVNULL)
    if os.path.exists("/root/reference/src/liorf/include/nanoflann.hpp") and (
            force or not os.path.exists(os.path.join(_HERE, "_ref", "liboracle_nf.so"))):
        subprocess.check_call(["make", "-C", _HERE, "_ref"], stdout=subprocess.DEVNULL)


def _f4(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    assert a.ndim == 2 and a.shape[1] == 4
    return a


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t)) if a is not None else None


class Oracle:
    """One loaded oracle library.  kind='port' (own KD-tree) or 'nanoflann' (oracle/_ref)."""

    def __init__(self, kind: str = "port"):
        if kind == "port":
            path, self.pre = os.path.join(_HERE, "liboracle.so"), "ref_"
            if not os.path.exists(path):
                build()
        elif kind == "nanoflann":
            path, self.pre = os.path.join(_HERE, "_ref", "liboracle_nf.so"), "refnf_"
            if not os.path.exists(path):
                build()
        else:
            raise ValueError(kind)
        self.kind = kind
        self.lib = C.CDLL(path)
        self._f("index_build").restype = C.c_void_p
        self._f("index_build").argtypes = [C.c_void_p, C.c_int]
        self._f("index_free").argtypes = [C.c_void_p]

    @staticmethod
    def available(kind: str) -> bool:
        if kind == "port":
            return True
        return os.path.exists(os.path.join(_HERE, "_ref", "liboracle_nf.so")) or \
            os.path.exists("/root/reference/src/liorf/include/nanoflann.hpp")

    def _f(self, name):
        return getattr(self.lib, self.pre + name)

    def max_threads(self) -> int:
        return int(self._f("omp_max_threads")())

    # -- a6 -------------------------------------------------------------------------------------
    def pose_to_T(self, pose6) -> np.ndarray:
        pose6 = np.ascontiguousarray(pose6, dtype=np.float32)
        T = np.zeros(12, dtype=np.float32)
        self._f("pose_to_T")(_p(pose6, C.c_float), _p(T, C.c_float))
        return T

    # -- a2 -------------------------------------------------------------------------------------
    def transform_cloud(self, cloud4, pose6, threads: int = 1) -> np.ndarray:
        cloud4 = _f4(cloud4)
        pose6 = np.ascontiguousarray(pose6, dtype=np.float32)
        out = np.empty_like(cloud4)
        self._f("transform_cloud")(_p(cloud4, C.c_float), C.c_int(cloud4.shape[0]), _p(pose6, C.c_float),
                                   _p(out, C.c_float), C.c_int(threads))
        return out

    # -- a3 / a4 --------------------------------------------------------------------------------
    def voxel_grid(self, cloud4, leaf: float):
        cloud4 = _f4(cloud4)
        out = np.empty_like(cloud4)
        n_out = C.c_int(0)
        ov = self._f("voxel_grid")(_p(cloud4, C.c_float), C.c_int(cloud4.shape[0]), C.c_float(leaf),
                                   _p(out, C.c_float), C.byref(n_out))
        return out[: n_out.value].copy(), bool(ov)

    def build_local_map(self, clouds, poses, leaf: float, threads: int = 1):
        offs = np.zeros(len(clouds) + 1, dtype=np.int32)
        offs[1:] = np.cumsum([c.shape[0] for c in clouds])
        cat = _f4(np.concatenate(clouds)) if clouds else np.zeros((0, 4), np.float32)
        poses = np.ascontiguousarray(poses, dtype=np.float32).reshape(-1, 6)
        out = np.empty_like(cat)
        n_out = C.c_int(0)
        ov = self._f("build_local_map")(_p(cat, C.c_float), _p(offs, C.c_int), _p(poses, C.c_float),
                                        C.c_int(len(clouds)), C.c_float(leaf), _p(out, C.c_float),
                                        C.byref(n_out), C.c_int(threads))
        return out[: n_out.value].copy(), bool(ov)

    # -- f2 -------------------------------------------------------------------------------------
    def yaw_frame_T(self, pose_now):
        pose_now = np.ascontiguousarray(pose_now, dtype=np.float32)
        m = np.zeros(12, np.float32)
        self._f("yaw_frame_T")(_p(pose_now, C.c_float), _p(m, C.c_float))
        return m

    def publish_local_map(self, clouds, poses, pose_now, left=40.0, right=40.0, front=70.0, back=20.0,
                          use_removing_outliers=True, mean_k=10, stddev_threshold=1.0, use_down_sampling=True,
                          leaf=0.01, brute=False, threads: int = 1):
        """publishLocalMap (MO:2442-2541) -> (cloud, info dict, mean distances of the cropped cloud)."""
        offs = np.zeros(len(clouds) + 1, dtype=np.int32)
        offs[1:] = np.cumsum([c.shape[0] for c in clouds])
        cat = _f4(np.concatenate(clouds)) if clouds else np.zeros((0, 4), np.float32)
        poses = np.ascontiguousarray(poses, dtype=np.float32).reshape(-1, 6)
        pose_now = np.ascontiguousarray(pose_now, dtype=np.float32)
        prm = LocalMapParams(left, right, front, back, int(use_removing_outliers), int(mean_k), stddev_threshold,
                             int(use_down_sampling), leaf)
        out = np.empty((max(cat.shape[0], 1), 4), np.float32)
        md = np.zeros(max(cat.shape[0], 1), np.float32)
        n_out = C.c_int(0)
        info = LocalMapInfo()
        self._f("publish_local_map")(_p(cat, C.c_float), _p(offs, C.c_int), _p(poses, C.c_float), C.c_int(len(clouds)),
                                     _p(pose_now, C.c_float), C.byref(prm), C.c_int(1 if brute else 0),
                                     _p(out, C.c_float), C.byref(n_out), C.byref(info), _p(md, C.c_float),
                                     C.c_int(threads))
        d = {k: getattr(info, k) for k, _ in LocalMapInfo._fields_ if k != "pad"}
        return out[: n_out.value].copy(), d, md[: info.n_cropped].copy()

    # -- f3 -------------------------------------------------------------------------------------
    def icp_align(self, source, target, max_correspondence_distance=20.0, max_iterations=100,
                  transformation_epsilon=1e-6, euclidean_fitness_epsilon=1e-6, brute=False, threads: int = 1):
        """pcl::IterativeClosestPoint as configured at MO:1111-1123 -> dict(T (4,4), iterations, converged, ...)."""
        source, target = _f4(source), _f4(target)
        prm = IcpParams(max_correspondence_distance, max_iterations, transformation_epsilon, euclidean_fitness_epsilon)
        res = IcpResult()
        self._f("icp_align")(_p(source, C.c_float), C.c_int(source.shape[0]), _p(target, C.c_float),
                             C.c_int(target.shape[0]), C.byref(prm), C.c_int(1 if brute else 0), C.byref(res),
                             C.c_int(threads))
        return dict(T=np.array(res.final_transformation, np.float32).reshape(4, 4), iterations=res.iterations,
                    converged=res.converged, state=res.state, n_correspondences=res.n_correspondences,
                    fitness_score=res.fitness_score, last_mse=res.last_mse)

    def make_scancontext(self, scan4, lidar_height=2.0, max_radius=80.0):
        """SCManager::makeScancontext + keys (Scancontext.cpp:151-225) -> (desc (20,60), ringkey (20,), sectorkey (60,))."""
        scan4 = _f4(scan4)
        desc = np.zeros((20, 60), np.float64)
        rk = np.zeros(20, np.float64)
        sk = np.zeros(60, np.float64)
        self._f("make_scancontext")(_p(scan4, C.c_float), C.c_int(scan4.shape[0]), C.c_double(lidar_height),
                                    C.c_double(max_radius), _p(desc, C.c_double), _p(rk, C.c_double), _p(sk, C.c_double))
        return desc, rk, sk

    def extract_nearby(self, key3d, key_time, time_cur, radius=50.0, density=2.0):
        """extractNearby + extractCloud's guard (MO:1519-1565) -> keyframe indices in concatenation order."""
        key3d = _f4(key3d)
        key_time = np.ascontiguousarray(key_time, dtype=np.float64)
        ids = np.zeros(2 * max(key3d.shape[0], 1), np.int32)
        n = self._f("extract_nearby")(_p(key3d, C.c_float), _p(key_time, C.c_double), C.c_int(key3d.shape[0]),
                                      C.c_double(time_cur), C.c_float(radius), C.c_float(density), _p(ids, C.c_int))
        return ids[:n].copy()

    # -- a5 / a7 --------------------------------------------------------------------------------
    def index_build(self, map4):
        map4 = _f4(map4)
        h = self._f("index_build")(map4.ctypes.data, C.c_int(map4.shape[0]))
        return (h, map4)  # keep the array alive with the handle

    def index_free(self, handle) -> None:
        self._f("index_free")(C.c_void_p(handle[0]))

    def knn5(self, map4, q4, handle=None, threads: int = 1):
        map4, q4 = _f4(map4), _f4(q4)
        n = q4.shape[0]
        idx = np.empty((n, 5), np.int32); d2 = np.empty((n, 5), np.float32); tie = np.empty(n, np.uint8)
        self._f("knn5")(_p(map4, C.c_float), C.c_int(map4.shape[0]), C.c_void_p(handle[0]) if handle else None,
                        _p(q4, C.c_float), C.c_int(n), _p(idx, C.c_int), _p(d2, C.c_float), _p(tie, C.c_ubyte),
                        C.c_int(threads))
        return idx, d2, tie

    def surf_optimization(self, map4, scan4, pose6=None, T12=None, handle=None, threads: int = 1):
        map4, scan4 = _f4(map4), _f4(scan4)
        n = scan4.shape[0]
        idx = np.empty((n, 5), np.int32); d2 = np.empty((n, 5), np.float32)
        coeff = np.empty((n, 4), np.float32); flag = np.empty(n, np.uint8); tie = np.empty(n, np.uint8)
        pose = np.ascontiguousarray(pose6, dtype=np.float32) if pose6 is not None else None
        T = np.ascontiguousarray(T12, dtype=np.float32) if T12 is not None else None
        self._f("surf_optimization")(_p(map4, C.c_float), C.c_int(map4.shape[0]),
                                     C.c_void_p(handle[0]) if handle else None, _p(scan4, C.c_float), C.c_int(n),
                                     _p(pose, C.c_float), _p(T, C.c_float), _p(idx, C.c_int), _p(d2, C.c_float),
                                     _p(coeff, C.c_float), _p(flag, C.c_ubyte), _p(tie, C.c_ubyte), C.c_int(threads))
        return dict(nn_idx=idx, nn_d2=d2, coeff=coeff, flag=flag, tie=tie)

    # -- a8 / a9 --------------------------------------------------------------------------------
    def normal_equations(self, scan4, coeff4, flag, pose6):
        scan4, coeff4 = _f4(scan4), _f4(coeff4)
        flag = np.ascontiguousarray(flag, dtype=np.uint8)
        pose6 = np.ascontiguousarray(pose6, dtype=np.float32)
        JtJ = np.zeros(36); Jtr = np.zeros(6)
        nsel = self._f("normal_equations")(_p(scan4, C.c_float), _p(coeff4, C.c_float), _p(flag, C.c_ubyte),
                                           C.c_int(scan4.shape[0]), _p(pose6, C.c_float), _p(JtJ, C.c_double),
                                           _p(Jtr, C.c_double))
        return int(nsel), JtJ.reshape(6, 6), Jtr

    def lm_solve_update(self, JtJ, Jtr, iter_count, pose6, matP, degenerate):
        JtJ = np.ascontiguousarray(JtJ, dtype=np.float64).reshape(36)
        Jtr = np.ascontiguousarray(Jtr, dtype=np.float64)
        pose = np.array(pose6, dtype=np.float32)
        P = np.array(matP, dtype=np.float32).reshape(36)
        deg = C.c_int(int(degenerate)); dr = C.c_float(0); dt = C.c_float(0)
        conv = self._f("lm_solve_update")(_p(JtJ, C.c_double), _p(Jtr, C.c_double), C.c_int(iter_count),
                                          _p(pose, C.c_float), _p(P, C.c_float), C.byref(deg), C.byref(dr), C.byref(dt))
        return bool(conv), pose, P.reshape(6, 6), deg.value, dr.value, dt.value

    def cv_solve6_qr(self, A, b):
        A = np.ascontiguousarray(A, np.float32).reshape(36); b = np.ascontiguousarray(b, np.float32)
        x = np.zeros(6, np.float32)
        ok = self._f("cv_solve6_qr")(_p(A, C.c_float), _p(b, C.c_float), _p(x, C.c_float))
        return bool(ok), x

    def cv_eigen6(self, A):
        A = np.ascontiguousarray(A, np.float32).reshape(36)
        W = np.zeros(6, np.float32); V = np.zeros(36, np.float32)
        self._f("cv_eigen6")(_p(A, C.c_float), _p(W, C.c_float), _p(V, C.c_float))
        return W, V.reshape(6, 6)

    def cv_inv6(self, A):
        A = np.ascontiguousarray(A, np.float32).reshape(36)
        out = np.zeros(36, np.float32)
        ok = self._f("cv_inv6")(_p(A, C.c_float), _p(out, C.c_float))
        return bool(ok), out.reshape(6, 6)

    def cv_gemm6(self, A, B):
        A = np.ascontiguousarray(A, np.float32).reshape(36); B = np.ascontiguousarray(B, np.float32).reshape(36)
        out = np.zeros(36, np.float32)
        self._f("cv_gemm6")(_p(A, C.c_float), _p(B, C.c_float), _p(out, C.c_float))
        return out.reshape(6, 6)

    def qr53_solve(self, A, b):
        A = np.ascontiguousarray(A, np.float32).reshape(15); b = np.ascontiguousarray(b, np.float32)
        x = np.zeros(3, np.float32)
        self._f("qr53_solve")(_p(A, C.c_float), _p(b, C.c_float), _p(x, C.c_float))
        return x

    def plane_residual(self, ori, sel, nbr, d2_4: float = 0.0):
        """surfOptimization's plane fit for one point (MO:1641-1684) -> (flag, coeff (4,)); coeff is zero when rejected."""
        ori = np.ascontiguousarray(ori, np.float32).reshape(4); sel = np.ascontiguousarray(sel, np.float32).reshape(4)
        nbr = np.ascontiguousarray(nbr, np.float32).reshape(20)
        coeff = np.zeros(4, np.float32)
        ok = self._f("plane_residual")(_p(ori, C.c_float), _p(sel, C.c_float), _p(nbr, C.c_float), C.c_float(d2_4),
                                       _p(coeff, C.c_float))
        return bool(ok), coeff

    def umeyama_rotation(self, sigma):
        """Eigen::umeyama's rotation (no scaling) of the 3x3 cross-covariance sigma -> R (3,3) float32."""
        sigma = np.ascontiguousarray(sigma, np.float32).reshape(9)
        R = np.zeros(9, np.float32)
        self._f("umeyama_rotation")(_p(sigma, C.c_float), _p(R, C.c_float))
        return R.reshape(3, 3)

    # -- a10 ------------------------------------------------------------------------------------
    def scan2map(self, map4, scan4, pose6, matP=None, degenerate: int = 0, max_iter: int = 30, threads: int = 1,
                 handle=None, brute: bool = False):
        map4, scan4 = _f4(map4), _f4(scan4)
        pose = np.array(pose6, dtype=np.float32)
        P = np.zeros(36, np.float32) if matP is None else np.array(matP, dtype=np.float32).reshape(36)
        deg = C.c_int(int(degenerate))
        res = S2MResult()
        st = self._f("scan2map")(_p(map4, C.c_float), C.c_int(map4.shape[0]),
                                 C.c_void_p(handle[0]) if handle else None, C.c_int(int(brute)),
                                 _p(scan4, C.c_float), C.c_int(scan4.shape[0]), _p(pose, C.c_float),
                                 _p(P, C.c_float), C.byref(deg), C.c_int(max_iter), C.c_int(threads), C.byref(res))
        info = dict(status=int(st), iterations=res.iterations, converged=bool(res.converged), n_sel=res.n_sel,
                    is_degenerate=deg.value, tie_queries=res.tie_queries, delta_r=res.delta_r, delta_t=res.delta_t,
                    JtJ=np.array(res.JtJ).reshape(6, 6), Jtr=np.array(res.Jtr),
                    pose_hist=np.array(res.pose_hist, dtype=np.float32).reshape(30, 6)[: res.iterations],
                    nsel_hist=np.array(res.nsel_hist)[: res.iterations], ms_build=res.ms_build, ms_loop=res.ms_loop)
        return pose, P.reshape(6, 6), info

    # -- a1 -------------------------------------------------------------------------------------
    def deskew(self, scan_xyzirt: np.ndarray, params: DeskewParams, time_scan_cur: float, imu_t, rx, ry, rz,
               deskew_enabled: bool = True) -> np.ndarray:
        raw = np.ascontiguousarray(scan_xyzirt)
        assert raw.dtype.itemsize == 32
        n = raw.shape[0]
        imu_t = np.ascontiguousarray(imu_t, np.float64); rx = np.ascontiguousarray(rx, np.float64)
        ry = np.ascontiguousarray(ry, np.float64); rz = np.ascontiguousarray(rz, np.float64)
        out = np.empty((max(n, 1), 4), np.float32)
        m = self._f("deskew")(C.c_void_p(raw.ctypes.data), C.c_int(n), C.byref(params), C.c_double(time_scan_cur),
                              _p(imu_t, C.c_double), _p(rx, C.c_double), _p(ry, C.c_double), _p(rz, C.c_double),
                              C.c_int(imu_t.shape[0]), C.c_int(int(deskew_enabled)), _p(out, C.c_float))
        return out[:m].copy()
