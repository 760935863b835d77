"""ctypes binding of libliogpu.so — the C ABI declared in include/liogpu.h.

This is plumbing for tests and bench.py; the product is the shared library.  There is no CPU path:
if the library is missing or no sm_100 GPU is usable, construction raises.

Clouds may be passed as
  * (n,4) float32 arrays  (packed x,y,z,intensity; stride 16), or
  * structured arrays with itemsize 32 (pcl::PointXYZI / PointXYZIRT records; stride 32), or
  * (device_ptr:int, n, stride) tuples for buffers already resident on the GPU.
"""
from __future__ import annotations

import ctypes as C
import os
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LIOGPU_LIB") or os.path.join(_HERE, "libliogpu.so")  # LIOGPU_LIB: A/B builds

LIOGPU_MAX_ITER = 30
OK = 0
E_INVALID, E_CUDA, E_NO_MAP, E_NO_KEYFRAME, E_CAPACITY = -1, -2, -3, -4, -5
W_LEAF_OVERFLOW, W_FEW_FEATURES, W_NO_KEYFRAMES = 1, 2, 3


class Params(C.Structure):
    _fields_ = [("device", C.c_int), ("n_scan", C.c_int), ("horizon_scan", C.c_int),
                ("mapping_surf_leaf_size", C.c_float), ("surrounding_keyframe_map_leaf_size", C.c_float),
                ("downsample_rate", C.c_int), ("point_filter_num", C.c_int),
                ("lidar_min_front", C.c_float), ("lidar_min_back", C.c_float), ("lidar_min_left", C.c_float),
                ("lidar_min_right", C.c_float), ("lidar_max_range", C.c_float), ("lidar_max_intensity", C.c_float),
                ("knn_cell_size", C.c_float), ("knn_phase1_radius", C.c_float), ("profile_kernels", C.c_int), ("s2m_path", C.c_int),
                ("s2m_no_certificate", C.c_int), ("reserved", C.c_int * 3)]


class S2MInfo(C.Structure):
    _fields_ = [("iterations", C.c_int), ("converged", C.c_int), ("n_query", C.c_int), ("n_sel", C.c_int),
                ("is_degenerate", C.c_int), ("tie_queries", C.c_int), ("delta_r_deg", C.c_float),
                ("delta_t_cm", C.c_float), ("JtJ", C.c_double * 36), ("Jtr", C.c_double * 6),
                ("pose_hist", (C.c_float * 6) * LIOGPU_MAX_ITER), ("nsel_hist", C.c_int * LIOGPU_MAX_ITER),
                ("gpu_ms", C.c_float), ("seeded", C.c_int), ("main_kernel_ms", C.c_float),
                ("left_kernel_ms", C.c_float), ("main_kernel_launches", C.c_int), ("left_kernel_launches", C.c_int),
                ("certified", C.c_int), ("leftovers", C.c_int), ("tail_ms", C.c_float), ("kernel_launches", C.c_int),
                ("certified_hist", C.c_int * LIOGPU_MAX_ITER), ("seeded_hist", C.c_int * LIOGPU_MAX_ITER),
                ("leftover_hist", C.c_int * LIOGPU_MAX_ITER), ("main_us_hist", C.c_float * LIOGPU_MAX_ITER),
                ("rest_us_hist", C.c_float * LIOGPU_MAX_ITER)]


class LocalMapParams(C.Structure):
    _fields_ = [("local_map_left", C.c_float), ("local_map_right", C.c_float), ("local_map_front", C.c_float),
                ("local_map_back", C.c_float), ("use_removing_outliers", C.c_int), ("mean_k", C.c_int),
                ("stddev_threshold", C.c_float), ("use_down_sampling", C.c_int),
                ("local_mapping_surf_leaf_size", C.c_float), ("sor_cell_size", C.c_float), ("reserved", C.c_int * 6)]


class LocalMapInfo(C.Structure):
    _fields_ = [("n_concat", C.c_int), ("n_cropped", C.c_int), ("n_after_sor", C.c_int), ("n_out", C.c_int),
                ("leaf_overflow", C.c_int), ("sor_borderline", C.c_int), ("sor_mean", C.c_double),
                ("sor_stddev", C.c_double), ("sor_threshold", C.c_double), ("gpu_ms", C.c_float),
                ("sor_leftover", C.c_int), ("sor_exhaustive", C.c_int), ("reserved", C.c_int * 4)]


class IcpParams(C.Structure):
    _fields_ = [("max_correspondence_distance", C.c_float), ("max_iterations", C.c_int),
                ("transformation_epsilon", C.c_double), ("euclidean_fitness_epsilon", C.c_double),
                ("cell_size", C.c_float), ("reserved", C.c_int * 5)]


class IcpInfo(C.Structure):
    _fields_ = [("iterations", C.c_int), ("converged", C.c_int), ("convergence_state", C.c_int),
                ("n_correspondences", C.c_int), ("fitness_score", C.c_double), ("last_mse", C.c_double),
                ("gpu_ms", C.c_float), ("reserved", C.c_int * 5)]


class LoopIcpResult(C.Structure):
    _fields_ = [("n_source", C.c_int), ("n_target", C.c_int), ("source_overflow", C.c_int), ("target_overflow", C.c_int),
                ("rejected_by_size", C.c_int), ("final_transformation", C.c_float * 16), ("icp", IcpInfo),
                ("reserved", C.c_int * 4)]


class TileInfo(C.Structure):
    _fields_ = [("n_points", C.c_int), ("n_rows", C.c_int), ("n_bins", C.c_int), ("bin_lo", C.c_int), ("bin_hi", C.c_int),
                ("n_tile_points", C.c_int), ("leaf_overflow", C.c_int), ("gpu_ms", C.c_float), ("plan_ms", C.c_float),
                ("reserved", C.c_int * 3)]


LIOGPU_SC_MAX_CANDIDATES = 32


class ScParams(C.Structure):
    _fields_ = [("num_exclude_recent", C.c_int), ("num_candidates_from_tree", C.c_int), ("tree_making_period", C.c_int),
                ("search_ratio", C.c_double), ("sc_dist_thres", C.c_double), ("reserved", C.c_int * 4)]


class ScInfo(C.Structure):
    _fields_ = [("n_stored", C.c_int), ("n_searchable", C.c_int), ("tree_rebuilt", C.c_int), ("n_candidates", C.c_int),
                ("candidates", C.c_int * LIOGPU_SC_MAX_CANDIDATES), ("candidate_key_d2", C.c_float * LIOGPU_SC_MAX_CANDIDATES),
                ("candidate_dist", C.c_double * LIOGPU_SC_MAX_CANDIDATES),
                ("candidate_shift", C.c_int * LIOGPU_SC_MAX_CANDIDATES), ("nn_idx", C.c_int), ("nn_align", C.c_int),
                ("min_dist", C.c_double), ("knn_ties", C.c_int), ("gpu_ms", C.c_float), ("reserved", C.c_int * 4)]


EXPORTS = ["liogpu_abi_version", "liogpu_default_params", "liogpu_create", "liogpu_destroy", "liogpu_last_error",
           "liogpu_host_alloc", "liogpu_host_free", "liogpu_deskew", "liogpu_transform_cloud",
           "liogpu_voxel_downsample", "liogpu_keyframe_put", "liogpu_keyframe_clear", "liogpu_keyframe_count",
           "liogpu_build_local_map", "liogpu_set_local_map", "liogpu_local_map_size", "liogpu_scan2map",
           "liogpu_downsample_scan2map", "liogpu_surf_optimization", "liogpu_last_gpu_ms", "liogpu_launch_count",
           "liogpu_stream", "liogpu_resident_size", "liogpu_default_local_map_params", "liogpu_publish_local_map", "liogpu_merge_keyframes", "liogpu_default_icp_params", "liogpu_icp_align", "liogpu_make_scancontext", "liogpu_extract_nearby",
           "liogpu_scan2map_trace", "liogpu_voxel_tile", "liogpu_upload_scan_async", "liogpu_fetch_result",
           "liogpu_default_sc_params", "liogpu_sc_add", "liogpu_sc_clear", "liogpu_sc_detect_loop", "liogpu_sc_detect_loops",
           "liogpu_detect_loop_distance", "liogpu_loop_closure_icp_batch", "liogpu_merge_keyframes_batch"]

RESIDENT = "resident"   # LIOGPU_DEVICE_RESIDENT: the cloud the context kept in HBM (include/liogpu.h)
UPLOADED = "uploaded"   # LIOGPU_UPLOADED_SCAN: the sweep liogpu_upload_scan_async put on its way

_lib = None


def load_library() -> C.CDLL:
    """Load libliogpu.so (built in-tree by __graft_entry__.build()).  Fails loudly when absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    lib.liogpu_last_error.restype = C.c_char_p
    lib.liogpu_last_error.argtypes = [C.c_void_p]
    lib.liogpu_host_alloc.restype = C.c_void_p
    lib.liogpu_host_alloc.argtypes = [C.c_ulonglong]
    lib.liogpu_host_free.argtypes = [C.c_void_p]
    lib.liogpu_create.argtypes = [C.POINTER(C.c_void_p), C.POINTER(Params)]
    lib.liogpu_destroy.argtypes = [C.c_void_p]
    lib.liogpu_last_gpu_ms.restype = C.c_float
    lib.liogpu_last_gpu_ms.argtypes = [C.c_void_p]
    lib.liogpu_launch_count.restype = C.c_ulonglong
    lib.liogpu_launch_count.argtypes = [C.c_void_p]
    lib.liogpu_stream.restype = C.c_void_p
    lib.liogpu_stream.argtypes = [C.c_void_p]
    lib.liogpu_keyframe_count.argtypes = [C.c_void_p]
    lib.liogpu_local_map_size.argtypes = [C.c_void_p]
    lib.liogpu_resident_size.argtypes = [C.c_void_p]
    lib.liogpu_keyframe_clear.argtypes = [C.c_void_p]
    lib.liogpu_deskew.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                  C.POINTER(C.c_int)]
    lib.liogpu_transform_cloud.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
    lib.liogpu_voxel_downsample.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_int,
                                            C.c_int, C.POINTER(C.c_int)]
    lib.liogpu_keyframe_put.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int]
    lib.liogpu_build_local_map.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_float,
                                           C.POINTER(C.c_int), C.c_void_p, C.c_int, C.c_int]
    lib.liogpu_set_local_map.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    lib.liogpu_merge_keyframes.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_void_p, C.c_int,
                                           C.c_int, C.POINTER(C.c_int)]
    lib.liogpu_merge_keyframes_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_float,
                                                 C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    lib.liogpu_upload_scan_async.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    lib.liogpu_fetch_result.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int)]
    lib.liogpu_voxel_tile.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_int, C.c_int, C.c_void_p,
                                      C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(TileInfo)]
    lib.liogpu_make_scancontext.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_void_p,
                                            C.c_void_p, C.c_void_p]
    lib.liogpu_extract_nearby.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_double,
                                          C.c_float, C.c_float, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
    lib.liogpu_default_sc_params.argtypes = [C.POINTER(ScParams)]
    lib.liogpu_default_sc_params.restype = None
    lib.liogpu_sc_add.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    lib.liogpu_sc_clear.argtypes = [C.c_void_p]
    lib.liogpu_sc_detect_loop.argtypes = [C.c_void_p, C.POINTER(ScParams), C.POINTER(C.c_int), C.POINTER(C.c_float),
                                          C.POINTER(ScInfo)]
    lib.liogpu_sc_detect_loops.argtypes = [C.c_void_p, C.POINTER(ScParams), C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                           C.c_void_p]
    lib.liogpu_detect_loop_distance.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_double,
                                                C.c_float, C.c_float, C.POINTER(C.c_int)]
    lib.liogpu_default_icp_params.argtypes = [C.POINTER(IcpParams), C.c_float]
    lib.liogpu_default_icp_params.restype = None
    lib.liogpu_icp_align.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                     C.POINTER(IcpParams), C.c_void_p, C.POINTER(IcpInfo)]
    lib.liogpu_loop_closure_icp_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                                  C.c_float, C.POINTER(IcpParams), C.c_void_p]
    lib.liogpu_default_local_map_params.argtypes = [C.POINTER(LocalMapParams)]
    lib.liogpu_default_local_map_params.restype = None
    lib.liogpu_publish_local_map.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                             C.POINTER(LocalMapParams), C.c_void_p, C.c_int, C.c_int,
                                             C.POINTER(C.c_int), C.POINTER(LocalMapInfo)]
    lib.liogpu_scan2map.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                    C.POINTER(C.c_int), C.c_int, C.POINTER(S2MInfo)]
    lib.liogpu_scan2map_trace.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                          C.POINTER(C.c_int), C.c_int, C.POINTER(S2MInfo), C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_void_p]
    lib.liogpu_downsample_scan2map.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                               C.POINTER(C.c_int), C.c_int, C.POINTER(S2MInfo), C.POINTER(C.c_int),
                                               C.c_void_p, C.c_int, C.c_int]
    lib.liogpu_surf_optimization.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    _lib = lib
    return lib


def default_params(**over) -> Params:
    p = Params()
    load_library().liogpu_default_params(C.byref(p))
    for k, v in over.items():
        setattr(p, k, v)
    return p


def local_map_params(**over) -> LocalMapParams:
    """utility.h:219-229 defaults, with keyword overrides."""
    p = LocalMapParams()
    load_library().liogpu_default_local_map_params(C.byref(p))
    for k, v in over.items():
        setattr(p, k, v)
    return p


def sc_params(**over) -> ScParams:
    """SCManager's constants (Scancontext.h) with keyword overrides; `num_candidates` is accepted for
    num_candidates_from_tree."""
    p = ScParams()
    load_library().liogpu_default_sc_params(C.byref(p))
    for k, v in over.items():
        setattr(p, "num_candidates_from_tree" if k == "num_candidates" else k, v)
    return p


class LioGpuError(RuntimeError):
    def __init__(self, status: int, msg: str):
        super().__init__(f"liogpu status {status}: {msg}")
        self.status = status


def _cloud_args(cloud):
    """-> (pointer:int, n, stride, keepalive)"""
    if isinstance(cloud, str) and cloud == RESIDENT:
        return 1, 0, 16, None
    if isinstance(cloud, str) and cloud == UPLOADED:
        return 2, 0, 16, None
    if isinstance(cloud, tuple):
        ptr, n, stride = cloud
        return int(ptr), int(n), int(stride), None
    a = cloud
    if a.dtype.fields is not None:
        a = np.ascontiguousarray(a)
        return a.ctypes.data, a.shape[0], a.dtype.itemsize, a
    a = np.ascontiguousarray(a, dtype=np.float32)
    assert a.ndim == 2 and a.shape[1] in (4, 8), "packed clouds are (n,4) float32 (or (n,8) for 32-byte records)"
    return a.ctypes.data, a.shape[0], a.shape[1] * 4, a


def info_to_dict(info: S2MInfo) -> dict:
    it = info.iterations
    return dict(iterations=it, converged=bool(info.converged), n_query=info.n_query, n_sel=info.n_sel,
                is_degenerate=info.is_degenerate, tie_queries=info.tie_queries, delta_r=info.delta_r_deg,
                delta_t=info.delta_t_cm, JtJ=np.array(info.JtJ).reshape(6, 6), Jtr=np.array(info.Jtr),
                pose_hist=np.array(info.pose_hist, dtype=np.float32).reshape(LIOGPU_MAX_ITER, 6)[:it],
                nsel_hist=np.array(info.nsel_hist)[:it], gpu_ms=info.gpu_ms, seeded=info.seeded,
                main_kernel_ms=info.main_kernel_ms, left_kernel_ms=info.left_kernel_ms,
                main_kernel_launches=info.main_kernel_launches, left_kernel_launches=info.left_kernel_launches,
                certified=info.certified, leftovers=info.leftovers, tail_ms=info.tail_ms,
                kernel_launches=info.kernel_launches, certified_hist=np.array(info.certified_hist)[:it],
                seeded_hist=np.array(info.seeded_hist)[:it], leftover_hist=np.array(info.leftover_hist)[:it],
                main_us_hist=np.array(info.main_us_hist)[:it], rest_us_hist=np.array(info.rest_us_hist)[:it])


class LioGpu:
    """One liogpu context (one GPU, one stream)."""

    def __init__(self, params: Params | None = None, **over):
        self.lib = load_library()
        self.params = params if params is not None else default_params(**over)
        h = C.c_void_p()
        st = self.lib.liogpu_create(C.byref(h), C.byref(self.params))
        if st != OK:
            raise LioGpuError(st, "liogpu_create failed (no usable sm_100 CUDA device? there is no CPU fallback)")
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.lib.liogpu_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, st: int) -> int:
        if st < 0:
            raise LioGpuError(st, self.lib.liogpu_last_error(self.h).decode())
        return st

    # --------------------------------------------------------------------------------------------
    def last_gpu_ms(self) -> float:
        return float(self.lib.liogpu_last_gpu_ms(self.h))

    def launch_count(self) -> int:
        return int(self.lib.liogpu_launch_count(self.h))

    def stream(self) -> int:
        return int(self.lib.liogpu_stream(self.h) or 0)

    def deskew(self, scan_xyzirt, time_scan_cur: float, imu_t, rx, ry, rz, deskew_enabled: bool = True,
               keep_on_device: bool = False):
        ptr, n, stride, keep = _cloud_args(scan_xyzirt)
        imu_t = np.ascontiguousarray(imu_t, np.float64); rx = np.ascontiguousarray(rx, np.float64)
        ry = np.ascontiguousarray(ry, np.float64); rz = np.ascontiguousarray(rz, np.float64)
        out = np.empty((max(n, 1), 4), np.float32)
        n_out = C.c_int(0)
        st = self._check(self.lib.liogpu_deskew(self.h, ptr, n, stride, C.c_double(time_scan_cur), imu_t.ctypes.data,
                                                rx.ctypes.data, ry.ctypes.data, rz.ctypes.data, imu_t.shape[0],
                                                int(deskew_enabled), 1 if keep_on_device else out.ctypes.data, 16,
                                                out.shape[0], C.byref(n_out)))
        if keep_on_device:
            return n_out.value, st
        return out[: n_out.value].copy(), st

    def resident_size(self) -> int:
        return int(self.lib.liogpu_resident_size(self.h))

    def transform_cloud(self, cloud, pose6) -> np.ndarray:
        ptr, n, stride, keep = _cloud_args(cloud)
        pose = np.ascontiguousarray(pose6, np.float32)
        out = np.empty((n, 4), np.float32)
        self._check(self.lib.liogpu_transform_cloud(self.h, ptr, n, stride, pose.ctypes.data, out.ctypes.data, 16))
        return out

    def voxel_downsample(self, cloud, leaf: float, out_stride: int = 16, keep_on_device: bool = False):
        ptr, n, stride, keep = _cloud_args(cloud)
        if cloud is RESIDENT or (isinstance(cloud, str) and cloud == RESIDENT):
            n = self.resident_size()
        out = np.empty((max(n, 1), out_stride // 4), np.float32)
        n_out = C.c_int(0)
        st = self._check(self.lib.liogpu_voxel_downsample(self.h, ptr, n, stride, C.c_float(leaf),
                                                          1 if keep_on_device else out.ctypes.data,
                                                          out_stride, out.shape[0], C.byref(n_out)))
        if keep_on_device:
            return n_out.value, st
        return out[: n_out.value].copy(), st

    def keyframe_put(self, kid: int, cloud) -> None:
        ptr, n, stride, keep = _cloud_args(cloud)
        self._check(self.lib.liogpu_keyframe_put(self.h, int(kid), ptr, n, stride))

    def keyframe_clear(self) -> None:
        self._check(self.lib.liogpu_keyframe_clear(self.h))

    def keyframe_count(self) -> int:
        return int(self.lib.liogpu_keyframe_count(self.h))

    def build_local_map(self, ids, poses, leaf: float, fetch: bool = True, cap: int | None = None):
        ids = np.ascontiguousarray(ids, np.int32)
        poses = np.ascontiguousarray(poses, np.float32).reshape(-1, 6)
        assert poses.shape[0] == ids.shape[0]
        n_map = C.c_int(0)
        if fetch:
            out = np.empty((int(cap or 1), 4), np.float32)
            st = self.lib.liogpu_build_local_map(self.h, ids.ctypes.data, poses.ctypes.data, ids.shape[0],
                                                 C.c_float(leaf), C.byref(n_map), out.ctypes.data, 16, out.shape[0])
            if st == E_CAPACITY:  # the map is built and installed: copy it out without rebuilding
                out = np.empty((n_map.value, 4), np.float32)
                st = self.lib.liogpu_fetch_result(self.h, out.ctypes.data, 16, out.shape[0], C.byref(n_map))
            self._check(st)
            return out[: n_map.value].copy(), st
        st = self._check(self.lib.liogpu_build_local_map(self.h, ids.ctypes.data, poses.ctypes.data, ids.shape[0],
                                                         C.c_float(leaf), C.byref(n_map), None, 16, 0))
        return n_map.value, st

    def voxel_tile(self, ids, poses, leaf: float, tile: int, n_tiles: int, out=None):
        """Tile `tile` of `n_tiles` of extractCloud's VoxelGrid (liogpu_voxel_tile).  out: None -> host array returned;
        (device_ptr, capacity) -> written there (packed float4), only the count returned.  -> (cloud | n, info, status)."""
        ids = np.ascontiguousarray(ids, np.int32)
        poses = np.ascontiguousarray(poses, np.float32).reshape(-1, 6)
        info = TileInfo()
        n_out = C.c_int(0)
        if out is None:
            st = self._check(self.lib.liogpu_voxel_tile(self.h, ids.ctypes.data, poses.ctypes.data, ids.shape[0], C.c_float(leaf),
                                                        tile, n_tiles, None, 16, 0, C.byref(n_out), C.byref(info)))
            host = np.empty((max(n_out.value, 1), 4), np.float32)
            st = self._check(self.lib.liogpu_fetch_result(self.h, host.ctypes.data, 16, host.shape[0], C.byref(n_out)))
            res = host[: n_out.value].copy()
        else:
            ptr, cap = out
            st = self._check(self.lib.liogpu_voxel_tile(self.h, ids.ctypes.data, poses.ctypes.data, ids.shape[0], C.c_float(leaf),
                                                        tile, n_tiles, int(ptr), 16, int(cap), C.byref(n_out), C.byref(info)))
            res = n_out.value
        d = {k: getattr(info, k) for k, _ in TileInfo._fields_ if k != "reserved"}
        return res, d, st

    def publish_local_map(self, ids, poses, pose_now, params: "LocalMapParams | None" = None, **over):
        """publishLocalMap (mapOptmization.cpp:2442-2541) -> (cloud (n,4), info dict, status)."""
        prm = params if params is not None else local_map_params(**over)
        ids = np.ascontiguousarray(ids, np.int32)
        poses = np.ascontiguousarray(poses, np.float32).reshape(-1, 6)
        assert poses.shape[0] == ids.shape[0]
        pose_now = np.ascontiguousarray(pose_now, np.float32)
        info = LocalMapInfo()
        n_out = C.c_int(0)
        out = np.empty((1, 4), np.float32)
        st = self.lib.liogpu_publish_local_map(self.h, ids.ctypes.data, poses.ctypes.data, ids.shape[0],
                                               pose_now.ctypes.data, C.byref(prm), out.ctypes.data, 16, out.shape[0],
                                               C.byref(n_out), C.byref(info))
        if st == E_CAPACITY:  # the cloud exists on the device: copy it out without recomputing
            out = np.empty((n_out.value, 4), np.float32)
            st = self.lib.liogpu_fetch_result(self.h, out.ctypes.data, 16, out.shape[0], C.byref(n_out))
        self._check(st)
        d = {k: getattr(info, k) for k, _ in LocalMapInfo._fields_ if k != "reserved"}
        return out[: n_out.value].copy(), d, st

    def merge_keyframes(self, ids, poses, leaf: float = 0.0):
        """saveMapService / publishGlobalMap / loopFindNearKeyframes cloud assembly -> (cloud (n,4), status)."""
        ids = np.ascontiguousarray(ids, np.int32)
        poses = np.ascontiguousarray(poses, np.float32).reshape(-1, 6)
        assert poses.shape[0] == ids.shape[0]
        n_out = C.c_int(0)
        out = np.empty((1, 4), np.float32)
        st = self.lib.liogpu_merge_keyframes(self.h, ids.ctypes.data, poses.ctypes.data, ids.shape[0], C.c_float(leaf),
                                             out.ctypes.data, 16, out.shape[0], C.byref(n_out))
        if st == E_CAPACITY:
            out = np.empty((n_out.value, 4), np.float32)
            st = self.lib.liogpu_fetch_result(self.h, out.ctypes.data, 16, out.shape[0], C.byref(n_out))
        self._check(st)
        return out[: n_out.value].copy(), st

    def merge_keyframes_batch(self, windows, leaf: float = 0.0):
        """merge_keyframes of many windows in one call (liogpu_merge_keyframes_batch); windows = [(ids, poses), ...]
        -> (list of clouds (n_w, 4), overflow flags (n_windows,) bool, status)."""
        ids = [np.ascontiguousarray(i, np.int32).reshape(-1) for i, _ in windows]
        poses = [np.ascontiguousarray(p, np.float32).reshape(-1, 6) for _, p in windows]
        assert all(p.shape[0] == i.shape[0] for i, p in zip(ids, poses))
        n = len(windows)
        win_off = np.zeros(n + 1, np.int32)
        win_off[1:] = np.cumsum([i.shape[0] for i in ids])
        flat_ids = np.concatenate(ids + [np.zeros(1, np.int32)])
        flat_poses = np.concatenate(poses + [np.zeros((1, 6), np.float32)])
        out_off = np.zeros(n + 1, np.int32)
        ovf = np.zeros(max(n, 1), np.int32)
        n_out = C.c_int(0)
        out = np.empty((1, 4), np.float32)
        st = self.lib.liogpu_merge_keyframes_batch(self.h, flat_ids.ctypes.data, flat_poses.ctypes.data,
                                                   win_off.ctypes.data, n, C.c_float(leaf), out.ctypes.data, 16,
                                                   out.shape[0], out_off.ctypes.data, ovf.ctypes.data)
        if st == E_CAPACITY:  # the clouds exist on the device: copy them out without recomputing
            out = np.empty((int(out_off[n]), 4), np.float32)
            st = self.lib.liogpu_fetch_result(self.h, out.ctypes.data, 16, out.shape[0], C.byref(n_out))
        self._check(st)
        return [out[out_off[w]:out_off[w + 1]].copy() for w in range(n)], ovf[:n].astype(bool), st

    def icp_align(self, source, target, history_keyframe_search_radius: float = 10.0, **over):
        """pcl::IterativeClosestPoint as configured at mapOptmization.cpp:1111-1123 -> (T (4,4), info dict)."""
        prm = IcpParams()
        self.lib.liogpu_default_icp_params(C.byref(prm), C.c_float(history_keyframe_search_radius))
        for k, v in over.items():
            setattr(prm, k, v)
        sp, sn, ss, keep_s = _cloud_args(source)
        tp, tn, ts, keep_t = _cloud_args(target)
        T = np.zeros(16, np.float32)
        info = IcpInfo()
        self._check(self.lib.liogpu_icp_align(self.h, sp, sn, ss, tp, tn, ts, C.byref(prm), T.ctypes.data, C.byref(info)))
        d = {k: getattr(info, k) for k, _ in IcpInfo._fields_ if k != "reserved"}
        return T.reshape(4, 4), d

    def loop_closure_icp_batch(self, key_cur, key_pre, key_pose6s, search_num: int = 25, icp_leaf: float = 0.3,
                               history_keyframe_search_radius: float = 10.0, **over):
        """loopFindNearKeyframes for both ends of every pair + the ICP of mapOptmization.cpp:1104-1123, many pairs in one
        call (liogpu_loop_closure_icp_batch) -> (T (n, 4, 4) float32, list of per-pair dicts: the submap sizes and
        overflow flags, rejected_by_size and the icp_align info keys)."""
        prm = IcpParams()
        self.lib.liogpu_default_icp_params(C.byref(prm), C.c_float(history_keyframe_search_radius))
        for k, v in over.items():
            setattr(prm, k, v)
        kc = np.ascontiguousarray(key_cur, np.int32).reshape(-1)
        kp = np.ascontiguousarray(key_pre, np.int32).reshape(-1)
        assert kc.shape == kp.shape
        poses = np.ascontiguousarray(key_pose6s, np.float32).reshape(-1, 6)
        n = kc.shape[0]
        res = (LoopIcpResult * max(n, 1))()
        self._check(self.lib.liogpu_loop_closure_icp_batch(self.h, kc.ctypes.data, kp.ctypes.data, n, poses.ctypes.data,
                                                           poses.shape[0], int(search_num), C.c_float(icp_leaf),
                                                           C.byref(prm), res))
        T = np.array([np.ctypeslib.as_array(r.final_transformation) for r in res[:n]], np.float32).reshape(n, 4, 4)
        out = []
        for r in res[:n]:
            d = {k: getattr(r, k) for k in ("n_source", "n_target", "source_overflow", "target_overflow", "rejected_by_size")}
            d.update({k: getattr(r.icp, k) for k, _ in IcpInfo._fields_ if k != "reserved"})
            out.append(d)
        return T, out

    def make_scancontext(self, cloud, lidar_height: float = 2.0, max_radius: float = 80.0):
        """SCManager::makeScancontext + keys (Scancontext.cpp:151-225) -> (desc (20,60), ringkey, sectorkey), f64."""
        ptr, n, stride, keep = _cloud_args(cloud)
        desc = np.zeros((20, 60), np.float64)
        rk = np.zeros(20, np.float64)
        sk = np.zeros(60, np.float64)
        self._check(self.lib.liogpu_make_scancontext(self.h, ptr, n, stride, lidar_height, max_radius, desc.ctypes.data,
                                                     rk.ctypes.data, sk.ctypes.data))
        return desc, rk, sk

    def extract_nearby(self, key3d, key_time, time_cur: float, radius: float = 50.0, density: float = 2.0):
        """extractNearby + extractCloud's guard (mapOptmization.cpp:1519-1565) -> keyframe indices, concatenation order."""
        ptr, n, stride, keep = _cloud_args(key3d)
        key_time = np.ascontiguousarray(key_time, np.float64)
        assert key_time.shape[0] == n
        ids = np.zeros(max(2 * n, 1), np.int32)
        n_ids = C.c_int(0)
        st = self._check(self.lib.liogpu_extract_nearby(self.h, ptr, n, stride, key_time.ctypes.data, 8, C.c_double(time_cur),
                                                        C.c_float(radius), C.c_float(density), ids.ctypes.data, ids.shape[0],
                                                        C.byref(n_ids)))
        return ids[: n_ids.value].copy(), st

    def sc_add(self, descs) -> None:
        """makeAndSaveScancontextAndKeys for descriptors as make_scancontext returns them: (20, 60) or (n, 20, 60) f64."""
        d = np.ascontiguousarray(descs, np.float64).reshape(-1, 1200)
        self._check(self.lib.liogpu_sc_add(self.h, d.ctypes.data, d.shape[0]))

    def sc_clear(self) -> None:
        self._check(self.lib.liogpu_sc_clear(self.h))

    def sc_detect_loop(self, params: "ScParams | None" = None, **over):
        """SCManager::detectLoopClosureID on the newest stored descriptor -> (loop_id, yaw_diff_rad, info dict)."""
        prm = params if params is not None else sc_params(**over)
        loop_id = C.c_int(0)
        yaw = C.c_float(0)
        info = ScInfo()
        self._check(self.lib.liogpu_sc_detect_loop(self.h, C.byref(prm), C.byref(loop_id), C.byref(yaw), C.byref(info)))
        n = info.n_candidates
        d = dict(n_stored=info.n_stored, n_searchable=info.n_searchable, tree_rebuilt=info.tree_rebuilt, n_candidates=n,
                 candidates=np.array(info.candidates[:n], np.int32),
                 candidate_key_d2=np.array(info.candidate_key_d2[:n], np.float32),
                 candidate_dist=np.array(info.candidate_dist[:n], np.float64),
                 candidate_shift=np.array(info.candidate_shift[:n], np.int32), nn_idx=info.nn_idx, nn_align=info.nn_align,
                 min_dist=info.min_dist, knn_ties=info.knn_ties, gpu_ms=info.gpu_ms)
        return loop_id.value, np.float32(yaw.value), d

    def sc_detect_loops(self, store_sizes, params: "ScParams | None" = None, **over):
        """detectLoopClosureID of a fresh SCManager at each store size -> (loop_ids, yaw_diff_rad, min_dist)."""
        prm = params if params is not None else sc_params(**over)
        sizes = np.ascontiguousarray(store_sizes, np.int32)
        n = sizes.shape[0]
        ids = np.zeros(max(n, 1), np.int32)
        yaw = np.zeros(max(n, 1), np.float32)
        md = np.zeros(max(n, 1), np.float64)
        self._check(self.lib.liogpu_sc_detect_loops(self.h, C.byref(prm), sizes.ctypes.data, n, ids.ctypes.data,
                                                    yaw.ctypes.data, md.ctypes.data))
        return ids[:n].copy(), yaw[:n].copy(), md[:n].copy()

    def detect_loop_distance(self, key3d, key_time, time_cur: float, radius: float = 10.0, time_diff: float = 30.0) -> int:
        """detectLoopClosureDistance (mapOptmization.cpp ~1271-1300) without the loopIndexContainer check -> id or -1."""
        ptr, n, stride, keep = _cloud_args(key3d)
        key_time = np.ascontiguousarray(key_time, np.float64)
        assert key_time.shape[0] == n
        out = C.c_int(-1)
        self._check(self.lib.liogpu_detect_loop_distance(self.h, ptr, n, stride, key_time.ctypes.data, 8, C.c_double(time_cur),
                                                         C.c_float(radius), C.c_float(time_diff), C.byref(out)))
        return out.value

    def upload_scan_async(self, cloud) -> None:
        """liogpu_upload_scan_async: the buffer must stay alive until the call that consumes UPLOADED returns."""
        ptr, n, stride, keep = _cloud_args(cloud)
        self._check(self.lib.liogpu_upload_scan_async(self.h, ptr, n, stride))

    def set_local_map(self, cloud) -> None:
        ptr, n, stride, keep = _cloud_args(cloud)
        self._check(self.lib.liogpu_set_local_map(self.h, ptr, n, stride))

    def local_map_size(self) -> int:
        return int(self.lib.liogpu_local_map_size(self.h))

    def scan2map(self, scan_ds, pose6, matP=None, degenerate: int = 0, max_iter: int = 30, raw_info: bool = False):
        ptr, n, stride, keep = _cloud_args(scan_ds)
        pose = np.array(pose6, dtype=np.float32)
        P = np.zeros(36, np.float32) if matP is None else np.array(matP, dtype=np.float32).reshape(36)
        deg = C.c_int(int(degenerate))
        info = S2MInfo()
        st = self._check(self.lib.liogpu_scan2map(self.h, ptr, n, stride, pose.ctypes.data, P.ctypes.data,
                                                  C.byref(deg), max_iter, C.byref(info)))
        d = info if raw_info else info_to_dict(info)
        if not raw_info:
            d["status"] = st
            d["is_degenerate"] = deg.value
        return pose, P.reshape(6, 6), d

    def scan2map_trace(self, scan_ds, pose6, matP=None, degenerate: int = 0, max_iter: int = 30):
        """liogpu_scan2map plus the per-point results of its last executed iteration -> (pose, matP, info, per-point dict)."""
        ptr, n, stride, keep = _cloud_args(scan_ds)
        if isinstance(scan_ds, str) and scan_ds == RESIDENT:
            n = self.resident_size()
        pose = np.array(pose6, dtype=np.float32)
        P = np.zeros(36, np.float32) if matP is None else np.array(matP, dtype=np.float32).reshape(36)
        deg = C.c_int(int(degenerate))
        info = S2MInfo()
        idx = np.empty((n, 5), np.int32); d2 = np.empty((n, 5), np.float32)
        coeff = np.empty((n, 4), np.float32); flag = np.empty(n, np.uint8); tie = np.empty(n, np.uint8)
        st = self._check(self.lib.liogpu_scan2map_trace(self.h, ptr, n, stride, pose.ctypes.data, P.ctypes.data,
                                                        C.byref(deg), max_iter, C.byref(info), idx.ctypes.data,
                                                        d2.ctypes.data, coeff.ctypes.data, flag.ctypes.data,
                                                        tie.ctypes.data))
        d = info_to_dict(info)
        d["status"] = st
        d["is_degenerate"] = deg.value
        return pose, P.reshape(6, 6), d, dict(nn_idx=idx, nn_d2=d2, coeff=coeff, flag=flag, tie=tie)

    def downsample_scan2map(self, scan, pose6, matP=None, degenerate: int = 0, max_iter: int = 30, fetch_ds=False,
                            keep_ds_on_device: bool = False):
        ptr, n, stride, keep = _cloud_args(scan)
        if isinstance(scan, str) and scan == RESIDENT:
            n = self.resident_size()
        pose = np.array(pose6, dtype=np.float32)
        P = np.zeros(36, np.float32) if matP is None else np.array(matP, dtype=np.float32).reshape(36)
        deg = C.c_int(int(degenerate))
        info = S2MInfo()
        n_ds = C.c_int(0)
        out = np.empty((max(n, 1), 4), np.float32) if fetch_ds else None
        st = self._check(self.lib.liogpu_downsample_scan2map(
            self.h, ptr, n, stride, pose.ctypes.data, P.ctypes.data, C.byref(deg), max_iter, C.byref(info),
            C.byref(n_ds), 1 if keep_ds_on_device else (out.ctypes.data if fetch_ds else None), 16,
            out.shape[0] if fetch_ds else 0))
        d = info_to_dict(info)
        d["status"] = st
        d["is_degenerate"] = deg.value
        d["n_ds"] = n_ds.value
        if fetch_ds:
            d["scan_ds"] = out[: n_ds.value].copy()
        return pose, P.reshape(6, 6), d

    def surf_optimization(self, scan_ds, pose6=None, T12=None):
        ptr, n, stride, keep = _cloud_args(scan_ds)
        if isinstance(scan_ds, str) and scan_ds == RESIDENT:
            n = self.resident_size()
        idx = np.empty((n, 5), np.int32); d2 = np.empty((n, 5), np.float32)
        coeff = np.empty((n, 4), np.float32); flag = np.empty(n, np.uint8); tie = np.empty(n, np.uint8)
        pose = np.ascontiguousarray(pose6, np.float32) if pose6 is not None else None
        T = np.ascontiguousarray(T12, np.float32) if T12 is not None else None
        self._check(self.lib.liogpu_surf_optimization(
            self.h, ptr, n, stride, pose.ctypes.data if pose is not None else None,
            T.ctypes.data if T is not None else None, idx.ctypes.data, d2.ctypes.data, coeff.ctypes.data,
            flag.ctypes.data, tie.ctypes.data))
        return dict(nn_idx=idx, nn_d2=d2, coeff=coeff, flag=flag, tie=tie)
