"""ctypes binding of libliorf_host.so (lio_slam_b200/host/liorf_replay.h): one call replays one sequence of raw sweeps
through the host mirror of the reference's per-scan path (cloudHandler -> laserCloudInfoHandler,
imageProjection.cpp:206 / mapOptmization.cpp:432-506) on one GPU.  ctypes releases the GIL during the call, so
several sequences can be replayed concurrently from Python threads (batch offline mapping, BASELINE configs[4])."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import liogpu

_HERE = os.path.dirname(os.path.abspath(__file__))
HOST_LIB_PATH = os.path.join(_HERE, "libliorf_host.so")


class Sweep(C.Structure):
    _fields_ = [("raw", C.c_void_p), ("n_raw", C.c_int), ("time_scan_cur", C.c_double), ("guess", C.c_float * 6),
                ("imu", C.c_void_p), ("n_imu", C.c_int)]


class ReplayOptions(C.Structure):
    _fields_ = [("select_key_poses_on_device", C.c_int), ("publish_local_map", C.c_int), ("keyframe_dist", C.c_float),
                ("keyframe_angle", C.c_float), ("search_radius", C.c_float), ("density", C.c_float),
                ("loop_detection_every", C.c_int), ("reserved", C.c_int * 5)]


class ReplayStats(C.Structure):
    _fields_ = [("scans", C.c_int), ("registered", C.c_int), ("keyframes", C.c_int), ("map_rebuilds", C.c_int),
                ("lm_iterations", C.c_int), ("map_points_last", C.c_int), ("wall_ms", C.c_double),
                ("deskew_ms", C.c_double), ("nearby_ms", C.c_double), ("register_ms", C.c_double),
                ("keyframe_ms", C.c_double), ("loop_gpu_ms", C.c_double), ("h2d_bytes", C.c_longlong),
                ("d2h_bytes", C.c_longlong), ("gpu_launches", C.c_ulonglong), ("loops_sc", C.c_int), ("loops_rs", C.c_int),
                ("reserved", C.c_int * 2)]


_lib = None


def load_host_library() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    liogpu.load_library()
    if not os.path.exists(HOST_LIB_PATH):
        raise RuntimeError(f"{HOST_LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'`")
    lib = C.CDLL(HOST_LIB_PATH)
    lib.liorf_replay_sequence.argtypes = [C.POINTER(liogpu.Params), C.POINTER(ReplayOptions), C.POINTER(Sweep), C.c_int,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(ReplayStats), C.c_char_p, C.c_int]
    lib.liorf_replay_sequence.restype = C.c_int
    lib.liorf_worker_create.argtypes = [C.POINTER(liogpu.Params), C.c_char_p, C.c_int]
    lib.liorf_worker_create.restype = C.c_void_p
    lib.liorf_worker_destroy.argtypes = [C.c_void_p]
    lib.liorf_worker_replay.argtypes = [C.c_void_p, C.POINTER(ReplayOptions), C.POINTER(Sweep), C.c_int, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.POINTER(ReplayStats), C.c_char_p, C.c_int]
    lib.liorf_worker_replay.restype = C.c_int
    _lib = lib
    return lib


def kitti_params(device: int = 0, **over) -> liogpu.Params:
    """The hot-path parameters of config/kitti.yaml (64-beam, lines 27-32, 56, 71)."""
    kw = dict(device=device, n_scan=64, horizon_scan=1800, downsample_rate=2, point_filter_num=5,
              mapping_surf_leaf_size=0.4, surrounding_keyframe_map_leaf_size=0.5,
              lidar_min_front=1.0, lidar_min_back=1.0, lidar_min_left=1.0, lidar_min_right=1.0, lidar_max_range=1000.0)
    kw.update(over)
    return liogpu.default_params(**kw)


class Worker:
    """liorf_worker: one liogpu context reused for sequence after sequence (one per host thread)."""

    def __init__(self, params: liogpu.Params):
        self.lib = load_host_library()
        err = C.create_string_buffer(256)
        self.h = self.lib.liorf_worker_create(C.byref(params), err, 256)
        if not self.h:
            raise liogpu.LioGpuError(liogpu.E_CUDA, err.value.decode() or "liorf_worker_create failed")

    def replay(self, seq: dict, first: int = 0, count: int | None = None, **options):
        return replay_sequence(None, seq, first, count, _worker=self, **options)

    def close(self):
        if getattr(self, "h", None):
            self.lib.liorf_worker_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def replay_sequence(params, seq: dict, first: int = 0, count: int | None = None, _worker: "Worker | None" = None, **options):
    """seq: the dict of synth_torch.make_sequence (raw pinned tensor or numpy uint8/float32 array of 32-byte records,
    offs, times, guesses, imu).  -> (poses (n,6) f32, iterations (n,), n_ds (n,), stats dict)"""
    lib = load_host_library()
    raw = seq["raw"]
    base = raw.data_ptr() if hasattr(raw, "data_ptr") else raw.ctypes.data
    offs = seq["offs"]
    n_all = len(offs) - 1
    n = n_all - first if count is None else count
    sweeps = (Sweep * n)()
    keep = []
    for k in range(n):
        s = first + k
        sw = sweeps[k]
        sw.raw = base + int(offs[s]) * 32
        sw.n_raw = int(offs[s + 1] - offs[s])
        sw.time_scan_cur = float(seq["times"][s])
        for q in range(6):
            sw.guess[q] = float(seq["guesses"][s][q])
        imu = np.ascontiguousarray(seq["imu"][s], np.float64)
        keep.append(imu)
        sw.imu = imu.ctypes.data
        sw.n_imu = imu.shape[1]
    opt = ReplayOptions()
    for k, v in options.items():
        setattr(opt, k, v)
    poses = np.zeros((n, 6), np.float32)
    iters = np.zeros(n, np.int32)
    nds = np.zeros(n, np.int32)
    stats = ReplayStats()
    err = C.create_string_buffer(512)
    if _worker is not None:
        rc = lib.liorf_worker_replay(_worker.h, C.byref(opt), sweeps, n, poses.ctypes.data, iters.ctypes.data,
                                     nds.ctypes.data, C.byref(stats), err, 512)
    else:
        rc = lib.liorf_replay_sequence(C.byref(params), C.byref(opt), sweeps, n, poses.ctypes.data, iters.ctypes.data,
                                       nds.ctypes.data, C.byref(stats), err, 512)
    if rc != 0:
        raise liogpu.LioGpuError(rc, err.value.decode() or "liorf_replay_sequence failed")
    d = {k: getattr(stats, k) for k, _ in ReplayStats._fields_ if k != "reserved"}
    return poses, iters, nds, d
