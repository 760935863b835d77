"""ctypes binding of the CPU oracle's loop-closure detection (oracle/libloop_oracle.so, built from
liorf_oracle_loop.cpp / liorf_oracle_loop.h on first use or by __graft_entry__.build()).

TEST INFRASTRUCTURE — imported only by tests/ and tests/perf/.  PARITY UNPINNED (see oracle/liorf_oracle_core.h)."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(_HERE, "libloop_oracle.so")
_SOURCES = ("liorf_oracle_loop.cpp", "liorf_oracle_loop.h", "liorf_oracle_core.h")
# the flags of oracle/Makefile: x86-64 baseline, no FMA contraction, OpenMP
CXXFLAGS = ["-O2", "-std=c++14", "-fPIC", "-shared", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-Wall",
            "-Wno-unused-function"]

# SCManager's constants (Scancontext.h of SC-LIO-SAM, which liorf vendors)
SC_DEFAULTS = dict(num_exclude_recent=30, num_candidates=3, tree_making_period=30, search_ratio=0.1, sc_dist_thres=0.2)


class ScParams(C.Structure):
    _fields_ = [("num_exclude_recent", C.c_int), ("num_candidates", C.c_int), ("tree_making_period", C.c_int),
                ("search_ratio", C.c_double), ("sc_dist_thres", C.c_double)]


class ScResult(C.Structure):
    _fields_ = [("loop_id", C.c_int), ("yaw", C.c_float), ("n_stored", C.c_int), ("n_searchable", C.c_int),
                ("tree_rebuilt", C.c_int), ("n_candidates", C.c_int), ("nn_idx", C.c_int), ("nn_align", C.c_int),
                ("knn_ties", C.c_int), ("min_dist", C.c_double), ("cand", C.c_int * 32), ("cand_d2", C.c_float * 32),
                ("cand_dist", C.c_double * 32), ("cand_shift", C.c_int * 32)]


def build(force: bool = False) -> None:
    """Compile libloop_oracle.so when it is missing or older than its sources."""
    if not force and os.path.exists(LIB):
        t = os.path.getmtime(LIB)
        if all(os.path.getmtime(os.path.join(_HERE, s)) <= t for s in _SOURCES):
            return
    subprocess.check_call(["/usr/bin/g++", *CXXFLAGS, "-o", LIB, os.path.join(_HERE, "liorf_oracle_loop.cpp")])


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


class LoopOracle:
    """SCManager::detectLoopClosureID and detectLoopClosureDistance restated on the CPU."""

    def __init__(self):
        build()
        self.lib = C.CDLL(LIB)
        self.lib.loop_detect_loop_distance.restype = C.c_int

    def max_threads(self) -> int:
        return int(self.lib.loop_omp_max_threads())

    def sc_detect_loops(self, descs, store_sizes, threads: int = 1, **params):
        """detectLoopClosureID of a fresh SCManager, call j after the store grew to store_sizes[j] descriptors
        (descs: (n, 20, 60) f64) -> list of dicts, one per call (loop_id, yaw, nn_idx, nn_align, min_dist, n_searchable,
        tree_rebuilt, candidates with their ring-key distances, distances and shifts, ...)."""
        descs = np.ascontiguousarray(descs, np.float64).reshape(-1, 1200)
        sizes = np.ascontiguousarray(store_sizes, np.int32)
        p = dict(SC_DEFAULTS)
        p.update(params)
        prm = ScParams(**p)
        res = (ScResult * max(len(sizes), 1))()
        st = self.lib.loop_sc_detect_loops(_p(descs, C.c_double), C.c_int(descs.shape[0]), _p(sizes, C.c_int),
                                           C.c_int(len(sizes)), C.byref(prm), C.c_int(threads), res)
        if st != 0:
            raise ValueError("store_sizes must be non-decreasing and <= the number of descriptors")
        out = []
        for j in range(len(sizes)):
            r = res[j]
            n = r.n_candidates
            out.append(dict(loop_id=r.loop_id, yaw=np.float32(r.yaw), n_stored=r.n_stored, n_searchable=r.n_searchable,
                            tree_rebuilt=r.tree_rebuilt, n_candidates=n, nn_idx=r.nn_idx, nn_align=r.nn_align,
                            knn_ties=r.knn_ties, min_dist=r.min_dist, candidates=np.array(r.cand[:n], np.int32),
                            candidate_key_d2=np.array(r.cand_d2[:n], np.float32),
                            candidate_dist=np.array(r.cand_dist[:n], np.float64),
                            candidate_shift=np.array(r.cand_shift[:n], np.int32)))
        return out

    def detect_loop_distance(self, key3d, key_time, time_cur, radius=10.0, time_diff=30.0) -> int:
        """detectLoopClosureDistance (MO ~1271-1300) without the loopIndexContainer check -> loop_key_pre or -1."""
        key3d = np.ascontiguousarray(key3d, dtype=np.float32)
        assert key3d.ndim == 2 and key3d.shape[1] == 4
        key_time = np.ascontiguousarray(key_time, dtype=np.float64)
        return int(self.lib.loop_detect_loop_distance(_p(key3d, C.c_float), _p(key_time, C.c_double),
                                                      C.c_int(key3d.shape[0]), C.c_double(time_cur), C.c_float(radius),
                                                      C.c_float(time_diff)))
