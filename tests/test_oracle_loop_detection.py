"""The oracle's restatement of loop-closure detection, checked on the CPU:
  * SCManager::detectLoopClosureID (include/Scancontext.cpp) against a small numpy restatement, call by call (counter,
    tree snapshot, ring-key kNN, sector-key alignment, search window, column-wise cosine distance);
  * detectLoopClosureDistance (mapOptmization.cpp ~1271-1300) against a numpy restatement, edges included;
  * the ctypes mirrors of the new structs of include/liogpu.h against a C compiler's layout."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from lio_slam_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NS = 60


# ---- numpy restatement ---------------------------------------------------------------------------------------------
def seqsum(x):
    """left-to-right f64 sum (np.sum is pairwise)"""
    return np.cumsum(x)[-1] if len(x) else 0.0


def redux4(x):
    """Eigen 3.3.7 linear-vectorised sum for SSE2 doubles: lanes j mod 4, (s0 + s2) + (s1 + s3)"""
    s = [seqsum(x[k::4]) for k in range(4)]
    return (s[0] + s[2]) + (s[1] + s[3])


def l2_adaptor(q, k):
    """nanoflann L2_Adaptor<float> over 20 dims: result += ((d0*d0 + d1*d1) + d2*d2) + d3*d3 per group, f32"""
    d = (q[None, :] - k).astype(np.float32)
    r = np.zeros(k.shape[0], np.float32)
    for g in range(0, 20, 4):
        r = r + (((d[:, g] * d[:, g] + d[:, g + 1] * d[:, g + 1]) + d[:, g + 2] * d[:, g + 2]) + d[:, g + 3] * d[:, g + 3])
    return r


class NumpySC:
    def __init__(self):
        self.descs, self.rkeys, self.vkeys, self.norms = [], [], [], []
        self.counter = 0
        self.snap = 0

    def add(self, desc):
        desc = np.asarray(desc, np.float64).reshape(20, NS)
        self.descs.append(desc)
        self.rkeys.append(np.array([seqsum(desc[r]) / NS for r in range(20)]).astype(np.float32))
        self.vkeys.append(np.array([seqsum(desc[:, c]) / 20 for c in range(NS)]))
        self.norms.append(np.array([np.sqrt(redux4(desc[:, c] * desc[:, c])) for c in range(NS)]))

    def distance(self, q, i, ratio):
        vq, vc = self.vkeys[q], self.vkeys[i]
        align, best = 0, 1e7
        for s in range(NS):
            d = vq - np.roll(vc, s)                        # circshift: column c -> (c + s) % 60
            n = np.sqrt(redux4(d * d))
            if n < best:
                align, best = s, n
        R = int(np.round(0.5 * ratio * NS))
        if 0.5 * ratio * NS % 1 == 0.5:                    # C's round: half away from zero
            R = int(np.floor(0.5 * ratio * NS + 0.5))
        space = sorted([align] + [x for ii in range(1, R + 1) for x in ((align + ii) % NS, (align - ii) % NS)])
        dq, dc, nq, nc = self.descs[q], self.descs[i], self.norms[q], self.norms[i]
        shift, dist = 0, 1e7
        for s in space:
            tot, n_eff = 0.0, 0
            for c in range(NS):
                cc = (c - s) % NS
                if nq[c] == 0 or nc[cc] == 0:
                    continue
                tot = tot + redux4(dq[:, c] * dc[:, cc]) / (nq[c] * nc[cc])
                n_eff += 1
            with np.errstate(invalid="ignore", divide="ignore"):
                d = 1.0 - (np.float64(tot) / np.float64(n_eff))
            if d < dist:
                shift, dist = s, d
        return dist, shift

    def detect(self, ne, k, period, ratio, thres):
        size = len(self.descs)
        if size < ne + 1:
            return dict(loop_id=-1, yaw=np.float32(0), rebuilt=0, m=self.snap, candidates=[], nn_idx=-1, min_dist=1e7)
        rebuilt = int(self.counter % period == 0)
        if rebuilt:
            self.snap = size - ne
        self.counter += 1
        q = size - 1
        d2 = l2_adaptor(self.rkeys[q], np.array(self.rkeys[: self.snap]))
        order = np.lexsort((np.arange(self.snap), d2))[: min(k, self.snap)]
        min_dist, nn_align, nn_idx = 1e7, 0, 0
        dists, shifts = [], []
        for i in order:
            dd, ss = self.distance(q, int(i), ratio)
            dists.append(dd)
            shifts.append(ss)
            if dd < min_dist:
                min_dist, nn_align, nn_idx = dd, ss, int(i)
        deg = np.float32(nn_align * (360.0 / NS))
        yaw = np.float32(np.float64(deg) * np.pi / 180.0)
        return dict(loop_id=nn_idx if min_dist < thres else -1, yaw=yaw, rebuilt=rebuilt, m=self.snap,
                    candidates=[int(i) for i in order], key_d2=d2[order], dists=dists, shifts=shifts, nn_idx=nn_idx,
                    nn_align=nn_align, min_dist=min_dist)


def compare_with_numpy(loop_oracle, descs, sizes, **prm):
    res = loop_oracle.sc_detect_loops(descs, sizes, **prm)
    ref = NumpySC()
    p = dict(num_exclude_recent=30, num_candidates=3, tree_making_period=30, search_ratio=0.1, sc_dist_thres=0.2)
    p.update(prm)
    for r, size in zip(res, sizes):
        while len(ref.descs) < size:
            ref.add(descs[len(ref.descs)])
        want = ref.detect(p["num_exclude_recent"], p["num_candidates"], p["tree_making_period"], p["search_ratio"],
                          p["sc_dist_thres"])
        assert r["loop_id"] == want["loop_id"] and r["yaw"] == want["yaw"], (size, r, want)
        assert r["tree_rebuilt"] == want["rebuilt"] and r["n_searchable"] == want["m"], size
        assert list(r["candidates"]) == want["candidates"], size
        assert r["nn_idx"] == want["nn_idx"], size
        assert np.float64(r["min_dist"]).view(np.uint64) == np.float64(want["min_dist"]).view(np.uint64), size
        if want["candidates"]:
            assert np.array_equal(r["candidate_key_d2"].view(np.uint32), want["key_d2"].view(np.uint32)), size
            assert np.array_equal(r["candidate_dist"].view(np.uint64), np.array(want["dists"]).view(np.uint64)), size
            assert list(r["candidate_shift"]) == want["shifts"], size
    return res


@pytest.fixture(scope="module")
def loop_oracle():
    """the oracle's restatement of loop-closure detection (oracle/liorf_oracle_loop.h)"""
    from oracle.loop_oracle import LoopOracle
    return LoopOracle()


# ---- descriptors ----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def sweep_descs(oracle, world):
    """Scan Context descriptors of 16-beam sweeps every 1.2 m along the 8 m circle (a lap and a bit)"""
    out = []
    for j in range(48):
        scan = synth.to_packed(synth.make_scan(world, synth.path_pose(1.2 * j), 16, seed=300 + j, cols=600))
        out.append(oracle.make_scancontext(scan)[0])
    return np.array(out)


def shifted(desc, s):
    return np.roll(desc, s, axis=1)


@pytest.mark.parametrize("prm", [dict(num_exclude_recent=5, num_candidates=3, tree_making_period=7),
                                 dict(num_exclude_recent=0, num_candidates=10, tree_making_period=1, search_ratio=0.5),
                                 dict(num_exclude_recent=12, num_candidates=1, tree_making_period=3, search_ratio=0.05,
                                      sc_dist_thres=0.35)])
def test_detect_loop_id_matches_numpy_restatement(loop_oracle, sweep_descs, prm):
    res = compare_with_numpy(loop_oracle, sweep_descs, np.arange(1, sweep_descs.shape[0] + 1), **prm)
    assert any(r["n_candidates"] > 0 for r in res)


def test_detect_loop_id_irregular_sizes(loop_oracle, sweep_descs):
    sizes = [1, 3, 3, 9, 10, 10, 10, 17, 30, 31, 40, 48, 48]
    compare_with_numpy(loop_oracle, sweep_descs, sizes, num_exclude_recent=8, num_candidates=4, tree_making_period=2)


def test_circshifted_copy_has_zero_distance_at_the_planted_shift(loop_oracle, sweep_descs):
    base = sweep_descs[5]
    for s in (0, 1, 17, 59):
        descs = np.array([sweep_descs[0], base, sweep_descs[20], shifted(base, s)])
        res = compare_with_numpy(loop_oracle, descs, [4], num_exclude_recent=1, num_candidates=3, tree_making_period=1,
                                 search_ratio=0.1)
        r = res[0]
        assert r["loop_id"] == 1 and r["min_dist"] < 1e-12 and r["nn_align"] == s, (s, r)
        assert r["yaw"] == np.float32(np.float64(np.float32(s * 6.0)) * np.pi / 180.0)


def test_all_zero_and_empty_column_descriptors(loop_oracle, sweep_descs):
    z = np.zeros((20, NS))
    # all-zero: every column pair is skipped -> NaN for every shift, the distances stay 1e7, no loop, nn_idx 0, shift 0
    r = compare_with_numpy(loop_oracle, np.array([z, z, z]), [3], num_exclude_recent=1, num_candidates=2, tree_making_period=1)[0]
    assert r["loop_id"] == -1 and r["min_dist"] == 1e7 and r["nn_idx"] == 0 and r["nn_align"] == 0
    assert (r["candidate_dist"] == 1e7).all()                 # distanceBtnScanContext keeps its initial 1e7
    e = sweep_descs[7].copy()
    e[:, 10:25] = 0.0
    e[:, 40] = 0.0
    descs = np.array([sweep_descs[3], e, sweep_descs[9], z, shifted(e, 3), sweep_descs[7]])
    compare_with_numpy(loop_oracle, descs, [2, 3, 4, 5, 6], num_exclude_recent=1, num_candidates=4, tree_making_period=1,
                       search_ratio=0.2)


def test_duplicates_give_logged_ties_and_the_lower_index(loop_oracle, sweep_descs):
    d = sweep_descs[11]
    descs = np.array([sweep_descs[0], d, sweep_descs[30], d, d, sweep_descs[2], d])
    r = compare_with_numpy(loop_oracle, descs, [7], num_exclude_recent=1, num_candidates=2, tree_making_period=1)[0]
    assert list(r["candidates"]) == [1, 3] and r["knn_ties"] >= 2 and r["loop_id"] == 1 and r["min_dist"] == 0.0


def test_early_return_does_not_advance_the_counter(loop_oracle, sweep_descs):
    res = loop_oracle.sc_detect_loops(sweep_descs, [1, 2, 3, 4, 5, 6, 7], num_exclude_recent=3, tree_making_period=3)
    assert [r["loop_id"] for r in res[:3]] == [-1, -1, -1] and [r["tree_rebuilt"] for r in res] == [0, 0, 0, 1, 0, 0, 1]
    assert [r["n_searchable"] for r in res[3:]] == [1, 1, 1, 4]
    with pytest.raises(ValueError):
        loop_oracle.sc_detect_loops(sweep_descs, [3, 2])


# ---- radius detector ------------------------------------------------------------------------------------------------
def numpy_loop_distance(key3d, key_time, t_cur, radius, time_diff):
    k = np.asarray(key3d, np.float32)
    d = k[:, :3] - k[-1, :3]
    d2 = ((d[:, 0] * d[:, 0]) + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
    ok = (d2 < np.float32(np.float64(radius) * np.float64(radius))) & \
        (np.abs(np.asarray(key_time, np.float64) - t_cur) > np.float64(np.float32(time_diff)))
    idx = np.nonzero(ok)[0]
    if idx.size == 0:
        return -1
    best = int(idx[np.lexsort((idx, d2[idx]))[0]])
    return -1 if best == k.shape[0] - 1 else best


def test_detect_loop_distance_matches_numpy(loop_oracle):
    rng = np.random.default_rng(8)
    for trial in range(30):
        n = int(rng.integers(1, 400))
        key = np.c_[rng.uniform(-20, 20, (n, 2)), rng.uniform(-1, 1, (n, 1)), np.arange(n)].astype(np.float32)
        key[rng.random(n) < 0.2, :3] = key[-1, :3] + np.float32(rng.choice([0.0, 3.0]))  # equal distances
        t = np.sort(rng.uniform(0, 200, n))
        t_cur = t[-1] + 0.05
        for radius, tdiff in ((10.0, 30.0), (3.0, 0.0), (25.0, 100.0)):
            assert loop_oracle.detect_loop_distance(key, t, t_cur, radius, tdiff) == numpy_loop_distance(key, t, t_cur, radius, tdiff)


def test_detect_loop_distance_edges(loop_oracle):
    key = np.array([[0, 0, 0, 0], [3, 4, 0, 1], [0, 5, 0, 2], [1, 0, 0, 3], [0, 0, 0, 4]], np.float32)
    t = np.array([0.0, 10.0, 20.0, 69.0, 100.0])
    assert loop_oracle.detect_loop_distance(key, t, 100.0, 5.0, 30.0) == 0         # d2 == r^2 (poses 1, 2) excluded
    assert loop_oracle.detect_loop_distance(key, t, 100.0, 5.01, 30.0) == 0        # 0 is nearer than 1 and 2
    assert loop_oracle.detect_loop_distance(key, t, 100.0, 5.01, 31.0) == 0
    assert loop_oracle.detect_loop_distance(key, t, 100.0, 1.5, 31.0) == 0         # |dt| == 31 of pose 3 excluded; 0 is at d 0
    key2 = key.copy()
    key2[0, :3] = 9
    assert loop_oracle.detect_loop_distance(key2, t, 100.0, 1.5, 31.0) == -1       # pose 3: |dt| == time_diff excluded
    assert loop_oracle.detect_loop_distance(key2, t, 100.0, 1.5, 30.9) == 3
    assert loop_oracle.detect_loop_distance(key2, t, 100.0, 6.0, 30.9) == 3        # nearest qualifying, not the lowest index
    assert loop_oracle.detect_loop_distance(key[:1], t[:1], 100.0, 5.0, 30.0) == -1  # n = 1: the newest itself
    assert loop_oracle.detect_loop_distance(key2, t, 200.0, 5.0, 30.0) == -1       # the newest pose wins -> -1
    assert loop_oracle.detect_loop_distance(key, t, 200.0, 5.0, 30.0) == 0         # ... unless an older pose ties with it
    for k, tt in ((key, t), (key2, t)):
        for r in (1.5, 5.0, 5.01, 6.0):
            for td in (30.0, 30.9, 31.0):
                assert loop_oracle.detect_loop_distance(k, tt, 100.0, r, td) == numpy_loop_distance(k, tt, 100.0, r, td)


# ---- C ABI structs --------------------------------------------------------------------------------------------------
def test_sc_struct_layouts_match_a_c_compiler(tmp_path):
    """sizeof / offsetof of liogpu_sc_params / liogpu_sc_info as a C compiler lays them out == the ctypes mirrors"""
    from lio_slam_b200 import liogpu
    pairs = [("liogpu_sc_params", liogpu.ScParams), ("liogpu_sc_info", liogpu.ScInfo)]
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "liogpu.h"', 'int main(void) {']
    for cname, ct in pairs:
        lines.append(f'  printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, _ in ct._fields_:
            lines.append(f'  printf("{cname}.{fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ['  printf("max_candidates %d\\n", LIOGPU_SC_MAX_CANDIDATES);', '  return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.check_call(["/usr/bin/gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = dict(l.split() for l in subprocess.check_output([str(exe)], text=True).splitlines())
    assert int(got["max_candidates"]) == liogpu.LIOGPU_SC_MAX_CANDIDATES
    for cname, ct in pairs:
        assert int(got[cname]) == C.sizeof(ct), cname
        for fname, _ in ct._fields_:
            assert int(got[f"{cname}.{fname}"]) == getattr(ct, fname).offset, f"{cname}.{fname}"


def test_sc_defaults():
    from lio_slam_b200 import liogpu
    from oracle.loop_oracle import SC_DEFAULTS
    p = liogpu.sc_params()
    assert (p.num_exclude_recent, p.num_candidates_from_tree, p.tree_making_period) == (30, 3, 30)
    assert p.search_ratio == 0.1 and p.sc_dist_thres == 0.2
    assert SC_DEFAULTS == dict(num_exclude_recent=30, num_candidates=3, tree_making_period=30, search_ratio=0.1,
                               sc_dist_thres=0.2)
