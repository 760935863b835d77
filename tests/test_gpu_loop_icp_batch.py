"""liogpu_loop_closure_icp_batch: loopFindNearKeyframes for both ends of many candidate pairs and the ICP of
mapOptmization.cpp:1104-1123, in one call with the submaps kept on the device.  The reference for every pair is the
two-call path on the same context (merge_keyframes of both windows, then icp_align), which test_gpu_icp.py holds to the
oracle: every pair must match it bit for bit (submap sizes, overflow flags, T, iterations, convergence state,
correspondence count, f64 fitness and last MSE), whatever the batch around it."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from lio_slam_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_LAP = 64            # keyframes every 1.6 m along two laps of synth.path_pose's 50.3 m circle
S_SMALL = 5           # historyKeyframeSearchNum of the mixed batches (the lattice block below has 2 * 5 + 1 keyframes)
INFO_KEYS = ("iterations", "convergence_state", "converged", "n_correspondences")


def lattice(step, nx, ny, nz, x0=0.0, y0=0.0):
    """points on a lattice coarser than the ICP leaf: VoxelGrid keeps every one of them unchanged"""
    g = np.stack(np.meshgrid(np.arange(nx) * step + x0, np.arange(ny) * step + y0, np.arange(nz) * step,
                             indexing="ij"), -1).reshape(-1, 3)
    return np.c_[g, np.zeros(len(g))].astype(np.float32)


@pytest.fixture(scope="module")
def g():
    from lio_slam_b200.liogpu import LioGpu
    ctx = LioGpu()
    yield ctx
    ctx.close()


@pytest.fixture(scope="module")
def kf(g, world):
    """Keyframes (sensor-frame sweeps) along two laps; the key poses of the second lap drift so that ICP has work.
    After them: 2 * S_SMALL + 1 copies of one integer lattice at the identity (their merged submap is the lattice
    itself), a sweep placed 500 m away, a 100-point cloud and a 73,500-point lattice (sources above 65,536 points)."""
    g.keyframe_clear()
    clouds, poses = [], []
    for j in range(N_LAP):
        s = 1.6 * j
        clouds.append(synth.to_packed(synth.make_scan(world, synth.path_pose(s), 16, seed=3000 + j, cols=900)))
        p = synth.path_pose(s).astype(np.float32)
        if j >= N_LAP // 2:
            f = (j - N_LAP // 2 + 1) / (N_LAP // 2)
            p[3] += 0.9 * f
            p[4] -= 0.6 * f
            p[2] += 0.04 * f
        poses.append(p)
    lat = lattice(1.0, 41, 41, 3, -20.0, -20.0)
    block0 = len(clouds)
    for _ in range(2 * S_SMALL + 1):
        clouds.append(lat)
        poses.append(np.zeros(6, np.float32))
    far = len(clouds)
    clouds.append(clouds[5])
    p = poses[5].copy()
    p[3] += 500.0
    poses.append(p)
    tiny = len(clouds)
    clouds.append(clouds[7][:100].copy())
    poses.append(poses[7].copy())
    big = len(clouds)
    clouds.append(lattice(0.5, 70, 70, 15, -17.0, -17.0))
    poses.append(poses[40].copy())
    for k, c in enumerate(clouds):
        g.keyframe_put(k, c)
    return dict(clouds=clouds, poses=np.array(poses, np.float32), block0=block0, far=far, tiny=tiny, big=big)


@pytest.fixture(scope="module")
def sc_pairs(g, kf):
    """(cur, pre) pairs found by Scan Context detection over the laps (SCManager defaults)"""
    descs = np.array([g.make_scancontext(c)[0] for c in kf["clouds"][:N_LAP]])
    g.sc_clear()
    g.sc_add(descs)
    ids, _, _ = g.sc_detect_loops(np.arange(1, N_LAP + 1))
    pairs = [(j, int(i)) for j, i in enumerate(ids) if i >= 0]
    g.sc_clear()
    assert len(pairs) >= 3, pairs
    return pairs


def rot_angle(Ra, Rb):
    return float(np.linalg.norm(Ra.astype(np.float64) - Rb.astype(np.float64)) / np.sqrt(2.0))


def window(key, s, n_key):
    return list(range(max(key - s, 0), min(key + s, n_key - 1) + 1))


class Reference:
    """the two-call path per pair (merge_keyframes for both windows, icp_align), memoised"""

    def __init__(self, g, poses):
        self.g, self.poses, self.memo = g, poses, {}

    def __call__(self, cur, pre, s, leaf=0.3, **over):
        key = (cur, pre, s, leaf, tuple(sorted(over.items())))
        if key not in self.memo:
            n_key = self.poses.shape[0]
            src, st_s = self.g.merge_keyframes([cur], self.poses[[cur]], leaf)
            w = window(pre, s, n_key)
            tgt, st_t = self.g.merge_keyframes(w, self.poses[w], leaf)
            r = dict(n_source=src.shape[0], n_target=tgt.shape[0], source_overflow=int(st_s == 1),
                     target_overflow=int(st_t == 1), src=src, tgt=tgt)
            if src.shape[0] < 300 or tgt.shape[0] < 1000:
                r.update(rejected_by_size=1, T=np.eye(4, dtype=np.float32), iterations=0, convergence_state=0,
                         converged=0, n_correspondences=0, fitness_score=0.0, last_mse=0.0)
            else:
                T, info = self.g.icp_align(src, tgt, **over)
                r.update(info, rejected_by_size=0, T=T)
            self.memo[key] = r
        return self.memo[key]


@pytest.fixture(scope="module")
def ref(g, kf):
    return Reference(g, kf["poses"])


def same(T, got, want, where):
    for k in ("n_source", "n_target", "source_overflow", "target_overflow", "rejected_by_size") + INFO_KEYS:
        assert got[k] == want[k], (where, k, got[k], want[k])
    assert np.array_equal(T.view(np.uint32), want["T"].view(np.uint32)), (where, T, want["T"])
    for k in ("fitness_score", "last_mse"):
        assert np.float64(got[k]).view(np.uint64) == np.float64(want[k]).view(np.uint64), (where, k, got[k], want[k])
    assert got["gpu_ms"] == 0.0


def run_and_check(g, ref, kf, pairs, s, **over):
    cur = [c for c, _ in pairs]
    pre = [p for _, p in pairs]
    T, res = g.loop_closure_icp_batch(cur, pre, kf["poses"], search_num=s, **over)
    assert T.shape == (len(pairs), 4, 4) and len(res) == len(pairs)
    for j, (c, p) in enumerate(pairs):
        same(T[j], res[j], ref(c, p, s, **over), f"pair {j} {(c, p)}")
    return T, res


def hand_picked(kf):
    return [(40, 8), (N_LAP - 1, 31), (33, 1), (50, 18), (45, 13), (kf["big"], 8), (60, 28)]


@pytest.mark.gpu
@pytest.mark.parametrize("b", [1, 7, 64])
def test_batch_bit_equal_to_two_calls(g, ref, kf, sc_pairs, b):
    pool = sc_pairs + hand_picked(kf)
    pairs = [pool[(3 * j) % len(pool)] for j in range(b)]
    T, res = run_and_check(g, ref, kf, pairs, 25)
    if b > 1:
        assert sum(r["converged"] for r in res) >= 1 and sum(r["iterations"] > 1 for r in res) >= 1


@pytest.mark.gpu
def test_batch_split_into_groups(g, ref, kf, sc_pairs, monkeypatch):
    """a batch that spans several groups (forced small groups) gives the same results"""
    pairs = (sc_pairs + hand_picked(kf))[:20]
    monkeypatch.setenv("LIOGPU_LOOP_ICP_GROUP", "3")
    T3, r3 = run_and_check(g, ref, kf, pairs, 25)
    monkeypatch.delenv("LIOGPU_LOOP_ICP_GROUP")
    T, r = g.loop_closure_icp_batch([c for c, _ in pairs], [p for _, p in pairs], kf["poses"])
    assert np.array_equal(T.view(np.uint32), T3.view(np.uint32)) and r == r3


def mixed_pairs(kf):
    n_key = kf["poses"].shape[0]
    centre = kf["block0"] + S_SMALL
    return [
        (kf["block0"], centre),       # the source is a subset of the target: converges in one iteration
        (40, 8),                      # drifted: runs into max_iterations
        (kf["far"], 5),               # 500 m away: no correspondences (state 5)
        (kf["tiny"], 7),              # 100-point source: rejected by the size guard
        (36, 2),                      # target window clipped at 0
        (44, n_key - 1),              # target window clipped at n_key
        (40, 8),                      # repeated pair
        (kf["big"], 8),               # 73,500-point source
        (kf["big"], 40),
        (57, 25),
    ]


@pytest.mark.gpu
@pytest.mark.parametrize("max_iterations", [3, 100])
def test_mixed_batch(g, ref, kf, max_iterations):
    pairs = mixed_pairs(kf)
    T, res = run_and_check(g, ref, kf, pairs, S_SMALL, max_iterations=max_iterations)
    one, drift, far, tiny = res[0], res[1], res[2], res[3]
    assert one["iterations"] == 1 and one["converged"] == 1 and one["fitness_score"] < 1e-10
    assert np.abs(T[0] - np.eye(4, dtype=np.float32)).max() < 1e-6
    assert far["convergence_state"] == 5 and far["iterations"] == 0 and far["converged"] == 0
    assert tiny["rejected_by_size"] == 1 and tiny["n_source"] <= 100 and tiny["iterations"] == 0
    assert np.array_equal(T[3], np.eye(4, dtype=np.float32))
    assert res[7]["n_source"] > 65536 and res[8]["n_source"] > 65536
    assert res[6] == res[1] and np.array_equal(T[6].view(np.uint32), T[1].view(np.uint32))
    if max_iterations == 3:
        assert drift["iterations"] == 3 and drift["convergence_state"] == 1
    else:
        assert drift["iterations"] > 3


@pytest.mark.gpu
def test_order_permutes_results(g, kf):
    pairs = mixed_pairs(kf)
    cur, pre = np.array([c for c, _ in pairs]), np.array([p for _, p in pairs])
    T, res = g.loop_closure_icp_batch(cur, pre, kf["poses"], search_num=S_SMALL)
    perm = np.random.default_rng(5).permutation(len(pairs))
    Tp, resp = g.loop_closure_icp_batch(cur[perm], pre[perm], kf["poses"], search_num=S_SMALL)
    assert np.array_equal(Tp.view(np.uint32), T[perm].view(np.uint32))
    assert resp == [res[k] for k in perm]


@pytest.mark.gpu
def test_matches_oracle(g, oracle, ref, kf):
    """two pairs against the oracle's restatement of the submaps and of the ICP, with test_gpu_icp.py's bars"""
    T, res = g.loop_closure_icp_batch([40, 50], [8, 18], kf["poses"], search_num=S_SMALL)
    for j, (c, p) in enumerate([(40, 8), (50, 18)]):
        w = window(p, S_SMALL, kf["poses"].shape[0])
        tgt, _ = oracle.build_local_map([kf["clouds"][k] for k in w], kf["poses"][w], 0.3, threads=4)
        src, _ = oracle.build_local_map([kf["clouds"][c]], kf["poses"][[c]], 0.3, threads=4)
        assert res[j]["n_source"] == src.shape[0] and res[j]["n_target"] == tgt.shape[0]
        want = oracle.icp_align(src, tgt, threads=8, max_correspondence_distance=20.0, max_iterations=100,
                                transformation_epsilon=1e-6, euclidean_fitness_epsilon=1e-6)
        assert res[j]["iterations"] == want["iterations"] and res[j]["convergence_state"] == want["state"]
        assert res[j]["n_correspondences"] == want["n_correspondences"]
        assert np.abs(T[j][:3, 3] - want["T"][:3, 3]).max() < 1e-4
        assert rot_angle(T[j][:3, :3], want["T"][:3, :3]) < 1e-5
        assert res[j]["fitness_score"] == pytest.approx(want["fitness_score"], rel=1e-6, abs=1e-12)


@pytest.mark.gpu
def test_keeps_registration_and_rejects_bad_calls(g, kf, small_case):
    from lio_slam_b200.liogpu import E_INVALID, E_NO_KEYFRAME, LioGpuError
    g.set_local_map(small_case["map4"])
    p0, _, i0 = g.scan2map(small_case["scan4"], small_case["guess"])
    n_res, _ = g.voxel_downsample(small_case["scan4"], 0.4, keep_on_device=True)
    q0, _, _ = g.scan2map("resident", small_case["guess"])
    g.loop_closure_icp_batch([40, 50, kf["big"]], [8, 18, 8], kf["poses"], search_num=S_SMALL)
    assert g.resident_size() == n_res
    q1, _, _ = g.scan2map("resident", small_case["guess"])
    assert np.array_equal(q0.view(np.uint32), q1.view(np.uint32))
    p1, _, i1 = g.scan2map(small_case["scan4"], small_case["guess"])
    assert np.array_equal(p0.view(np.uint32), p1.view(np.uint32)) and i0["iterations"] == i1["iterations"]
    # errors are found before any work: no launch
    poses_plus = np.vstack([kf["poses"], np.zeros((1, 6), np.float32)])  # id n_key - 1 was never put
    for args, kw, status in [(([40], [8], kf["poses"]), dict(search_num=-1), E_INVALID),
                             (([40], [kf["poses"].shape[0]], kf["poses"]), {}, E_INVALID),
                             (([-1], [8], kf["poses"]), {}, E_INVALID),
                             (([40, 41], [8, poses_plus.shape[0] - 1], poses_plus), dict(search_num=0), E_NO_KEYFRAME),
                             (([40], [8], kf["poses"]), dict(icp_leaf=0.0), E_INVALID),
                             (([40], [8], kf["poses"]), dict(max_iterations=0), E_INVALID)]:
        before = g.launch_count()
        with pytest.raises(LioGpuError) as e:
            g.loop_closure_icp_batch(*args, **kw)
        assert e.value.status == status and g.launch_count() == before, (args, kw)
    T, res = g.loop_closure_icp_batch([], [], kf["poses"])
    assert T.shape == (0, 4, 4) and res == []


@pytest.mark.gpu
def test_icp_launches_do_not_grow_with_the_batch(g, ref, kf, sc_pairs):
    pairs = (sc_pairs + hand_picked(kf))[:16]
    n_key = kf["poses"].shape[0]
    sub = 0
    for c, p in pairs:  # the submap launches, as liogpu_merge_keyframes makes them
        for w in ([c], window(p, 25, n_key)):
            before = g.launch_count()
            g.merge_keyframes(w, kf["poses"][w], 0.3)
            sub += g.launch_count() - before
    single = []
    for c, p in pairs:
        r = ref(c, p, 25)
        before = g.launch_count()
        g.icp_align(r["src"], r["tgt"])
        single.append(g.launch_count() - before)
    before = g.launch_count()
    g.loop_closure_icp_batch([c for c, _ in pairs], [p for _, p in pairs], kf["poses"])
    icp = g.launch_count() - before - sub
    assert icp <= max(single) + 6, (icp, single)


def test_result_struct_layout_matches_a_c_compiler(tmp_path):
    """sizeof / offsetof of liogpu_loop_icp_result as gcc lays it out == the ctypes mirror (no GPU needed)"""
    from lio_slam_b200 import liogpu
    ct = liogpu.LoopIcpResult
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "liogpu.h"', 'int main(void) {',
             '  printf("size %zu\\n", sizeof(liogpu_loop_icp_result));']
    for fname, _ in ct._fields_:
        lines.append(f'  printf("{fname} %zu\\n", offsetof(liogpu_loop_icp_result, {fname}));')
    lines += ['  return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.check_call(["/usr/bin/gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = dict(l.split() for l in subprocess.check_output([str(exe)], text=True).splitlines())
    assert int(got["size"]) == C.sizeof(ct)
    for fname, _ in ct._fields_:
        assert int(got[fname]) == getattr(ct, fname).offset, fname
    assert "liogpu_loop_closure_icp_batch" in liogpu.EXPORTS


MIRROR_SRC = r'''
// loopClosureICPBatch / loopClosureICP of the host mirror against the two C calls they replace
#include <cstdio>
#include <cstring>
#include "map_optimization_gpu.h"
using namespace liorf_gpu;

int main(int argc, char** argv) {
  FILE* f = std::fopen(argv[1], "rb");
  int n_key = 0, n_pairs = 0;
  if (std::fread(&n_key, 4, 1, f) != 1) return 2;
  liogpu_params prm;
  liogpu_default_params(&prm);
  mapOptimization mo(prm);
  mo.historyKeyframeSearchNum = 5;
  std::vector<Cloud> clouds(n_key);
  for (int k = 0; k < n_key; ++k) {
    int n = 0;
    if (std::fread(&n, 4, 1, f) != 1) return 2;
    std::vector<float> xyzi((size_t)n * 4);
    if (std::fread(xyzi.data(), 4, xyzi.size(), f) != xyzi.size()) return 2;
    clouds[k].resize(n);
    for (int i = 0; i < n; ++i) {
      PointType p{};
      p.x = xyzi[4 * i]; p.y = xyzi[4 * i + 1]; p.z = xyzi[4 * i + 2]; p.intensity = xyzi[4 * i + 3];
      clouds[k][i] = p;
    }
    if (liogpu_keyframe_put(mo.context(), k, clouds[k].data(), n, sizeof(PointType)) != LIOGPU_OK) return 3;
  }
  for (int k = 0; k < n_key; ++k) {
    float p6[6];
    if (std::fread(p6, 4, 6, f) != 6) return 2;
    PointTypePose p{};
    p.roll = p6[0]; p.pitch = p6[1]; p.yaw = p6[2]; p.x = p6[3]; p.y = p6[4]; p.z = p6[5];
    mo.cloudKeyPoses6D.push_back(p);
  }
  if (std::fread(&n_pairs, 4, 1, f) != 1) return 2;
  std::vector<std::pair<int, int>> pairs(n_pairs);
  for (auto& pr : pairs)
    if (std::fread(&pr.first, 4, 1, f) != 1 || std::fread(&pr.second, 4, 1, f) != 1) return 2;
  std::fclose(f);
  std::vector<mapOptimization::LoopClosureOutcome> batch;
  if (mo.loopClosureICPBatch(pairs, batch) < 0) { std::printf("batch failed: %s\n", mo.lastError()); return 4; }
  int accepted = 0, rejected = 0, bad = 0;
  for (int j = 0; j < n_pairs; ++j) {
    // the two C calls: loopFindNearKeyframes (merge + fetch to the host) for both ends, the guard, icp_align
    Cloud cur, pre;
    mo.loopFindNearKeyframes(cur, pairs[j].first, 0);
    mo.loopFindNearKeyframes(pre, pairs[j].second, mo.historyKeyframeSearchNum);
    bool want = false;
    float Tw[16], noise_w = 0.f;
    for (int q = 0; q < 16; ++q) Tw[q] = (q % 5 == 0) ? 1.f : 0.f;
    if (cur.size() >= 300 && pre.size() >= 1000) {
      liogpu_icp_params ip;
      liogpu_default_icp_params(&ip, mo.historyKeyframeSearchRadius);
      liogpu_icp_info info;
      if (liogpu_icp_align(mo.context(), cur.data(), (int)cur.size(), sizeof(PointType), pre.data(), (int)pre.size(),
                           sizeof(PointType), &ip, Tw, &info) != LIOGPU_OK) return 5;
      want = info.converged && info.fitness_score <= mo.historyKeyframeFitnessScore;
      noise_w = (float)info.fitness_score;
    }
    float T1[16];
    float noise1 = -1.f;
    const bool one = mo.loopClosureICP(pairs[j].first, pairs[j].second, T1, &noise1);
    const auto& b = batch[j];
    bool ok = one == want && b.accepted == want && std::memcmp(b.correctionLidarFrame, Tw, sizeof(Tw)) == 0 &&
              b.result.n_source == (int)cur.size() && b.result.n_target == (int)pre.size();
    if (want) ok = ok && std::memcmp(T1, Tw, sizeof(Tw)) == 0 && noise1 == noise_w && b.noiseScore == noise_w;
    if (!ok) { std::printf("mismatch pair %d (%d, %d)\n", j, pairs[j].first, pairs[j].second); ++bad; }
    (want ? accepted : rejected)++;
  }
  std::printf("accepted %d rejected %d mismatched %d\n", accepted, rejected, bad);
  return bad ? 1 : 0;
}
'''


@pytest.mark.gpu
def test_host_mirror_batch_and_one_pair(tmp_path, kf, sc_pairs):
    """loopClosureICPBatch and the one-pair loopClosureICP give the accept / reject, correction and noise score of the
    two C calls (liogpu_merge_keyframes through the host, liogpu_icp_align)"""
    host = os.path.join(ROOT, "lio_slam_b200", "host")
    src = tmp_path / "mirror.cpp"
    src.write_text(MIRROR_SRC)
    exe = tmp_path / "mirror"
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++14", "-I", host, str(src),
                           os.path.join(host, "map_optimization_gpu.cpp"), "-L", os.path.join(ROOT, "lio_slam_b200"),
                           "-lliogpu", "-Wl,-rpath," + os.path.join(ROOT, "lio_slam_b200"), "-o", str(exe)])
    pairs = sc_pairs[:12] + [(kf["tiny"], 7), (kf["far"], 5), (40, 8), (kf["block0"], kf["block0"] + S_SMALL)]
    blob = tmp_path / "case.bin"
    with open(blob, "wb") as f:
        f.write(np.int32(len(kf["clouds"])).tobytes())
        for c in kf["clouds"]:
            f.write(np.int32(c.shape[0]).tobytes())
            f.write(np.ascontiguousarray(c, np.float32).tobytes())
        f.write(kf["poses"].astype(np.float32).tobytes())
        f.write(np.int32(len(pairs)).tobytes())
        f.write(np.array(pairs, np.int32).tobytes())
    r = subprocess.run([str(exe), str(blob)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    acc, rej = int(r.stdout.split()[1]), int(r.stdout.split()[3])
    assert acc >= 1 and rej >= 2, r.stdout
