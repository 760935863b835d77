"""The thread-per-point pass of liogpu_icp_align (icp_nn_kernel, the left-list indirection of icp_left_kernel, the
grid-stride loop of icp_reduce_kernel).  Sources of up to 65,536 points go straight to the warp-per-point search; larger
ones, and every source when LIOGPU_ICP_THREAD_PASS is set, take the thread pass first.  Both passes find the same exact
nearest target point (ties: lower index) and the reduction sums in a fixed order whichever kernel wrote the
correspondences, so a forced thread pass must reproduce the default bit for bit.  Above 65,536 points the results are
held to the oracle with the tolerances of test_gpu_icp.check."""
import numpy as np
import pytest

from lio_slam_b200 import synth
from test_gpu_icp import check, loop_case  # noqa: F401  (loop_case is a fixture used here)

pytestmark = pytest.mark.gpu

THREAD_PASS_ABOVE = 65536   # icp_align_dev: all_warp = ns <= 65536
CHUNK = 10                  # iterations enqueued per host round trip
INFO_KEYS = ("iterations", "converged", "convergence_state", "n_correspondences", "fitness_score", "last_mse")


def same_result(a, b):
    (Ta, ia), (Tb, ib) = a, b
    assert np.array_equal(Ta.view(np.uint32), Tb.view(np.uint32))
    for k in INFO_KEYS:
        assert ia[k] == ib[k], (k, ia[k], ib[k])


def enqueued_iterations(info, max_iterations):
    """ICP iterations the host enqueued: whole chunks until the one whose last reduction finished the loop, plus the
    getFitnessScore pass.  A loop that stopped for lack of correspondences (state 5) ran one reduction past `iterations`."""
    ran = info["iterations"] + (1 if info["convergence_state"] == 5 else 0)
    return min(max_iterations, CHUNK * -(-ran // CHUNK)) + 1


def default_and_forced(gpu, monkeypatch, src, tgt, radius=10.0, **over):
    """the same alignment with the default pass choice and with the thread pass forced; returns both results and the
    launch counts of each call"""
    c0 = gpu.launch_count()
    a = gpu.icp_align(src, tgt, radius, **over)
    c1 = gpu.launch_count()
    monkeypatch.setenv("LIOGPU_ICP_THREAD_PASS", "1")
    try:
        b = gpu.icp_align(src, tgt, radius, **over)
    finally:
        monkeypatch.delenv("LIOGPU_ICP_THREAD_PASS")
    c2 = gpu.launch_count()
    return a, b, c1 - c0, c2 - c1


def sparse_target(seed=3, n=3000):
    rng = np.random.default_rng(seed)
    return rng, np.c_[rng.uniform(-40, 40, (n, 2)), rng.normal(0, 0.3, (n, 1)), np.zeros((n, 1))].astype(np.float32)


def strays(rng, n):
    """points 10-18 m above the plane: no target point within the warp's six shells, so they go to the exhaustive search"""
    return np.c_[rng.uniform(-40, 40, (n, 2)), rng.uniform(10, 18, (n, 1)), np.zeros((n, 1))].astype(np.float32)


# ---------------------------------------------------------------- every case of test_gpu_icp.py, thread pass forced
def _loop(o, lc):
    tgt, _ = o.build_local_map(lc["clouds"], lc["poses"], 0.4, threads=4)
    src, _ = o.build_local_map([lc["cur"]], lc["wrong"].reshape(1, 6), 0.4, threads=4)
    return src, tgt, dict(radius=10.0)


def _exhaustive(o, lc):
    tgt, _ = o.build_local_map(lc["clouds"][3:8], lc["poses"][3:8], 0.6, threads=4)
    return o.transform_cloud(lc["cur"][::3], lc["wrong"]), tgt, dict(radius=15.0)


def _maxd(d):
    def case(o, lc):
        tgt, _ = o.build_local_map(lc["clouds"], lc["poses"], 0.4, threads=4)
        return o.transform_cloud(lc["cur"], lc["wrong"]), tgt, dict(max_correspondence_distance=d)
    return case


def _iteration_limit(o, lc):
    tgt, _ = o.build_local_map(lc["clouds"], lc["poses"], 0.4, threads=4)
    return o.transform_cloud(lc["cur"], lc["wrong"]), tgt, dict(max_iterations=3)


def _subset(o, lc):
    tgt, _ = o.build_local_map(lc["clouds"], lc["poses"], 0.4, threads=4)
    return tgt[::7].copy(), tgt, dict()


def _no_correspondences(o, lc):
    tgt, _ = o.build_local_map(lc["clouds"][:3], lc["poses"][:3], 0.4, threads=4)
    far = lc["cur"].copy()
    far[:, 0] += 500.0
    return far, tgt, dict(max_correspondence_distance=5.0)


def _sparse(maxd):
    def case(o, lc):
        rng, tgt = sparse_target()
        src = tgt[rng.choice(3000, 1200, replace=False)].copy()
        src[:, 0] += 0.4
        src[:, 1] -= 0.2
        return np.vstack([src, strays(rng, 60)]), tgt, (dict(max_correspondence_distance=maxd) if maxd else dict())
    return case


CASES = {"loop": _loop, "exhaustive": _exhaustive, "maxd_0.3": _maxd(0.3), "maxd_1": _maxd(1.0), "maxd_3": _maxd(3.0),
         "max_iterations_3": _iteration_limit, "source_in_target": _subset, "no_correspondences": _no_correspondences,
         "sparse_strays": _sparse(None), "sparse_strays_maxd_4": _sparse(4.0)}


@pytest.mark.parametrize("case", list(CASES))
def test_forced_thread_pass_matches_default(gpu, oracle, loop_case, monkeypatch, case):  # noqa: F811
    src, tgt, kw = CASES[case](oracle, loop_case)
    assert src.shape[0] <= THREAD_PASS_ABOVE            # the default is the all-warp search
    radius = kw.pop("radius", 10.0)
    a, b, n_warp, n_thread = default_and_forced(gpu, monkeypatch, src, tgt, radius, **kw)
    same_result(a, b)
    # 3 launches per enqueued iteration in all-warp mode, 4 with the thread pass: the forced run took it
    extra = enqueued_iterations(a[1], kw.get("max_iterations", 100))
    assert n_thread > n_warp and n_thread - n_warp == extra, (n_warp, n_thread, extra)
    print(f"{case}: ns={src.shape[0]} iterations={a[1]['iterations']} launches all-warp {n_warp}, thread pass {n_thread}")


# ---------------------------------------------------------------- sources above 65,536 points
@pytest.fixture(scope="module")
def dense_case(world, oracle, loop_case):  # noqa: F811
    """raw 64- and 128-beam sweeps (1800 columns, every ray returns in the synthetic world) at loop_case's drifted pose,
    in the map frame, and the merged 0.4 m submap of loop_case's 11 keyframes as the target"""
    tgt, _ = oracle.build_local_map(loop_case["clouds"], loop_case["poses"], 0.4, threads=4)
    p = synth.path_pose(5.3)
    sweeps = {}
    for beams in (64, 128):
        sw = synth.to_packed(synth.make_scan(world, p, beams, seed=901, cols=1800))
        sweeps[beams] = oracle.transform_cloud(sw, loop_case["wrong"])
    assert sweeps[64].shape[0] == 115200 and sweeps[128].shape[0] == 230400
    return dict(tgt=tgt, sweeps=sweeps)


def test_at_the_switch(gpu, oracle, dense_case):
    """the last all-warp source size and the first thread-pass size, on the same points"""
    setup = []
    for n, per_iteration in ((THREAD_PASS_ABOVE, 3), (THREAD_PASS_ABOVE + 1, 4)):
        src = dense_case["sweeps"][64][:n]
        c0 = gpu.launch_count()
        T, info, want = check(gpu, oracle, src, dense_case["tgt"], radius=10.0)
        launches = gpu.launch_count() - c0
        assert info["converged"] == 1 and 2 <= info["convergence_state"] <= 4
        # the same target grid and source upload, then 3 (all-warp) or 4 (thread pass) kernels per enqueued iteration
        setup.append(launches - per_iteration * enqueued_iterations(info, 100))
        print(f"ns={n}: iterations={info['iterations']} launches={launches} fitness={info['fitness_score']:.6f}")
    assert setup[0] == setup[1] and setup[0] >= 0, setup


def test_dense_sweep_far_above_the_switch(gpu, oracle, dense_case):
    """230,400 source points: 256 reduce blocks of 256 threads, each thread loops 3.5 times"""
    src = dense_case["sweeps"][128]
    T, info, want = check(gpu, oracle, src, dense_case["tgt"], radius=10.0)
    assert info["converged"] == 1 and info["n_correspondences"] == src.shape[0]


def big_sparse_source(n_samples=66000, n_strays=300, nonfinite=True):
    """target samples jittered and shifted, strays high above the plane (the exhaustive list, written at offset ns of
    the left list), and non-finite points, which PCL's correspondence search drops"""
    rng, tgt = sparse_target()
    src = tgt[rng.integers(0, tgt.shape[0], n_samples)].copy()
    src[:, :3] += rng.normal(0, 0.05, (n_samples, 3)).astype(np.float32)
    src[:, 0] += 0.4
    src[:, 1] -= 0.2
    src = np.vstack([src, strays(rng, n_strays)]).astype(np.float32)
    if nonfinite:
        src[5::997, 0] = np.nan
        src[7::1999, 2] = np.inf
        src[11::2503, 1] = -np.inf
    return src, tgt


@pytest.mark.parametrize("maxd", [None, 4.0])
def test_sparse_target_strays_and_nonfinite_above_the_switch(gpu, oracle, maxd):
    src, tgt = big_sparse_source()
    assert src.shape[0] > THREAD_PASS_ABOVE
    over = dict(max_correspondence_distance=maxd) if maxd else dict()
    T, info, want = check(gpu, oracle, src, tgt, radius=10.0, brute=True, **over)
    n_bad = int((~np.isfinite(src[:, :3]).all(axis=1)).sum())
    assert n_bad > 90 and info["n_correspondences"] <= src.shape[0] - n_bad
    if maxd:   # the strays are farther than 4 m from every target point
        assert info["n_correspondences"] <= src.shape[0] - n_bad - 300


def test_buffer_reuse_large_small_large(oracle, loop_case):  # noqa: F811
    """one context: a thread-pass source, an all-warp source, the thread-pass source again; each bit-equal to a fresh
    context"""
    from lio_slam_b200.liogpu import LioGpu
    big_src, big_tgt = big_sparse_source()
    small_src, small_tgt, kw = _exhaustive(oracle, loop_case)
    runs = [(big_src, big_tgt, 10.0), (small_src, small_tgt, kw["radius"]), (big_src, big_tgt, 10.0)]
    fresh = []
    for s, t, r in runs[:2]:
        g = LioGpu()
        try:
            fresh.append(g.icp_align(s, t, r))
        finally:
            g.close()
    g = LioGpu()
    try:
        reused = [g.icp_align(s, t, r) for s, t, r in runs]
    finally:
        g.close()
    same_result(reused[0], fresh[0])
    same_result(reused[1], fresh[1])
    same_result(reused[2], fresh[0])
