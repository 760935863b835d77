"""Point records of every stride the C ABI accepts, in host memory and in device memory.  Cloud calls take 16 or any
multiple of 4 from 32 up; liogpu_deskew takes any multiple of 4 from 28 up.  Strides other than 16 and 32 reach the
scalar branches of unpack_kernel / pack_kernel / load_raw (28, 36, 40, 44) and the wide-record branches (48, 64).
Every record here carries a NaN sentinel in each byte that is not a field, so a wrong field offset or an unmasked ring
shows up in the results.  The reference is the same call on packed stride-16 input (clouds) or on plain 32-byte
PointXYZIRT records (deskew), which the parity tests pin to the oracle."""
import ctypes as C

import numpy as np
import pytest

from lio_slam_b200 import synth

pytestmark = pytest.mark.gpu

SENTINEL = 0x7FA5A5A5            # a quiet NaN whose bytes read 0xA5
ONE = 0x3F800000                 # 1.0f: PCL keeps data[3] = 1
CLOUD_STRIDES = [32, 36, 40, 44, 48, 64]
DESKEW_STRIDES = [28, 32, 36, 44, 48, 64]
OUT_STRIDES = [36, 48, 64]
WHERE = ["host", "device"]


def u32(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def xyzi_records(p4, stride):
    """packed (n,4) f32 -> (n, stride/4) u32 words: x y z at byte 0, intensity at byte 16, sentinel elsewhere"""
    w = np.full((p4.shape[0], stride // 4), SENTINEL, np.uint32)
    w[:, 0:3] = u32(p4[:, 0:3])
    w[:, 4] = u32(p4[:, 3])
    return w


def xyzirt_records(scan, stride):
    """PointXYZIRT (x y z pad intensity ring:u16 time) -> (n, stride/4) u32 words with the sentinel in the pad word, in
    bytes 22-23 after the ring and in the tail"""
    w = np.full((scan.shape[0], stride // 4), SENTINEL, np.uint32)
    for k, f in enumerate(("x", "y", "z")):
        w[:, k] = u32(scan[f])
    w[:, 4] = u32(scan["intensity"])
    w[:, 5] = (SENTINEL & 0xFFFF0000) | scan["ring"].astype(np.uint32)
    w[:, 6] = u32(scan["time"])
    return w


class Placed:
    """a record array in host memory or in a torch CUDA tensor; .arg is the (pointer, n, stride) tuple of the binding"""

    def __init__(self, words, where):
        import torch
        self.host = np.ascontiguousarray(words)
        self.n, self.stride = self.host.shape[0], self.host.shape[1] * 4
        if where == "device":
            self.dev = torch.from_numpy(self.host.view(np.int32)).cuda()
            torch.cuda.synchronize()
            self.ptr = self.dev.data_ptr()
        else:
            self.ptr = self.host.ctypes.data
        self.arg = (self.ptr, self.n, self.stride)

    def words(self):
        return self.dev.cpu().numpy().view(np.uint32) if hasattr(self, "dev") else self.host


@pytest.fixture(scope="module")
def clouds(oracle, small_case):
    scan4 = small_case["scan4"]
    ds, _ = oracle.voxel_grid(scan4, 0.4)
    n_key = 400
    key3d = np.c_[np.array([synth.path_pose(0.7 * k)[3:6] for k in range(n_key)]), np.arange(n_key)].astype(np.float32)
    return dict(scan=scan4, ds=ds, map=small_case["map4"], kf0=ds, kf1=oracle.voxel_grid(scan4[1::2], 0.5)[0],
                icp_src=oracle.transform_cloud(ds, synth.perturbed_guess(small_case["pose_gt"], 5, trans=(0.4, 0.3, 0.05))),
                key3d=key3d, key_time=100.0 + 0.35 * np.arange(n_key), guess=small_case["guess"])


def run_cloud_calls(g, cl, arg):
    """every entry point that reads a cloud; arg(name) is the cloud `name` in the layout under test"""
    pose = np.array([0.03, -0.02, 1.2, 10.5, -3.25, 0.7], np.float32)
    r = {}
    r["transform"] = u32(g.transform_cloud(arg("scan"), pose))
    out, st = g.voxel_downsample(arg("scan"), 0.4)
    r["voxel"] = (u32(out), st)
    g.keyframe_clear()
    g.keyframe_put(0, arg("kf0"))
    g.keyframe_put(1, arg("kf1"))
    kposes = np.array([synth.path_pose(0.0), synth.path_pose(1.5)], np.float32)
    out, st = g.build_local_map([0, 1], kposes, 0.4)
    r["local_map"] = (u32(out), st)
    for side in ("map", "query"):
        g.set_local_map(arg("map") if side == "map" else cl["map"])
        q = arg("ds") if side == "query" else cl["ds"]
        surf = g.surf_optimization(q, pose6=cl["guess"])
        r[f"surf_{side}"] = (surf["nn_idx"], u32(surf["nn_d2"]), u32(surf["coeff"]), surf["flag"], surf["tie"])
        p, P, info = g.scan2map(q, cl["guess"])
        r[f"s2m_{side}"] = (u32(p), u32(P), info["iterations"], info["converged"], info["n_sel"], info["is_degenerate"],
                            info["JtJ"], info["Jtr"], u32(info["pose_hist"]), info["nsel_hist"])
    T, info = g.icp_align(arg("icp_src"), arg("map"))
    r["icp"] = (u32(T),) + tuple(info[k] for k in ("iterations", "convergence_state", "n_correspondences", "fitness_score",
                                                   "last_mse"))
    r["scancontext"] = g.make_scancontext(arg("ds"))
    ids, st = g.extract_nearby(arg("key3d"), cl["key_time"], cl["key_time"][-1] + 0.1)
    r["nearby"] = (ids, st)
    return r


def assert_same(got, want, path=""):
    if isinstance(want, dict):
        assert got.keys() == want.keys()
        for k in want:
            assert_same(got[k], want[k], f"{path}.{k}")
    elif isinstance(want, tuple):
        assert len(got) == len(want), path
        for k, (a, b) in enumerate(zip(got, want)):
            assert_same(a, b, f"{path}[{k}]")
    elif isinstance(want, np.ndarray):
        assert got.shape == want.shape and np.array_equal(got, want), path
    else:
        assert got == want, (path, got, want)


@pytest.fixture(scope="module")
def packed_results(gpu, clouds):
    return run_cloud_calls(gpu, clouds, lambda name: clouds[name])


@pytest.mark.parametrize("where", WHERE)
@pytest.mark.parametrize("stride", CLOUD_STRIDES)
def test_cloud_input_strides(gpu, clouds, packed_results, stride, where):
    keep = []   # every buffer stays alive until the last call has returned

    def arg(name):
        keep.append(Placed(xyzi_records(clouds[name], stride), where))
        return keep[-1].arg

    got = run_cloud_calls(gpu, clouds, arg)
    assert_same(got, packed_results)


def check_out_records(words, ref4, n_out, cap):
    """x y z, 1.0f at byte 12, intensity at byte 16, zeros to the end of each written record; untouched after n_out"""
    assert n_out == ref4.shape[0]
    w = words[:n_out]
    assert np.array_equal(w[:, 0:3], u32(ref4[:, 0:3]))
    assert (w[:, 3] == ONE).all()
    assert np.array_equal(w[:, 4], u32(ref4[:, 3]))
    assert (w[:, 5:] == 0).all()
    assert (words[n_out:cap] == SENTINEL).all()


@pytest.mark.parametrize("where", WHERE)
@pytest.mark.parametrize("out_stride", OUT_STRIDES)
def test_voxel_output_strides(gpu, clouds, out_stride, where):
    scan = clouds["scan"]
    want, _ = gpu.voxel_downsample(scan, 0.4)
    cap = want.shape[0] + 8
    out = Placed(np.full((cap, out_stride // 4), SENTINEL, np.uint32), where)
    n_out = C.c_int(0)
    st = gpu.lib.liogpu_voxel_downsample(gpu.h, scan.ctypes.data, scan.shape[0], 16, C.c_float(0.4), out.ptr, out_stride,
                                         cap, C.byref(n_out))
    assert st == 0
    check_out_records(out.words(), want, n_out.value, cap)


# ---------------------------------------------------------------- deskew
DSK = dict(n_scan=32, downsample_rate=1, point_filter_num=1, lidar_min_front=2.0, lidar_min_back=10.0, lidar_min_left=2.0,
           lidar_min_right=2.0, lidar_max_range=100.0, lidar_max_intensity=90.0)


@pytest.fixture(scope="module")
def deskew_case(world, oracle):
    from lio_slam_b200.liogpu import LioGpu
    from oracle.oracle import DeskewParams
    scan = synth.make_scan(world, synth.path_pose(1.0), 32, seed=77, cols=600)
    t0 = 1700000000.25
    imu = synth.make_imu_table(t0, seed=8)
    g = LioGpu(**DSK)
    want = oracle.deskew(scan, DeskewParams(*DSK.values()), t0, *imu, True)
    got, st = g.deskew(scan, t0, *imu, True)
    assert np.array_equal(u32(got), u32(want)) and want.shape[0] > 1000
    yield dict(g=g, scan=scan, t0=t0, imu=imu, want=want)
    g.close()


def deskew_raw(g, ptr, n, stride, t0, imu, out_ptr, out_stride, cap):
    imu = [np.ascontiguousarray(a, np.float64) for a in imu]
    n_out = C.c_int(0)
    st = g.lib.liogpu_deskew(g.h, ptr, n, stride, C.c_double(t0), *[a.ctypes.data for a in imu], imu[0].shape[0], 1,
                             out_ptr, out_stride, cap, C.byref(n_out))
    return st, n_out.value


@pytest.mark.parametrize("where", WHERE)
@pytest.mark.parametrize("stride", DESKEW_STRIDES)
def test_deskew_input_strides(deskew_case, stride, where):
    d = deskew_case
    rec = Placed(xyzirt_records(d["scan"], stride), where)
    got, st = d["g"].deskew(rec.arg, d["t0"], *d["imu"], True)
    assert st == 0 and np.array_equal(u32(got), u32(d["want"]))


@pytest.mark.parametrize("where", WHERE)
@pytest.mark.parametrize("out_stride", OUT_STRIDES)
def test_deskew_output_strides(deskew_case, out_stride, where):
    d = deskew_case
    scan = np.ascontiguousarray(d["scan"])
    cap = d["want"].shape[0] + 8
    out = Placed(np.full((cap, out_stride // 4), SENTINEL, np.uint32), where)
    st, n_out = deskew_raw(d["g"], scan.ctypes.data, scan.shape[0], 32, d["t0"], d["imu"], out.ptr, out_stride, cap)
    assert st == 0
    check_out_records(out.words(), d["want"], n_out, cap)


def test_strides_outside_the_abi_are_refused(gpu, deskew_case, clouds):
    from lio_slam_b200.liogpu import E_INVALID, LioGpuError
    d = deskew_case
    buf = np.zeros((d["scan"].shape[0], 16), np.uint32)   # room for 64-byte records
    for stride in (24, 30):
        with pytest.raises(LioGpuError) as e:
            d["g"].deskew((buf.ctypes.data, d["scan"].shape[0], stride), d["t0"], *d["imu"], True)
        assert e.value.status == E_INVALID
    for stride in (20, 24, 28, 34):
        arg = (buf.ctypes.data, 1000, stride)
        with pytest.raises(LioGpuError) as e:
            gpu.voxel_downsample(arg, 0.4)
        assert e.value.status == E_INVALID
        with pytest.raises(LioGpuError) as e:
            gpu.transform_cloud(arg, np.zeros(6, np.float32))
        assert e.value.status == E_INVALID
    scan = clouds["scan"]
    out = np.zeros((scan.shape[0], 16), np.uint32)
    scan32 = np.ascontiguousarray(d["scan"])
    dsk_out = np.zeros((scan32.shape[0], 16), np.uint32)
    n_out = C.c_int(0)
    for out_stride in (20, 34):
        assert gpu.lib.liogpu_voxel_downsample(gpu.h, scan.ctypes.data, scan.shape[0], 16, C.c_float(0.4), out.ctypes.data,
                                               out_stride, scan.shape[0], C.byref(n_out)) == E_INVALID
        assert deskew_raw(d["g"], scan32.ctypes.data, scan32.shape[0], 32, d["t0"], d["imu"], dsk_out.ctypes.data,
                          out_stride, dsk_out.shape[0])[0] == E_INVALID
