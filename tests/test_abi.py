"""The C-ABI shared library loads and exports every symbol include/liogpu.h declares.  No compute call is
made here (this container has no GPU); without a device liogpu_create must fail loudly, not fall back."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_functions():
    src = open(os.path.join(ROOT, "include", "liogpu.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(liogpu_[a-z0-9_]+)\s*\(", src)))


def test_header_declares_expected_entry_points():
    names = declared_functions()
    for must in ("liogpu_create", "liogpu_destroy", "liogpu_deskew", "liogpu_voxel_downsample", "liogpu_keyframe_put",
                 "liogpu_build_local_map", "liogpu_set_local_map", "liogpu_scan2map", "liogpu_surf_optimization"):
        assert must in names


def test_library_exports_every_declared_symbol():
    from lio_slam_b200 import liogpu
    lib = liogpu.load_library()
    names = declared_functions()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/liogpu.h but not exported by libliogpu.so"
    assert sorted(liogpu.EXPORTS) == names
    assert lib.liogpu_abi_version() == 2


def test_struct_layouts_match_header():
    from lio_slam_b200 import liogpu
    # liogpu_params: 3 int + 2 float + 2 int + 6 float + 2 float + 6 int reserved
    assert C.sizeof(liogpu.Params) == 4 * 21
    # liogpu_s2m_info: 6 int + 2 float + 36 + 6 double + 30*6 float + 30 int + float (+ padding to 8)
    # ... + gpu_ms, seeded, 2 float kernel times, 2 int launch counts (6 x 4 bytes)
    # ... + certified, leftovers, tail_ms, kernel_launches (4 x 4 bytes) + five per-iteration histories
    assert C.sizeof(liogpu.S2MInfo) == 8 * 4 + 42 * 8 + 180 * 4 + 30 * 4 + 6 * 4 + 4 * 4 + 5 * 30 * 4


def test_struct_layouts_match_a_c_compiler(tmp_path):
    """sizeof / offsetof of every struct of include/liogpu.h as a C compiler lays them out == the ctypes mirrors"""
    import os
    import subprocess
    from lio_slam_b200 import liogpu
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    pairs = [("liogpu_params", liogpu.Params), ("liogpu_s2m_info", liogpu.S2MInfo),
             ("liogpu_local_map_params", liogpu.LocalMapParams), ("liogpu_local_map_info", liogpu.LocalMapInfo),
             ("liogpu_icp_params", liogpu.IcpParams), ("liogpu_icp_info", liogpu.IcpInfo)]
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "liogpu.h"', 'int main(void) {']
    for cname, ct in pairs:
        lines.append(f'  printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, _ in ct._fields_:
            lines.append(f'  printf("{cname}.{fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ['  return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.check_call(["/usr/bin/gcc", "-std=c99", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)])
    got = dict(l.split() for l in subprocess.check_output([str(exe)], text=True).splitlines())
    for cname, ct in pairs:
        assert int(got[cname]) == C.sizeof(ct), cname
        for fname, _ in ct._fields_:
            assert int(got[f"{cname}.{fname}"]) == getattr(ct, fname).offset, f"{cname}.{fname}"


def test_local_map_and_icp_defaults_follow_the_reference():
    from lio_slam_b200 import liogpu
    lp = liogpu.local_map_params()
    assert (lp.local_map_front, lp.local_map_left, lp.local_map_back, lp.local_map_right) == (70.0, 40.0, 20.0, 40.0)  # utility.h:220-223
    assert lp.use_down_sampling == 1 and lp.use_removing_outliers == 1 and lp.mean_k == 10            # :224, 227, 228
    assert abs(lp.local_mapping_surf_leaf_size - 0.01) < 1e-9 and lp.stddev_threshold == 1.0          # :226, 229
    ip = liogpu.IcpParams()
    liogpu.load_library().liogpu_default_icp_params(C.byref(ip), C.c_float(15.0))
    assert ip.max_correspondence_distance == 30.0 and ip.max_iterations == 100                         # mapOptmization.cpp:1112-1113
    assert ip.transformation_epsilon == 1e-6 and ip.euclidean_fitness_epsilon == 1e-6                  # :1114-1115


def test_defaults_follow_utility_h():
    from lio_slam_b200 import liogpu
    p = liogpu.default_params()
    assert (p.n_scan, p.horizon_scan, p.downsample_rate, p.point_filter_num) == (16, 1800, 1, 3)  # utility.h:275-278
    assert abs(p.mapping_surf_leaf_size - 0.2) < 1e-7 and abs(p.surrounding_keyframe_map_leaf_size - 0.2) < 1e-7
    assert (p.lidar_min_front, p.lidar_min_back, p.lidar_min_left, p.lidar_min_right) == (1.0, 5.0, 2.0, 2.0)
    assert p.lidar_max_range == 1000.0 and p.lidar_max_intensity == 100.0


def test_no_cpu_fallback_without_gpu():
    # in a child process that sees no device (CUDA_VISIBLE_DEVICES empty), so that it runs on GPU machines too
    import subprocess
    import sys
    child = ("import sys; sys.path.insert(0, %r)\n"
             "from lio_slam_b200 import liogpu\n"
             "try:\n"
             "    liogpu.LioGpu()\n"
             "except liogpu.LioGpuError as e:\n"
             "    print('status', e.status, e.status == liogpu.E_CUDA)\n" % ROOT)
    r = subprocess.run([sys.executable, "-c", child], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True,
                       text=True, timeout=120)
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.split()[-1] == "True", r.stdout


def test_product_never_touches_oracle():
    # the product path must not import, link or call anything under oracle/
    pkg = os.path.join(ROOT, "lio_slam_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp", "Makefile")):
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "liboracle" not in text and "from oracle" not in text and "import oracle" not in text, f
                assert "liorf_oracle" not in text, f
