"""The two extremes of the collecting walk's threshold (LIOGPU_COLLECT_MOVE, s2m.cu) must not change a single bit: the
threshold is read once per process from the environment, so each extreme runs the same dense-map registration in a child
process and its outputs are held against the default threshold's, run here —
  * one surfOptimization pass (mode 1): neighbour indices, squared distances, coefficients, flags, tie bits;
  * the whole loop: pose history, nsel history, JtJ / Jtr of the last iteration, tie count, matP, isDegenerate.
"collect_always" makes every seeded iteration collect, so loose bounds overflow the candidate lists and the insertion-walk
fallback runs; "collect_never" takes the insertion walk everywhere.  The default itself is checked against the CPU oracle
by tests/test_gpu_parity.py and tests/test_gpu_edge.py."""
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CHILD = r"""
import sys, numpy as np
sys.path.insert(0, {root!r})
from lio_slam_b200 import synth
from lio_slam_b200.liogpu import LioGpu
world = synth.make_world(1234)
pose_gt = synth.path_pose(1.0)
scan4 = synth.to_packed(synth.make_scan(world, pose_gt, 32, seed=77, cols=900))
map4 = synth.make_local_map(world, 32, 60000, 0.2, seed=9, s0=0.5, cols=900, max_poses=16)
guess = synth.perturbed_guess(pose_gt, 33)
g = LioGpu(surrounding_keyframe_map_leaf_size=0.2)
g.set_local_map(map4)
so = g.surf_optimization(scan4, pose6=guess)
pose, P, info = g.scan2map(scan4, guess)
g.close()
np.savez({out!r}, pose=pose, P=P, pose_hist=info["pose_hist"], nsel_hist=info["nsel_hist"], JtJ=info["JtJ"], Jtr=info["Jtr"],
         ties=info["tie_queries"], deg=info["is_degenerate"], iters=info["iterations"], seeded=info["seeded"], **so)
"""


def run_variant(variant, tmpdir):
    out = os.path.join(tmpdir, f"{variant or 'default'}.npz")
    env = dict(os.environ)
    env.pop("LIOGPU_COLLECT_MOVE", None)
    if variant == "collect_always":      # every seeded iteration collects: loose bounds overflow the lists -> fallback walk
        env["LIOGPU_COLLECT_MOVE"] = "1e9"
    elif variant == "collect_never":     # the insertion walk everywhere
        env["LIOGPU_COLLECT_MOVE"] = "0"
    r = subprocess.run([sys.executable, "-c", CHILD.format(root=ROOT, out=out)], env=env, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return dict(np.load(out))


@pytest.fixture(scope="module")
def reference_run():
    with tempfile.TemporaryDirectory() as d:
        yield run_variant("", d)


@pytest.mark.parametrize("variant", ["collect_always", "collect_never"])
def test_main_kernel_variant_is_bit_identical_to_the_default(reference_run, variant):
    with tempfile.TemporaryDirectory() as d:
        got = run_variant(variant, d)
    ref = reference_run
    assert int(ref["iters"]) >= 3 and int(got["iters"]) == int(ref["iters"])
    for k in ("nn_idx", "nn_d2", "coeff", "flag", "tie"):           # one surfOptimization pass, point by point
        assert np.array_equal(got[k].view(np.uint8), ref[k].view(np.uint8)), k
    for k in ("pose", "P", "pose_hist"):                             # the whole loop, bit for bit
        assert np.array_equal(got[k].view(np.uint8), ref[k].view(np.uint8)), k
    for k in ("JtJ", "Jtr"):                                         # same partial rows, same order: bit-equal sums
        assert np.array_equal(got[k].view(np.uint8), ref[k].view(np.uint8)), k
    assert np.array_equal(got["nsel_hist"], ref["nsel_hist"])
    assert int(got["ties"]) == int(ref["ties"]) and int(got["deg"]) == int(ref["deg"])
    assert int(got["seeded"]) > 0.5 * got["flag"].shape[0]            # the seeded path was taken
