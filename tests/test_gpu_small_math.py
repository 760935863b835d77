"""The device's small-matrix routines one call at a time against the CPU oracle (bit for bit) and f64 references:
the 6x6 tail of LMOptimization (lm_tail.cuh: QR solve, Jacobi eigen-decomposition, LU inverse, matP, the
non-degeneracy certificate, lm_finalize_warp), the 5x3 plane fit (pose_math.cuh: plane_qr53 / plane_residual),
Eigen::umeyama's rotation (umeyama_rotation_dev) and pose_to_T / warp_refresh_transform.

Whole registrations only reach well-conditioned normal equations; these tests feed the routines OpenCV's stored
outputs (tests/golden/cv2_6x6.npz, cv2_live.npz) and built families at the edges where such code goes wrong: the
eigenvalue threshold of 100 and the certificate's margin, repeated eigenvalues and exact pivot ties, scales from
1e-8 to 1e10, rank deficiency, the LU singularity epsilon, NaN / inf, degenerate neighbour sets.  The routines run
from tests/small_math_harness.cu (`make -C lio_slam_b200/csrc harness`), one warp per case."""
import ctypes as C
import math
import os
import subprocess
import time

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "lio_slam_b200", "csrc")
GOLD = os.path.join(ROOT, "tests", "golden")
FLT_EPS = float(np.finfo(np.float32).eps)
MAX_ITER = 30  # LIOGPU_MAX_ITER

pytestmark = pytest.mark.gpu


def _fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _ip(a):
    return a.ctypes.data_as(C.POINTER(C.c_int))


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


class Harness:
    def __init__(self, path):
        self.lib = C.CDLL(path)

    def _run(self, name, n, *args):
        rc = getattr(self.lib, name)(C.c_int(n), *args)
        assert rc == 0, f"{name}: CUDA error {rc}"

    def solve6(self, A, b):
        A = np.ascontiguousarray(A, np.float32).reshape(-1, 36); b = np.ascontiguousarray(b, np.float32).reshape(-1, 6)
        x = np.zeros((len(A), 6), np.float32)
        self._run("smh_solve6", len(A), _fp(A), _fp(b), _fp(x))
        return x

    def eigen6(self, A):
        A = np.ascontiguousarray(A, np.float32).reshape(-1, 36)
        W = np.zeros((len(A), 6), np.float32); V = np.zeros((len(A), 36), np.float32)
        self._run("smh_eigen6", len(A), _fp(A), _fp(W), _fp(V))
        return W, V.reshape(-1, 6, 6)

    def inv6(self, V):
        V = np.ascontiguousarray(V, np.float32).reshape(-1, 36)
        Vi = np.zeros((len(V), 36), np.float32)
        self._run("smh_inv6", len(V), _fp(V), _fp(Vi))
        return Vi.reshape(-1, 6, 6)

    def matp(self, A):
        A = np.ascontiguousarray(A, np.float32).reshape(-1, 36)
        P = np.zeros((len(A), 36), np.float32); deg = np.zeros(len(A), np.int32)
        self._run("smh_matp", len(A), _fp(A), _fp(P), _ip(deg))
        return P.reshape(-1, 6, 6), deg

    def certify(self, A):
        A = np.ascontiguousarray(A, np.float32).reshape(-1, 36)
        cert = np.zeros(len(A), np.int32)
        self._run("smh_certify", len(A), _fp(A), _ip(cert))
        return cert.astype(bool)

    def lm_tail(self, JtJ, Jtr, nsel, it, pose, matP, degenerate):
        JtJ = np.asarray(JtJ, np.float64).reshape(-1, 6, 6); n = len(JtJ)
        sums = np.zeros((n, 32), np.float64)
        iu = np.triu_indices(6)  # row by row: the layout of the main kernels' 21 AtA sums
        sums[:, :21] = JtJ[:, iu[0], iu[1]]
        sums[:, 21:27] = np.asarray(Jtr, np.float64).reshape(n, 6)
        sums[:, 27] = np.broadcast_to(np.asarray(nsel, np.float64), n)
        it = np.ascontiguousarray(np.broadcast_to(np.asarray(it, np.int32), n))
        deg = np.ascontiguousarray(np.broadcast_to(np.asarray(degenerate, np.int32), n))
        pose = np.ascontiguousarray(np.broadcast_to(np.asarray(pose, np.float32).reshape(-1, 6), (n, 6)))
        matP = np.ascontiguousarray(np.broadcast_to(np.asarray(matP, np.float32).reshape(-1, 6, 6), (n, 6, 6)))
        f = np.zeros((n, 62), np.float32); i = np.zeros((n, 6), np.int32)
        self._run("smh_lm_tail", n, _dp(sums), _ip(it), _fp(pose), _fp(matP), _ip(deg), _fp(f), _ip(i))
        return dict(pose=f[:, :6], matP=f[:, 6:42].reshape(n, 6, 6), T=f[:, 42:54], trig=f[:, 54:60], delta_r=f[:, 60],
                    delta_t=f[:, 61], degenerate=i[:, 0], certified=i[:, 1].astype(bool), cert_mismatch=i[:, 2],
                    converged=i[:, 3].astype(bool), done=i[:, 4].astype(bool), iter=i[:, 5])

    def pose_to_T(self, pose):
        pose = np.ascontiguousarray(pose, np.float32).reshape(-1, 6); n = len(pose)
        T = np.zeros((n, 12), np.float32); Tw = np.zeros((n, 12), np.float32); trig = np.zeros((n, 6), np.float32)
        self._run("smh_pose_to_T", n, _fp(pose), _fp(T), _fp(Tw), _fp(trig))
        return T, Tw, trig

    def plane_qr53(self, A):
        A = np.ascontiguousarray(A, np.float32).reshape(-1, 15)
        x = np.zeros((len(A), 3), np.float32)
        self._run("smh_plane_qr53", len(A), _fp(A), _fp(x))
        return x

    def plane_residual(self, ori, sel, nbr):
        ori = np.ascontiguousarray(ori, np.float32).reshape(-1, 4); n = len(ori)
        sel = np.ascontiguousarray(sel, np.float32).reshape(n, 4); nbr = np.ascontiguousarray(nbr, np.float32).reshape(n, 20)
        coeff = np.zeros((n, 4), np.float32); flag = np.zeros(n, np.int32)
        self._run("smh_plane_residual", n, _fp(ori), _fp(sel), _fp(nbr), _fp(coeff), _ip(flag))
        return flag.astype(bool), coeff

    def umeyama(self, sigma):
        sigma = np.ascontiguousarray(sigma, np.float32).reshape(-1, 9)
        R = np.zeros((len(sigma), 9), np.float32)
        self._run("smh_umeyama", len(sigma), _fp(sigma), _fp(R))
        return R.reshape(-1, 3, 3)


@pytest.fixture(scope="module")
def harness():
    r = subprocess.run(["make", "-C", CSRC, "harness"], capture_output=True, text=True)
    assert r.returncode == 0, "building the small-math harness failed:\n" + r.stdout[-4000:] + r.stderr[-4000:]
    return Harness(os.path.join(CSRC, "build", "libsmall_math_harness.so"))


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def biteq(a, b):
    """bit-equal, except that any NaN equals any NaN (payloads and signs of NaN differ between x86 and the GPU)"""
    a = np.ascontiguousarray(a, np.float32); b = np.ascontiguousarray(b, np.float32)
    return a.shape == b.shape and bool(np.all((bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b))))


def first_diff(a, b):
    a = np.ascontiguousarray(a, np.float32).reshape(len(a), -1); b = np.ascontiguousarray(b, np.float32).reshape(len(b), -1)
    bad = np.where(~np.all((bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b)), axis=1))[0]
    return (len(bad), bad[:5].tolist())


def degeneracy_V2(W, V):
    """the degeneracy loop of LMOptimization (MO:1797-1806): zero the rows of the trailing eigenvalues below 100"""
    V2 = np.array(V, np.float32)
    for i in range(5, -1, -1):
        if W[i] < np.float32(100):
            V2[i, :] = 0
        else:
            break
    return V2


def oracle_6x6(oracle, A, b):
    """the oracle's cv::solve / cv::eigen / Mat::inv / matP on one f32 system"""
    ok, X = oracle.cv_solve6_qr(A, b)
    W, V = oracle.cv_eigen6(A)
    _, Vi = oracle.cv_inv6(V)
    V2 = degeneracy_V2(W, V)
    deg = int(bool(W[5] < np.float32(100)))
    return dict(X=X, W=W, V=V, Vi=Vi, P=oracle.cv_gemm6(Vi, V2), deg=deg)


def check_6x6_family(harness, oracle, name, A, b=None, tail=True):
    """device solve / eigen / inverse / matP / (tail) against the oracle, bit for bit; returns the case count"""
    A = np.ascontiguousarray(A, np.float32).reshape(-1, 6, 6); n = len(A)
    if b is None:
        b = np.random.default_rng(n).normal(size=(n, 6)).astype(np.float32)
    ref = [oracle_6x6(oracle, A[k], b[k]) for k in range(n)]
    X = harness.solve6(A, b)
    W, V = harness.eigen6(A)
    P, deg = harness.matp(A)
    Vr = np.array([r["V"] for r in ref])
    Vi = harness.inv6(Vr)
    for key, got in (("X", X), ("W", W), ("V", V), ("Vi", Vi), ("P", P)):
        want = np.array([r[key] for r in ref])
        assert biteq(got, want), f"{name}: {key} differs from the oracle in (count, first cases) {first_diff(got, want)}"
    assert np.array_equal(deg, [r["deg"] for r in ref]), f"{name}: isDegenerate"
    if tail:
        check_tail(harness, oracle, name, A.astype(np.float64), b.astype(np.float64))
    return n


def tail_reference(oracle, JtJ, Jtr, nsel, it, pose, matP, deg):
    if nsel < 50:  # MO:1721-1724: the pose is untouched and the remaining iterations repeat
        return dict(conv=False, pose=np.array(pose, np.float32), P=np.array(matP, np.float32), deg=deg, dr=None, dt=None)
    conv, p, P, d, dr, dt = oracle.lm_solve_update(JtJ, Jtr, it, pose, matP, deg)
    return dict(conv=conv, pose=p, P=P, deg=d, dr=dr, dt=dt)


def check_tail(harness, oracle, name, JtJ, Jtr, nsel=1000, iters=((0, 0), (3, 0), (3, 1))):
    """lm_finalize_warp (+ the side computation of matP when the certificate fired) against oracle.lm_solve_update"""
    JtJ = np.asarray(JtJ, np.float64).reshape(-1, 6, 6); n = len(JtJ)
    # the device holds the 21 sums of the upper triangle only (AtA(a,b) and AtA(b,a) are the same sum): hand the
    # oracle the same symmetric matrix
    JtJ = np.triu(JtJ) + np.triu(JtJ, 1).transpose(0, 2, 1)
    rng = np.random.default_rng(n + 17)
    pose = rng.uniform(-0.5, 0.5, (n, 6)).astype(np.float32)
    matP_in = np.array([oracle_6x6(oracle, J.astype(np.float32), np.zeros(6, np.float32))["P"] for J in JtJ])
    nsel = np.broadcast_to(np.asarray(nsel), n)
    for it, deg_in in iters:
        got = harness.lm_tail(JtJ, Jtr, nsel, it, pose, matP_in, deg_in)
        assert not got["cert_mismatch"].any(), f"{name}: the certificate contradicted the eigenvalues"
        for k in range(n):
            ref = tail_reference(oracle, JtJ[k], Jtr[k], int(nsel[k]), it, pose[k], matP_in[k], deg_in)
            tag = f"{name} case {k} iter {it} degenerate {deg_in}"
            assert biteq(got["pose"][k], ref["pose"]), (tag, got["pose"][k], ref["pose"])
            assert biteq(got["matP"][k], ref["P"]), tag
            assert got["degenerate"][k] == ref["deg"], tag
            assert got["converged"][k] == ref["conv"], tag
            done = ref["conv"] or it + 1 >= MAX_ITER or nsel[k] < 50
            assert got["done"][k] == done and got["iter"][k] == (MAX_ITER if nsel[k] < 50 else it + 1), tag
            if ref["dr"] is not None:
                assert biteq(got["delta_r"][k], ref["dr"]) and biteq(got["delta_t"][k], ref["dt"]), tag
            if not done:
                assert biteq(got["T"][k], oracle.pose_to_T(ref["pose"])), tag
            if it == 0 and got["certified"][k]:
                assert ref["deg"] == 0, tag


# ---------------------------------------------------------------------------------------------------------------
# matrix families


def sym_from_eigs(lams, rng, q=None):
    """Q diag(lam) Q^T in f64 (Q random orthogonal, or q), rounded once to f32"""
    lams = np.asarray(lams, np.float64)
    Q = q if q is not None else np.linalg.qr(rng.normal(size=(6, 6)))[0]
    A = (Q * lams) @ Q.T
    return ((A + A.T) * 0.5).astype(np.float32)


def ulp_sweep_family(rng):
    """lambda_min swept across 100 in single-f32-ulp steps: diagonal (W is the diagonal, exactly) and rotated"""
    out = []
    base = np.float32(100)
    for k in range(-24, 25):
        lam = np.float32(base + np.float32(k) * np.spacing(base)) if k else base
        lam = np.nextafter(base, np.float32(np.inf if k > 0 else -np.inf), dtype=np.float32) if abs(k) == 1 else lam
        lams = [3.0e3, 1.2e3, 700.0, 300.0, 150.0, float(lam)]
        out.append(np.diag(np.array(rng.permutation(lams), np.float32)))
        out.append(sym_from_eigs(lams, rng))
        out.append(sym_from_eigs([4e6, 9e5, 2e5, 3e4, 2e3, float(lam)], rng))  # large spread: W[5] off by ~1
    return np.array(out)


def cert_mu(lams_other, eps):
    """lambda_min with lambda_min = (1 + eps) * (100 + 1e-4 * trace)"""
    S = float(np.sum(lams_other))
    return (100.0 + 1e-4 * S) * (1 + eps) / (1 - 1e-4 * (1 + eps))


def cert_boundary_family(rng):
    out = []
    for eps in np.concatenate([-np.logspace(-9, -1, 17), [0.0], np.logspace(-9, 0.5, 20)]):
        for others in ([5e3, 2e3, 1e3, 600.0, 300.0], [1e7, 1e6, 1e5, 1e4, 1e3], [400.0, 300.0, 250.0, 200.0, 150.0]):
            out.append(sym_from_eigs(list(others) + [cert_mu(others, eps)], rng))
    return np.array(out)


def repeated_family(rng):
    out = []
    for lams in ([500, 500, 300, 200, 150, 120], [900, 400, 400, 400, 250, 50], [700, 700, 700, 90, 90, 30],
                 [250.0] * 6, [99.0] * 6, [100.0] * 6, [1e-3] * 6, [7e5, 7e5, 7e5, 7e5, 100, 100]):
        out.append(sym_from_eigs(lams, rng))
        out.append(np.diag(np.array(lams, np.float32)))  # exact diagonal: the first pivot already passes <= FLT_EPSILON
    for c in (0.0, 1.0, 100.0, 1e6):
        out.append(np.eye(6, dtype=np.float32) * np.float32(c))
    # exact ties of the Jacobi pivot: equal off-diagonal magnitudes (c I + b 11^T), small-integer symmetric matrices
    for c, b in ((300.0, 20.0), (300.0, -20.0), (50.0, 10.0), (1000.0, 1.0)):
        out.append((np.eye(6) * c + b).astype(np.float32))
    for _ in range(60):
        M = rng.integers(-3, 4, size=(6, 6)).astype(np.float64)
        M = np.triu(M, 1); M = M + M.T + np.diag(rng.integers(1, 40, size=6) * 10.0)
        out.append(M.astype(np.float32))
    return np.array(out)


def scale_family(rng):
    out = []
    for s in np.logspace(-8, 10, 37):
        for _ in range(2):
            out.append(sym_from_eigs(s * rng.uniform(1, 10, size=6), rng))
    return np.array(out)


def rank_family(rng):
    """A^T A of integer matrices whose columns are dependent (rank 0..5): exact in f32, solve fails, X = 0"""
    out = []
    for r in range(6):
        for _ in range(6):
            Bm = rng.integers(-4, 5, size=(40, r)).astype(np.float64) if r else np.zeros((40, 0))
            Cm = rng.integers(-2, 3, size=(r, 6)).astype(np.float64) if r else np.zeros((0, 6))
            M = Bm @ Cm
            out.append((M.T @ M).astype(np.float32))
    return np.array(out)


def lu_eps_family(rng):
    """matrices whose LU pivot lands on either side of the singularity epsilon FLT_EPSILON * 10"""
    out = []
    thr = np.float32(FLT_EPS * 10)
    for d in (thr, np.nextafter(thr, np.float32(0)), np.nextafter(thr, np.float32(1)), np.float32(FLT_EPS),
              np.float32(5 * FLT_EPS), np.float32(20 * FLT_EPS), np.float32(0)):
        M = np.eye(6, dtype=np.float32); M[5, 5] = d
        out.append(M)
        out.append(M[rng.permutation(6)])  # row exchanges on the way
        M2 = np.eye(6, dtype=np.float32); M2[3, 3] = d; M2[3, 4] = np.float32(0.5); M2[4, 3] = d * np.float32(0.5)
        out.append(M2)
    return np.array(out)


def nonfinite_family(rng):
    out = []
    base = sym_from_eigs([800, 600, 400, 300, 200, 150], rng)
    for v in (np.nan, np.inf, -np.inf):
        for (i, j) in ((0, 0), (2, 3), (0, 5), (4, 5), (5, 5), (1, 4)):
            M = base.copy(); M[i, j] = v; M[j, i] = v
            out.append(M)
    return np.array(out)


# ---------------------------------------------------------------------------------------------------------------


def test_opencv_fixtures(harness, oracle):
    """all 24 + 60 stored OpenCV systems: the device's solve, eigen (W and V), inverse and matP equal OpenCV's outputs;
    the tail equals oracle.lm_solve_update at iteration 0 and at a later iteration for both values of isDegenerate"""
    t0 = time.time()
    G = np.load(os.path.join(GOLD, "cv2_6x6.npz")); L = np.load(os.path.join(GOLD, "cv2_live.npz"))
    cases = []
    for k in range(int(G["n_cases"])):
        A64, b64 = G[f"A_{k}"].astype(np.float64), G[f"b_{k}"].astype(np.float64)
        cases.append(dict(AtA=G[f"AtA_{k}"], Atb=G[f"Atb_{k}"], ok=bool(G[f"ok_{k}"]), X=G[f"X_{k}"], E=G[f"E_{k}"],
                          V=G[f"V_{k}"], Vi=G[f"Vi_{k}"], P=G[f"P_{k}"], JtJ=A64.T @ A64, Jtr=A64.T @ b64))
    for t in range(60):
        V2 = degeneracy_V2(L[f"E_{t}"], L[f"V_{t}"])
        cases.append(dict(AtA=L[f"AtA_{t}"], Atb=L[f"Atb_{t}"], ok=bool(L[f"ok_{t}"]), X=L[f"X_{t}"], E=L[f"E_{t}"],
                          V=L[f"V_{t}"], Vi=L[f"Vi_{t}"], P=oracle.cv_gemm6(L[f"Vi_{t}"], V2),
                          JtJ=L[f"AtA_{t}"].astype(np.float64), Jtr=L[f"Atb_{t}"].astype(np.float64)))
    st = lambda key: np.array([c[key] for c in cases])
    X = harness.solve6(st("AtA"), st("Atb"))
    for k, c in enumerate(cases):
        assert biteq(X[k], c["X"] if c["ok"] else np.zeros(6)), f"cv::solve case {k}"
    W, V = harness.eigen6(st("AtA"))
    assert biteq(W, st("E")) and biteq(V, st("V")), ("cv::eigen", first_diff(W, st("E")), first_diff(V, st("V")))
    assert biteq(harness.inv6(st("V")), st("Vi")), "Mat::inv"
    P, deg = harness.matp(st("AtA"))
    assert biteq(P, st("P")), ("matP", first_diff(P, st("P")))
    assert np.array_equal(deg, (st("E")[:, 5] < 100).astype(np.int32))
    check_tail(harness, oracle, "opencv fixtures", st("JtJ"), st("Jtr"))
    print(f"OpenCV fixtures: {len(cases)} systems, {time.time() - t0:.2f} s")


FAMILIES = dict(ulp_sweep=ulp_sweep_family, cert_boundary=cert_boundary_family, repeated=repeated_family,
                scales=scale_family, rank=rank_family, lu_eps=lu_eps_family, nonfinite=nonfinite_family)


@pytest.mark.parametrize("family", list(FAMILIES))
def test_6x6_family(harness, oracle, family):
    """built 6x6 families against the oracle's cv_solve6_qr / cv_eigen6 / cv_inv6 / cv_gemm6 / lm_solve_update"""
    t0 = time.time()
    A = FAMILIES[family](np.random.default_rng(len(family)))
    n = check_6x6_family(harness, oracle, family, A)
    if family == "lu_eps":  # the inverse on the matrices themselves, not only on eigenvector matrices
        got = harness.inv6(A)
        want = np.array([oracle.cv_inv6(M)[1] for M in A])
        assert biteq(got, want), ("Mat::inv at the singularity epsilon", first_diff(got, want))
    if family == "rank":
        X = harness.solve6(A, np.ones((len(A), 6), np.float32))
        fails = [not oracle.cv_solve6_qr(M, np.ones(6, np.float32))[0] for M in A]
        assert sum(fails) >= 4 and not X[np.array(fails)].any(), "a failed solve leaves X = 0"
    print(f"{family}: {n} matrices, {time.time() - t0:.2f} s")


def test_tail_nsel_threshold(harness, oracle):
    """nsel just below 50 leaves the pose untouched and ends the loop; at 50 the update runs"""
    rng = np.random.default_rng(3)
    A = np.array([sym_from_eigs(rng.uniform(150, 900, 6), rng) for _ in range(8)]).astype(np.float64)
    b = rng.normal(size=(8, 6))
    for nsel in (0, 49, 50, 51):
        check_tail(harness, oracle, f"nsel={nsel}", A, b, nsel=nsel)


def test_certificate_soundness(harness, oracle):
    """a certified matrix has an oracle W[5] >= 100 and an f64 lambda_min above 100; every matrix with
    lambda_min >= 2 (100 + 1e-4 trace) is certified (a tighter bound can fail for small traces: the LDL^T pivot floor
    is 1e-3 mu); the side computation never contradicts the certificate"""
    rng = np.random.default_rng(11)
    fams = [f(np.random.default_rng(len(name))) for name, f in FAMILIES.items()]
    n_rand = 100_000
    lam_min = 100.0 * np.exp(rng.uniform(-3, 3, n_rand))
    spread = np.exp(rng.uniform(0, np.log(1e5), (n_rand, 5)))
    lams = np.concatenate([lam_min[:, None], lam_min[:, None] * spread], 1)
    Q = np.linalg.qr(rng.normal(size=(n_rand, 6, 6)))[0]
    R = np.einsum("nij,nj,nkj->nik", Q, lams, Q)
    R = (0.5 * (R + R.transpose(0, 2, 1))).astype(np.float32)
    A = np.concatenate(fams + [R]).astype(np.float32)
    finite = np.isfinite(A).all(axis=(1, 2))
    cert = harness.certify(A)
    assert not cert[~finite].any(), "a matrix with NaN / inf entries was certified"
    A64 = A[finite].astype(np.float64)
    ev = np.linalg.eigvalsh(A64)[:, 0]
    c = cert[finite]
    tr = np.trace(A64, axis1=1, axis2=2)
    margin = ev[c] - 100.0
    assert (margin > 0).all(), f"certified with f64 lambda_min <= 100: {ev[c][margin <= 0][:5]}"
    for M in A[finite][c]:
        W, _ = oracle.cv_eigen6(M)
        assert W[5] >= np.float32(100), (M, W)
    must = ev >= 2 * (100 + 1e-4 * tr)
    assert c[must].all(), f"not certified although lambda_min >= 2 mu: {np.where(must & ~c)[0][:5]}"
    # the boundary sweep: lambda_min = (1 + eps) mu
    B = cert_boundary_family(np.random.default_rng(len("cert_boundary")))
    frac = harness.certify(B).mean()
    print(f"certificate: {len(A)} matrices ({len(A) - n_rand} built + {n_rand} random), {int(c.sum())} certified, "
          f"smallest certified margin lambda_min - 100 = {margin.min():.4g} (relative to mu: "
          f"{(ev[c] / (100 + 1e-4 * tr[c]) - 1).min():.3g}); certified across the mu boundary sweep: {frac:.3f}")


# ---------------------------------------------------------------------------------------------------------------
# 5x3 plane fit


def plane_sets(rng):
    """(name, nbr (n,5,4), sel (n,4), ori (n,4)) neighbour sets"""
    sets = []

    def on_plane(normal, dist, spread, noise, n, centre=None):
        normal = np.asarray(normal, np.float64); normal = normal / np.linalg.norm(normal)
        t1 = np.cross(normal, [1.0, 0.0, 0.0] if abs(normal[0]) < 0.9 else [0.0, 1.0, 0.0]); t1 /= np.linalg.norm(t1)
        t2 = np.cross(normal, t1)
        base = dist * normal if centre is None else np.asarray(centre, np.float64)
        uv = rng.normal(size=(n, 2)) * spread
        p = base + uv[:, :1] * t1 + uv[:, 1:] * t2 + rng.normal(size=(n, 1)) * noise * normal
        return p

    def pack(p5, sel, ori):
        nbr = np.concatenate([p5, np.zeros((len(p5), 5, 1))], 2).astype(np.float32)
        return nbr, np.concatenate([sel, np.zeros((len(sel), 1))], 1).astype(np.float32), \
            np.concatenate([ori, np.zeros((len(ori), 1))], 1).astype(np.float32)

    # planes at 1e-3 .. 1e4 m from the origin, and through it
    nb, sl, orr = [], [], []
    for dist in np.concatenate([[0.0], np.logspace(-3, 4, 15)]):
        for _ in range(12):
            nrm = rng.normal(size=3)
            p = on_plane(nrm, dist, rng.uniform(0.05, 0.5), rng.uniform(0, 0.05), 6)
            nb.append(p[:5]); sl.append(p[5] + rng.normal(size=3) * 0.1); orr.append(rng.normal(size=3) * 10)
    sets.append(("distance", *pack(np.array(nb), np.array(sl), np.array(orr))))
    # axis-aligned planes: exact zeros below the diagonal (the tail <= FLT_MIN branch of the Householder step)
    nb, sl, orr = [], [], []
    for axis in range(3):
        for c in (0.0, 0.5, -3.0, 40.0):
            for _ in range(8):
                p = rng.normal(size=(6, 3)) * 0.3 + rng.normal(size=3) * 5; p[:, axis] = c
                nb.append(p[:5]); sl.append(p[5]); orr.append(rng.normal(size=3) * 10)
        for _ in range(8):  # unit-vector neighbours: columns with exact zeros
            p = np.zeros((5, 3)); p[0, axis] = rng.uniform(0.5, 2); p[1, (axis + 1) % 3] = rng.uniform(0.5, 2)
            p[2, (axis + 2) % 3] = rng.uniform(0.5, 2); p[3] = p[0] + p[1]; p[4] = p[1] + p[2]
            nb.append(p); sl.append(p[0]); orr.append(p[0])
    sets.append(("axis_aligned", *pack(np.array(nb), np.array(sl), np.array(orr))))
    # neighbour sets below FLT_MIN in their squares: every Householder step takes the tail <= FLT_MIN branch
    nb, sl, orr = [], [], []
    for s in (1e-18, 3e-19, 1e-19, 3e-20, 1e-20):
        for _ in range(10):
            p = rng.normal(size=(5, 3)) * s; p[0] += rng.normal(size=3) * 10 * s
            nb.append(p); sl.append(p[0]); orr.append(np.ones(3))
    sets.append(("subnormal_scale", *pack(np.array(nb), np.array(sl), np.array(orr))))
    # collinear, two-point and all-coincident sets (nonzero < 3)
    nb, sl, orr = [], [], []
    for _ in range(30):
        a, d = rng.normal(size=3) * 5, rng.normal(size=3)
        nb.append(a + np.outer(rng.normal(size=5), d)); sl.append(a); orr.append(a)
        two = np.array([a, a, a + d, a + d, a]); nb.append(two); sl.append(a); orr.append(a)
        nb.append(np.repeat(a[None], 5, 0)); sl.append(a); orr.append(a)
    nb.append(np.zeros((5, 3))); sl.append(np.zeros(3)); orr.append(np.zeros(3))
    sets.append(("collinear_coincident", *pack(np.array(nb), np.array(sl), np.array(orr))))
    # clusters 1e4 m out with centimetre spread
    nb, sl, orr = [], [], []
    for _ in range(80):
        centre = rng.normal(size=3); centre = centre / np.linalg.norm(centre) * 1e4
        p = on_plane(rng.normal(size=3), 0, 0.01, 0.001, 6, centre=centre)
        nb.append(p[:5]); sl.append(p[5]); orr.append(p[5] - centre * 0.999)
    sets.append(("far_cluster", *pack(np.array(nb), np.array(sl), np.array(orr))))
    # residuals straddling 0.2, weight s straddling 0.1, the sweep point at the origin
    nb, sl, orr = [], [], []
    for off in np.linspace(0.17, 0.23, 25):
        p = on_plane([0, 0, 1], 2.0, 0.3, 0, 5); p[2, 2] += off * 2.5  # lifts one residual to about `off`
        nb.append(p); sl.append(p[0]); orr.append(p[0])
    for pd2 in np.linspace(0.85, 1.15, 31):  # s = 1 - 0.9 |pd2| / r^(1/4) with r^(1/4) = 1: straddles 0.1 at 1.0
        p = on_plane([0, 0, 1], 2.0, 0.3, 0, 5)
        nb.append(p); sl.append(p[0] + np.array([0, 0, pd2])); orr.append(np.array([1.0, 0, 0]))
    for _ in range(10):
        p = on_plane(rng.normal(size=3), 3.0, 0.3, 0.01, 6)
        nb.append(p[:5]); sl.append(p[5]); orr.append(np.zeros(3))
    sets.append(("thresholds", *pack(np.array(nb), np.array(sl), np.array(orr))))
    return sets


def test_plane_fit(harness, oracle):
    """plane_qr53 equals the oracle's qr53_solve and plane_residual's flag (and coeff where accepted) equal the
    oracle's plane_residual, bit for bit; well-conditioned sets also agree with f64 lstsq to 1e-5 * cond"""
    t0 = time.time()
    total = 0
    for name, nbr, sel, ori in plane_sets(np.random.default_rng(21)):
        n = len(nbr)
        x = harness.plane_qr53(nbr[:, :, :3])
        want = np.array([oracle.qr53_solve(nbr[k, :, :3], -np.ones(5, np.float32)) for k in range(n)])
        assert biteq(x, want), (name, "plane_qr53", first_diff(x, want))
        flag, coeff = harness.plane_residual(ori, sel, nbr)
        for k in range(n):
            ok, c = oracle.plane_residual(ori[k], sel[k], nbr[k])
            assert flag[k] == ok, (name, k, "flag")
            if ok:
                assert biteq(coeff[k], c), (name, k, coeff[k], c)
        A = nbr[:, :, :3].astype(np.float64)
        for k in range(n):
            cond = np.linalg.cond(A[k])
            if cond < 1e4 and np.abs(A[k]).max() > 1e-3:
                ref = np.linalg.lstsq(A[k], -np.ones(5), rcond=None)[0]
                err = np.linalg.norm(x[k] - ref) / np.linalg.norm(ref)
                assert err <= 1e-5 * cond + 1e-6, (name, k, err, cond)
        print(f"plane fit {name}: {n} sets, {int(flag.sum())} accepted")
        total += n
    print(f"plane fit: {total} sets, {time.time() - t0:.2f} s")


# ---------------------------------------------------------------------------------------------------------------
# Umeyama and pose_to_T


def rot(axis, angle):
    axis = np.asarray(axis, np.float64); axis = axis / np.linalg.norm(axis)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    return np.eye(3) + math.sin(angle) * K + (1 - math.cos(angle)) * K @ K


def test_umeyama(harness, oracle):
    """umeyama_rotation_dev equals the oracle's umeyama_rotation bit for bit, and f64 Kabsch within 2e-6 where the
    rotation is unique (sigma of rank >= 2 with distinct or repeated but well separated-from-zero singular values)"""
    rng = np.random.default_rng(31)
    sig, unique = [], []
    for t in range(300):  # rotations up to and including 180 degrees, full-rank and coplanar clouds, reflections
        angle = math.pi if t % 30 == 0 else rng.uniform(0, math.pi)
        R = rot(rng.normal(size=3), angle)
        Cs = np.diag(rng.uniform(0.5, 5, 3) ** 2)
        if t % 3 == 1:
            Cs[2, 2] = 0.0  # coplanar: rank 2
        S = R @ Cs
        if t % 3 == 2:
            S = np.diag([1.0, 1.0, -1.0]) @ S  # reflection: det(U) det(V) < 0
        sig.append(S); unique.append(True)
    for t in range(40):  # near-identity and repeated singular values (c R)
        R = rot(rng.normal(size=3), 10.0 ** rng.uniform(-7, -2))
        sig.append(R * rng.uniform(0.1, 10)); unique.append(True)
        sig.append(rot(rng.normal(size=3), rng.uniform(0, 3)) @ np.diag([2.0, 2.0, 0.5])); unique.append(True)
    for t in range(40):  # collinear (rank 1) and zero sigma: no unique answer, only the oracle
        a, b = rng.normal(size=3), rng.normal(size=3)
        sig.append(np.outer(a, b)); unique.append(False)
    sig.append(np.zeros((3, 3))); unique.append(False)
    sig = np.array(sig).astype(np.float32); unique = np.array(unique)
    got = harness.umeyama(sig)
    want = np.array([oracle.umeyama_rotation(s) for s in sig])
    assert biteq(got, want), ("umeyama", first_diff(got, want))
    worst = 0.0
    for k in np.where(unique)[0]:
        U, s, Vt = np.linalg.svd(sig[k].astype(np.float64))
        d = np.sign(np.linalg.det(U) * np.linalg.det(Vt))
        R = U @ np.diag([1.0, 1.0, d]) @ Vt
        err = np.abs(got[k] - R).max(); worst = max(worst, err)
        assert err <= 2e-6, (k, err)
    print(f"umeyama: {len(sig)} cross-covariances, max |R - Kabsch| = {worst:.3g} over {int(unique.sum())} unique ones")


def test_pose_to_T(harness, oracle):
    """pose_to_T and warp_refresh_transform against oracle.pose_to_T (f64 sin / cos rounded to f32, as glibc's)"""
    rng = np.random.default_rng(41)
    n = 100_000
    pose = rng.uniform(-math.pi, math.pi, (n, 6)).astype(np.float32)
    pose[:, 3:] = rng.normal(size=(n, 3)) * 50
    special = np.array([0.0, math.pi / 2, -math.pi / 2, math.pi, -math.pi, 1e-30, -0.0, 1e3, -1e3, 999.9, 3 * math.pi],
                       np.float32)
    m = len(special)
    extra = np.zeros((m * 3 + 2000, 6), np.float32)
    for a in range(3):
        extra[a * m:(a + 1) * m, a] = special
    extra[3 * m:, :3] = rng.uniform(-1e3, 1e3, (2000, 3))
    pose = np.concatenate([pose, extra])
    T, Tw, trig = harness.pose_to_T(pose)
    want = np.array([oracle.pose_to_T(p) for p in pose])
    assert biteq(T, want), ("pose_to_T", first_diff(T, want))
    assert biteq(Tw, want), ("warp_refresh_transform", first_diff(Tw, want))
    s = np.array([[math.sin(float(p[2])), math.cos(float(p[2])), math.sin(float(p[1])), math.cos(float(p[1])),
                   math.sin(float(p[0])), math.cos(float(p[0]))] for p in pose], np.float64).astype(np.float32)
    assert biteq(trig, s), ("LM trig", first_diff(trig, s))
    print(f"pose_to_T: {len(pose)} poses")
