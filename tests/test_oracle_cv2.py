"""The oracle's restatement of the OpenCV pieces of LMOptimization (mapOptmization.cpp:1781-1814) against
the real library: committed fixtures produced by Python cv2 (tests/golden/make_golden.py) and, when cv2 is
importable, the live library on fresh random inputs.  Bit-exact."""
import os

import numpy as np
import pytest

G = np.load(os.path.join(os.path.dirname(__file__), "golden", "cv2_6x6.npz"))
N = int(G["n_cases"])


def biteq(a, b):
    return np.array_equal(np.ascontiguousarray(a, np.float32).view(np.uint32), np.ascontiguousarray(b, np.float32).view(np.uint32))


@pytest.mark.parametrize("k", range(N))
def test_fixture_case(oracle, k):
    A, b = G[f"A_{k}"], G[f"b_{k}"]
    # cv::gemm on CV_32F = f64 accumulation of exact f32 products, rounded once
    AtA = (A.astype(np.float64).T @ A.astype(np.float64)).astype(np.float32)
    Atb = (A.astype(np.float64).T @ b.astype(np.float64)).astype(np.float32)
    assert biteq(AtA, G[f"AtA_{k}"]) and biteq(Atb, G[f"Atb_{k}"])
    ok, X = oracle.cv_solve6_qr(G[f"AtA_{k}"], G[f"Atb_{k}"])
    assert ok == bool(G[f"ok_{k}"])
    if ok:
        assert biteq(X, G[f"X_{k}"]), "cv::solve(DECOMP_QR)"
    W, V = oracle.cv_eigen6(G[f"AtA_{k}"])
    assert biteq(W, G[f"E_{k}"]) and biteq(V, G[f"V_{k}"]), "cv::eigen"
    ok, Vi = oracle.cv_inv6(G[f"V_{k}"])
    assert ok and biteq(Vi, G[f"Vi_{k}"]), "Mat::inv"
    V2 = G[f"V_{k}"].copy()
    for i in range(5, -1, -1):
        if G[f"E_{k}"][i] < 100:
            V2[i, :] = 0
        else:
            break
    assert biteq(oracle.cv_gemm6(Vi, V2), G[f"P_{k}"]), "matP = V.inv() * V2"


def test_normal_equations_match_cv_gemm(oracle):
    # the oracle's AtA/AtB accumulation (f64) rounded to f32 equals cv::gemm's result on the same rows
    rng = np.random.default_rng(1)
    n = 5000
    scan = rng.normal(0, 20, (n, 4)).astype(np.float32)
    coeff = rng.normal(0, 1, (n, 4)).astype(np.float32)
    flag = (rng.uniform(size=n) < 0.8).astype(np.uint8)
    pose = np.array([0.01, -0.02, 0.5, 1, 2, 3], np.float32)
    nsel, JtJ, Jtr = oracle.normal_equations(scan, coeff, flag, pose)
    assert nsel == int(flag.sum())
    assert np.allclose(JtJ, JtJ.T, rtol=0, atol=0)
    # JtJ = At*A cannot be rebuilt without the rows: check symmetry + a round trip through cv::solve(QR), against the
    # outputs make_golden.py stored and, when cv2 is importable, against the library itself
    L = np.load(os.path.join(os.path.dirname(__file__), "golden", "cv2_live.npz"))
    assert np.array_equal(JtJ, L["ne_JtJ"]) and np.array_equal(Jtr, L["ne_Jtr"])
    wants = [(bool(L["ne_ok"]), L["ne_X"])]
    cv2 = import_cv2()
    if cv2 is not None:
        ok, X = cv2.solve(JtJ.astype(np.float32), Jtr.astype(np.float32).reshape(6, 1), flags=cv2.DECOMP_QR)
        wants.append((ok, X[:, 0]))
    ok2, X2 = oracle.cv_solve6_qr(JtJ.astype(np.float32), Jtr.astype(np.float32))
    for ok, X in wants:
        assert ok == ok2 and biteq(X, X2)


def import_cv2():
    try:
        import cv2
        return cv2
    except ImportError:
        return None


def live_cases():
    """the seeded systems of test_live_cv2_random (tests/golden/make_golden.py stores OpenCV's outputs for them)"""
    rng = np.random.default_rng(77)
    for t in range(60):
        n = int(rng.integers(60, 2000))
        A = (rng.normal(size=(n, 6)) * rng.uniform(0.05, 20, size=6)).astype(np.float32)
        yield A, rng.normal(size=(n, 1)).astype(np.float32)


def cv2_live_outputs(cv2, A, b):
    AtA = cv2.gemm(np.ascontiguousarray(A.T), A, 1.0, None, 0.0)
    Atb = cv2.gemm(np.ascontiguousarray(A.T), b, 1.0, None, 0.0)
    ok, X = cv2.solve(AtA, Atb, flags=cv2.DECOMP_QR)
    _, E, V = cv2.eigen(AtA)
    _, Vi = cv2.invert(V, flags=cv2.DECOMP_LU)
    return dict(AtA=AtA, Atb=Atb[:, 0], ok=ok, X=X[:, 0], E=E[:, 0], V=V, Vi=Vi)


def test_live_cv2_random(oracle):
    """the oracle against OpenCV on 60 seeded random systems: against the outputs make_golden.py stored
    (cv2_live.npz) and, when cv2 is importable, against the library itself"""
    L = np.load(os.path.join(os.path.dirname(__file__), "golden", "cv2_live.npz"))
    cv2 = import_cv2()
    for t, (A, b) in enumerate(live_cases()):
        AtA = (A.astype(np.float64).T @ A.astype(np.float64)).astype(np.float32)
        assert biteq(AtA, L[f"AtA_{t}"]), t                   # the stored outputs belong to these inputs
        wants = [{k: L[f"{k}_{t}"] for k in ("AtA", "Atb", "ok", "X", "E", "V", "Vi")}]
        if cv2 is not None:
            wants.append(cv2_live_outputs(cv2, A, b))
        for w in wants:
            ok2, X2 = oracle.cv_solve6_qr(w["AtA"], w["Atb"])
            assert bool(w["ok"]) == ok2 and biteq(w["X"], X2)
            W2, V2 = oracle.cv_eigen6(w["AtA"])
            assert biteq(w["E"], W2) and biteq(w["V"], V2)
            assert biteq(w["Vi"], oracle.cv_inv6(w["V"])[1])
