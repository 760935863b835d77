// lm_tail.cuh — the 6x6 tail of LMOptimization (mapOptmization.cpp:1721-1835) on the device: the QR solve, OpenCV's
// Jacobi eigen-decomposition and LU inverse, the f64 non-degeneracy certificate, matP, the pose update and the
// convergence test.  Shared by both LM paths (s2m.cu, s2m_fused.cuh) and by tests/small_math_harness.cu, which runs
// each routine on its own against the CPU oracle.
#pragma once
#include "common.cuh"
#include "pose_math.cuh"
#include <limits.h>

namespace liogpu {

// ---- the 6x6 tail of LMOptimization (mapOptmization.cpp:1721-1835), executed by ONE WARP ----
// A single thread walking these 6x6 routines through local memory cost ~90 us per iteration (~170 us on
// iteration 0) — more than the search itself.  Here the matrices live in shared memory and the lanes
// take independent elements (columns of the Householder update, Jacobi rotation indices, columns of the
// LU elimination), while every individual element still sees exactly the operation sequence of the
// sequential OpenCV routine restated in pose_math.cuh — so the results stay bit-identical to it.
struct FinSmem {
  float AtA[36], AtB[6], X[6];
  float QA[36], qb[6], vl[6], hf[6];
  float JA[36], W[6], V[36], V2[36], Vi[36];
  int indR[6], indC[6];
};
constexpr unsigned FULL = 0xffffffffu;

// cv::solve(AtA, AtB, X, DECOMP_QR) (:1784) — hal::QR32f Householder (no pivoting), executed by ONE lane
// with every loop fully unrolled: all indices are compile-time constants, so the 6x6 matrix, the rhs and the
// reflector live in registers and the ~600 f32 operations run as straight-line code (about 1 us), in
// exactly the operation order of OpenCV's QRImpl.  (A warp-parallel version over shared memory was 5x
// slower: every step paid a shared-memory round trip and a __syncwarp.)
__device__ __forceinline__ void solve6_qr_reg(const float* __restrict__ Ain, const float* __restrict__ bin,
                                              float* __restrict__ x) {
  const float eps = FLT_EPSILON * 10;
  float A[6][6], b[6], hf[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) {
#pragma unroll
    for (int j = 0; j < 6; ++j) A[i][j] = Ain[i * 6 + j];
    b[i] = bin[i];
  }
#pragma unroll
  for (int l = 0; l < 6; ++l) {
    float vl[6];
    float vn = 0.f;
#pragma unroll
    for (int i = 0; i < 6 - l; ++i) { vl[i] = A[l + i][l]; vn += vl[i] * vl[i]; }
    const float t0 = vl[0];
    vl[0] = vl[0] + (vl[0] >= 0.f ? 1.f : -1.f) * sqrtf(vn);
    vn = sqrtf(vn + vl[0] * vl[0] - t0 * t0);
#pragma unroll
    for (int i = 0; i < 6 - l; ++i) vl[i] /= vn;
#pragma unroll
    for (int j = l; j < 6; ++j) {
      float va = 0.f;
#pragma unroll
      for (int i = l; i < 6; ++i) va += vl[i - l] * A[i][j];
#pragma unroll
      for (int i = l; i < 6; ++i) A[i][j] -= 2 * vl[i - l] * va;
    }
    hf[l] = vl[0] * vl[0];
#pragma unroll
    for (int i = 1; i < 6 - l; ++i) A[l + i][l] = vl[i] / vl[0];
  }
#pragma unroll
  for (int l = 0; l < 6; ++l) {
    float vb = 0.f;
#pragma unroll
    for (int i = l; i < 6; ++i) vb += (i == l ? 1.f : A[i][l]) * b[i];
#pragma unroll
    for (int i = l; i < 6; ++i) b[i] -= 2 * (i == l ? 1.f : A[i][l]) * vb * hf[l];
  }
  bool ok = true;
#pragma unroll
  for (int i = 5; i >= 0; --i) {
#pragma unroll
    for (int j = 5; j > i; --j) b[i] -= b[j] * A[i][j];
    if (fabsf(A[i][i]) < eps) ok = false;  // cv::solve returns false; the reference ignores it and X stays 0
    b[i] /= A[i][i];
  }
#pragma unroll
  for (int i = 0; i < 6; ++i) x[i] = ok ? b[i] : 0.f;
}
__device__ __forceinline__ void warp_solve6_qr(FinSmem& m, const int lane) {
  if (lane == 0) solve6_qr_reg(m.AtA, m.AtB, m.X);
  __syncwarp();
}

__device__ __forceinline__ int jacobi_argmax_row(const float* A, int idx) {  // indR[idx]: first max of |A[idx][idx+1..5]|
  int mI = idx + 1;
  float mv = fabsf(A[6 * idx + mI]);
  for (int i = idx + 2; i < 6; ++i) {
    const float val = fabsf(A[6 * idx + i]);
    if (mv < val) { mv = val; mI = i; }
  }
  return mI;
}
__device__ __forceinline__ int jacobi_argmax_col(const float* A, int idx) {  // indC[idx]: first max of |A[0..idx-1][idx]|
  int mI = 0;
  float mv = fabsf(A[idx]);
  for (int i = 1; i < idx; ++i) {
    const float val = fabsf(A[6 * i + idx]);
    if (mv < val) { mv = val; mI = i; }
  }
  return mI;
}

// cv::eigen(matAtA, matE, matV) (:1792) — JacobiImpl_<float>: W descending, eigenvectors as rows of V.
__device__ __forceinline__ void warp_eigen6(FinSmem& m, const int lane) {
  for (int e = lane; e < 36; e += 32) { m.JA[e] = m.AtA[e]; m.V[e] = (e / 6 == e % 6) ? 1.f : 0.f; }
  __syncwarp();
  if (lane < 6) {
    m.W[lane] = m.JA[7 * lane];
    if (lane < 5) m.indR[lane] = jacobi_argmax_row(m.JA, lane);
    if (lane > 0) m.indC[lane] = jacobi_argmax_col(m.JA, lane);
  }
  __syncwarp();
  for (int it = 0; it < 6 * 6 * 30; ++it) {
    // pivot: first strict maximum over |A[i][indR[i]]| (i=0..4) then |A[indC[i]][i]| (i=1..5)
    float cand = -1.f;
    if (lane < 5) cand = fabsf(m.JA[6 * lane + m.indR[lane]]);
    else if (lane < 10) cand = fabsf(m.JA[6 * m.indC[lane - 4] + (lane - 4)]);
    // as OpenCV's `if (mv < val)`: a NaN candidate never wins, except the first one, which then stays the pivot
    int cb = __float_as_int(cand);
    if (cand != cand) cb = lane == 0 ? INT_MAX : -1;
    const int mb = __reduce_max_sync(FULL, cb);
    const int pl = __ffs(__ballot_sync(FULL, cb == mb)) - 1;
    int k, l;
    if (pl < 5) { k = pl; l = m.indR[k]; } else { l = pl - 4; k = m.indC[l]; }
    const float p = m.JA[6 * k + l];
    if (fabsf(p) <= FLT_EPSILON) break;
    const float y = (float)((m.W[l] - m.W[k]) * 0.5);
    float t = fabsf(y) + cv_hypotf(p, y);
    float s = cv_hypotf(p, t);
    const float c = t / s;
    s = p / s;
    t = (p / t) * p;
    if (y < 0) { s = -s; t = -t; }
    __syncwarp();
    if (lane == 0) { m.JA[6 * k + l] = 0; m.W[k] -= t; m.W[l] += t; }
    if (lane < 6 && lane != k && lane != l) {  // rotate rows and columns k and l of the upper triangle
      const int i = lane;
      const int r0 = i < k ? 6 * i + k : 6 * k + i;
      const int r1 = i < l ? 6 * i + l : 6 * l + i;
      const float a0 = m.JA[r0], b0 = m.JA[r1];
      m.JA[r0] = a0 * c - b0 * s;
      m.JA[r1] = a0 * s + b0 * c;
    } else if (lane >= 8 && lane < 14) {        // rotate the eigenvectors
      const int i = lane - 8;
      const float a0 = m.V[6 * k + i], b0 = m.V[6 * l + i];
      m.V[6 * k + i] = a0 * c - b0 * s;
      m.V[6 * l + i] = a0 * s + b0 * c;
    }
    __syncwarp();
    if (lane == 0 && k < 5) m.indR[k] = jacobi_argmax_row(m.JA, k);
    if (lane == 1 && k > 0) m.indC[k] = jacobi_argmax_col(m.JA, k);
    if (lane == 2 && l < 5) m.indR[l] = jacobi_argmax_row(m.JA, l);
    if (lane == 3 && l > 0) m.indC[l] = jacobi_argmax_col(m.JA, l);
    __syncwarp();
  }
  __syncwarp();
  for (int k = 0; k < 5; ++k) {  // sort eigenvalues (descending) and eigenvectors
    int mI = k;
    for (int i = k + 1; i < 6; ++i)
      if (m.W[mI] < m.W[i]) mI = i;
    __syncwarp();
    if (k != mI) {
      if (lane == 0) { const float tw = m.W[mI]; m.W[mI] = m.W[k]; m.W[k] = tw; }
      if (lane >= 8 && lane < 14) {
        const int i = lane - 8;
        const float tv = m.V[6 * mI + i]; m.V[6 * mI + i] = m.V[6 * k + i]; m.V[6 * k + i] = tv;
      }
    }
    __syncwarp();
  }
}

// matV.inv() (:1807) — cv::invert DECOMP_LU = hal::LU32f on [V | I].  Lane c < 6 owns column c of V,
// lane 6 + c owns column c of the right-hand side; row operations are identical on every column.
__device__ __forceinline__ void warp_inv6_lu(FinSmem& m, const int lane) {
  float x[6];
  const bool isA = lane < 6, isB = lane >= 6 && lane < 12;
#pragma unroll
  for (int r = 0; r < 6; ++r) x[r] = isA ? m.V[r * 6 + lane] : ((isB && r == lane - 6) ? 1.f : 0.f);
  bool ok = true;
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    int k = i;  // pivot: first row with the largest |A[j][i]|, j >= i (computed by the owner of column i)
    float best = fabsf(x[i]);
#pragma unroll
    for (int j = i + 1; j < 6; ++j) {
      const float v = fabsf(x[j]);
      if (v > best) { best = v; k = j; }
    }
    k = __shfl_sync(FULL, k, i);
    best = __shfl_sync(FULL, best, i);
    if (best < FLT_EPSILON * 10) { ok = false; break; }
#pragma unroll
    for (int j = i + 1; j < 6; ++j)
      if (k == j) { const float tv = x[i]; x[i] = x[j]; x[j] = tv; }
    const float d = -1 / __shfl_sync(FULL, x[i], i);
#pragma unroll
    for (int j = i + 1; j < 6; ++j) {
      const float alpha = __shfl_sync(FULL, x[j], i) * d;
      if (lane != i) x[j] += alpha * x[i];  // column i itself is left as LUImpl leaves it (never read again)
    }
  }
  if (ok) {
#pragma unroll
    for (int i = 5; i >= 0; --i) {
      float sacc = x[i];
#pragma unroll
      for (int k = i + 1; k < 6; ++k) {
        const float aik = __shfl_sync(FULL, x[i], k);  // A[i][k] lives in lane k
        sacc -= aik * x[k];
      }
      const float aii = __shfl_sync(FULL, x[i], i);
      if (isB) x[i] = sacc / aii;
    }
  }
  if (isB) {
#pragma unroll
    for (int r = 0; r < 6; ++r) m.Vi[r * 6 + (lane - 6)] = ok ? x[r] : 0.f;
  }
  __syncwarp();
}

// transPointAssociateToMap and the LM trig terms of the current pose, computed ONCE per iteration
// instead of once per thread block; lanes 0-2 evaluate the f64 sin/cos of roll, pitch, yaw in parallel.
__device__ __forceinline__ void warp_refresh_transform(LmDevState* st, const int lane, const float pose_l) {
  // pose_l: lane k < 6 holds pose[k] = {roll, pitch, yaw, x, y, z}
  float sn = 0.f, cs = 0.f;
  if (lane < 3) {
    const double a = (double)pose_l;
    sn = (float)sin(a);
    cs = (float)cos(a);
  }
  const float F = __shfl_sync(FULL, sn, 0), E = __shfl_sync(FULL, cs, 0);  // roll
  const float D = __shfl_sync(FULL, sn, 1), C = __shfl_sync(FULL, cs, 1);  // pitch
  const float B = __shfl_sync(FULL, sn, 2), A = __shfl_sync(FULL, cs, 2);  // yaw
  const float px = __shfl_sync(FULL, pose_l, 3), py = __shfl_sync(FULL, pose_l, 4), pz = __shfl_sync(FULL, pose_l, 5);
  if (lane == 0) {  // pcl::getTransformation — same products as pose_to_T
    const float DE = D * E, DF = D * F;
    float* T = st->T;
    T[0] = A * C;  T[1] = A * DF - B * E;  T[2] = B * F + A * DE;  T[3] = px;
    T[4] = B * C;  T[5] = A * E + B * DF;  T[6] = B * DE - A * F;  T[7] = py;
    T[8] = -D;     T[9] = C * F;           T[10] = C * E;          T[11] = pz;
    // srx,crx = sin,cos(yaw); sry,cry = (pitch); srz,crz = (roll)  (:1714-1719)
    st->trig[0] = B; st->trig[1] = A; st->trig[2] = D; st->trig[3] = C; st->trig[4] = F; st->trig[5] = E;
  }
}

// lambda_min(A) > mu  <=>  A - mu*I is positive definite  <=>  its LDL^T has positive pivots (f64, static
// indices: everything stays in registers).  mu = 100 + 1e-4 * trace(A).
__device__ __forceinline__ bool certify_min_eig(const float* A32) {
  double a[6][6];
  double tr = 0;
#pragma unroll
  for (int i = 0; i < 6; ++i) tr += (double)A32[i * 6 + i];
  if (!(tr > 0)) return false;
  const double mu = 100.0 + 1e-4 * tr;
#pragma unroll
  for (int i = 0; i < 6; ++i)
#pragma unroll
    for (int j = 0; j < 6; ++j) a[i][j] = (double)A32[i * 6 + j] - (i == j ? mu : 0.0);
  bool ok = true;
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    const double piv = a[k][k];
    if (!(piv > 1e-3 * mu)) ok = false;  // also rejects NaN; keeps a margin against cancellation
    const double inv = 1.0 / piv;
#pragma unroll
    for (int i = k + 1; i < 6; ++i) {
      const double f = a[i][k] * inv;
#pragma unroll
      for (int j = k + 1; j <= i; ++j) a[i][j] -= f * a[j][k];
    }
  }
  return ok;
}

// cv::eigen + the degeneracy loop + matP = matV.inv() * matV2 (:1792-1808) on m.AtA, one warp.  Returns isDegenerate
// on every lane; the callers decide where it goes (st->degenerate, or the certificate's tripwire).
__device__ __forceinline__ int lm_eigen_matp(FinSmem& m, const int lane, float* matP_out) {
  warp_eigen6(m, lane);
  for (int e = lane; e < 36; e += 32) m.V2[e] = m.V[e];
  __syncwarp();
  int deg = 0;
  if (lane == 0) {
    for (int i = 5; i >= 0; --i) {
      if (m.W[i] < 100.f) {
        for (int j = 0; j < 6; ++j) m.V2[i * 6 + j] = 0.f;
        deg = 1;
      } else {
        break;
      }
    }
  }
  deg = __shfl_sync(FULL, deg, 0);
  __syncwarp();
  warp_inv6_lu(m, lane);
  for (int e = lane; e < 36; e += 32) {  // f64 accumulation, as cv::gemm does
    const int i = e / 6, j = e % 6;
    double acc = 0;
    for (int k = 0; k < 6; ++k) acc += (double)m.Vi[i * 6 + k] * (double)m.V2[k * 6 + j];
    matP_out[e] = (float)acc;
  }
  return deg;
}

__device__ __noinline__ void lm_finalize_warp(LmDevState* st, const double* sums, FinSmem& m, const int lane) {
  // one batch of loads for every state field the tail needs (instead of a chain of dependent L2 reads)
  float pose_l = lane < 6 ? st->pose[lane] : 0.f;
  const int it = st->iter, max_iter = st->max_iter;
  int degenerate = st->degenerate;
  const int nsel = (int)sums[27];
  // expand the upper triangle; AtA(a,b) and AtA(b,a) are the same f64 sum of the same products
  for (int e = lane; e < 36; e += 32) {
    int a = e / 6, b = e % 6;
    if (a > b) { const int tt = a; a = b; b = tt; }
    const double v = sums[a * 6 - (a * (a - 1)) / 2 + (b - a)];
    st->JtJ[e] = v;
    m.AtA[e] = (float)v;
  }
  if (lane < 6) { st->Jtr[lane] = sums[21 + lane]; m.AtB[lane] = (float)sums[21 + lane]; }
  if (lane == 0) { st->n_sel = nsel; st->tie_queries = (int)sums[28]; st->nsel_hist[it] = nsel; st->seeded = (int)sums[29]; }
  __syncwarp();
  bool conv = false;
  if (nsel >= 50) {  // :1721-1724 — below 50 the pose is untouched and the loop just repeats
    warp_solve6_qr(m, lane);
    if (it == 0) {  // :1786-1808
      // cv::eigen (a few hundred dependent steps) is only needed to DECIDE isDegenerate and, if so, to
      // build matP.  A rigorous certificate settles the common case at once: if AtA - mu*I is positive
      // definite (LDL^T in f64, mu = 100 + 1e-4*trace, i.e. >1000 f32 ulps of ||AtA|| above the threshold)
      // every eigenvalue OpenCV's f32 Jacobi can report is >= 100, so isDegenerate = false and matP is not
      // read by this scan.  The exact matP (= V^-1 * V2) is then computed from the saved AtA by
      // lm_matp_kernel on a second stream while iterations 1.. run; otherwise the exact path runs here.
      bool certified = false;
      if (lane == 0) certified = certify_min_eig(m.AtA);
      certified = __shfl_sync(FULL, (int)certified, 0) != 0;
      for (int e = lane; e < 36; e += 32) st->AtA0[e] = m.AtA[e];
      if (certified) {
        degenerate = 0;
        if (lane == 0) { st->degenerate = 0; st->eig_pending = 1; }
      } else {
        degenerate = lm_eigen_matp(m, lane, st->matP);
        if (lane == 0) st->degenerate = degenerate;
      }
      __threadfence_block();
      __syncwarp();
    }
    float xi = lane < 6 ? m.X[lane] : 0.f;
    if (degenerate && lane < 6) {  // :1810-1815
      double acc = 0;
      for (int k = 0; k < 6; ++k) acc += (double)st->matP[lane * 6 + k] * (double)m.X[k];
      xi = (float)acc;
    }
    pose_l += xi;
    if (lane < 6) st->pose[lane] = pose_l;
    const float r2d = 57.29578f;  // pcl::rad2deg(float)
    const float x0 = __shfl_sync(FULL, xi, 0), x1 = __shfl_sync(FULL, xi, 1), x2 = __shfl_sync(FULL, xi, 2);
    const float x3 = __shfl_sync(FULL, xi, 3), x4 = __shfl_sync(FULL, xi, 4), x5 = __shfl_sync(FULL, xi, 5);
    const float rx = x0 * r2d, ry = x1 * r2d, rz = x2 * r2d;
    const float dr = (float)sqrt((double)rx * rx + (double)ry * ry + (double)rz * rz);
    const float tx = x3 * 100, ty = x4 * 100, tz = x5 * 100;
    const float dt = (float)sqrt((double)tx * tx + (double)ty * ty + (double)tz * tz);
    if (lane == 0) { st->delta_r = dr; st->delta_t = dt; }
    conv = ((double)dr < 0.05) && ((double)dt < 0.05);
  }
  if (lane < 6) st->pose_hist[it][lane] = pose_l;
  int iter = it + 1;
  if (nsel < 50) {
    // Nothing changed, so every remaining iteration of the reference's loop would redo identical work
    // and bail out at :1722 again (quirk q2): record them and stop instead of burning launches.
    for (int k = it + 1; k < max_iter; ++k) {
      if (lane < 6) st->pose_hist[k][lane] = pose_l;
      if (lane == 0) st->nsel_hist[k] = nsel;
    }
    iter = max_iter;
  }
  const bool done = conv || iter >= max_iter;
  if (!done) warp_refresh_transform(st, lane, pose_l);
  if (lane == 0) {
    st->iter = iter;
    if (conv) st->converged = 1;
    if (done) st->done = 1;
  }
}

}  // namespace liogpu
