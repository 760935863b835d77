// pose_math.cuh — device-side small math of the scan-to-map path.  Compiled with -fmad=false: every
// f32 expression keeps the reference's operation order and rounding (an x86-64 baseline build of the
// reference has no FMA contraction), so results can be compared bit for bit with the CPU oracle.
#pragma once
#include <cuda_runtime.h>
#include <float.h>

namespace liogpu {

// pcl::getTransformation(x,y,z,roll,pitch,yaw) as used by trans2Affine3f (mapOptmization.cpp:887-890)
// and transformPointCloud (:856): Rz*Ry*Rx with f32 products.  Trig: f64 sin/cos rounded to f32 (the
// canonical choice shared with the oracle; DESIGN.md "transform drift").  T row-major 3x4.
__device__ __forceinline__ void pose_to_T(const float* pose, float* T) {
  const float roll = pose[0], pitch = pose[1], yaw = pose[2];
  const float A = (float)cos((double)yaw), B = (float)sin((double)yaw);
  const float C = (float)cos((double)pitch), D = (float)sin((double)pitch);
  const float E = (float)cos((double)roll), F = (float)sin((double)roll);
  const float DE = D * E, DF = D * F;
  T[0] = A * C;  T[1] = A * DF - B * E;  T[2] = B * F + A * DE;  T[3] = pose[3];
  T[4] = B * C;  T[5] = A * E + B * DF;  T[6] = B * DE - A * F;  T[7] = pose[4];
  T[8] = -D;     T[9] = C * F;           T[10] = C * E;          T[11] = pose[5];
}

// pointAssociateToMap (mapOptmization.cpp:841-847)
__device__ __forceinline__ float4 apply_T(const float* T, const float4 p) {
  float4 o;
  o.x = T[0] * p.x + T[1] * p.y + T[2] * p.z + T[3];
  o.y = T[4] * p.x + T[5] * p.y + T[6] * p.z + T[7];
  o.z = T[8] * p.x + T[9] * p.y + T[10] * p.z + T[11];
  o.w = p.w;
  return o;
}

// ---------------------------------------------------------------------------------------------
// Eigen::Matrix<float,5,3>::colPivHouseholderQr().solve(-1) (mapOptmization.cpp:1633-1648), the
// unblocked column-pivoted Householder QR of Eigen 3.3.7 (SURVEY A.3).  a[r][c] lives in registers:
// every loop is fully unrolled and the dynamic pivot column is resolved with predicated swaps.
__device__ __forceinline__ void swapf(float& a, float& b) { const float t = a; a = b; b = t; }
__device__ __forceinline__ void swapi(int& a, int& b) { const int t = a; a = b; b = t; }

__device__ __forceinline__ void plane_qr53(float a[5][3], float x[3]) {
  float hc[3], nu[3], nd[3];
  int perm[3] = {0, 1, 2};
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 5; ++i) s += a[i][j] * a[i][j];
    nd[j] = nu[j] = sqrtf(s);
  }
  float maxn = nu[0];
  if (nu[1] > maxn) maxn = nu[1];
  if (nu[2] > maxn) maxn = nu[2];
  const float th = (maxn * FLT_EPSILON) * (maxn * FLT_EPSILON) / 5.0f;
  const float downdate_th = sqrtf(FLT_EPSILON);
  int nonzero = 3;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    int big = k;
#pragma unroll
    for (int j = k + 1; j < 3; ++j) {
      // nu[big] with dynamic big: resolve through selects so everything stays in registers
      const float cur = (big == 0) ? nu[0] : ((big == 1) ? nu[1] : nu[2]);
      if (nu[j] > cur) big = j;
    }
    const float nb = (big == 0) ? nu[0] : ((big == 1) ? nu[1] : nu[2]);
    const float bigsq = nb * nb;
    if (nonzero == 3 && bigsq < th * (float)(5 - k)) nonzero = k;
#pragma unroll
    for (int j = k + 1; j < 3; ++j) {
      if (big == j) {
#pragma unroll
        for (int i = 0; i < 5; ++i) swapf(a[i][k], a[i][j]);
        swapf(nu[k], nu[j]);
        swapf(nd[k], nd[j]);
        swapi(perm[k], perm[j]);
      }
    }
    float tail = 0.f;
#pragma unroll
    for (int i = k + 1; i < 5; ++i) tail += a[i][k] * a[i][k];
    const float c0 = a[k][k];
    float beta, tau;
    if (tail <= FLT_MIN) {
      tau = 0.f; beta = c0;
#pragma unroll
      for (int i = k + 1; i < 5; ++i) a[i][k] = 0.f;
    } else {
      beta = sqrtf(c0 * c0 + tail);
      if (c0 >= 0.f) beta = -beta;
      const float den = c0 - beta;
#pragma unroll
      for (int i = k + 1; i < 5; ++i) a[i][k] = a[i][k] / den;
      tau = (beta - c0) / beta;
    }
    a[k][k] = beta;
    hc[k] = tau;
    if (tau != 0.f) {
#pragma unroll
      for (int j = k + 1; j < 3; ++j) {
        float tmp = 0.f;
#pragma unroll
        for (int i = k + 1; i < 5; ++i) tmp += a[i][k] * a[i][j];
        tmp += a[k][j];
        a[k][j] -= tau * tmp;
#pragma unroll
        for (int i = k + 1; i < 5; ++i) a[i][j] -= (tau * a[i][k]) * tmp;
      }
    }
#pragma unroll
    for (int j = k + 1; j < 3; ++j) {
      if (nu[j] != 0.f) {
        float temp = fabsf(a[k][j]) / nu[j];
        temp = (1.f + temp) * (1.f - temp);
        temp = temp < 0.f ? 0.f : temp;
        const float ratio = nu[j] / nd[j];
        const float temp2 = temp * (ratio * ratio);
        if (temp2 <= downdate_th) {
          float s = 0.f;
#pragma unroll
          for (int i = k + 1; i < 5; ++i) s += a[i][j] * a[i][j];
          nd[j] = sqrtf(s);
          nu[j] = nd[j];
        } else {
          nu[j] *= sqrtf(temp);
        }
      }
    }
  }
  x[0] = x[1] = x[2] = 0.f;
  if (nonzero == 0) return;
  float c[5] = {-1.f, -1.f, -1.f, -1.f, -1.f};  // matB0.fill(-1), :1638
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    if (k < nonzero && hc[k] != 0.f) {
      float tmp = 0.f;
#pragma unroll
      for (int i = k + 1; i < 5; ++i) tmp += a[i][k] * c[i];
      tmp += c[k];
      c[k] -= hc[k] * tmp;
#pragma unroll
      for (int i = k + 1; i < 5; ++i) c[i] -= (hc[k] * a[i][k]) * tmp;
    }
  }
#pragma unroll
  for (int i = 2; i >= 0; --i) {
    if (i < nonzero) {
      c[i] = c[i] / a[i][i];
#pragma unroll
      for (int r = 0; r < i; ++r) c[r] -= c[i] * a[r][i];
    }
  }
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    if (i < nonzero) {
      if (perm[i] == 0) x[0] = c[i];
      else if (perm[i] == 1) x[1] = c[i];
      else x[2] = c[i];
    }
  }
}

// Body of the OpenMP loop of surfOptimization after the k-NN (mapOptmization.cpp:1641-1684).
// nbr = the five neighbours (ascending distance); returns the accept flag, coeff = (s pa, s pb, s pc, s pd2).
__device__ __forceinline__ bool plane_residual(const float4 ori, const float4 sel, const float4 nbr[5], float4& coeff) {
  float a[5][3], x[3];
#pragma unroll
  for (int j = 0; j < 5; ++j) { a[j][0] = nbr[j].x; a[j][1] = nbr[j].y; a[j][2] = nbr[j].z; }
  plane_qr53(a, x);
  float pa = x[0], pb = x[1], pc = x[2], pd = 1.f;
  const float ps = sqrtf(pa * pa + pb * pb + pc * pc);
  pa /= ps; pb /= ps; pc /= ps; pd /= ps;
  bool valid = true;
#pragma unroll
  for (int j = 0; j < 5; ++j) {
    const float r = pa * nbr[j].x + pb * nbr[j].y + pc * nbr[j].z + pd;
    if ((double)fabsf(r) > 0.2) valid = false;  // :1662 compares against a double literal
  }
  const float pd2 = pa * sel.x + pb * sel.y + pc * sel.z + pd;
  const float r2 = ori.x * ori.x + ori.y * ori.y + ori.z * ori.z;
  // :1671 — the 0.9 literal makes the quotient f64; sqrt(sqrt(float)) stays f32 (std:: overloads)
  const float s = (float)(1.0 - 0.9 * (double)fabsf(pd2) / (double)sqrtf(sqrtf(r2)));
  coeff = make_float4(s * pa, s * pb, s * pc, s * pd2);
  return valid && ((double)s > 0.1);
}

// ---------------------------------------------------------------------------------------------
// LMOptimization (mapOptmization.cpp:1702-1837)
struct LmTrig { float srx, crx, sry, cry, srz, crz; };
__device__ __forceinline__ LmTrig lm_trig(const float* pose) {  // :1714-1719
  LmTrig t;
  t.srx = (float)sin((double)pose[2]); t.crx = (float)cos((double)pose[2]);
  t.sry = (float)sin((double)pose[1]); t.cry = (float)cos((double)pose[1]);
  t.srz = (float)sin((double)pose[0]); t.crz = (float)cos((double)pose[0]);
  return t;
}
// One row of matA and matB (:1760-1778): row = (arz, ary, arx, cx, cy, cz), rhs = -coeff.intensity.
__device__ __forceinline__ void jacobian_row(const LmTrig g, const float4 o, const float4 c, float row[6], float& rhs) {
  const float srx = g.srx, crx = g.crx, sry = g.sry, cry = g.cry, srz = g.srz, crz = g.crz;
  const float arx = (-srx * cry * o.x - (srx * sry * srz + crx * crz) * o.y + (crx * srz - srx * sry * crz) * o.z) * c.x
                  + (crx * cry * o.x - (srx * crz - crx * sry * srz) * o.y + (crx * sry * crz + srx * srz) * o.z) * c.y;
  const float ary = (-crx * sry * o.x + crx * cry * srz * o.y + crx * cry * crz * o.z) * c.x
                  + (-srx * sry * o.x + srx * sry * srz * o.y + srx * cry * crz * o.z) * c.y
                  + (-cry * o.x - sry * srz * o.y - sry * crz * o.z) * c.z;
  const float arz = ((crx * sry * crz + srx * srz) * o.y + (srx * crz - crx * sry * srz) * o.z) * c.x
                  + ((-crx * srz + srx * sry * crz) * o.y + (-srx * sry * srz - crx * crz) * o.z) * c.y
                  + (cry * crz * o.y - cry * srz * o.z) * c.z;
  row[0] = arz; row[1] = ary; row[2] = arx; row[3] = c.x; row[4] = c.y; row[5] = c.z;
  rhs = -c.w;
}

// ---- OpenCV 4.x 6x6 pieces (SURVEY A.4): the solve / eigen / inverse routines live in lm_tail.cuh ----
__device__ __forceinline__ float cv_hypotf(float a, float b) {
  a = fabsf(a); b = fabsf(b);
  if (a > b) { b /= a; return a * sqrtf(1 + b * b); }
  if (b > 0) { a /= b; return b * sqrtf(1 + a * a); }
  return 0.f;
}

// ---------------------------------------------------------------------------------------------
// Eigen::umeyama (no scaling), the rotation of every ICP iteration (icp.cu) from the cross-covariance sigma (row-major
// 3x3): one-sided Jacobi SVD in f64, then R = U diag(1, 1, d) V^T; same operation order as the oracle's restatement.
__device__ __forceinline__ void umeyama_rotation_dev(const float sigma[9], float R[9]) {
  double A[3][3], V[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) A[i][j] = (double)sigma[3 * i + j];
  for (int sweep = 0; sweep < 60; ++sweep) {
    bool rotated = false;
    for (int p = 0; p < 2; ++p)
      for (int q = p + 1; q < 3; ++q) {
        double alpha = 0, beta = 0, gamma = 0;
        for (int i = 0; i < 3; ++i) { alpha += A[i][p] * A[i][p]; beta += A[i][q] * A[i][q]; gamma += A[i][p] * A[i][q]; }
        if (gamma == 0.0 || fabs(gamma) <= 1e-17 * sqrt(alpha * beta)) continue;
        rotated = true;
        const double zeta = (beta - alpha) / (2.0 * gamma);
        const double t = (zeta >= 0.0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
        const double c = 1.0 / sqrt(1.0 + t * t), sn = c * t;
        for (int i = 0; i < 3; ++i) {
          const double ap = A[i][p], aq = A[i][q];
          A[i][p] = c * ap - sn * aq; A[i][q] = sn * ap + c * aq;
          const double vp = V[i][p], vq = V[i][q];
          V[i][p] = c * vp - sn * vq; V[i][q] = sn * vp + c * vq;
        }
      }
    if (!rotated) break;
  }
  double sv[3], U[3][3];
  for (int j = 0; j < 3; ++j) sv[j] = sqrt(A[0][j] * A[0][j] + A[1][j] * A[1][j] + A[2][j] * A[2][j]);
  int lo = 0;
  if (sv[1] < sv[lo]) lo = 1;
  if (sv[2] < sv[lo]) lo = 2;
  const int a = (lo + 1) % 3, b = (lo + 2) % 3;
  for (int j = 0; j < 3; ++j)
    for (int i = 0; i < 3; ++i) U[i][j] = sv[j] > 0.0 ? A[i][j] / sv[j] : 0.0;
  if (!(sv[lo] > 1e-12 * (sv[a] > sv[b] ? sv[a] : sv[b]))) {  // rank-deficient: complete U right-handed
    U[0][lo] = U[1][a] * U[2][b] - U[2][a] * U[1][b];
    U[1][lo] = U[2][a] * U[0][b] - U[0][a] * U[2][b];
    U[2][lo] = U[0][a] * U[1][b] - U[1][a] * U[0][b];
  }
  const double detU = U[0][0] * (U[1][1] * U[2][2] - U[1][2] * U[2][1]) - U[0][1] * (U[1][0] * U[2][2] - U[1][2] * U[2][0]) +
                      U[0][2] * (U[1][0] * U[2][1] - U[1][1] * U[2][0]);
  const double detV = V[0][0] * (V[1][1] * V[2][2] - V[1][2] * V[2][1]) - V[0][1] * (V[1][0] * V[2][2] - V[1][2] * V[2][0]) +
                      V[0][2] * (V[1][0] * V[2][1] - V[1][1] * V[2][0]);
  const double d = detU * detV < 0.0 ? -1.0 : 1.0;
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      const double r = U[i][a] * V[j][a] + U[i][b] * V[j][b] + d * (U[i][lo] * V[j][lo]);
      R[3 * i + j] = (float)r;
    }
}

}  // namespace liogpu
