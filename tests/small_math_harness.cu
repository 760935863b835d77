// small_math_harness.cu — test-only entry points into the device's small-matrix routines (lm_tail.cuh,
// pose_math.cuh), so that tests/test_gpu_small_math.py can compare each one with the CPU oracle case by case.
// Built by `make -C lio_slam_b200/csrc harness` with the library's flags into its own shared object; nothing here is
// part of libliogpu.so or its C ABI.  Every entry takes n cases in host arrays, runs ONE WARP per case (the warp
// routines need a full warp; the single-thread routines run on lane 0), copies the results back and returns a
// cudaError_t (0 = success).
#include "../lio_slam_b200/csrc/lm_tail.cuh"

using namespace liogpu;

namespace {

template <class T>
cudaError_t to_dev(T** d, const T* h, size_t count) {
  cudaError_t e = cudaMalloc((void**)d, count * sizeof(T) + 16);
  if (e != cudaSuccess) return e;
  return h ? cudaMemcpy(*d, h, count * sizeof(T), cudaMemcpyHostToDevice) : cudaMemset(*d, 0, count * sizeof(T) + 16);
}
template <class T>
cudaError_t to_host(T* h, const T* d, size_t count) {
  return cudaMemcpy(h, d, count * sizeof(T), cudaMemcpyDeviceToHost);
}

// one warp per case
__global__ void k_solve6(int n, const float* A, const float* b, float* x) {
  __shared__ FinSmem m;
  const int c = blockIdx.x, lane = threadIdx.x;
  if (c >= n) return;
  for (int e = lane; e < 36; e += 32) m.AtA[e] = A[36 * c + e];
  if (lane < 6) m.AtB[lane] = b[6 * c + lane];
  __syncwarp();
  warp_solve6_qr(m, lane);
  if (lane < 6) x[6 * c + lane] = m.X[lane];
}

__global__ void k_eigen6(int n, const float* A, float* W, float* V) {
  __shared__ FinSmem m;
  const int c = blockIdx.x, lane = threadIdx.x;
  if (c >= n) return;
  for (int e = lane; e < 36; e += 32) m.AtA[e] = A[36 * c + e];
  __syncwarp();
  warp_eigen6(m, lane);
  for (int e = lane; e < 36; e += 32) V[36 * c + e] = m.V[e];
  if (lane < 6) W[6 * c + lane] = m.W[lane];
}

__global__ void k_inv6(int n, const float* V, float* Vi) {
  __shared__ FinSmem m;
  const int c = blockIdx.x, lane = threadIdx.x;
  if (c >= n) return;
  for (int e = lane; e < 36; e += 32) m.V[e] = V[36 * c + e];
  __syncwarp();
  warp_inv6_lu(m, lane);
  for (int e = lane; e < 36; e += 32) Vi[36 * c + e] = m.Vi[e];
}

__global__ void k_matp(int n, const float* A, float* P, int* deg) {
  __shared__ FinSmem m;
  const int c = blockIdx.x, lane = threadIdx.x;
  if (c >= n) return;
  for (int e = lane; e < 36; e += 32) m.AtA[e] = A[36 * c + e];
  __syncwarp();
  const int d = lm_eigen_matp(m, lane, P + 36 * c);
  if (lane == 0) deg[c] = d;
}

__global__ void k_certify(int n, const float* A, int* cert) {
  const int c = blockIdx.x, lane = threadIdx.x;
  if (c >= n || lane != 0) return;
  cert[c] = certify_min_eig(A + 36 * c) ? 1 : 0;
}

// lm_finalize_warp on a state filled from the inputs; when the certificate fired, iteration 0's matP is then computed
// the way lm_matp_kernel does it (the same helper, the same tripwire)
__global__ void k_lm_tail(int n, const double* sums, const int* iter, const float* pose, const float* matP,
                          const int* degenerate, LmDevState* st, float* out_f, int* out_i) {
  __shared__ FinSmem m;
  const int c = blockIdx.x, lane = threadIdx.x;
  if (c >= n) return;
  LmDevState* s = st + c;
  if (lane < 6) s->pose[lane] = pose[6 * c + lane];
  for (int e = lane; e < 36; e += 32) s->matP[e] = matP[36 * c + e];
  if (lane == 0) { s->iter = iter[c]; s->max_iter = LIOGPU_MAX_ITER; s->degenerate = degenerate[c]; }
  __syncwarp();
  __threadfence_block();
  lm_finalize_warp(s, sums + 32 * c, m, lane);
  __syncwarp();
  __threadfence_block();
  const int certified = s->eig_pending;
  __syncwarp();
  if (certified) {
    for (int e = lane; e < 36; e += 32) m.AtA[e] = s->AtA0[e];
    __syncwarp();
    const int deg = lm_eigen_matp(m, lane, s->matP);
    if (lane == 0) {
      if (deg) s->cert_mismatch = 1;
      s->eig_pending = 0;
    }
  }
  __syncwarp();
  __threadfence_block();
  // out_f: pose[6], matP[36], T[12], trig[6], delta_r, delta_t;  out_i: degenerate, certified, cert_mismatch,
  // converged, done, iter
  float* f = out_f + 62 * c;
  if (lane < 6) f[lane] = s->pose[lane];
  for (int e = lane; e < 36; e += 32) f[6 + e] = s->matP[e];
  if (lane < 12) f[42 + lane] = s->T[lane];
  if (lane < 6) f[54 + lane] = s->trig[lane];
  if (lane == 0) {
    f[60] = s->delta_r; f[61] = s->delta_t;
    int* o = out_i + 6 * c;
    o[0] = s->degenerate; o[1] = certified; o[2] = s->cert_mismatch; o[3] = s->converged; o[4] = s->done; o[5] = s->iter;
  }
}

__global__ void k_pose_to_T(int n, const float* pose, float* T, LmDevState* st, float* T_warp, float* trig) {
  const int c = blockIdx.x, lane = threadIdx.x;
  if (c >= n) return;
  if (lane == 0) pose_to_T(pose + 6 * c, T + 12 * c);
  warp_refresh_transform(st + c, lane, lane < 6 ? pose[6 * c + lane] : 0.f);
  __syncwarp();
  __threadfence_block();
  if (lane < 12) T_warp[12 * c + lane] = st[c].T[lane];
  if (lane < 6) trig[6 * c + lane] = st[c].trig[lane];
}

__global__ void k_plane_qr53(int n, const float* A15, float* x3) {
  const int c = blockIdx.x, lane = threadIdx.x;
  if (c >= n || lane != 0) return;
  float a[5][3], x[3];
  for (int i = 0; i < 5; ++i)
    for (int j = 0; j < 3; ++j) a[i][j] = A15[15 * c + 3 * i + j];
  plane_qr53(a, x);
  for (int j = 0; j < 3; ++j) x3[3 * c + j] = x[j];
}

__global__ void k_plane_residual(int n, const float4* ori, const float4* sel, const float4* nbr, float4* coeff,
                                 int* flag) {
  const int c = blockIdx.x, lane = threadIdx.x;
  if (c >= n || lane != 0) return;
  float4 nb[5];
  for (int j = 0; j < 5; ++j) nb[j] = nbr[5 * c + j];
  float4 co;
  flag[c] = plane_residual(ori[c], sel[c], nb, co) ? 1 : 0;
  coeff[c] = co;
}

__global__ void k_umeyama(int n, const float* sigma, float* R) {
  const int c = blockIdx.x, lane = threadIdx.x;
  if (c >= n || lane != 0) return;
  umeyama_rotation_dev(sigma + 9 * c, R + 9 * c);
}

#define SMH_TRY(x) do { const cudaError_t e_ = (x); if (e_ != cudaSuccess) { rc = e_; goto out; } } while (0)
#define SMH_LAUNCH(kern, ...) do { kern<<<n, 32>>>(__VA_ARGS__); SMH_TRY(cudaGetLastError()); SMH_TRY(cudaDeviceSynchronize()); } while (0)

}  // namespace

extern "C" {

int smh_solve6(int n, const float* A, const float* b, float* x) {
  cudaError_t rc = cudaSuccess;
  float *dA = nullptr, *db = nullptr, *dx = nullptr;
  if (n <= 0) return 0;
  SMH_TRY(to_dev(&dA, A, 36 * (size_t)n)); SMH_TRY(to_dev(&db, b, 6 * (size_t)n)); SMH_TRY(to_dev<float>(&dx, nullptr, 6 * (size_t)n));
  SMH_LAUNCH(k_solve6, n, dA, db, dx);
  SMH_TRY(to_host(x, dx, 6 * (size_t)n));
out:
  cudaFree(dA); cudaFree(db); cudaFree(dx);
  return (int)rc;
}

int smh_eigen6(int n, const float* A, float* W, float* V) {
  cudaError_t rc = cudaSuccess;
  float *dA = nullptr, *dW = nullptr, *dV = nullptr;
  if (n <= 0) return 0;
  SMH_TRY(to_dev(&dA, A, 36 * (size_t)n)); SMH_TRY(to_dev<float>(&dW, nullptr, 6 * (size_t)n)); SMH_TRY(to_dev<float>(&dV, nullptr, 36 * (size_t)n));
  SMH_LAUNCH(k_eigen6, n, dA, dW, dV);
  SMH_TRY(to_host(W, dW, 6 * (size_t)n)); SMH_TRY(to_host(V, dV, 36 * (size_t)n));
out:
  cudaFree(dA); cudaFree(dW); cudaFree(dV);
  return (int)rc;
}

int smh_inv6(int n, const float* V, float* Vi) {
  cudaError_t rc = cudaSuccess;
  float *dV = nullptr, *dVi = nullptr;
  if (n <= 0) return 0;
  SMH_TRY(to_dev(&dV, V, 36 * (size_t)n)); SMH_TRY(to_dev<float>(&dVi, nullptr, 36 * (size_t)n));
  SMH_LAUNCH(k_inv6, n, dV, dVi);
  SMH_TRY(to_host(Vi, dVi, 36 * (size_t)n));
out:
  cudaFree(dV); cudaFree(dVi);
  return (int)rc;
}

int smh_matp(int n, const float* A, float* P, int* deg) {
  cudaError_t rc = cudaSuccess;
  float *dA = nullptr, *dP = nullptr;
  int* dd = nullptr;
  if (n <= 0) return 0;
  SMH_TRY(to_dev(&dA, A, 36 * (size_t)n)); SMH_TRY(to_dev<float>(&dP, nullptr, 36 * (size_t)n)); SMH_TRY(to_dev<int>(&dd, nullptr, (size_t)n));
  SMH_LAUNCH(k_matp, n, dA, dP, dd);
  SMH_TRY(to_host(P, dP, 36 * (size_t)n)); SMH_TRY(to_host(deg, dd, (size_t)n));
out:
  cudaFree(dA); cudaFree(dP); cudaFree(dd);
  return (int)rc;
}

int smh_certify(int n, const float* A, int* cert) {
  cudaError_t rc = cudaSuccess;
  float* dA = nullptr;
  int* dc = nullptr;
  if (n <= 0) return 0;
  SMH_TRY(to_dev(&dA, A, 36 * (size_t)n)); SMH_TRY(to_dev<int>(&dc, nullptr, (size_t)n));
  SMH_LAUNCH(k_certify, n, dA, dc);
  SMH_TRY(to_host(cert, dc, (size_t)n));
out:
  cudaFree(dA); cudaFree(dc);
  return (int)rc;
}

// sums: n x 32 (upper triangle of JtJ row by row, Jtr, nsel, ties, seeded, 0, 0)
int smh_lm_tail(int n, const double* sums, const int* iter, const float* pose, const float* matP, const int* degenerate,
                float* out_f, int* out_i) {
  cudaError_t rc = cudaSuccess;
  double* ds = nullptr;
  int *di = nullptr, *dd = nullptr, *doi = nullptr;
  float *dp = nullptr, *dm = nullptr, *dof = nullptr;
  LmDevState* st = nullptr;
  if (n <= 0) return 0;
  SMH_TRY(to_dev(&ds, sums, 32 * (size_t)n)); SMH_TRY(to_dev(&di, iter, (size_t)n)); SMH_TRY(to_dev(&dd, degenerate, (size_t)n));
  SMH_TRY(to_dev(&dp, pose, 6 * (size_t)n)); SMH_TRY(to_dev(&dm, matP, 36 * (size_t)n));
  SMH_TRY(to_dev<float>(&dof, nullptr, 62 * (size_t)n)); SMH_TRY(to_dev<int>(&doi, nullptr, 6 * (size_t)n));
  SMH_TRY(to_dev<LmDevState>(&st, nullptr, (size_t)n));
  SMH_LAUNCH(k_lm_tail, n, ds, di, dp, dm, dd, st, dof, doi);
  SMH_TRY(to_host(out_f, dof, 62 * (size_t)n)); SMH_TRY(to_host(out_i, doi, 6 * (size_t)n));
out:
  cudaFree(ds); cudaFree(di); cudaFree(dd); cudaFree(dp); cudaFree(dm); cudaFree(dof); cudaFree(doi); cudaFree(st);
  return (int)rc;
}

// T: pose_to_T (one thread), T_warp / trig: warp_refresh_transform (lanes 0-2 evaluate the trig)
int smh_pose_to_T(int n, const float* pose, float* T, float* T_warp, float* trig) {
  cudaError_t rc = cudaSuccess;
  float *dp = nullptr, *dT = nullptr, *dTw = nullptr, *dg = nullptr;
  LmDevState* st = nullptr;
  if (n <= 0) return 0;
  SMH_TRY(to_dev(&dp, pose, 6 * (size_t)n)); SMH_TRY(to_dev<float>(&dT, nullptr, 12 * (size_t)n));
  SMH_TRY(to_dev<float>(&dTw, nullptr, 12 * (size_t)n)); SMH_TRY(to_dev<float>(&dg, nullptr, 6 * (size_t)n));
  SMH_TRY(to_dev<LmDevState>(&st, nullptr, (size_t)n));
  SMH_LAUNCH(k_pose_to_T, n, dp, dT, st, dTw, dg);
  SMH_TRY(to_host(T, dT, 12 * (size_t)n)); SMH_TRY(to_host(T_warp, dTw, 12 * (size_t)n)); SMH_TRY(to_host(trig, dg, 6 * (size_t)n));
out:
  cudaFree(dp); cudaFree(dT); cudaFree(dTw); cudaFree(dg); cudaFree(st);
  return (int)rc;
}

int smh_plane_qr53(int n, const float* A15, float* x3) {
  cudaError_t rc = cudaSuccess;
  float *dA = nullptr, *dx = nullptr;
  if (n <= 0) return 0;
  SMH_TRY(to_dev(&dA, A15, 15 * (size_t)n)); SMH_TRY(to_dev<float>(&dx, nullptr, 3 * (size_t)n));
  SMH_LAUNCH(k_plane_qr53, n, dA, dx);
  SMH_TRY(to_host(x3, dx, 3 * (size_t)n));
out:
  cudaFree(dA); cudaFree(dx);
  return (int)rc;
}

// ori, sel: n x 4; nbr: n x 5 x 4; coeff: n x 4
int smh_plane_residual(int n, const float* ori, const float* sel, const float* nbr, float* coeff, int* flag) {
  cudaError_t rc = cudaSuccess;
  float4 *dori = nullptr, *dsel = nullptr, *dnbr = nullptr, *dco = nullptr;
  int* dfl = nullptr;
  if (n <= 0) return 0;
  SMH_TRY(to_dev(&dori, (const float4*)ori, (size_t)n)); SMH_TRY(to_dev(&dsel, (const float4*)sel, (size_t)n));
  SMH_TRY(to_dev(&dnbr, (const float4*)nbr, 5 * (size_t)n)); SMH_TRY(to_dev<float4>(&dco, nullptr, (size_t)n));
  SMH_TRY(to_dev<int>(&dfl, nullptr, (size_t)n));
  SMH_LAUNCH(k_plane_residual, n, dori, dsel, dnbr, dco, dfl);
  SMH_TRY(to_host((float4*)coeff, dco, (size_t)n)); SMH_TRY(to_host(flag, dfl, (size_t)n));
out:
  cudaFree(dori); cudaFree(dsel); cudaFree(dnbr); cudaFree(dco); cudaFree(dfl);
  return (int)rc;
}

int smh_umeyama(int n, const float* sigma, float* R) {
  cudaError_t rc = cudaSuccess;
  float *ds = nullptr, *dR = nullptr;
  if (n <= 0) return 0;
  SMH_TRY(to_dev(&ds, sigma, 9 * (size_t)n)); SMH_TRY(to_dev<float>(&dR, nullptr, 9 * (size_t)n));
  SMH_LAUNCH(k_umeyama, n, ds, dR);
  SMH_TRY(to_host(R, dR, 9 * (size_t)n));
out:
  cudaFree(ds); cudaFree(dR);
  return (int)rc;
}

}  // extern "C"
