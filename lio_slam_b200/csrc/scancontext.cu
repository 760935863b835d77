// scancontext.cu — the Scan Context descriptor of a keyframe cloud: SCManager::makeScancontext
// (include/Scancontext.cpp:151-195, xy2theta :23-36) and its ring / sector keys (:198-225), which the reference
// computes at every keyframe from the full deskewed sweep (mapOptmization.cpp:2151-2166).  SURVEY §8 row f3.
//
// One thread per point: polar bin (ring, sector) in the arithmetic of the source (f32 range, f64 atan narrowed to
// f32, f64 ceil), height z + LIDAR_HEIGHT narrowed to f32, atomicMax on an order-preserving integer image of the
// float into a 20 x 60 table in shared memory, one global atomicMax per occupied bin and block.  A one-block
// epilogue kernel turns the table into doubles (empty bins -> 0) and forms the row / column means.
#include "scancontext.cuh"

#include <math_constants.h>

namespace liogpu {

namespace {

__device__ __forceinline__ unsigned sc_f2ord(float f) {
  const unsigned u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float sc_ord2f(unsigned o) {
  return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
}

__device__ __forceinline__ float sc_xy2theta(float x, float y) {  // Scancontext.cpp:23-36
  const double k = 180.0 / 3.14159265358979323846;
  if ((x >= 0) & (y >= 0)) return (float)(k * atan((double)(y / x)));
  if ((x < 0) & (y >= 0)) return (float)(180.0 - (k * atan((double)(y / (-x)))));
  if ((x < 0) & (y < 0)) return (float)(180.0 + (k * atan((double)(y / x))));
  return (float)(360.0 - (k * atan((double)((-y) / x))));
}

__global__ void sc_init_kernel(unsigned* __restrict__ table) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k < SC_BINS) table[k] = sc_f2ord(-1000.0f);  // NO_POINT (:158)
}

__global__ void __launch_bounds__(256)
sc_bin_kernel(const float4* __restrict__ pts, int n, double lidar_height, double max_radius, unsigned* __restrict__ table) {
  __shared__ unsigned sh[SC_BINS];
  const unsigned none = sc_f2ord(-1000.0f);
  for (int k = threadIdx.x; k < SC_BINS; k += blockDim.x) sh[k] = none;
  __syncthreads();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 p = pts[i];
    if (!(isfinite(p.x) && isfinite(p.y) && isfinite(p.z))) continue;
    const float z = (float)((double)p.z + lidar_height);                 // :167
    const float azim_range = (float)sqrt((double)(p.x * p.x + p.y * p.y));  // :170
    const float azim_angle = sc_xy2theta(p.x, p.y);
    if ((double)azim_range > max_radius) continue;                       // :174
    int ring = (int)ceil(((double)azim_range / max_radius) * SC_RING);   // :177
    ring = max(min(SC_RING, ring), 1);
    const double sc = ceil(((double)azim_angle / 360.0) * SC_SECTOR);    // :178
    int sector = isnan(sc) ? 0 : (int)sc;
    sector = max(min(SC_SECTOR, sector), 1);
    atomicMax(&sh[(ring - 1) * SC_SECTOR + (sector - 1)], sc_f2ord(z));  // :181-182
  }
  __syncthreads();
  for (int k = threadIdx.x; k < SC_BINS; k += blockDim.x)
    if (sh[k] != none) atomicMax(&table[k], sh[k]);
}

__global__ void __launch_bounds__(256)
sc_keys_kernel(const unsigned* __restrict__ table, double* __restrict__ out) {
  // out: desc [SC_BINS] | ringkey [SC_RING] | sectorkey [SC_SECTOR]
  __shared__ double d[SC_BINS];
  for (int k = threadIdx.x; k < SC_BINS; k += blockDim.x) {
    const float v = sc_ord2f(table[k]);
    const double dv = v == -1000.0f ? 0.0 : (double)v;  // :186-189
    d[k] = dv;
    out[k] = dv;
  }
  __syncthreads();
  const int k = threadIdx.x;
  if (k < SC_RING + SC_SECTOR) out[SC_BINS + k] = sc_key(d, k);
}

}  // namespace

int scancontext_dev(Ctx* c, const float4* pts, int n, double lidar_height, double max_radius, double* h_out) {
  LIOGPU_CUDA_OK(c, c->lm_stats.reserve(65536));
  unsigned* table = reinterpret_cast<unsigned*>((char*)c->lm_stats.p + 8192);
  double* d_out = reinterpret_cast<double*>((char*)c->lm_stats.p + 16384);
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
  sc_init_kernel<<<div_up(SC_BINS, 256), 256, 0, c->stream>>>(table);
  if (n > 0) {
    int grid = div_up(n, 256);
    if (grid > c->sm_count * 4) grid = c->sm_count * 4;
    sc_bin_kernel<<<grid, 256, 0, c->stream>>>(pts, n, lidar_height, max_radius, table);
    c->launches++;
  }
  sc_keys_kernel<<<1, 256, 0, c->stream>>>(table, d_out);
  c->launches += 2;
  LIOGPU_CUDA_OK(c, cudaGetLastError());
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
  double* h = reinterpret_cast<double*>((char*)c->h_pinned + 16384);
  const size_t bytes = (size_t)(SC_BINS + SC_RING + SC_SECTOR) * sizeof(double);
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(h, d_out, bytes, cudaMemcpyDeviceToHost, c->stream));
  LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1);
  memcpy(h_out, h, bytes);
  return LIOGPU_OK;
}

}  // namespace liogpu
