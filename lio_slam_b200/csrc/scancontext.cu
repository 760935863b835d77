// scancontext.cu — the Scan Context descriptor of a keyframe cloud: SCManager::makeScancontext
// (include/Scancontext.cpp:151-195, xy2theta :23-36) and its ring / sector keys (:198-225), which the reference
// computes at every keyframe from the full deskewed sweep (mapOptmization.cpp:2151-2166).  SURVEY §8 row f3.
//
// One thread per point: polar bin (ring, sector) in the arithmetic of the source (f32 range, f64 atan narrowed to
// f32, f64 ceil), height z + LIDAR_HEIGHT narrowed to f32, atomicMax on an order-preserving integer image of the
// float into a 20 x 60 table in shared memory, one global atomicMax per occupied bin and block.  A one-block
// epilogue kernel turns the table into doubles (empty bins -> 0) and forms the row / column means.
//
// Many resident keyframes at once (liogpu_sc_add_keyframes): a grid over (keyframe, chunk of SC_CHUNK points); the
// block-offset table is the prefix sum of ceil(n_f / SC_CHUNK), so a 230k-point keyframe among small ones spreads over
// as many blocks as its size needs.  The clouds are read in place through the srcs / offs tables of stage_keyframes.
// Table memory (option "in the slot"): each new store entry's f64 slot (9.6 KB) holds the keyframe's u32 image
// (4.8 KB) in its first half while the blocks bin into it; sc_store_kernel (loopdetect.cu) then loads the image into
// shared memory, overwrites the slot with the doubles and derives the keys.  No memory beyond the store itself.  Passes
// exist only because the staged tables address a pass's clouds with 32-bit offsets: a call covers 2^31 - 1 points per
// pass (loopdetect.cu: sc_add_keyframes_dev).  Max is order-independent: every entry is exact whatever the decomposition.
#include "scancontext.cuh"

#include <math_constants.h>

namespace liogpu {

namespace {

__device__ __forceinline__ float sc_xy2theta(float x, float y) {  // Scancontext.cpp:23-36
  const double k = 180.0 / 3.14159265358979323846;
  if ((x >= 0) & (y >= 0)) return (float)(k * atan((double)(y / x)));
  if ((x < 0) & (y >= 0)) return (float)(180.0 - (k * atan((double)(y / (-x)))));
  if ((x < 0) & (y < 0)) return (float)(180.0 + (k * atan((double)(y / x))));
  return (float)(360.0 - (k * atan((double)((-y) / x))));
}

__global__ void sc_init_kernel(unsigned* __restrict__ table) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k < SC_BINS) table[k] = sc_none();  // NO_POINT (:158)
}

// Bins points first, first + step, ... < end into the block's shared table, then one global atomicMax per occupied
// bin into `table`.
__device__ __forceinline__ void sc_bin_block(const float4* __restrict__ pts, long long first, long long end, int step,
                                             double lidar_height, double max_radius, unsigned* sh, unsigned* table) {
  const unsigned none = sc_none();
  for (int k = threadIdx.x; k < SC_BINS; k += blockDim.x) sh[k] = none;
  __syncthreads();
  for (long long i = first; i < end; i += step) {
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
    atomicMax(&sh[(ring - 1) * SC_SECTOR + (sector - 1)], f2ord(z));  // :181-182
  }
  __syncthreads();
  for (int k = threadIdx.x; k < SC_BINS; k += blockDim.x)
    if (sh[k] != none) atomicMax(&table[k], sh[k]);
}

__global__ void __launch_bounds__(256)
sc_bin_kernel(const float4* __restrict__ pts, int n, double lidar_height, double max_radius, unsigned* __restrict__ table) {
  __shared__ unsigned sh[SC_BINS];
  sc_bin_block(pts, blockIdx.x * blockDim.x + threadIdx.x, n, gridDim.x * blockDim.x, lidar_height, max_radius, sh, table);
}

// image of entry e: the first SC_BINS words of its f64 slot (2 * SC_BINS words)
__global__ void sc_slot_init_kernel(unsigned* __restrict__ slots, int n) {
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k < (long long)n * SC_BINS) slots[(k / SC_BINS) * (2 * SC_BINS) + k % SC_BINS] = sc_none();
}

// block b bins chunk b - blk_off[f] of keyframe f (blk_off[f] <= b < blk_off[f + 1]) into entry f's image
__global__ void __launch_bounds__(256)
sc_bin_keyframes_kernel(const float4* const* __restrict__ srcs, const int* __restrict__ offs, const int* __restrict__ blk_off,
                        int n, double lidar_height, double max_radius, unsigned* __restrict__ slots) {
  __shared__ unsigned sh[SC_BINS];
  const int b = blockIdx.x;
  int lo = 0, hi = n - 1;  // the last f with blk_off[f] <= b (empty keyframes own no block)
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (blk_off[mid] <= b) lo = mid; else hi = mid - 1;
  }
  const int f = lo;
  const long long first = (long long)(b - blk_off[f]) * SC_CHUNK;
  const long long end = min((long long)(offs[f + 1] - offs[f]), first + SC_CHUNK);
  sc_bin_block(srcs[f], first + threadIdx.x, end, blockDim.x, lidar_height, max_radius, sh,
               slots + (size_t)f * (2 * SC_BINS));
}

__global__ void __launch_bounds__(256)
sc_keys_kernel(const unsigned* __restrict__ table, double* __restrict__ out) {
  // out: desc [SC_BINS] | ringkey [SC_RING] | sectorkey [SC_SECTOR]
  __shared__ double d[SC_BINS];
  for (int k = threadIdx.x; k < SC_BINS; k += blockDim.x) {
    const double dv = sc_bin_value(table[k]);
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

cudaError_t launch_sc_bin_keyframes(Ctx* c, const float4* const* srcs, const int* offs, const int* blk_off, int n,
                                    int n_blocks, double lidar_height, double max_radius, double* slots) {
  unsigned* img = reinterpret_cast<unsigned*>(slots);
  sc_slot_init_kernel<<<div_up((long long)n * SC_BINS, 256), 256, 0, c->stream>>>(img, n);
  c->launches++;
  if (n_blocks > 0) {
    sc_bin_keyframes_kernel<<<n_blocks, 256, 0, c->stream>>>(srcs, offs, blk_off, n, lidar_height, max_radius, img);
    c->launches++;
  }
  return cudaGetLastError();
}

}  // namespace liogpu
