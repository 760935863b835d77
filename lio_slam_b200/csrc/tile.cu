// tile.cu — full-map VoxelGrid rebuild sharded by spatial tile (BASELINE configs[3]; SURVEY §8e): the
// downSizeFilterLocalMapSurf pass of extractCloud (mapOptmization.cpp:1556-1588) over ~50 keyframes / ~5 M points,
// split over 2/4/8 GPUs with no collective on the way in.
//
// pcl::VoxelGrid emits its voxels in ascending idx = ix + iy*dx + iz*dx*dy, i.e. lexicographic in (iz, iy, ix).  A
// contiguous range of the voxel-ROW index (iz, iy) therefore owns a contiguous slice of the output, a voxel never
// spans two ranges, and a STABLE selection of a range's points keeps the canonical within-voxel summation order:
// the tiles' outputs concatenated in tile order are bit-identical to the single-GPU output.
//
// Every GPU holds the keyframes (they are uploaded to each as they are created, 1-2 MB apiece) and runs the SAME
// deterministic plan on the same bytes, so no plan has to be exchanged:
//   transform + concatenate (transform_multi_kernel)                16n B written
//   global f32 bounding box (vox_minmax_kernel) -> overflow guard of the WHOLE cloud, row-index origin
//   tile_hist_kernel   coarse histogram of the row index (<= 65,536 bins, global atomics)       16n B read
//   exclusive scan of the bins; tile_bounds_kernel: tile t = bins [b_t, b_t+1) with b_t the first bin whose
//                      cumulative count reaches t*n/N  (balanced by points, not by area)
//   tile_flag_kernel + exclusive scan + tile_compact_kernel: this tile's points, input order kept   ~40n B
//   VoxelGrid of the tile (voxel.cu) — the only part whose cost shrinks with the number of tiles
#include "common.cuh"

namespace liogpu {

constexpr unsigned TILE_MAX_BINS = 65536;

struct TilePlan {
  float inv_leaf;
  int iy0, iz0, dy, dz;
  unsigned nrows;     // dy * dz
  int shift;          // bin = row >> shift
  unsigned nbins;
  int overflow;       // the VoxelGrid guard of the whole cloud fired (output = input, q4)
  int n_valid;        // finite points of the whole cloud
  unsigned lo, hi;    // this tile's bin range [lo, hi)
  unsigned n_tile;    // finite points of this tile
};

__global__ void tile_setup_kernel(const unsigned* __restrict__ mm, float leaf, TilePlan* __restrict__ plan) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  TilePlan p;
  p.n_valid = (int)mm[6];
  float mn[3], mx[3];
  for (int a = 0; a < 3; ++a) { mn[a] = ord2f(mm[a]); mx[a] = ord2f(mm[3 + a]); }
  const float inv = 1.0f / leaf;
  p.inv_leaf = inv;
  long long d[3];
  for (int a = 0; a < 3; ++a) d[a] = (long long)((mx[a] - mn[a]) * inv) + 1;  // SURVEY A.1 step 3
  p.overflow = (p.n_valid > 0 && d[0] * d[1] * d[2] > 2147483647LL) ? 1 : 0;
  p.iy0 = (int)floorf(mn[1] * inv);
  p.iz0 = (int)floorf(mn[2] * inv);
  p.dy = (int)floorf(mx[1] * inv) - p.iy0 + 1;
  p.dz = (int)floorf(mx[2] * inv) - p.iz0 + 1;
  if (p.n_valid <= 0 || p.overflow) { p.dy = 1; p.dz = 1; }
  p.nrows = (unsigned)p.dy * (unsigned)p.dz;
  p.shift = 0;
  while ((((p.nrows - 1u) >> p.shift) + 1u) > TILE_MAX_BINS) ++p.shift;
  p.nbins = ((p.nrows - 1u) >> p.shift) + 1u;
  p.lo = 0; p.hi = 0; p.n_tile = 0;
  *plan = p;
}

__device__ __forceinline__ bool tile_bin_of(const float4 p, const TilePlan& s, unsigned& bin) {
  if (!(isfinite(p.x) && isfinite(p.y) && isfinite(p.z))) return false;
  const int iy = (int)floorf(p.y * s.inv_leaf) - s.iy0;   // the same f32 products and floors as A.1 step 5
  const int iz = (int)floorf(p.z * s.inv_leaf) - s.iz0;
  bin = ((unsigned)iz * (unsigned)s.dy + (unsigned)iy) >> s.shift;
  return true;
}

__global__ void __launch_bounds__(256)
tile_hist_kernel(const float4* __restrict__ pts, int n, const TilePlan* __restrict__ plan, uint32_t* __restrict__ hist) {
  __shared__ TilePlan s;
  if (threadIdx.x == 0) s = *plan;
  __syncthreads();
  if (s.overflow) return;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    unsigned bin;
    if (tile_bin_of(pts[i], s, bin)) {
      // neighbouring points of a sweep usually share a row: one atomic per run of equal bins in the warp
      const unsigned act = __activemask();
      const unsigned peers = __match_any_sync(act, bin);
      if ((int)(__ffs(peers) - 1) == (int)(threadIdx.x & 31)) atomicAdd(&hist[bin], (uint32_t)__popc(peers));
    }
  }
}

// cum = exclusive scan of hist (nbins entries) ; tile t = [b_t, b_t+1), b_t = first bin with cum[bin] >= t*n/N
__global__ void tile_bounds_kernel(const uint32_t* __restrict__ cum, const uint32_t* __restrict__ hist, int tile, int n_tiles,
                                   TilePlan* __restrict__ plan) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  TilePlan p = *plan;
  if (p.overflow) return;
  unsigned b[2];
  for (int q = 0; q < 2; ++q) {
    const int t = tile + q;
    if (t <= 0) { b[q] = 0; continue; }
    if (t >= n_tiles) { b[q] = p.nbins; continue; }
    const unsigned long long want = ((unsigned long long)(unsigned)p.n_valid * (unsigned long long)t) / (unsigned long long)n_tiles;
    unsigned lo = 0, hi = p.nbins;  // first bin with cum[bin] >= want
    while (lo < hi) {
      const unsigned mid = (lo + hi) >> 1;
      if ((unsigned long long)cum[mid] >= want) hi = mid; else lo = mid + 1;
    }
    b[q] = lo;
  }
  p.lo = b[0]; p.hi = b[1] < b[0] ? b[0] : b[1];
  unsigned cnt = 0;
  if (p.hi > p.lo) cnt = (p.hi < p.nbins ? cum[p.hi] : (unsigned)p.n_valid) - cum[p.lo];
  p.n_tile = cnt;
  (void)hist;
  *plan = p;
}

__global__ void __launch_bounds__(256)
tile_flag_kernel(const float4* __restrict__ pts, int n, const TilePlan* __restrict__ plan, uint32_t* __restrict__ flag) {
  __shared__ TilePlan s;
  if (threadIdx.x == 0) s = *plan;
  __syncthreads();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  unsigned bin = 0;
  const bool ok = tile_bin_of(pts[i], s, bin);
  flag[i] = (ok && bin >= s.lo && bin < s.hi) ? 1u : 0u;
}

__global__ void __launch_bounds__(256)
tile_compact_kernel(const float4* __restrict__ pts, int n, const TilePlan* __restrict__ plan, const uint32_t* __restrict__ pos,
                    float4* __restrict__ out) {
  __shared__ TilePlan s;
  if (threadIdx.x == 0) s = *plan;
  __syncthreads();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 p = pts[i];
  unsigned bin = 0;
  if (tile_bin_of(p, s, bin) && bin >= s.lo && bin < s.hi) out[pos[i]] = p;  // pos = exclusive scan of the flags: input order kept
}

// pts: the transformed concatenation (n points).  Leaves this tile's voxels in `out`.
int voxel_tile_dev(Ctx* c, const float4* pts, int n, float leaf, int tile, int n_tiles, DevBuf& out, int* n_out,
                   bool* overflow, liogpu_tile_info* info) {
  *n_out = 0;
  *overflow = false;
  if (n <= 0) return LIOGPU_OK;
  LIOGPU_CUDA_OK(c, c->minmax.reserve(64));
  LIOGPU_CUDA_OK(c, c->tile_plan.reserve(sizeof(TilePlan)));
  LIOGPU_CUDA_OK(c, c->tile_hist.reserve(((size_t)TILE_MAX_BINS + 2) * 2 * sizeof(uint32_t)));
  LIOGPU_CUDA_OK(c, c->seg_flag.reserve((size_t)n * 4 + 16));
  unsigned* mm = c->minmax.as<unsigned>();
  TilePlan* d_plan = c->tile_plan.as<TilePlan>();
  uint32_t* hist = c->tile_hist.as<uint32_t>();
  uint32_t* cum = hist + TILE_MAX_BINS + 2;
  LIOGPU_CUDA_OK(c, launch_minmax(c, pts, n, mm));
  tile_setup_kernel<<<1, 32, 0, c->stream>>>(mm, leaf, d_plan);
  LIOGPU_CUDA_OK(c, cudaMemsetAsync(hist, 0, ((size_t)TILE_MAX_BINS + 2) * sizeof(uint32_t), c->stream));
  int grid = div_up(n, 256);
  if (grid > c->sm_count * 16) grid = c->sm_count * 16;
  tile_hist_kernel<<<grid, 256, 0, c->stream>>>(pts, n, d_plan, hist);
  c->launches += 2;
  LIOGPU_CUDA_OK(c, exclusive_scan_u32(c, hist, cum, (int)TILE_MAX_BINS + 1, nullptr));
  tile_bounds_kernel<<<1, 32, 0, c->stream>>>(cum, hist, tile, n_tiles, d_plan);
  uint32_t* flag = c->seg_flag.as<uint32_t>();
  tile_flag_kernel<<<div_up(n, 256), 256, 0, c->stream>>>(pts, n, d_plan, flag);
  c->launches += 2;
  LIOGPU_CUDA_OK(c, exclusive_scan_u32(c, flag, flag, n, nullptr));
  TilePlan* h_plan = reinterpret_cast<TilePlan*>((char*)c->h_pinned + 1024);
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(h_plan, d_plan, sizeof(TilePlan), cudaMemcpyDeviceToHost, c->stream));
  LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  const TilePlan plan = *h_plan;
  if (info) {
    info->n_points = n;
    info->n_rows = (int)plan.nrows;
    info->n_bins = (int)plan.nbins;
    info->bin_lo = (int)plan.lo;
    info->bin_hi = (int)plan.hi;
    info->n_tile_points = (int)plan.n_tile;
    info->leaf_overflow = plan.overflow;
  }
  if (plan.overflow) {
    // q4: PCL returns the input unchanged; tile t owns the t-th contiguous slice so the concatenation is the input
    const long long b = (long long)n * tile / n_tiles, e = (long long)n * (tile + 1) / n_tiles;
    const int m = (int)(e - b);
    LIOGPU_CUDA_OK(c, out.reserve((size_t)(m > 0 ? m : 1) * sizeof(float4)));
    if (m > 0) LIOGPU_CUDA_OK(c, cudaMemcpyAsync(out.p, pts + b, (size_t)m * sizeof(float4), cudaMemcpyDeviceToDevice, c->stream));
    *n_out = m;
    *overflow = true;
    if (info) info->n_tile_points = m;
    if (c->ev_mid) LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev_mid, c->stream));
    return LIOGPU_OK;
  }
  const int m = (int)plan.n_tile;
  if (m <= 0) { if (c->ev_mid) LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev_mid, c->stream)); return LIOGPU_OK; }
  LIOGPU_CUDA_OK(c, c->tile_pts.reserve((size_t)m * sizeof(float4)));
  tile_compact_kernel<<<div_up(n, 256), 256, 0, c->stream>>>(pts, n, d_plan, flag, c->tile_pts.as<float4>());
  c->launches++;
  LIOGPU_CUDA_OK(c, cudaGetLastError());
  if (c->ev_mid) LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev_mid, c->stream));
  bool ov = false;
  return voxel_downsample_dev(c, c->tile_pts.as<float4>(), m, leaf, out, n_out, &ov);
}

}  // namespace liogpu
