// grid.cu — the sorted-grid index that replaces pcl::KdTreeFLANN for the local map
// (kdtreeSurfFromMap->setInputCloud, mapOptmization.cpp:1846; built once per local-map change
// instead of once per scan — SURVEY quirk q1).
//
// surfOptimization only keeps a query whose 5th neighbour is closer than 1 m (dist^2 < 1.0, :1641),
// so an EXACT 5-NN inside that gate needs nothing beyond the cells within 1 m of the query.  Points
// are bucketed into cubic cells of edge h (default 0.5 m), sorted by cell key z-major / x-minor so
// that a run of x-adjacent cells is one contiguous range of the sorted array:
//     candidates(row y,z ; x in [xlo,xhi]) = sorted[cell_start[row+xlo] .. cell_start[row+xhi+1])
// Layout in HBM: map4 (float4 x,y,z,intensity, map order), map_sorted (float4 x,y,z,bits(map index)),
// cell_start (u32, n_cells+1).  For a 500k-point map: 8 + 8 MB + ~4 MB, all L2-resident on B200.
#include "common.cuh"

namespace liogpu {

// mm = output of vox_minmax_kernel (ordered-uint min[3], max[3], finite count)
__global__ void grid_setup_kernel(const unsigned* __restrict__ mm, float cell, float gate_d2, float gate1_d2,
                                  unsigned max_cells, GridParams* __restrict__ gp) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  float mn[3], mx[3];
  for (int a = 0; a < 3; ++a) { mn[a] = ord2f(mm[a]); mx[a] = ord2f(mm[3 + a]); }
  *gp = grid_setup_compute(mn, mx, (int)mm[6], cell, max_cells, gate_d2, gate1_d2);
}

__global__ void __launch_bounds__(256)
grid_key_kernel(const float4* __restrict__ map4, int n, const GridParams* __restrict__ gp,
                uint32_t* __restrict__ keys, uint32_t* __restrict__ cell_count) {
  __shared__ GridParams g;
  if (threadIdx.x == 0) g = *gp;
  __syncthreads();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 p = map4[i];
  uint32_t key = g.n_cells;  // non-finite points sort last and are never referenced
  if (isfinite(p.x) && isfinite(p.y) && isfinite(p.z)) {
    const int cx = cell_coord(p.x, g.ox, g.inv_h, g.nx);
    const int cy = cell_coord(p.y, g.oy, g.inv_h, g.ny);
    const int cz = cell_coord(p.z, g.oz, g.inv_h, g.nz);
    key = ((uint32_t)cz * (uint32_t)g.ny + (uint32_t)cy) * (uint32_t)g.nx + (uint32_t)cx;
    atomicAdd(&cell_count[key], 1u);
  }
  keys[i] = key;
}

__global__ void __launch_bounds__(256)
grid_gather_kernel(const float4* __restrict__ map4, const uint32_t* __restrict__ perm, int n_valid,
                   float4* __restrict__ map_sorted) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_valid) return;
  const uint32_t src = perm[j];
  const float4 p = map4[src];
  map_sorted[j] = make_float4(p.x, p.y, p.z, __int_as_float((int)src));
}

// Builds the sorted-grid index of `pts` into the given buffers (the local-map index of the registration and the
// self-index of publishLocalMap's outlier filter are two instances).  Synchronises the stream once to learn
// the grid dimensions.
int grid_build_core(Ctx* c, const float4* pts, int n, float cell, float gate_d2, float gate1_d2, DevBuf& setup,
                    DevBuf& sorted, DevBuf& cell_start_buf, GridParams& host_gp) {
  LIOGPU_CUDA_OK(c, c->minmax.reserve(64));
  LIOGPU_CUDA_OK(c, setup.reserve(sizeof(GridParams)));
  LIOGPU_CUDA_OK(c, c->keys0.reserve((size_t)n * 4));
  LIOGPU_CUDA_OK(c, c->keys1.reserve((size_t)n * 4));
  LIOGPU_CUDA_OK(c, c->vals0.reserve((size_t)n * 4));
  LIOGPU_CUDA_OK(c, c->vals1.reserve((size_t)n * 4));
  LIOGPU_CUDA_OK(c, sorted.reserve((size_t)n * sizeof(float4)));
  unsigned* mm = c->minmax.as<unsigned>();
  GridParams* d_gp = setup.as<GridParams>();
  LIOGPU_CUDA_OK(c, launch_minmax(c, pts, n, mm));
  grid_setup_kernel<<<1, 32, 0, c->stream>>>(mm, cell, gate_d2, gate1_d2, 1u << 25, d_gp);
  c->launches += 1;
  GridParams* h_gp = reinterpret_cast<GridParams*>((char*)c->h_pinned + 2048);
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(h_gp, d_gp, sizeof(GridParams), cudaMemcpyDeviceToHost, c->stream));
  LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  host_gp = *h_gp;
  const GridParams& g = host_gp;
  if (g.n_points <= 0) return LIOGPU_OK;
  LIOGPU_CUDA_OK(c, cell_start_buf.reserve(((size_t)g.n_cells + 2) * sizeof(uint32_t)));
  uint32_t* cell_start = cell_start_buf.as<uint32_t>();
  LIOGPU_CUDA_OK(c, cudaMemsetAsync(cell_start, 0, ((size_t)g.n_cells + 2) * sizeof(uint32_t), c->stream));
  grid_key_kernel<<<div_up(n, 256), 256, 0, c->stream>>>(pts, n, d_gp, c->keys0.as<uint32_t>(), cell_start);
  c->launches++;
  LIOGPU_CUDA_OK(c, exclusive_scan_u32(c, cell_start, cell_start, (int)g.n_cells + 1, nullptr));
  int bits = 0;
  while (bits < 32 && (g.n_cells >> bits) != 0u) ++bits;
  uint32_t *skeys = nullptr, *sperm = nullptr;
  LIOGPU_CUDA_OK(c, radix_sort_pairs(c, n, bits, nullptr, &skeys, &sperm));
  grid_gather_kernel<<<div_up(g.n_points, 256), 256, 0, c->stream>>>(pts, sperm, g.n_points, sorted.as<float4>());
  c->launches++;
  LIOGPU_CUDA_OK(c, cudaGetLastError());
  return LIOGPU_OK;
}

int grid_build_dev(Ctx* c, const float4* map4, int n, float leaf_hint) {
  c->grid_valid = false;
  c->n_map = n;
  if (n <= 0) return LIOGPU_OK;
  // Tuning (results never depend on it): the first search phase looks inside r1 ~ twice the map's point
  // spacing (the VoxelGrid leaf), where a query on a mapped surface already finds its 5 neighbours; the
  // cell edge follows r1 so that phase 1 touches a 3x3x3 block of cells.
  const float gate_d2 = 1.0f;  // mapOptmization.cpp:1641
  const float spacing = leaf_hint > 0.f ? leaf_hint : 0.2f;
  float r1 = c->prm.knn_phase1_radius > 0.f ? c->prm.knn_phase1_radius : 2.0f * spacing;
  float gate1_d2 = r1 * r1;
  if (c->prm.knn_phase1_radius < 0.f || gate1_d2 >= 0.64f * gate_d2) gate1_d2 = gate_d2;  // single phase
  float cell = c->prm.knn_cell_size;
  // dense map: cell edge = phase-1 radius (its reach box is then at most 3 x 3 rows of cells);
  // sparse map (single phase): 1 m cells so that the full 1 m gate also fits a 3 x 3 box
  if (!(cell > 0.f)) cell = (gate1_d2 < gate_d2) ? fminf(fmaxf(r1, 0.25f), 0.5f) : 1.0f;
  const int rc = grid_build_core(c, map4, n, cell, gate_d2, gate1_d2, c->grid_setup, c->map_sorted, c->cell_start, c->grid);
  if (rc) return rc;
  c->grid_valid = true;
  return LIOGPU_OK;
}

}  // namespace liogpu
