// shell_search.cuh — exact nearest-neighbour search on the sorted uniform grid (grid.cu) by growing shells of
// cells around the query's home cell, shared by the outlier filter of publishLocalMap (localmap.cu: the K
// smallest distances) and the loop-closure ICP (icp.cu: the nearest point).  `Acc` is the running result:
// Acc::push(d2, w) receives every inspected point's squared distance and the w word of its sorted record
// (bits of the point's original index).
#pragma once
#include "common.cuh"

#include <math_constants.h>

namespace liogpu {

// FLANN L2_Simple<float> (same expression as the registration's search)
__device__ __forceinline__ float sor_d2(const float4& a, const float4& b) {
  float r = 0.f;
  float d = a.x - b.x; r += d * d;
  d = a.y - b.y;       r += d * d;
  d = a.z - b.z;       r += d * d;
  return r;
}

struct HomeCell {
  int cx, cy, cz;
  float fx, fy, fz;  // position of the point inside its cell: distance to the cell's lower faces
};
__device__ __forceinline__ HomeCell home_cell(const GridParams& g, const float4& p) {
  HomeCell hc;
  hc.cx = cell_coord(p.x, g.ox, g.inv_h, g.nx);
  hc.cy = cell_coord(p.y, g.oy, g.inv_h, g.ny);
  hc.cz = cell_coord(p.z, g.oz, g.inv_h, g.nz);
  hc.fx = (p.x - g.ox) - (float)hc.cx * g.h;
  hc.fy = (p.y - g.oy) - (float)hc.cy * g.h;
  hc.fz = (p.z - g.oz) - (float)hc.cz * g.h;
  return hc;
}

// After all cells within R rings of the home cell have been inspected, every point NOT inspected lies at least
// `covered` away.  Returns the square of a safe lower bound of it (slack: f32 rounding of the cell assignment;
// the relative margin covers the rounding of the squared distances), or +inf when the box is the whole grid.
__device__ __forceinline__ float covered_d2(const GridParams& g, const HomeCell& hc, int R) {
  const float Rh = (float)R * g.h;
  float cov = CUDART_INF_F;
  if (hc.cx - R > 0) cov = fminf(cov, Rh + hc.fx);
  if (hc.cx + R < g.nx - 1) cov = fminf(cov, Rh + (g.h - hc.fx));
  if (hc.cy - R > 0) cov = fminf(cov, Rh + hc.fy);
  if (hc.cy + R < g.ny - 1) cov = fminf(cov, Rh + (g.h - hc.fy));
  if (hc.cz - R > 0) cov = fminf(cov, Rh + hc.fz);
  if (hc.cz + R < g.nz - 1) cov = fminf(cov, Rh + (g.h - hc.fz));
  if (cov == CUDART_INF_F) return cov;
  cov = fmaxf(cov - g.slack, 0.f) * 0.999999f;
  return cov * cov;
}

template <class Acc>
__device__ __forceinline__ void scan_range(const float4* __restrict__ sorted, unsigned b, unsigned e, const float4& p,
                                           Acc& top) {
  for (unsigned t = b; t < e; ++t) {
    const float4 q = __ldg(sorted + t);
    top.push(sor_d2(p, q), q.w);
  }
}

// the part of shell R (cells at Chebyshev distance exactly R from the home cell) that lies in row (y, z)
template <class Acc>
__device__ __forceinline__ void scan_shell_row(const float4* __restrict__ sorted, const uint32_t* __restrict__ cs,
                                               const GridParams& g, const HomeCell& hc, int R, int y, int z,
                                               const float4& p, Acc& top) {
  const unsigned row = ((unsigned)z * (unsigned)g.ny + (unsigned)y) * (unsigned)g.nx;
  const int ady = y > hc.cy ? y - hc.cy : hc.cy - y, adz = z > hc.cz ? z - hc.cz : hc.cz - z;
  if (ady == R || adz == R) {  // the whole x-run of the box is new: one contiguous range of the sorted array
    const int x0 = max(hc.cx - R, 0), x1 = min(hc.cx + R, g.nx - 1);
    scan_range(sorted, __ldg(cs + row + x0), __ldg(cs + row + x1 + 1), p, top);
  } else {                     // interior row: only the two end cells are new
    if (hc.cx - R >= 0) scan_range(sorted, __ldg(cs + row + hc.cx - R), __ldg(cs + row + hc.cx - R + 1), p, top);
    if (hc.cx + R <= g.nx - 1) scan_range(sorted, __ldg(cs + row + hc.cx + R), __ldg(cs + row + hc.cx + R + 1), p, top);
  }
}

}  // namespace liogpu
