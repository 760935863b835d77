// s2m.cu — the scan-to-map hot loop: surfOptimization + combineOptimizationCoeffs + LMOptimization
// (mapOptmization.cpp:1618-1687, 1689-1700, 1702-1837), two kernels per Gauss-Newton iteration, the whole loop
// on the device.
//
//   s2m_main_kernel   one thread per sweep point
//     1. pointAssociateToMap (:841-847) with the device-resident 3x4 transform
//     2. exact 5-NN on the sorted grid (grid.cu): rows of x-adjacent cells are contiguous ranges of map_sorted;
//        rows are visited centre-out and pruned against the running 5th-best distance; distances are FLANN
//        L2_Simple in f32 without FMA; ties -> lower map index.  Iteration 0 searches inside a small phase-1
//        gate; iterations >= 1 inside the bound given by the previous iteration's neighbours (seeded search) —
//        as the insertion walk after a large pose step, as collect-then-select (grid_knn5_collect) after a small
//        one; points with too few map points around are skipped by the exact "hopeless" rule
//     3. 5x3 column-pivoted Householder plane fit, validity, weight s, coefficient (:1633-1684)
//     4. Jacobian row (:1760-1778) staged in shared memory; the block reduces the 27 sums of A^T A (upper
//        triangle) and A^T b in FP64 (cv::gemm accumulates f32 products in double)
//     5. points phase 1 could not settle go to a per-block segment of the leftover list
//   s2m_left_kernel   offsets of the leftover segments (parallel scan in every block), warp-cooperative full-gate
//     search of the leftovers (one per warp), fold of all partial sums in a fixed order, and — in the last block
//     to finish — the 6x6 tail of LMOptimization
//     (lm_finalize_warp): QR solve, degeneracy decision / matP on iteration 0, projection, pose update,
//     convergence test (:1784-1835), next iteration's transform
//   lm_matp_kernel    iteration 0's Jacobi eigen-decomposition + matP on a second stream when a rigorous
//     certificate has already decided isDegenerate = false
//   s2m_fused.cuh is the whole loop as one cooperative launch (params.s2m_path = 2).  Other main kernels (persistent
//   warps, warp-cooperative candidate evaluation, search and fit split) were measured slower: DESIGN.md §4.
//
// The pose, matP, isDegenerate and the iteration counter stay in HBM (LmDevState); the host enqueues a chunk of
// iterations back to back and reads the 2.5 KB state once — a launch that finds `done` set returns immediately.
// Compaction (:1689-1700) is unnecessary: rejected points contribute exact zeros to the FP64 sums.
//
// Algorithmic HBM bytes per launch: 16 B query + 5 x 16 B neighbours = 96 B per sweep point.
#include "common.cuh"
#include "pose_math.cuh"
#include "lm_tail.cuh"
#include <stdio.h>
#include <stdlib.h>

namespace liogpu {

#ifndef S2M_THREADS_CFG
#define S2M_THREADS_CFG 256
#endif
#ifndef S2M_MINBLOCKS_CFG
#define S2M_MINBLOCKS_CFG 4
#endif
constexpr int S2M_THREADS = S2M_THREADS_CFG;
// The leftover kernel turns the main kernel's per-block leftover counts into segment offsets itself, in shared memory,
// when the table fits; the main kernel then ends without a ticket and without the serial scan of its last block (which
// still runs for sweeps of more than (LEFT_OFF_CAP - 1) x S2M_THREADS points).
constexpr int LEFT_OFF_CAP = 8192;
constexpr int S2M_SUMS = 32;  // 21 (upper AtA) + 6 (AtB) + nsel + ties, padded to 32

struct SurfDebugOut {
  int* nn_idx;          // n*5
  float* nn_d2;         // n*5
  float4* coeff;        // n
  unsigned char* flag;  // n
  unsigned char* tie;   // n
};

// Running 5 best (d2, map index) pairs as 64-bit keys: (bits of d2) << 32 | index.  d2 >= +0 so the
// bit pattern orders like the value, and the low word breaks ties toward the lower map index — one
// unsigned 64-bit compare per test, branch-free compare-exchange bubble on insertion.
typedef unsigned long long u64;
struct Top5 {
  u64 k0, k1, k2, k3, k4;
  float rej;  // best distance among candidates that did not stay in the top 5 (tie logging)
  __device__ __forceinline__ void init(float gate) {
    // sentinel (gate, index 0): a candidate at exactly the gate distance never compares below it
    k0 = k1 = k2 = k3 = k4 = ((u64)__float_as_uint(gate)) << 32;
    rej = FLT_MAX;
  }
  __device__ __forceinline__ void offer(float d, int id) {
    const u64 key = (((u64)__float_as_uint(d)) << 32) | (u64)(unsigned)id;
    if (key < k4) {
      rej = fminf(rej, __uint_as_float((unsigned)(k4 >> 32)));
      u64 lo;
      k4 = key;
      lo = min(k3, k4); k4 = max(k3, k4); k3 = lo;
      lo = min(k2, k3); k3 = max(k2, k3); k2 = lo;
      lo = min(k1, k2); k2 = max(k1, k2); k1 = lo;
      lo = min(k0, k1); k1 = max(k0, k1); k0 = lo;
    } else {
      rej = fminf(rej, d);
    }
  }
  __device__ __forceinline__ float d(const u64 k) const { return __uint_as_float((unsigned)(k >> 32)); }
  __device__ __forceinline__ int i(const u64 k) const { return (int)(unsigned)(k & 0xffffffffull); }
  __device__ __forceinline__ bool tie() const {
    return d(k0) == d(k1) || d(k1) == d(k2) || d(k2) == d(k3) || d(k3) == d(k4) || d(k4) == rej;
  }
};

// FLANN L2_Simple<float>: result = 0; result += diff*diff for x, y, z — f32, no FMA (-fmad=false)
__device__ __forceinline__ float l2_simple(const float4 q, const float4 p) {
  float d = q.x - p.x;
  float acc = d * d;
  d = q.y - p.y; acc = acc + d * d;
  d = q.z - p.z; acc = acc + d * d;
  return acc;
}

__device__ __forceinline__ int zigzag(int k) { return (k & 1) ? -((k + 1) >> 1) : (k >> 1); }  // 0,-1,+1,-2,+2,...

// Exact 5 nearest map points of q among those closer than sqrt(gate_d2), ascending (d2, map index).
// On return t.d(t.k4) < gate_d2 iff at least 5 such points exist (then the answer is exact).
__device__ __forceinline__ void grid_knn5(const float4 q, const GridParams& g, const float gate_d2,
                                          const float4* __restrict__ map_sorted,
                                          const uint32_t* __restrict__ cell_start, Top5& t) {
  t.init(gate_d2);
  const float s2 = 2.0f * g.slack;
  const float reach = sqrtf(gate_d2) * 1.000001f + s2;
  int zmin = (int)floorf((q.z - reach - g.oz) * g.inv_h), zmax = (int)floorf((q.z + reach - g.oz) * g.inv_h);
  int ymin = (int)floorf((q.y - reach - g.oy) * g.inv_h), ymax = (int)floorf((q.y + reach - g.oy) * g.inv_h);
  zmin = max(zmin, 0); zmax = min(zmax, g.nz - 1);
  ymin = max(ymin, 0); ymax = min(ymax, g.ny - 1);
  if (zmin > zmax || ymin > ymax) return;
  const int cz = min(max((int)floorf((q.z - g.oz) * g.inv_h), zmin), zmax);
  const int cy = min(max((int)floorf((q.y - g.oy) * g.inv_h), ymin), ymax);
  const int nzs = zmax - zmin + 1, nys = ymax - ymin + 1;
  for (int kz = 0, seen_z = 0; seen_z < nzs; ++kz) {  // centre-out over the z slabs in reach
    const int z = cz + zigzag(kz);
    if (z < zmin || z > zmax) continue;
    ++seen_z;
    const float zlo = g.oz + (float)z * g.h;
    const float gz = fmaxf(fmaxf(zlo - q.z, q.z - (zlo + g.h)) - s2, 0.f);
    const float gz2 = gz * gz;
    if (gz2 > t.d(t.k4)) continue;
    for (int ky = 0, seen_y = 0; seen_y < nys; ++ky) {
      const int y = cy + zigzag(ky);
      if (y < ymin || y > ymax) continue;
      ++seen_y;
      const float ylo = g.oy + (float)y * g.h;
      const float gy = fmaxf(fmaxf(ylo - q.y, q.y - (ylo + g.h)) - s2, 0.f);
      const float m2 = (gz2 + gy * gy) * 0.999999f;
      const float worst = t.d(t.k4);
      if (m2 > worst) continue;
      const float r = sqrtf(worst - m2) * 1.000001f + s2;
      int xlo = (int)floorf((q.x - r - g.ox) * g.inv_h);
      int xhi = (int)floorf((q.x + r - g.ox) * g.inv_h);
      xlo = max(xlo, 0);
      xhi = min(xhi, g.nx - 1);
      if (xlo > xhi) continue;
      const uint32_t row = ((uint32_t)z * (uint32_t)g.ny + (uint32_t)y) * (uint32_t)g.nx;
      const uint32_t s = __ldg(cell_start + row + xlo);
      const uint32_t e = __ldg(cell_start + row + xhi + 1);
      for (uint32_t j = s; j < e; j += 4) {
        // four independent 16-byte loads in flight per thread (clamped, so no predicate on the loads)
        const uint32_t last = e - 1;
        const float4 p0 = __ldg(map_sorted + j);
        const float4 p1 = __ldg(map_sorted + min(j + 1, last));
        const float4 p2 = __ldg(map_sorted + min(j + 2, last));
        const float4 p3 = __ldg(map_sorted + min(j + 3, last));
        t.offer(l2_simple(q, p0), __float_as_int(p0.w));
        if (j + 1 < e) t.offer(l2_simple(q, p1), __float_as_int(p1.w));
        if (j + 2 < e) t.offer(l2_simple(q, p2), __float_as_int(p2.w));
        if (j + 3 < e) t.offer(l2_simple(q, p3), __float_as_int(p3.w));
      }
    }
  }
}

// Collect variant of the walk for a TIGHT bound (a late seeded iteration: the bound is the previous neighbours' largest
// distance to the barely moved point, i.e. already the answer's 5th distance): every candidate closer than the bound is
// appended to the thread's list in shared memory by a few predicated instructions — no top-5 insertion inside the walk,
// where it runs ~30 times per warp at 5 of 32 lanes; the five are selected afterwards with all lanes in step.  The bound
// is not tightened during the walk (nothing to gain when it is tight from the start).  Returns the number of candidates
// inside the bound; more than S2M_COLLECT_CAP means the list overflowed (the caller repeats with the insertion walk).
#ifndef S2M_COLLECT_CAP_CFG
#define S2M_COLLECT_CAP_CFG 16
#endif
constexpr int S2M_COLLECT_CAP = S2M_COLLECT_CAP_CFG;
// When is a seeded bound tight?  When the point has barely moved since its neighbours were found.  The last pose
// increment (deltaR in degrees, deltaT in cm: mapOptmization.cpp:1826-1833, kept in LmDevState) bounds that move by
// deltaT + deltaR x range; a warp collects when at least three quarters of its seeded lanes moved less than this.
#ifndef S2M_COLLECT_MOVE_CFG
#define S2M_COLLECT_MOVE_CFG 0.20f
#endif
constexpr float S2M_COLLECT_MOVE = S2M_COLLECT_MOVE_CFG;  // metres
template <int STRIDE>
__device__ __forceinline__ int grid_knn5_collect(const float4 q, const GridParams& g, const float bound,
                                                 const float4* __restrict__ map_sorted,
                                                 const uint32_t* __restrict__ cell_start, u64* __restrict__ list) {
  int cnt = 0;
  const float s2 = 2.0f * g.slack;
  const float reach = sqrtf(bound) * 1.000001f + s2;
  int zmin = (int)floorf((q.z - reach - g.oz) * g.inv_h), zmax = (int)floorf((q.z + reach - g.oz) * g.inv_h);
  int ymin = (int)floorf((q.y - reach - g.oy) * g.inv_h), ymax = (int)floorf((q.y + reach - g.oy) * g.inv_h);
  zmin = max(zmin, 0); zmax = min(zmax, g.nz - 1);
  ymin = max(ymin, 0); ymax = min(ymax, g.ny - 1);
  for (int z = zmin; z <= zmax; ++z) {
    const float zlo = g.oz + (float)z * g.h;
    const float gz = fmaxf(fmaxf(zlo - q.z, q.z - (zlo + g.h)) - s2, 0.f);
    const float gz2 = gz * gz;
    if (gz2 > bound) continue;
    for (int y = ymin; y <= ymax; ++y) {
      const float ylo = g.oy + (float)y * g.h;
      const float gy = fmaxf(fmaxf(ylo - q.y, q.y - (ylo + g.h)) - s2, 0.f);
      const float m2 = (gz2 + gy * gy) * 0.999999f;
      if (m2 > bound) continue;
      const float r = sqrtf(bound - m2) * 1.000001f + s2;
      int xlo = (int)floorf((q.x - r - g.ox) * g.inv_h);
      int xhi = (int)floorf((q.x + r - g.ox) * g.inv_h);
      xlo = max(xlo, 0);
      xhi = min(xhi, g.nx - 1);
      if (xlo > xhi) continue;
      const uint32_t row = ((uint32_t)z * (uint32_t)g.ny + (uint32_t)y) * (uint32_t)g.nx;
      const uint32_t s = __ldg(cell_start + row + xlo);
      const uint32_t e = __ldg(cell_start + row + xhi + 1);
      // (issuing the next row's look-ups before this row's candidates are evaluated was measured: no change)
      for (uint32_t j = s; j < e; j += 4) {
        const uint32_t last = e - 1;
        const float4 p0 = __ldg(map_sorted + j);
        const float4 p1 = __ldg(map_sorted + min(j + 1, last));
        const float4 p2 = __ldg(map_sorted + min(j + 2, last));
        const float4 p3 = __ldg(map_sorted + min(j + 3, last));
        const float d0 = l2_simple(q, p0), d1 = l2_simple(q, p1), d2 = l2_simple(q, p2), d3 = l2_simple(q, p3);
        if (d0 < bound) { list[min(cnt, S2M_COLLECT_CAP - 1) * STRIDE] = (((u64)__float_as_uint(d0)) << 32) | (u64)__float_as_uint(p0.w); ++cnt; }
        if ((j + 1 < e) & (d1 < bound)) { list[min(cnt, S2M_COLLECT_CAP - 1) * STRIDE] = (((u64)__float_as_uint(d1)) << 32) | (u64)__float_as_uint(p1.w); ++cnt; }
        if ((j + 2 < e) & (d2 < bound)) { list[min(cnt, S2M_COLLECT_CAP - 1) * STRIDE] = (((u64)__float_as_uint(d2)) << 32) | (u64)__float_as_uint(p2.w); ++cnt; }
        if ((j + 3 < e) & (d3 < bound)) { list[min(cnt, S2M_COLLECT_CAP - 1) * STRIDE] = (((u64)__float_as_uint(d3)) << 32) | (u64)__float_as_uint(p3.w); ++cnt; }
      }
    }
  }
  return cnt;
}

// Fast path of the per-thread search when the reach box covers at most 3 x 3 rows of cells (always the case
// for the phase-1 gate and for a seeded search on a grid whose cell edge is the phase-1 radius): the
// cell_start look-ups of ALL rows are issued together — one memory round trip instead of one per visited row —
// and the rows are then walked centre-out with the usual pruning against the running 5th-best distance.
// The x range of a row is fixed from the initial bound (a superset of what the tightened bound would give);
// the extra candidates cost one compare each.  Returns false when the box is larger (caller falls back).
__device__ __forceinline__ bool grid_knn5_box9(const float4 q, const GridParams& g, const float gate_d2,
                                               const float4* __restrict__ map_sorted,
                                               const uint32_t* __restrict__ cell_start, Top5& t) {
  t.init(gate_d2);
  const float s2 = 2.0f * g.slack;
  const float reach = sqrtf(gate_d2) * 1.000001f + s2;
  int zmin = (int)floorf((q.z - reach - g.oz) * g.inv_h), zmax = (int)floorf((q.z + reach - g.oz) * g.inv_h);
  int ymin = (int)floorf((q.y - reach - g.oy) * g.inv_h), ymax = (int)floorf((q.y + reach - g.oy) * g.inv_h);
  zmin = max(zmin, 0); zmax = min(zmax, g.nz - 1);
  ymin = max(ymin, 0); ymax = min(ymax, g.ny - 1);
  if (zmin > zmax || ymin > ymax) return true;  // nothing in reach
  if (zmax - zmin > 2 || ymax - ymin > 2) return false;
  // centre row first; the box is [c-1, c+1] at most, clipped
  const int cz = min(max((int)floorf((q.z - g.oz) * g.inv_h), zmin), zmax);
  const int cy = min(max((int)floorf((q.y - g.oy) * g.inv_h), ymin), ymax);
  if (cz - zmin > 1 || zmax - cz > 1 || cy - ymin > 1 || ymax - cy > 1) return false;
  uint32_t rs[9], re[9];
  float rm2[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) {
    const int dz = (k / 3 == 0) ? 0 : ((k / 3 == 1) ? -1 : 1);
    const int dy = (k % 3 == 0) ? 0 : ((k % 3 == 1) ? -1 : 1);
    const int z = cz + dz, y = cy + dy;
    rs[k] = 0; re[k] = 0; rm2[k] = FLT_MAX;
    if (z >= zmin && z <= zmax && y >= ymin && y <= ymax) {
      const float zlo = g.oz + (float)z * g.h, ylo = g.oy + (float)y * g.h;
      const float gz = fmaxf(fmaxf(zlo - q.z, q.z - (zlo + g.h)) - s2, 0.f);
      const float gy = fmaxf(fmaxf(ylo - q.y, q.y - (ylo + g.h)) - s2, 0.f);
      const float m2 = (gz * gz + gy * gy) * 0.999999f;
      if (m2 <= gate_d2) {
        const float r = sqrtf(gate_d2 - m2) * 1.000001f + s2;
        int xlo = (int)floorf((q.x - r - g.ox) * g.inv_h);
        int xhi = (int)floorf((q.x + r - g.ox) * g.inv_h);
        xlo = max(xlo, 0);
        xhi = min(xhi, g.nx - 1);
        if (xlo <= xhi) {
          const uint32_t row = ((uint32_t)z * (uint32_t)g.ny + (uint32_t)y) * (uint32_t)g.nx;
          rs[k] = __ldg(cell_start + row + xlo);
          re[k] = __ldg(cell_start + row + xhi + 1);
          rm2[k] = m2;
        }
      }
    }
  }
#pragma unroll
  for (int k = 0; k < 9; ++k) {
    if (rm2[k] > t.d(t.k4)) continue;  // also skips the rows that were never loaded (rm2 = FLT_MAX)
    const uint32_t s = rs[k], e = re[k];
    for (uint32_t j = s; j < e; j += 4) {
      const uint32_t last = e - 1;
      const float4 p0 = __ldg(map_sorted + j);
      const float4 p1 = __ldg(map_sorted + min(j + 1, last));
      const float4 p2 = __ldg(map_sorted + min(j + 2, last));
      const float4 p3 = __ldg(map_sorted + min(j + 3, last));
      t.offer(l2_simple(q, p0), __float_as_int(p0.w));
      if (j + 1 < e) t.offer(l2_simple(q, p1), __float_as_int(p1.w));
      if (j + 2 < e) t.offer(l2_simple(q, p2), __float_as_int(p2.w));
      if (j + 3 < e) t.offer(l2_simple(q, p3), __float_as_int(p3.w));
    }
  }
  return true;
}

__device__ __forceinline__ u64 warp_min_u64(const u64 v) {
  const unsigned hi = (unsigned)(v >> 32), lo = (unsigned)v;
  const unsigned mhi = __reduce_min_sync(0xffffffffu, hi);
  const unsigned mlo = __reduce_min_sync(0xffffffffu, hi == mhi ? lo : 0xffffffffu);
  return ((u64)mhi << 32) | (u64)mlo;
}

// Warp-cooperative exact 5-NN of ONE query inside the full gate (phase 2: the few queries whose
// neighbours are not within the phase-1 radius).  Lanes take the (y,z) rows in reach, 32 at a time: all
// the cell_start look-ups are in flight together; the rows' candidates are then flattened with a warp
// prefix sum and handed out one per lane, so the candidate loads are in flight together too.  Each lane
// keeps the best 5 of the candidates it saw; the lanes' lists are merged with five warp-wide minima.
// The result is identical to the sequential search: a set selection under the total order (d2, index).
// gate_ext_d2 >= gate_d2: every map point closer than sqrt(gate_ext_d2) is visited and COUNTED (return value,
// warp-uniform), while only points inside gate_d2 compete for the five slots.  The count feeds the
// "hopeless point" rule of the main kernel (see HOPELESS_* below).
// init_d2 (< 0: the gate): the sentinel of the lists, i.e. only points closer than sqrt(init_d2) compete for the five
// slots; the fused loop passes the search radius itself to learn the 5th distance even when it lies beyond the gate.
__device__ __forceinline__ int warp_knn5(const float4 q, const GridParams& g, const float gate_ext_d2,
                                         const float4* __restrict__ map_sorted,
                                         const uint32_t* __restrict__ cell_start, const int lane, Top5& out,
                                         const float init_d2 = -1.f) {
  Top5 t;
  t.init(init_d2 < 0.f ? g.gate_d2 : init_d2);
  out.init(init_d2 < 0.f ? g.gate_d2 : init_d2);
  int n_ext = 0;
  const float s2 = 2.0f * g.slack;
  const float reach = sqrtf(gate_ext_d2) * 1.000001f + s2;
  int zmin = (int)floorf((q.z - reach - g.oz) * g.inv_h), zmax = (int)floorf((q.z + reach - g.oz) * g.inv_h);
  int ymin = (int)floorf((q.y - reach - g.oy) * g.inv_h), ymax = (int)floorf((q.y + reach - g.oy) * g.inv_h);
  zmin = max(zmin, 0); zmax = min(zmax, g.nz - 1);
  ymin = max(ymin, 0); ymax = min(ymax, g.ny - 1);
  if (zmin > zmax || ymin > ymax) return 0;
  const int nys = ymax - ymin + 1;
  const int nrows = (zmax - zmin + 1) * nys;
  for (int base = 0; base < nrows; base += 32) {
    const int r = base + lane;
    uint32_t s = 0, cnt = 0;
    if (r < nrows) {
      const int z = zmin + r / nys, y = ymin + r % nys;
      const float zlo = g.oz + (float)z * g.h, ylo = g.oy + (float)y * g.h;
      const float gz = fmaxf(fmaxf(zlo - q.z, q.z - (zlo + g.h)) - s2, 0.f);
      const float gy = fmaxf(fmaxf(ylo - q.y, q.y - (ylo + g.h)) - s2, 0.f);
      const float m2 = (gz * gz + gy * gy) * 0.999999f;
      if (m2 <= gate_ext_d2) {
        const float rr = sqrtf(gate_ext_d2 - m2) * 1.000001f + s2;
        int xlo = (int)floorf((q.x - rr - g.ox) * g.inv_h);
        int xhi = (int)floorf((q.x + rr - g.ox) * g.inv_h);
        xlo = max(xlo, 0);
        xhi = min(xhi, g.nx - 1);
        if (xlo <= xhi) {
          const uint32_t row = ((uint32_t)z * (uint32_t)g.ny + (uint32_t)y) * (uint32_t)g.nx;
          s = __ldg(cell_start + row + xlo);
          cnt = __ldg(cell_start + row + xhi + 1) - s;
        }
      }
    }
    uint32_t incl = cnt;  // inclusive prefix sum of the rows' candidate counts
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
    for (uint32_t c0 = 0; c0 < total; c0 += 32) {
      const uint32_t c = c0 + lane;
      // owner row of candidate c: the first lane whose inclusive sum exceeds c (binary search by shuffles)
      int lo = 0;
#pragma unroll
      for (int step = 16; step > 0; step >>= 1) {
        const uint32_t v = __shfl_sync(0xffffffffu, incl, lo + step - 1);
        if (v <= c) lo += step;
      }
      lo = min(lo, 31);
      const uint32_t row_s = __shfl_sync(0xffffffffu, s, lo);
      const uint32_t row_incl = __shfl_sync(0xffffffffu, incl, lo);
      const uint32_t row_cnt = __shfl_sync(0xffffffffu, cnt, lo);
      if (c < total) {
        const uint32_t j = row_s + (c - (row_incl - row_cnt));
        const float4 p = __ldg(map_sorted + j);
        const float d2 = l2_simple(q, p);
        if (d2 < gate_ext_d2) ++n_ext;
        t.offer(d2, __float_as_int(p.w));
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) n_ext += __shfl_xor_sync(0xffffffffu, n_ext, o);
  // merge: five times take the smallest head over the lanes and pop it from its owner's list
  u64 res[5];
#pragma unroll
  for (int k = 0; k < 5; ++k) {
    const u64 m = warp_min_u64(t.k0);
    res[k] = m;
    const unsigned owners = __ballot_sync(0xffffffffu, t.k0 == m);
    if (lane == __ffs(owners) - 1) {
      t.rej = fminf(t.rej, FLT_MAX);
      t.k0 = t.k1; t.k1 = t.k2; t.k2 = t.k3; t.k3 = t.k4; t.k4 = ~0ull;
    }
  }
  // best candidate that is NOT in the result (tie logging): a remaining head or something a lane dropped
  const u64 next = warp_min_u64(t.k0);
  float rj = fminf(t.rej, next == ~0ull ? FLT_MAX : __uint_as_float((unsigned)(next >> 32)));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) rj = fminf(rj, __shfl_xor_sync(0xffffffffu, rj, o));
  out.k0 = res[0]; out.k1 = res[1]; out.k2 = res[2]; out.k3 = res[3]; out.k4 = res[4];
  out.rej = rj;
  return n_ext;
}

// "Hopeless" points.  A sweep point with fewer than five map points within 1 m is dropped by surfOptimization
// (:1641) — typically the far part of a sweep that lies outside the 50 m local map — but finding that out costs a
// full-gate search in every iteration.  The leftover kernel therefore also counts the map points within
// 1 m + HOPELESS_MARGIN of the point; if even that count is below five, then for as long as the point has moved
// less than the margin (minus 1 mm for rounding) since then, fewer than five map points can lie within 1 m of
// it (triangle inequality), and the main kernel skips it without searching.  Exact, not heuristic.
constexpr float HOPELESS_MARGIN = 0.25f;
// Generalised (round 2): the leftover search now learns the distance of the 5th-nearest map point even when it lies
// beyond the gate (up to 1 m + HOPELESS_MARGIN); a point whose 5th neighbour is sqrt(d5) > 1 m away cannot have five
// neighbours within the gate until it has moved sqrt(d5) - 1 m.  hopeless[i] = (position at search time, that margin
// minus 1 mm; 0 = no claim).  The old rule is the special case "fewer than five points inside the extended gate".
constexpr float HOPELESS_REL = 1e-5f;

// Full-gate search of a point the phase-1 gate could not settle, warp-cooperative, in two stages: most such points
// have their five neighbours within 0.7 m, so a first pass over that ball usually settles them (a quarter of the rows
// and candidates of the 1.25 m ball); only the rest walk the extended gate.  On return t holds the five nearest map
// points closer than sqrt(r2) (ascending), r2 = the squared radius that was enumerated completely, and t.rej the
// best distance among everything else that was visited.
constexpr float LEFT_STAGE1 = 0.7f;
__device__ __forceinline__ void leftover_search(const float4 q, const GridParams& g, const float ge2,
                                                   const float4* __restrict__ map_sorted, const uint32_t* __restrict__ cell_start,
                                                   const int lane, Top5& t, float& r2) {
  r2 = LEFT_STAGE1 * LEFT_STAGE1;
  if (r2 < g.gate_d2 && g.gate1_d2 < g.gate_d2) {  // dense map only: on a sparse one the five are usually farther (measured)
    warp_knn5(q, g, r2, map_sorted, cell_start, lane, t, r2);
    if (t.d(t.k4) < r2) return;  // five points inside the ball, all of it enumerated: exact
  }
  r2 = ge2;
  warp_knn5(q, g, ge2, map_sorted, cell_start, lane, t, ge2);
}

// The loop's initial state travels as LAUNCH PARAMETERS, not as a host-to-device copy: a copy would queue on the copy
// engine behind a sweep upload that may be in flight (liogpu_upload_scan_async) and hold the whole loop back.
struct LmInit {
  float pose[6];
  float matP[36];
  int degenerate;
  int max_iter;
};
__global__ void __launch_bounds__(256)
lm_prepare_kernel(LmDevState* st, const LmInit init) {
  if (blockIdx.x != 0) return;
  unsigned* w = reinterpret_cast<unsigned*>(st);
  for (int k = threadIdx.x; k < (int)(sizeof(LmDevState) / sizeof(unsigned)); k += blockDim.x) w[k] = 0u;
  __syncthreads();
  if (threadIdx.x < 6) st->pose[threadIdx.x] = init.pose[threadIdx.x];
  if (threadIdx.x < 36) st->matP[threadIdx.x] = init.matP[threadIdx.x];
  if (threadIdx.x == 40) { st->degenerate = init.degenerate; st->max_iter = init.max_iter; }
  __syncthreads();
  if (threadIdx.x < 32) warp_refresh_transform(st, threadIdx.x, threadIdx.x < 6 ? init.pose[threadIdx.x] : 0.f);
}

// Side computation of iteration 0's matP when the certificate let the loop go ahead (second stream).
__global__ void lm_matp_kernel(LmDevState* st) {
  __shared__ FinSmem m;
  const int lane = threadIdx.x;
  if (blockIdx.x != 0 || lane >= 32) return;
  if (!st->eig_pending) return;
  for (int e = lane; e < 36; e += 32) m.AtA[e] = st->AtA0[e];
  __syncwarp();
  // st->degenerate is not touched here: iterations 1.. read it concurrently
  const int deg = lm_eigen_matp(m, lane, st->matP);
  if (lane == 0) {
    if (deg) st->cert_mismatch = 1;  // cannot happen: the certificate is 1000+ ulps away from the threshold (tests/test_gpu_small_math.py)
    st->eig_pending = 0;
  }
}


// ------------------------------------------------------------------------------------------------
// Per-iteration launches (mode 0: LM iteration on the device state; mode 1: one surfOptimization pass
// with per-point outputs and no state update, T_override replacing the pose-derived transform):
//
//   s2m_main_kernel  one thread per scan point: transform, phase-1 search (small gate), plane fit, Jacobian
//                    row, FP64 block reduction -> partials[block].  A point whose 5 neighbours are not all
//                    inside the phase-1 radius is NOT searched further here: its index goes to the block's
//                    segment of `fail_seg` (deterministic order) so no warp ever waits for a straggler.
//                    The leftover kernel turns the per-block counts into segment offsets (only when that table
//                    exceeds its shared memory does the main kernel's last block still do it).
//   s2m_left_kernel  the leftover points (about 2 % on a dense map, all of them on a sparse one), 32 per
//                    warp: warp-cooperative full-gate search per point, then the plane fit lane-parallel.
//                    Its blocks also fold the main kernel's partials; the last block adds everything in a
//                    fixed order and runs the 6x6 tail of LMOptimization (lm_finalize_warp).
struct S2mArgs {
  const float4* scan;
  int nq;
  const float4* map4;
  const float4* map_sorted;
  const uint32_t* cell_start;
  GridParams g;
  LmDevState* st;
  double* partials_main;   // [main blocks][S2M_SUMS]
  double* partials_left;   // [left blocks][S2M_SUMS]
  int* block_nfail;        // [main blocks]
  int* fail_seg;           // [main blocks][S2M_THREADS]
  int* fail_off;           // [main blocks + 1] exclusive scan of block_nfail
  int* fail_total;         // [1]
  unsigned* ticket;        // [2]: main, left
  const float* T_override;
  SurfDebugOut dbg;
  int mode;
  int main_blocks;         // main kernel blocks: partial rows of the main phase and leftover segments
  float collect_move;      // metres: a warp collects when most of its seeded points moved less than this (see main_point)
  int* prev_nn;            // [5][nq] neighbours found by the previous iteration (-1: none), SoA
  float4* hopeless;        // [nq] (x,y,z of the point when it was found hopeless, w = 1) or w = 0
};

struct RowAcc {  // which product of the staged row a reducing thread owns
  int a, b;
  bool live;
};
__device__ __forceinline__ RowAcc row_acc_of(const int p) {
  RowAcc r;
  r.live = p <= 27;
  if (p < 21) {  // upper-triangle pair index -> (a, b)
    int q = p, a = 0;
    while (q >= 6 - a) { q -= 6 - a; ++a; }
    r.a = a; r.b = a + q;
  } else if (p < 27) {
    r.a = p - 21; r.b = 6;
  } else {
    r.a = 7; r.b = 7;  // p == 27: accepted count (flag * flag)
  }
  return r;
}

// plane fit + Jacobian row of one point whose neighbours are known; writes the debug outputs in mode 1
__device__ __forceinline__ void finish_point(const S2mArgs& A, const int i, const float4 ori, const float4 sel,
                                             const Top5& t, const LmTrig& trig, float row[6], float& rhs, bool& flag,
                                             bool& tie) {
  float4 coeff = make_float4(0.f, 0.f, 0.f, 0.f);
  const bool found = t.d(t.k4) < A.g.gate_d2;  // :1641 (the gate is the reference's 1.0)
  flag = false; tie = false;
  if (found) {
    float4 nbr[5];
    nbr[0] = __ldg(A.map4 + t.i(t.k0)); nbr[1] = __ldg(A.map4 + t.i(t.k1)); nbr[2] = __ldg(A.map4 + t.i(t.k2));
    nbr[3] = __ldg(A.map4 + t.i(t.k3)); nbr[4] = __ldg(A.map4 + t.i(t.k4));
    flag = plane_residual(ori, sel, nbr, coeff);
    tie = t.tie();
    if (!flag) coeff = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  if (flag) jacobian_row(trig, ori, coeff, row, rhs);
  if (A.mode == 0) {  // seeds of the next iteration
    A.prev_nn[i] = found ? t.i(t.k0) : -1;
    A.prev_nn[(size_t)A.nq + i] = t.i(t.k1);
    A.prev_nn[2 * (size_t)A.nq + i] = t.i(t.k2);
    A.prev_nn[3 * (size_t)A.nq + i] = t.i(t.k3);
    A.prev_nn[4 * (size_t)A.nq + i] = t.i(t.k4);
  }
  if (A.mode == 1) {
    if (A.dbg.nn_idx) {
      int* o = A.dbg.nn_idx + (size_t)i * 5;
      o[0] = found ? t.i(t.k0) : -1; o[1] = found ? t.i(t.k1) : -1; o[2] = found ? t.i(t.k2) : -1;
      o[3] = found ? t.i(t.k3) : -1; o[4] = found ? t.i(t.k4) : -1;
    }
    if (A.dbg.nn_d2) {
      float* o = A.dbg.nn_d2 + (size_t)i * 5;
      o[0] = t.d(t.k0); o[1] = t.d(t.k1); o[2] = t.d(t.k2); o[3] = t.d(t.k3); o[4] = t.d(t.k4);
    }
    if (A.dbg.coeff) A.dbg.coeff[i] = coeff;
    if (A.dbg.flag) A.dbg.flag[i] = flag ? 1 : 0;
    if (A.dbg.tie) A.dbg.tie[i] = tie ? 1 : 0;
  }
}

// One sweep point of surfOptimization: transform, exact search (phase-1 gate, seeded bound or skip), plane fit, Jacobian row.
// need2: the phase-1 gate could not settle the point (it goes to the leftover list).
__device__ __forceinline__ void main_point(const S2mArgs& A, const float* sT, const LmTrig& sTrig, const int s_iter, const int i,
                                           float row[6], float& rhs, bool& flag, bool& tie, bool& need2, int& seeded,
                                           u64* __restrict__ slist, const float step_t, const float step_r) {
    const float4 ori = A.scan[i];
    const float4 sel = apply_T(sT, ori);
    Top5 t;
    const bool dense = A.g.gate1_d2 < A.g.gate_d2;     // phase-1 gate active (cell edge = its radius)
    float gate_use = fminf(A.g.gate1_d2, A.g.gate_d2);
    const float gate1_use = gate_use;
    bool can_search = dense, is_seeded = false, skip = false;
    if (s_iter > 0) {
      // Seeded search: the five neighbours of the previous iteration are real map points, so their
      // largest distance to the moved query bounds the true 5th-neighbour distance.  Searching inside
      // that bound is exact, prunes almost every row, and needs no second phase.
      const int p0 = A.prev_nn[i];
      if (p0 < 0) {
        const float4 hr = A.hopeless[i];
        if (hr.w > 0.f) {
          const float dx = sel.x - hr.x, dy = sel.y - hr.y, dz = sel.z - hr.z;
          skip = (dx * dx + dy * dy + dz * dz) * (1.f + HOPELESS_REL) < hr.w * hr.w;  // still cannot have 5 neighbours within the gate
        }
      }
      if (p0 >= 0) {
        const int p1 = A.prev_nn[(size_t)A.nq + i], p2 = A.prev_nn[2 * (size_t)A.nq + i];
        const int p3 = A.prev_nn[3 * (size_t)A.nq + i], p4 = A.prev_nn[4 * (size_t)A.nq + i];
        const float d0 = l2_simple(sel, __ldg(A.map4 + p0)), d1 = l2_simple(sel, __ldg(A.map4 + p1));
        const float d2 = l2_simple(sel, __ldg(A.map4 + p2)), d3 = l2_simple(sel, __ldg(A.map4 + p3));
        const float d4 = l2_simple(sel, __ldg(A.map4 + p4));
        const float D = fmaxf(fmaxf(fmaxf(d0, d1), fmaxf(d2, d3)), d4);
        const float bound = __uint_as_float(__float_as_uint(D) + 1u);  // next float above D: the seeds stay inside
        if (bound <= A.g.gate_d2) {
          gate_use = bound;
          can_search = true;
          is_seeded = true;
          ++seeded;
        }
      }
    }
    // How the seeded points of this warp search (all three are exact; the choice only moves time):
    //   the last pose step was small for most of them -> collect, then select (grid_knn5_collect): 58 vs 70 us per launch;
    //   otherwise -> the insertion walk that tightens its bound as it goes (after a large step the seeds' bound is loose:
    //   collecting then costs 130 us instead of 77).
    bool use_collect = false;
    if (s_iter > 0 && dense) {
      const float range = sqrtf(ori.x * ori.x + ori.y * ori.y + ori.z * ori.z);
      const unsigned act = __activemask();
      const unsigned ms = __ballot_sync(act, is_seeded);
      const unsigned mt = __ballot_sync(act, is_seeded && step_t + step_r * range < A.collect_move);
      use_collect = 4 * __popc(mt) >= 3 * __popc(ms);
    }
    if (skip) {
      t.init(A.g.gate_d2);  // "not found": flag false, no seeds for the next iteration, marker kept
      need2 = false;
    } else if (can_search) {
      bool searched = false;
      if (is_seeded && use_collect) {
        const int cnt = grid_knn5_collect<S2M_THREADS>(sel, A.g, gate_use, A.map_sorted, A.cell_start, slist);
        if (cnt <= S2M_COLLECT_CAP) {  // else: the list overflowed, the insertion walk below repeats the search
          t.init(gate_use);
          for (int j = 0; j < cnt; ++j) {
            const u64 key = slist[j * S2M_THREADS];
            t.offer(__uint_as_float((unsigned)(key >> 32)), (int)(unsigned)(key & 0xffffffffull));
          }
          searched = true;
        }
      }
      if (!searched) {
        // dense map: the row-by-row walk (x ranges tightened as the bound shrinks) executes fewer instructions
        // and the kernel is issue bound; sparse map (1 m cells, few points per row): the search is latency
        // bound and the all-rows-at-once variant wins
        if (dense || !grid_knn5_box9(sel, A.g, gate_use, A.map_sorted, A.cell_start, t))
          grid_knn5(sel, A.g, gate_use, A.map_sorted, A.cell_start, t);
      }
      need2 = !is_seeded && !(t.d(t.k4) < gate1_use);
    } else {
      need2 = true;
    }
    if (!need2) finish_point(A, i, ori, sel, t, sTrig, row, rhs, flag, tie);
}

__global__ void __launch_bounds__(S2M_THREADS, S2M_MINBLOCKS_CFG)
s2m_main_kernel(const S2mArgs A) {
  __shared__ float sT[12];
  __shared__ LmTrig sTrig;
  __shared__ float rows[S2M_THREADS][8];  // 6 Jacobian entries, rhs, accepted flag
  __shared__ u64 s_list[S2M_COLLECT_CAP][S2M_THREADS];  // candidates inside the bound (grid_knn5_collect), slot-major
  __shared__ float s_step[2];
  __shared__ double red[S2M_THREADS / 32][S2M_SUMS];
  __shared__ int s_ties, s_wfail[S2M_THREADS / 32], s_iter, s_seeded;
  __shared__ bool s_last;

  __shared__ int s_done0;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // Programmatic dependent launch: this grid may have been scheduled while the previous kernel of the stream
  // was still in its single-block tail; nothing it wrote may be read before this returns.
  cudaGridDependencySynchronize();
  // a launch enqueued beyond the loop's last iteration: every thread sees the flag itself and leaves at once
  if (A.mode == 0 && __ldcg(&A.st->done)) return;
  if (tid < 12) sT[tid] = A.T_override ? A.T_override[tid] : A.st->T[tid];  // updatePointAssociateToMap (:1613-1616)
  if (tid == 32) {
    sTrig.srx = A.st->trig[0]; sTrig.crx = A.st->trig[1]; sTrig.sry = A.st->trig[2];
    sTrig.cry = A.st->trig[3]; sTrig.srz = A.st->trig[4]; sTrig.crz = A.st->trig[5];
    s_ties = 0;
    s_seeded = 0;
  }
  if (tid == 64) { s_done0 = A.st->done; s_iter = A.mode == 0 ? A.st->iter : 0; }
  if (tid == 96) { s_step[0] = A.st->delta_t * 0.01f; s_step[1] = A.st->delta_r * 0.01745329f; }  // last step: metres, radians
  __syncthreads();
  if (A.mode == 0 && s_done0) return;

  const int i = blockIdx.x * S2M_THREADS + tid;
  float row[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  float rhs = 0.f;
  bool flag = false, tie = false, need2 = false;
  int seeded = 0;
  if (i < A.nq) main_point(A, sT, sTrig, s_iter, i, row, rhs, flag, tie, need2, seeded, &s_list[0][tid], s_step[0], s_step[1]);
  // leftover indices, in thread order, into this block's segment
  const unsigned fm = __ballot_sync(0xffffffffu, need2);
  if (lane == 0) s_wfail[warp] = __popc(fm);
#pragma unroll
  for (int k = 0; k < 6; ++k) rows[tid][k] = row[k];
  rows[tid][6] = rhs;
  rows[tid][7] = flag ? 1.f : 0.f;
  if (flag && tie) atomicAdd(&s_ties, 1);
  {
    const int ws = __popc(__ballot_sync(0xffffffffu, seeded != 0));
    if (lane == 0 && ws) atomicAdd(&s_seeded, ws);
  }
  __syncthreads();
  if (need2) {
    int base = 0;
    for (int w = 0; w < warp; ++w) base += s_wfail[w];
    A.fail_seg[(size_t)blockIdx.x * S2M_THREADS + base + __popc(fm & ((1u << lane) - 1u))] = i;
  }
  // 27 FP64 sums + count: thread (slice, p) adds its 32 rows' product p; products of two floats are
  // exact in double, so only the order of additions differs from cv::gemm's.
  {
    const int p = lane, slice = warp;
    const RowAcc ra = row_acc_of(p);
    double acc = 0.0;
    if (ra.live) {
#pragma unroll 8
      for (int r = 0; r < 32; ++r) {
        const float* rr = rows[slice * 32 + r];
        acc += (double)rr[ra.a] * (double)rr[ra.b];
      }
    }
    red[slice][p] = acc;
  }
  __syncthreads();
  if (tid < S2M_SUMS) {
    double sum = 0.0;
#pragma unroll
    for (int k = 0; k < S2M_THREADS / 32; ++k) sum += red[k][tid];
    if (tid == 28) sum = (double)s_ties;
    if (tid == 29) sum = (double)s_seeded;
    A.partials_main[(size_t)blockIdx.x * S2M_SUMS + tid] = sum;
  }
  if (tid == 0) {
    int nf = 0;
    for (int w = 0; w < S2M_THREADS / 32; ++w) nf += s_wfail[w];
    A.block_nfail[blockIdx.x] = nf;
  }
  if (A.main_blocks + 1 <= LEFT_OFF_CAP) return;  // the leftover kernel derives the offsets itself
  __threadfence();
  __syncthreads();
  if (tid == 0) s_last = (atomicAdd(A.ticket, 1u) == gridDim.x - 1);
  __syncthreads();
  if (!s_last) return;
  // ---- last block: exclusive scan of the per-block leftover counts -> fail_off (block order) ----
  __threadfence();
  __shared__ int s_wsum[S2M_THREADS / 32];
  __shared__ int s_carry;
  if (tid == 0) s_carry = 0;
  __syncthreads();
  for (int b0 = 0; b0 < (int)gridDim.x; b0 += S2M_THREADS) {
    const int b = b0 + tid;
    const int cnt = b < (int)gridDim.x ? __ldcg(A.block_nfail + b) : 0;
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    if (lane == 31) s_wsum[warp] = incl;
    __syncthreads();
    int base = s_carry;
    for (int w = 0; w < warp; ++w) base += s_wsum[w];
    if (b < (int)gridDim.x) A.fail_off[b] = base + incl - cnt;
    __syncthreads();
    if (tid == S2M_THREADS - 1) s_carry = base + incl;
    __syncthreads();
  }
  if (tid == 0) {
    A.fail_off[gridDim.x] = s_carry;
    *A.fail_total = s_carry;
    *A.ticket = 0u;
  }
}

constexpr int LEFT_THREADS = 256;
__global__ void __launch_bounds__(LEFT_THREADS, 2)
s2m_left_kernel(const S2mArgs A) {
  __shared__ float sT[12];
  __shared__ LmTrig sTrig;
  __shared__ float rows[LEFT_THREADS][8];
  __shared__ double red[LEFT_THREADS / 32][S2M_SUMS];
  __shared__ int s_ties;
  __shared__ bool s_last;
  __shared__ FinSmem s_fin;

  __shared__ int s_done0, s_iter0, s_total0;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  cudaGridDependencySynchronize();  // see s2m_main_kernel
  if (A.mode == 0 && __ldcg(&A.st->done)) return;  // enqueued beyond the last iteration (before the offset scan below)
  // every global value the block needs is requested in one go (one L2 round trip instead of four)
  if (tid < 12) sT[tid] = A.T_override ? A.T_override[tid] : A.st->T[tid];
  if (tid == 32) {
    sTrig.srx = A.st->trig[0]; sTrig.crx = A.st->trig[1]; sTrig.sry = A.st->trig[2];
    sTrig.cry = A.st->trig[3]; sTrig.srz = A.st->trig[4]; sTrig.crz = A.st->trig[5];
    s_ties = 0;
  }
  const bool off_in_smem = A.main_blocks + 1 <= LEFT_OFF_CAP;
  if (tid == 64) { s_done0 = A.st->done; s_iter0 = A.st->iter; s_total0 = off_in_smem ? 0 : *A.fail_total; }
  // The offsets of the leftover segments (exclusive scan of the main kernel's per-block counts), computed HERE by every
  // block in shared memory: every thread sums a contiguous slice of the counts (all loads in flight), one block-wide scan
  // of the 256 slice sums, then the slice's prefixes are written out.  The binary search below runs on shared memory.
  __shared__ int s_off[LEFT_OFF_CAP];
  __shared__ int s_wsum[LEFT_THREADS / 32];
  if (off_in_smem) {
    for (int k = tid; k < A.main_blocks; k += LEFT_THREADS) s_off[k] = __ldcg(A.block_nfail + k);  // one round trip
    __syncthreads();
    const int per = (A.main_blocks + LEFT_THREADS - 1) / LEFT_THREADS;
    const int k0 = min(tid * per, A.main_blocks), k1 = min(k0 + per, A.main_blocks);
    int sum = 0;
    for (int k = k0; k < k1; ++k) sum += s_off[k];
    int incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    if (lane == 31) s_wsum[warp] = incl;
    __syncthreads();
    int run = incl - sum;
    for (int w = 0; w < warp; ++w) run += s_wsum[w];
    for (int k = k0; k < k1; ++k) { const int v = s_off[k]; s_off[k] = run; run += v; }
    if (tid == LEFT_THREADS - 1) { s_off[A.main_blocks] = run; s_total0 = run; }
  }
  __syncthreads();
  if (A.mode == 0 && s_done0) return;
  // sparse map (no phase-1 gate): on iteration 0 (and in mode 1) the main kernel did not run at all
  const bool all_points = !(A.g.gate1_d2 < A.g.gate_d2) && (A.mode == 1 || s_iter0 == 0);
  const int total = all_points ? A.nq : s_total0;
  if (A.mode == 0 && blockIdx.x == 0 && tid == 0 && s_iter0 < LIOGPU_MAX_ITER) {  // statistics
    A.st->left_hist[s_iter0] = total;
    A.st->leftovers = total;
  }
  const int warps_per_grid = gridDim.x * (LEFT_THREADS / 32);
  // points per warp: as few as possible (each point is a serial chain of dependent look-ups, so spreading
  // them over all resident warps hides that latency), up to 32 when there are more points than warps
  const int per_warp = min(32, max(1, (total + warps_per_grid - 1) / warps_per_grid));
  const int nbatch = (total + per_warp - 1) / per_warp;
  const RowAcc ra = row_acc_of(lane);
  double acc = 0.0;  // this thread's share of the block's sums, kept across rounds
  int ties = 0;
  // rounds: in round r, warp w of the grid owns batch r * warps_per_grid + (block, warp) — a static map,
  // so the order of every addition is fixed.
  for (int r0 = 0; r0 < nbatch; r0 += warps_per_grid) {
    const int batch = r0 + blockIdx.x * (LEFT_THREADS / 32) + warp;
    float row[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    float rhs = 0.f;
    bool flag = false, tie = false;
    if (batch < nbatch) {
      const int e0 = batch * per_warp;
      const int cnt = min(per_warp, total - e0);
      int mine = -1;
      if (lane < cnt) {
        const int e = e0 + lane;
        if (all_points) {
          mine = e;
        } else {  // leftover e lives in the segment of the main block whose offset range contains it
          int lo = 0, hi = A.main_blocks;  // invariant: fail_off[lo] <= e < fail_off[hi]
          while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            const int v = off_in_smem ? s_off[mid] : __ldg(A.fail_off + mid);
            if (v <= e) lo = mid; else hi = mid;
          }
          mine = A.fail_seg[(size_t)lo * S2M_THREADS + (e - (off_in_smem ? s_off[lo] : __ldg(A.fail_off + lo)))];
        }
      }
      float4 ori = make_float4(0.f, 0.f, 0.f, 0.f), sel = ori;
      if (mine >= 0) { ori = A.scan[mine]; sel = apply_T(sT, ori); }
      Top5 t;
      t.init(A.g.gate_d2);
      const float ge = sqrtf(A.g.gate_d2) + HOPELESS_MARGIN;
      for (int j = 0; j < cnt; ++j) {  // the warp searches for point j; lane j keeps the answer
        float4 q;
        q.x = __shfl_sync(0xffffffffu, sel.x, j); q.y = __shfl_sync(0xffffffffu, sel.y, j);
        q.z = __shfl_sync(0xffffffffu, sel.z, j); q.w = 0.f;
        Top5 tj;
        float r2;
        leftover_search(q, A.g, ge * ge, A.map_sorted, A.cell_start, lane, tj, r2);
        if (lane == j) t = tj;
      }
      if (mine >= 0) {
        finish_point(A, mine, ori, sel, t, sTrig, row, rhs, flag, tie);
        // d(k4) = the 5th-nearest distance^2 when five points lie inside the enumerated ball, else its radius^2
        const bool found = t.d(t.k4) < A.g.gate_d2;
        const float margin = found ? 0.f : sqrtf(t.d(t.k4)) * (1.f - HOPELESS_REL) - sqrtf(A.g.gate_d2) - 1e-3f;
        A.hopeless[mine] = make_float4(sel.x, sel.y, sel.z, margin > 0.f ? margin : 0.f);
      }
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) rows[tid][k] = row[k];
    rows[tid][6] = rhs;
    rows[tid][7] = flag ? 1.f : 0.f;
    if (flag && tie) ++ties;
    __syncthreads();
    if (ra.live) {  // every warp owns the slice of rows its own lanes staged
#pragma unroll 8
      for (int r = 0; r < 32; ++r) {
        const float* rr = rows[warp * 32 + r];
        acc += (double)rr[ra.a] * (double)rr[ra.b];
      }
    }
    __syncthreads();
  }
  // fold this block's share of the main kernel's partial rows (same (slice, p) ownership)
#pragma unroll 4
  for (int b = blockIdx.x * (LEFT_THREADS / 32) + warp; !all_points && b < A.main_blocks; b += warps_per_grid)
    acc += __ldcg(A.partials_main + (size_t)b * S2M_SUMS + lane);
  if (ties) atomicAdd(&s_ties, ties);
  red[warp][lane] = acc;
  __syncthreads();
  if (tid < S2M_SUMS) {
    double sum = 0.0;
#pragma unroll
    for (int k = 0; k < LEFT_THREADS / 32; ++k) sum += red[k][tid];
    if (tid == 28) sum += (double)s_ties;  // main kernel's tie counts arrive through slot 28 of its partials
    A.partials_left[(size_t)blockIdx.x * S2M_SUMS + tid] = sum;
  }
  if (A.mode == 1) return;
  __threadfence();
  __syncthreads();
  if (tid == 0) s_last = (atomicAdd(A.ticket + 1, 1u) == gridDim.x - 1);
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  {  // fixed-order sum over the left blocks: 8 slices of blocks, then the slices
    // sixteen independent accumulators: the pass is L2-latency bound, so the loads of a group are all in flight together
    // (fixed order of additions: accumulator k takes blocks warp + (16 j + k) W, then the accumulators are added pairwise)
    constexpr unsigned W = LEFT_THREADS / 32, U = 16;
    double a[U];
#pragma unroll
    for (unsigned k = 0; k < U; ++k) a[k] = 0.0;
    unsigned b = warp;
    for (; b + (U - 1) * W < gridDim.x; b += U * W) {
      double v[U];
#pragma unroll
      for (unsigned k = 0; k < U; ++k) v[k] = __ldcg(A.partials_left + (size_t)(b + k * W) * S2M_SUMS + lane);
#pragma unroll
      for (unsigned k = 0; k < U; ++k) a[k] += v[k];
    }
    {
      double v[U];
#pragma unroll
      for (unsigned k = 0; k < U; ++k) v[k] = (b + k * W < gridDim.x) ? __ldcg(A.partials_left + (size_t)(b + k * W) * S2M_SUMS + lane) : 0.0;
#pragma unroll
      for (unsigned k = 0; k < U; ++k) a[k] += v[k];
    }
#pragma unroll
    for (unsigned o = U / 2; o > 0; o >>= 1) {
#pragma unroll
      for (unsigned k = 0; k < o; ++k) a[k] += a[k + o];
    }
    red[warp][lane] = a[0];
  }
  __syncthreads();
  if (tid < S2M_SUMS) {
    double sum = 0.0;
#pragma unroll
    for (int k = 0; k < LEFT_THREADS / 32; ++k) sum += red[k][tid];
    red[0][tid] = sum;
  }
  __syncthreads();
  if (tid < 32) {
    lm_finalize_warp(A.st, red[0], s_fin, tid);
    if (tid == 0) A.ticket[1] = 0u;
  }
}

}  // namespace liogpu
#include "s2m_fused.cuh"
namespace liogpu {

// Both kernels of an iteration are launched with programmatic stream serialization: the next grid is scheduled
// as the previous one drains (its last block is still reducing / solving the 6x6 system) and waits in
// cudaGridDependencySynchronize(), which hides the launch latency between dependent kernels.
template <class K>
static cudaError_t launch_pdl(K kernel, int blocks, int threads, cudaStream_t stream, const S2mArgs& A) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)blocks);
  cfg.blockDim = dim3((unsigned)threads);
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, A);
}

static int check_grid(Ctx* c) {
  if (!c->grid_valid) { c->err = "no local map installed (call liogpu_set_local_map / liogpu_build_local_map)"; return LIOGPU_E_NO_MAP; }
  return LIOGPU_OK;
}

// device scratch shared by both entry points.  fail_buf: fail_seg[main_blocks][S2M_THREADS] | fail_off[main_blocks + 1] |
// block_nfail[main_blocks] | fail_total[1]; block_counter: word 0 the main kernel's ticket, word 1 the leftover kernel's.
static int prepare_args(Ctx* c, const float4* scan4, int n, S2mArgs& A, int& main_blocks, int& left_blocks) {
  A = S2mArgs{};
  main_blocks = div_up(n, S2M_THREADS);
  // two CTAs per SM: a leftover point is a serial chain of dependent look-ups (~5 us), so they are spread
  // over as many resident warps as possible (one point per warp up to 2368 points)
  left_blocks = c->sm_count * 2;
  LIOGPU_CUDA_OK(c, c->lm_state.reserve(sizeof(LmDevState)));
  LIOGPU_CUDA_OK(c, c->partials.reserve(((size_t)main_blocks + left_blocks) * S2M_SUMS * sizeof(double)));
  LIOGPU_CUDA_OK(c, c->fail_buf.reserve(((size_t)main_blocks * S2M_THREADS + 2 * (size_t)main_blocks + 64) * sizeof(int)));
  if (!c->block_counter.p) {
    LIOGPU_CUDA_OK(c, c->block_counter.reserve(64));
    LIOGPU_CUDA_OK(c, cudaMemsetAsync(c->block_counter.p, 0, 64, c->stream));
  }
  A.scan = scan4; A.nq = n;
  A.map4 = c->map4.as<float4>(); A.map_sorted = c->map_sorted.as<float4>(); A.cell_start = c->cell_start.as<uint32_t>();
  A.g = c->grid;
  A.st = c->lm_state.as<LmDevState>();
  A.partials_main = c->partials.as<double>();
  A.partials_left = A.partials_main + (size_t)main_blocks * S2M_SUMS;
  int* fb = c->fail_buf.as<int>();
  A.fail_seg = fb;
  // LIOGPU_COLLECT_MOVE (metres) overrides the threshold of the collecting walk: 0 = never collect, a huge value = every
  // seeded iteration collects (tests/test_gpu_variants.py uses both to exercise the list-overflow fallback)
  static const float collect_move = [] { const char* e = getenv("LIOGPU_COLLECT_MOVE"); return e ? (float)atof(e) : S2M_COLLECT_MOVE; }();
  A.collect_move = collect_move;
  A.fail_off = fb + (size_t)main_blocks * S2M_THREADS;
  A.block_nfail = A.fail_off + main_blocks + 1;
  A.fail_total = A.block_nfail + main_blocks;
  A.ticket = c->block_counter.as<unsigned>();
  LIOGPU_CUDA_OK(c, c->prev_nn.reserve((size_t)5 * (size_t)(n > 0 ? n : 1) * sizeof(int)));
  A.prev_nn = c->prev_nn.as<int>();
  LIOGPU_CUDA_OK(c, c->hopeless.reserve((size_t)(n > 0 ? n : 1) * sizeof(float4)));
  A.hopeless = c->hopeless.as<float4>();
  A.T_override = nullptr;
  A.dbg = SurfDebugOut{nullptr, nullptr, nullptr, nullptr, nullptr};
  A.mode = 0;
  A.main_blocks = main_blocks;
  return LIOGPU_OK;
}

static void fill_info(Ctx* c, const LmDevState* h, int n, liogpu_s2m_info* info) {
  info->iterations = h->iter;
  info->converged = h->converged;
  info->n_query = n;
  info->n_sel = h->n_sel;
  info->is_degenerate = h->degenerate;
  info->tie_queries = h->tie_queries;
  info->delta_r_deg = h->delta_r;
  info->delta_t_cm = h->delta_t;
  memcpy(info->JtJ, h->JtJ, sizeof(info->JtJ));
  memcpy(info->Jtr, h->Jtr, sizeof(info->Jtr));
  memcpy(info->pose_hist, h->pose_hist, sizeof(info->pose_hist));
  memcpy(info->nsel_hist, h->nsel_hist, sizeof(info->nsel_hist));
  info->gpu_ms = c->last_ms;
  info->seeded = h->seeded;
  info->certified = h->certified;
  info->leftovers = h->leftovers;
}

// CTAs of the cooperative launch: every slot the kernel can occupy (cached per context)
static int fused_grid(Ctx* c) {
  if (c->fz_grid != 0) return c->fz_grid;
  int coop = 0, per_sm = 0;
  if (cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, c->device) != cudaSuccess || !coop ||
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, s2m_fused_kernel, FZ_THREADS, 0) != cudaSuccess || per_sm < 1) {
    cudaGetLastError();
    c->fz_grid = -1;
    return -1;
  }
  c->fz_grid = per_sm * c->sm_count;
  return c->fz_grid;
}

// The whole loop as one persistent cooperative launch (s2m_fused.cuh).  dbg: per-point outputs of the last executed
// iteration (device pointers), or null.
static int scan2map_fused_dev(Ctx* c, const float4* scan4, int n, float pose_io[6], float matP_io[36], int* degenerate_io,
                              int max_iter, liogpu_s2m_info* info, const SurfDebugOut* dbg) {
  const int grid = fused_grid(c);
  const int nchunks = div_up(n, FZ_THREADS);
  FusedArgs A;
  LIOGPU_CUDA_OK(c, c->lm_state.reserve(sizeof(LmDevState)));
  LIOGPU_CUDA_OK(c, c->fz_rows.reserve(((size_t)nchunks + (size_t)grid) * S2M_SUMS * sizeof(double)));
  LIOGPU_CUDA_OK(c, c->fz_left.reserve(((size_t)nchunks * FZ_THREADS + (size_t)nchunks + 64) * sizeof(int)));
  LIOGPU_CUDA_OK(c, c->prev_nn.reserve((size_t)FZ_K * (size_t)n * sizeof(int)));
  LIOGPU_CUDA_OK(c, c->fz_lb.reserve((size_t)n * sizeof(float)));
  LIOGPU_CUDA_OK(c, c->hopeless.reserve((size_t)n * sizeof(float4)));
  A.scan = scan4; A.nq = n;
  A.map4 = c->map4.as<float4>(); A.map_sorted = c->map_sorted.as<float4>(); A.cell_start = c->cell_start.as<uint32_t>();
  A.g = c->grid;
  A.st = c->lm_state.as<LmDevState>();
  A.chunk_rows = c->fz_rows.as<double>();
  A.cta_rows = A.chunk_rows + (size_t)nchunks * S2M_SUMS;
  A.left_list = c->fz_left.as<int>();
  A.chunk_nleft = A.left_list + (size_t)nchunks * FZ_THREADS;
  A.prev_nn = c->prev_nn.as<int>();
  A.prev_lb = c->fz_lb.as<float>();
  A.hopeless = c->hopeless.as<float4>();
  A.probe = nullptr;
  A.dbg = dbg ? *dbg : SurfDebugOut{nullptr, nullptr, nullptr, nullptr, nullptr};
  A.nchunks = nchunks;
  A.use_cert = c->prm.s2m_no_certificate ? 0 : 1;
  const bool prof = c->prm.profile_kernels != 0;
  unsigned long long* h_probe = reinterpret_cast<unsigned long long*>((char*)c->h_pinned + 8192);
  if (prof) {
    LIOGPU_CUDA_OK(c, c->fz_probe.reserve(LIOGPU_MAX_ITER * FZ_PROBES * sizeof(unsigned long long)));
    A.probe = c->fz_probe.as<unsigned long long>();
    LIOGPU_CUDA_OK(c, cudaMemsetAsync(A.probe, 0, LIOGPU_MAX_ITER * FZ_PROBES * sizeof(unsigned long long), c->stream));
  }
  LmDevState* h = reinterpret_cast<LmDevState*>((char*)c->h_pinned + 4096);
  LmInit init;
  for (int k = 0; k < 6; ++k) init.pose[k] = pose_io[k];
  for (int k = 0; k < 36; ++k) init.matP[k] = matP_io[k];
  init.degenerate = *degenerate_io;
  init.max_iter = max_iter;
  LmDevState* d = A.st;
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
  lm_prepare_kernel<<<1, 256, 0, c->stream>>>(d, init);
  c->launches++;
  void* kargs[] = {(void*)&A};
  LIOGPU_CUDA_OK(c, cudaLaunchCooperativeKernel((const void*)s2m_fused_kernel, dim3((unsigned)grid), dim3(FZ_THREADS), kargs, 0, c->stream));
  c->launches++;
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(h, d, sizeof(LmDevState), cudaMemcpyDeviceToHost, c->stream));
  if (prof) LIOGPU_CUDA_OK(c, cudaMemcpyAsync(h_probe, A.probe, LIOGPU_MAX_ITER * FZ_PROBES * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
  LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  LIOGPU_CUDA_OK(c, cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1));
  for (int k = 0; k < 6; ++k) pose_io[k] = h->pose[k];
  for (int k = 0; k < 36; ++k) matP_io[k] = h->matP[k];
  *degenerate_io = h->degenerate;
  if (info) {
    fill_info(c, h, n, info);
    info->kernel_launches = 1;  // the loop itself (plus the 2.5 KB state initialisation)
    for (int it = 0; it < LIOGPU_MAX_ITER; ++it) {
      info->certified_hist[it] = h->cert_hist[it]; info->seeded_hist[it] = h->seed_hist[it];
      info->leftover_hist[it] = h->left_hist[it];
    }
    if (prof) {
      // probes (ns, %globaltimer): 0 iteration start, 2 last CTA out of the main phase, 5 last CTA out of the
      // deferred-leftover phase (if it ran), 6 sums complete, 7 6x6 tail done
      double m = 0, l = 0, t = 0;
      int cnt = 0;
      for (int it = 0; it < h->iter && it < LIOGPU_MAX_ITER; ++it) {
        const unsigned long long* p = h_probe + it * FZ_PROBES;
        if (!p[0] || !p[2] || !p[7]) break;
        const unsigned long long arrive = p[5] ? p[5] : p[2];
        m += (double)(p[2] - p[0]); l += (double)(p[7] - p[2]); t += (double)(p[7] - arrive);
        info->main_us_hist[it] = (float)((double)(p[2] - p[0]) * 1e-3);
        info->rest_us_hist[it] = (float)((double)(p[7] - p[2]) * 1e-3);
        ++cnt;
      }
      info->main_kernel_ms = (float)(m * 1e-6); info->left_kernel_ms = (float)(l * 1e-6); info->tail_ms = (float)(t * 1e-6);
      info->main_kernel_launches = cnt; info->left_kernel_launches = cnt;
      if (getenv("LIOGPU_PRINT_PROBES")) {  // development aid: every stamp relative to the iteration's start, us
        for (int it = 0; it < cnt; ++it) {
          const unsigned long long* p = h_probe + it * FZ_PROBES;
          fprintf(stderr, "[liogpu probes] it %d:", it);
          for (int k = 1; k < FZ_PROBES; ++k) fprintf(stderr, " p%d=%.1f", k, p[k] ? (double)(p[k] - p[0]) * 1e-3 : -1.0);
          fprintf(stderr, "  cert=%d seeded=%d left=%d\n", h->cert_hist[it], h->seed_hist[it], h->left_hist[it]);
        }
      }
    }
  }
  if (h->cert_mismatch) { c->err = "internal: eigen certificate contradicted by the exact computation"; return LIOGPU_E_INVALID; }
  return LIOGPU_OK;
}

static int scan2map_legacy_dev(Ctx* c, const float4* scan4, int n, float pose_io[6], float matP_io[36], int* degenerate_io,
                               int max_iter, liogpu_s2m_info* info);

int scan2map_dev(Ctx* c, const float4* scan4, int n, float pose_io[6], float matP_io[36], int* degenerate_io,
                 int max_iter, liogpu_s2m_info* info) {
  int rc = check_grid(c);
  if (rc != LIOGPU_OK) return rc;
  if (max_iter < 1 || max_iter > LIOGPU_MAX_ITER) { c->err = "max_iter out of range"; return LIOGPU_E_INVALID; }
  // the fused loop keeps its chunk-offset table in shared memory: sweeps beyond 1,048,576 points (none of the
  // reference's sensors) take the two-kernel path
  if (c->prm.s2m_path == 2 && div_up(n, FZ_THREADS) <= FZ_MAXCHUNKS && fused_grid(c) > 1)
    return scan2map_fused_dev(c, scan4, n, pose_io, matP_io, degenerate_io, max_iter, info, nullptr);
  return scan2map_legacy_dev(c, scan4, n, pose_io, matP_io, degenerate_io, max_iter, info);
}

// One registration with the per-point results of its LAST executed iteration (parity tests of the fused loop).
int scan2map_trace_dev(Ctx* c, const float4* scan4, int n, float pose_io[6], float matP_io[36], int* degenerate_io,
                       int max_iter, liogpu_s2m_info* info, int* nn_idx, float* nn_d2, float* coeff, unsigned char* flag,
                       unsigned char* tie) {
  int rc = check_grid(c);
  if (rc != LIOGPU_OK) return rc;
  if (max_iter < 1 || max_iter > LIOGPU_MAX_ITER) { c->err = "max_iter out of range"; return LIOGPU_E_INVALID; }
  if (div_up(n, FZ_THREADS) > FZ_MAXCHUNKS || fused_grid(c) <= 1) { c->err = "fused loop unavailable for this size / device"; return LIOGPU_E_INVALID; }
  LIOGPU_CUDA_OK(c, c->dbg_idx.reserve((size_t)n * 5 * sizeof(int)));
  LIOGPU_CUDA_OK(c, c->dbg_d2.reserve((size_t)n * 5 * sizeof(float)));
  LIOGPU_CUDA_OK(c, c->dbg_coeff.reserve((size_t)n * sizeof(float4)));
  LIOGPU_CUDA_OK(c, c->dbg_flag.reserve((size_t)n));
  LIOGPU_CUDA_OK(c, c->dbg_tie.reserve((size_t)n));
  const SurfDebugOut dbg{c->dbg_idx.as<int>(), c->dbg_d2.as<float>(), c->dbg_coeff.as<float4>(),
                         c->dbg_flag.as<unsigned char>(), c->dbg_tie.as<unsigned char>()};
  rc = scan2map_fused_dev(c, scan4, n, pose_io, matP_io, degenerate_io, max_iter, info, &dbg);
  if (rc != LIOGPU_OK) return rc;
  if (nn_idx) LIOGPU_CUDA_OK(c, cudaMemcpyAsync(nn_idx, dbg.nn_idx, (size_t)n * 5 * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  if (nn_d2) LIOGPU_CUDA_OK(c, cudaMemcpyAsync(nn_d2, dbg.nn_d2, (size_t)n * 5 * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  if (coeff) LIOGPU_CUDA_OK(c, cudaMemcpyAsync(coeff, dbg.coeff, (size_t)n * sizeof(float4), cudaMemcpyDeviceToHost, c->stream));
  if (flag) LIOGPU_CUDA_OK(c, cudaMemcpyAsync(flag, dbg.flag, (size_t)n, cudaMemcpyDeviceToHost, c->stream));
  if (tie) LIOGPU_CUDA_OK(c, cudaMemcpyAsync(tie, dbg.tie, (size_t)n, cudaMemcpyDeviceToHost, c->stream));
  LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  return LIOGPU_OK;
}

static int scan2map_legacy_dev(Ctx* c, const float4* scan4, int n, float pose_io[6], float matP_io[36], int* degenerate_io,
                               int max_iter, liogpu_s2m_info* info) {
  int rc = LIOGPU_OK;
  S2mArgs A;
  int main_blocks = 0, left_blocks = 0;
  rc = prepare_args(c, scan4, n, A, main_blocks, left_blocks);
  if (rc != LIOGPU_OK) return rc;
  LmDevState* h = reinterpret_cast<LmDevState*>((char*)c->h_pinned + 4096);
  LmInit init;
  for (int k = 0; k < 6; ++k) init.pose[k] = pose_io[k];
  for (int k = 0; k < 36; ++k) init.matP[k] = matP_io[k];
  init.degenerate = *degenerate_io;
  init.max_iter = max_iter;
  LmDevState* d = A.st;
  const unsigned long long launches_before = c->launches;
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
  lm_prepare_kernel<<<1, 256, 0, c->stream>>>(d, init);
  c->launches++;
  // The loop never waits for the host inside a chunk: S2M_CHUNK iterations are enqueued back to back
  // (a launch that finds `done` set exits at once), then the state block is read back — the same single
  // read-back a converged registration needs anyway.  Only scans that need more than S2M_CHUNK iterations
  // pay a second round trip.
  // (Sizing the first chunk from the previous registration's iteration count — 2.8 on the 64-beam sequences, where a
  // chunk of 5 spends two launch pairs of ~5 us per scan on nothing — was tried: a misprediction costs a second host
  // round trip, and the batch-mapping throughput moved by +0.5 % (6,362 vs 6,331 scans/s, 8 workers on one GPU).)
  const int S2M_CHUNK = 5;
  int launched = 0;
  float prof_main_ms = 0.f, prof_left_ms = 0.f;
  int prof_main_n = 0, prof_left_n = 0;
  for (;;) {
    const int todo = (max_iter - launched) < S2M_CHUNK ? (max_iter - launched) : S2M_CHUNK;
    // on a sparse map (no phase-1 gate) iteration 0 has nothing for the main kernel to do, but from
    // iteration 1 on the seeded search runs there
    const bool two_phase = A.g.gate1_d2 < A.g.gate_d2;
    const bool prof = c->prm.profile_kernels != 0 && launched == 0;
    if (prof && c->prof_ev.empty()) {
      c->prof_ev.resize(3 * S2M_CHUNK);
      for (cudaEvent_t& e : c->prof_ev) LIOGPU_CUDA_OK(c, cudaEventCreate(&e));
    }
    for (int it = 0; it < todo; ++it) {
      const bool first = launched + it == 0;
      if (prof) LIOGPU_CUDA_OK(c, cudaEventRecord(c->prof_ev[3 * it], c->stream));
      if (two_phase || !first) LIOGPU_CUDA_OK(c, launch_pdl(s2m_main_kernel, main_blocks, S2M_THREADS, c->stream, A));
      if (prof) LIOGPU_CUDA_OK(c, cudaEventRecord(c->prof_ev[3 * it + 1], c->stream));
      LIOGPU_CUDA_OK(c, launch_pdl(s2m_left_kernel, left_blocks, LEFT_THREADS, c->stream, A));
      if (prof) LIOGPU_CUDA_OK(c, cudaEventRecord(c->prof_ev[3 * it + 2], c->stream));
      c->launches += (two_phase || !first) ? 2 : 1;
      if (first) {  // iteration 0's eigen analysis / matP off the critical path
        LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev_it0, c->stream));
        LIOGPU_CUDA_OK(c, cudaStreamWaitEvent(c->side_stream, c->ev_it0, 0));
        lm_matp_kernel<<<1, 32, 0, c->side_stream>>>(d);
        c->launches++;
        LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev_side, c->side_stream));
      }
    }
    launched += todo;
    LIOGPU_CUDA_OK(c, cudaGetLastError());
    LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
    LIOGPU_CUDA_OK(c, cudaStreamWaitEvent(c->stream, c->ev_side, 0));
    LIOGPU_CUDA_OK(c, cudaMemcpyAsync(h, d, sizeof(LmDevState), cudaMemcpyDeviceToHost, c->stream));
    LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
    LIOGPU_CUDA_OK(c, cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1));
    if (prof) {
      for (int it = 0; it < todo && it < h->iter; ++it) {
        float a = 0.f, b = 0.f;
        cudaEventElapsedTime(&a, c->prof_ev[3 * it], c->prof_ev[3 * it + 1]);
        cudaEventElapsedTime(&b, c->prof_ev[3 * it + 1], c->prof_ev[3 * it + 2]);
        if (two_phase || it > 0) { prof_main_ms += a; ++prof_main_n; }
        prof_left_ms += b; ++prof_left_n;
        if (info && launched - todo + it < LIOGPU_MAX_ITER) {
          info->main_us_hist[launched - todo + it] = a * 1e3f;
          info->rest_us_hist[launched - todo + it] = b * 1e3f;
        }
      }
    }
    if (h->done || launched >= max_iter) break;
  }
  for (int k = 0; k < 6; ++k) pose_io[k] = h->pose[k];
  for (int k = 0; k < 36; ++k) matP_io[k] = h->matP[k];
  *degenerate_io = h->degenerate;
  if (info) {
    fill_info(c, h, n, info);
    info->kernel_launches = (int)(c->launches - launches_before);
    info->main_kernel_ms = prof_main_ms; info->left_kernel_ms = prof_left_ms;
    info->main_kernel_launches = prof_main_n; info->left_kernel_launches = prof_left_n;
    for (int it = 0; it < LIOGPU_MAX_ITER; ++it) info->leftover_hist[it] = h->left_hist[it];
  }
  if (h->cert_mismatch) { c->err = "internal: eigen certificate contradicted by the exact computation"; return LIOGPU_E_INVALID; }
  return LIOGPU_OK;
}

int surf_optimization_dev(Ctx* c, const float4* scan4, int n, const float* pose6, const float* T12, int* nn_idx,
                          float* nn_d2, float* coeff, unsigned char* flag, unsigned char* tie) {
  int rc = check_grid(c);
  if (rc != LIOGPU_OK) return rc;
  if ((pose6 == nullptr) == (T12 == nullptr)) { c->err = "exactly one of pose6 / T12 must be given"; return LIOGPU_E_INVALID; }
  if (n <= 0) return LIOGPU_OK;
  S2mArgs A;
  int main_blocks = 0, left_blocks = 0;
  rc = prepare_args(c, scan4, n, A, main_blocks, left_blocks);
  if (rc != LIOGPU_OK) return rc;
  LIOGPU_CUDA_OK(c, c->misc.reserve(256));
  LIOGPU_CUDA_OK(c, c->dbg_idx.reserve((size_t)n * 5 * sizeof(int)));
  LIOGPU_CUDA_OK(c, c->dbg_d2.reserve((size_t)n * 5 * sizeof(float)));
  LIOGPU_CUDA_OK(c, c->dbg_coeff.reserve((size_t)n * sizeof(float4)));
  LIOGPU_CUDA_OK(c, c->dbg_flag.reserve((size_t)n));
  LIOGPU_CUDA_OK(c, c->dbg_tie.reserve((size_t)n));
  LmInit init;
  memset(&init, 0, sizeof(init));
  if (pose6) for (int k = 0; k < 6; ++k) init.pose[k] = pose6[k];
  LmDevState* d = A.st;
  lm_prepare_kernel<<<1, 256, 0, c->stream>>>(d, init);
  c->launches++;
  if (T12) {
    float* d_T = c->misc.as<float>() + 16;
    float* hT = reinterpret_cast<float*>((char*)c->h_pinned + 3072);
    for (int k = 0; k < 12; ++k) hT[k] = T12[k];
    LIOGPU_CUDA_OK(c, cudaMemcpyAsync(d_T, hT, 12 * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    A.T_override = d_T;
  }
  A.dbg = SurfDebugOut{c->dbg_idx.as<int>(), c->dbg_d2.as<float>(), c->dbg_coeff.as<float4>(),
                       c->dbg_flag.as<unsigned char>(), c->dbg_tie.as<unsigned char>()};
  A.mode = 1;
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
  if (A.g.gate1_d2 < A.g.gate_d2) s2m_main_kernel<<<main_blocks, S2M_THREADS, 0, c->stream>>>(A);
  s2m_left_kernel<<<left_blocks, LEFT_THREADS, 0, c->stream>>>(A);
  c->launches += 2;
  LIOGPU_CUDA_OK(c, cudaGetLastError());
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
  const SurfDebugOut& dbg = A.dbg;
  if (nn_idx) LIOGPU_CUDA_OK(c, cudaMemcpyAsync(nn_idx, dbg.nn_idx, (size_t)n * 5 * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  if (nn_d2) LIOGPU_CUDA_OK(c, cudaMemcpyAsync(nn_d2, dbg.nn_d2, (size_t)n * 5 * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  if (coeff) LIOGPU_CUDA_OK(c, cudaMemcpyAsync(coeff, dbg.coeff, (size_t)n * sizeof(float4), cudaMemcpyDeviceToHost, c->stream));
  if (flag) LIOGPU_CUDA_OK(c, cudaMemcpyAsync(flag, dbg.flag, (size_t)n, cudaMemcpyDeviceToHost, c->stream));
  if (tie) LIOGPU_CUDA_OK(c, cudaMemcpyAsync(tie, dbg.tie, (size_t)n, cudaMemcpyDeviceToHost, c->stream));
  LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  LIOGPU_CUDA_OK(c, cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1));
  return LIOGPU_OK;
}

}  // namespace liogpu
static_assert(sizeof(liogpu::LmDevState) == 2520, "bench.py counts sizeof(LmDevState) bytes of H2D/D2H per registration");
