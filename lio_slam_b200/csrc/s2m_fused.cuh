// s2m_fused.cuh — the whole loop of scan2MapOptimization (mapOptmization.cpp:1848-1859) as ONE persistent
// cooperative launch per registration.  Included by s2m.cu (same translation unit: it reuses the search and plane-fit
// routines defined there and the 6x6 tail of lm_tail.cuh).
//
// Grid: every CTA slot of the GPU (occupancy x SM count), co-resident by cooperative launch.  CTA `gridDim.x - 1`
// is a service CTA (iteration 0's eigen-decomposition / matP, off the critical path); the others loop:
//
//   per Gauss-Newton iteration
//     main phase   chunks of 256 sweep points pulled from an atomic queue (no wave tail: a CTA that finishes
//                  early takes the next chunk).  Inside a chunk every WARP works on its 32 points on its own (no
//                  block-wide step until the final reduction, so warps of a CTA overlap freely):
//                    1 classify  lane = point.  From iteration 1 on every point carries a CANDIDATE SET: the (up
//                                to) 8 nearest map points found by its last search and a lower bound `lb` on the
//                                distance from the point to every map point outside the set.  The set members'
//                                distances to the moved point are evaluated exactly; if the 5th smallest is
//                                below lb - |move| (triangle inequality, rounding margins included) the five
//                                nearest neighbours of the moved point are certainly inside the set: they are
//                                selected and ordered by (d2, map index) with no grid walk at all — an exact
//                                certificate, not a heuristic.  Otherwise the point needs a search.
//                    2 search    iteration 0 (no sets yet, and the first step is too large for a set to survive):
//                                the 5-nearest walk of the sorted grid inside the phase-1 gate, lane = point.
//                                Later iterations: the 9-nearest walk inside the seeded bound (exact 5-NN + the next
//                                candidate set + its bound), lane = point when many lanes need it; when only a
//                                few do (the usual case once the certificate bites) the warp serves them one by
//                                one COOPERATIVELY (lanes share rows and candidates: ~2 us instead of a ~13 us
//                                single-lane chain).
//                    3 leftovers points phase 1 cannot settle: up to 4 per warp are finished on the spot by the
//                                warp-cooperative full-gate search, more are deferred to the grid-wide phase.
//                    4 fit       lane = point: 5x3 plane fit, weight, Jacobian row; FP64 reduction of the 27 sums
//                                of A^T A / A^T b over the warp's rows, then over the chunk's warps.
//     ticket A     the last CTA to finish the main phase looks at the number of deferred leftovers:
//                    none (the usual case from iteration 1 on): it adds the chunk rows in a fixed order, runs the
//                          6x6 tail of LMOptimization (lm_finalize_warp) and releases the others — ONE grid-wide
//                          synchronisation per iteration;
//                    some: it opens the leftover phase: warp-cooperative full-gate search, one point per warp over
//                          the whole grid (static map -> fixed summation order), per-CTA partial rows, ticket B, the
//                          last CTA adds chunk rows + CTA rows, runs the tail and releases the others.
//
// Nothing returns to the host inside the loop; the 1.8 KB state block is read back once.
#pragma once

namespace liogpu {

constexpr int FZ_THREADS = 256;
constexpr int FZ_WARPS = FZ_THREADS / 32;
#ifndef FZ_MINBLOCKS_CFG
#define FZ_MINBLOCKS_CFG 3
#endif
constexpr int FZ_K = LIOGPU_FZ_K;        // members of a candidate set
constexpr int FZ_MAXCHUNKS = 4096;       // chunk-offset table of the leftover phase lives in shared memory
constexpr float FZ_REL = 1e-5f;          // relative safety margin of every bound (f32 rounding is < 3e-7)
constexpr float FZ_SEED_MARGIN = 0.10f;  // a seeded search enumerates this far (m) beyond the seeds' 5th distance
constexpr int FZ_WCOOP_MAX = 4;          // a warp with at most this many search requests serves them cooperatively, one by one
constexpr int FZ_INPLACE = 4;            // a warp with at most this many leftovers finishes them on the spot
constexpr int FZ_PROBES = 8;             // %globaltimer stamps per iteration (profile_kernels)

// ---- 9 best (d2, map index) pairs, same 64-bit keys as Top5; slot FZ_K is the pruning threshold ----
struct TopN {
  u64 k[FZ_K + 1];
  __device__ __forceinline__ void init(float gate) {
#pragma unroll
    for (int j = 0; j <= FZ_K; ++j) k[j] = ((u64)__float_as_uint(gate)) << 32;
  }
  __device__ __forceinline__ void offer(float d, int id) {
    const u64 key = (((u64)__float_as_uint(d)) << 32) | (u64)(unsigned)id;
    if (key < k[FZ_K]) {
      k[FZ_K] = key;
#pragma unroll
      for (int j = FZ_K; j > 0; --j) {
        const u64 lo = min(k[j - 1], k[j]), hi = max(k[j - 1], k[j]);
        k[j - 1] = lo; k[j] = hi;
      }
    }
  }
  __device__ __forceinline__ float d(int j) const { return __uint_as_float((unsigned)(k[j] >> 32)); }
  __device__ __forceinline__ int i(int j) const { return (int)(unsigned)(k[j] & 0xffffffffull); }
  __device__ __forceinline__ float worst() const { return d(FZ_K); }
};

// grid_knn5 with the wider list: on return every map point that is NOT in k[0..FZ_K-1] has d2 >= worst(), and
// k[0..4] are the exact 5 nearest among the points closer than sqrt(gate_d2) (ascending (d2, index)).
__device__ __forceinline__ void grid_knn_topn(const float4 q, const GridParams& g, const float gate_d2,
                                              const float4* __restrict__ map_sorted,
                                              const uint32_t* __restrict__ cell_start, TopN& t) {
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
  for (int kz = 0, seen_z = 0; seen_z < nzs; ++kz) {
    const int z = cz + zigzag(kz);
    if (z < zmin || z > zmax) continue;
    ++seen_z;
    const float zlo = g.oz + (float)z * g.h;
    const float gz = fmaxf(fmaxf(zlo - q.z, q.z - (zlo + g.h)) - s2, 0.f);
    const float gz2 = gz * gz;
    if (gz2 > t.worst()) continue;
    for (int ky = 0, seen_y = 0; seen_y < nys; ++ky) {
      const int y = cy + zigzag(ky);
      if (y < ymin || y > ymax) continue;
      ++seen_y;
      const float ylo = g.oy + (float)y * g.h;
      const float gy = fmaxf(fmaxf(ylo - q.y, q.y - (ylo + g.h)) - s2, 0.f);
      const float m2 = (gz2 + gy * gy) * 0.999999f;
      const float worst = t.worst();
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

#define FZ_CE(a, b) { const u64 lo_ = min(a, b), hi_ = max(a, b); a = lo_; b = hi_; }
// 19-comparator sorting network for 8 keys (Batcher odd-even merge sort), ascending
__device__ __forceinline__ void sort8(u64 k[8]) {
  FZ_CE(k[0], k[1]); FZ_CE(k[2], k[3]); FZ_CE(k[4], k[5]); FZ_CE(k[6], k[7]);
  FZ_CE(k[0], k[2]); FZ_CE(k[1], k[3]); FZ_CE(k[4], k[6]); FZ_CE(k[5], k[7]);
  FZ_CE(k[1], k[2]); FZ_CE(k[5], k[6]);
  FZ_CE(k[0], k[4]); FZ_CE(k[1], k[5]); FZ_CE(k[2], k[6]); FZ_CE(k[3], k[7]);
  FZ_CE(k[2], k[4]); FZ_CE(k[3], k[5]);
  FZ_CE(k[1], k[2]); FZ_CE(k[3], k[4]); FZ_CE(k[5], k[6]);
}

struct FusedArgs {
  const float4* scan;
  int nq;
  const float4* map4;
  const float4* map_sorted;
  const uint32_t* cell_start;
  GridParams g;
  LmDevState* st;
  double* chunk_rows;      // [nchunks][S2M_SUMS]  partial sums of a chunk (deterministic: a chunk is a fixed set of points)
  double* cta_rows;        // [compute CTAs][S2M_SUMS]
  int* left_list;          // [nchunks][FZ_THREADS] leftover point indices, per chunk segment
  int* chunk_nleft;        // [nchunks]
  int* prev_nn;            // [FZ_K][nq] candidate set of every point (-1: empty slot; prev_nn[0][i] < 0: no set)
  float* prev_lb;          // [nq] lower bound on the distance to every map point outside the set
  float4* hopeless;        // [nq] see HOPELESS_MARGIN
  unsigned long long* probe;  // [LIOGPU_MAX_ITER][FZ_PROBES] %globaltimer stamps (profile_kernels), or null
  SurfDebugOut dbg;        // per-point outputs of the last executed iteration (trace entry point), or nulls
  int nchunks;
  int use_cert;            // 0: never take the certificate (A/B switch: every point with a set is searched)
};

__device__ __forceinline__ unsigned long long fz_globaltimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ unsigned fz_ld_acquire(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}


// transPointAssociateToMap + LM trig of `pose` into caller storage (same arithmetic as warp_refresh_transform)
__device__ __forceinline__ void fz_warp_transform(const int lane, const float pose_l, float* T, float* trig) {
  float sn = 0.f, cs = 0.f;
  if (lane < 3) {
    const double a = (double)pose_l;
    sn = (float)sin(a);
    cs = (float)cos(a);
  }
  const float F = __shfl_sync(FULL, sn, 0), E = __shfl_sync(FULL, cs, 0);
  const float D = __shfl_sync(FULL, sn, 1), C = __shfl_sync(FULL, cs, 1);
  const float B = __shfl_sync(FULL, sn, 2), A = __shfl_sync(FULL, cs, 2);
  const float px = __shfl_sync(FULL, pose_l, 3), py = __shfl_sync(FULL, pose_l, 4), pz = __shfl_sync(FULL, pose_l, 5);
  if (lane == 0) {
    const float DE = D * E, DF = D * F;
    T[0] = A * C;  T[1] = A * DF - B * E;  T[2] = B * F + A * DE;  T[3] = px;
    T[4] = B * C;  T[5] = A * E + B * DF;  T[6] = B * DE - A * F;  T[7] = py;
    T[8] = -D;     T[9] = C * F;           T[10] = C * E;          T[11] = pz;
    trig[0] = B; trig[1] = A; trig[2] = D; trig[3] = C; trig[4] = F; trig[5] = E;
  }
}

// iteration 0's matP when the certificate let the loop go ahead (body of lm_matp_kernel), one warp
__device__ __forceinline__ void fz_matp_warp(LmDevState* st, FinSmem& m, const int lane) {
  for (int e = lane; e < 36; e += 32) m.AtA[e] = __ldcg(st->AtA0 + e);
  __syncwarp();
  const int deg = lm_eigen_matp(m, lane, st->matP);
  if (lane == 0) {
    if (deg) st->cert_mismatch = 1;
    st->eig_pending = 0;
  }
}

// Warp-cooperative exact search of ONE query inside gate_d2 (all lanes pass the same q): the five nearest in
// ascending (d2, index), up to FZ_K - 5 further candidates, lb2 = a lower bound on d2 of every map point that is not
// returned, d6 = the best d2 among the points outside the five (tie logging).  Same row / candidate hand-out as
// warp_knn5; every lane returns the same values.  Empty slots of `out` hold ~0.
__device__ __forceinline__ void warp_knn_set(const float4 q, const GridParams& g, const float gate_d2,
                                             const float4* __restrict__ map_sorted, const uint32_t* __restrict__ cell_start,
                                             const int lane, u64 out[FZ_K], float& lb2, float& d6) {
  Top5 t;
  t.init(gate_d2);
  const float s2 = 2.0f * g.slack;
  const float reach = sqrtf(gate_d2) * 1.000001f + s2;
  int zmin = (int)floorf((q.z - reach - g.oz) * g.inv_h), zmax = (int)floorf((q.z + reach - g.oz) * g.inv_h);
  int ymin = (int)floorf((q.y - reach - g.oy) * g.inv_h), ymax = (int)floorf((q.y + reach - g.oy) * g.inv_h);
  zmin = max(zmin, 0); zmax = min(zmax, g.nz - 1);
  ymin = max(ymin, 0); ymax = min(ymax, g.ny - 1);
  const int nys = ymax - ymin + 1;
  const int nrows = (zmin > zmax || ymin > ymax) ? 0 : (zmax - zmin + 1) * nys;
  for (int base = 0; base < nrows; base += 32) {
    const int r = base + lane;
    uint32_t s = 0, cnt = 0;
    if (r < nrows) {
      const int z = zmin + r / nys, y = ymin + r % nys;
      const float zlo = g.oz + (float)z * g.h, ylo = g.oy + (float)y * g.h;
      const float gz = fmaxf(fmaxf(zlo - q.z, q.z - (zlo + g.h)) - s2, 0.f);
      const float gy = fmaxf(fmaxf(ylo - q.y, q.y - (ylo + g.h)) - s2, 0.f);
      const float m2 = (gz * gz + gy * gy) * 0.999999f;
      if (m2 <= gate_d2) {
        const float rr = sqrtf(gate_d2 - m2) * 1.000001f + s2;
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
    uint32_t incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t v = __shfl_up_sync(FULL, incl, o);
      if (lane >= o) incl += v;
    }
    const uint32_t total = __shfl_sync(FULL, incl, 31);
    for (uint32_t c0 = 0; c0 < total; c0 += 32) {
      const uint32_t c = c0 + lane;
      int lo = 0;
#pragma unroll
      for (int step = 16; step > 0; step >>= 1) {
        const uint32_t v = __shfl_sync(FULL, incl, lo + step - 1);
        if (v <= c) lo += step;
      }
      lo = min(lo, 31);
      const uint32_t row_s = __shfl_sync(FULL, s, lo);
      const uint32_t row_incl = __shfl_sync(FULL, incl, lo);
      const uint32_t row_cnt = __shfl_sync(FULL, cnt, lo);
      if (c < total) {
        const float4 p = __ldg(map_sorted + (row_s + (c - (row_incl - row_cnt))));
        t.offer(l2_simple(q, p), __float_as_int(p.w));
      }
    }
  }
  // FZ_K + 1 smallest heads over the lanes, popped from their owners' lists
  const unsigned gbits = __float_as_uint(gate_d2);
  u64 res[FZ_K + 1];
#pragma unroll
  for (int k = 0; k <= FZ_K; ++k) {
    const u64 m = warp_min_u64(t.k0);
    res[k] = m;
    const unsigned owners = __ballot_sync(FULL, t.k0 == m);
    if (lane == __ffs(owners) - 1) { t.k0 = t.k1; t.k1 = t.k2; t.k2 = t.k3; t.k3 = t.k4; t.k4 = ~0ull; }
  }
  float rj = t.rej;  // best candidate a lane saw but dropped (its own 6th or worse, or beyond the gate)
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) rj = fminf(rj, __shfl_xor_sync(FULL, rj, o));
#pragma unroll
  for (int k = 0; k < FZ_K; ++k) out[k] = ((unsigned)(res[k] >> 32) < gbits) ? res[k] : ~0ull;
  const float d9 = ((unsigned)(res[FZ_K] >> 32) < gbits) ? __uint_as_float((unsigned)(res[FZ_K] >> 32)) : gate_d2;
  lb2 = fminf(fminf(gate_d2, rj), d9);
  const float dn = ((unsigned)(res[5] >> 32) < gbits) ? __uint_as_float((unsigned)(res[5] >> 32)) : FLT_MAX;
  d6 = fminf(dn, rj);
}

// shared-memory carve-up: the main phase and the leftover phase never overlap in time
struct FzMainSmem {
  float rows[FZ_THREADS][8];               // Jacobian row, rhs, accepted flag
  unsigned char llist[FZ_WARPS][32];       // per warp: slots deferred to the grid-wide leftover phase
  int nl[FZ_WARPS];
};
struct FzLeftSmem {
  int off[FZ_MAXCHUNKS + 1];
  float rows[FZ_THREADS][8];
};
union FzSmem {
  FzMainSmem m;
  FzLeftSmem l;
};

// what a leftover search leaves behind for the next iteration: the candidate set (its five neighbours), the bound
// (everything else it visited was >= rej away, everything it did not visit is beyond the enumerated radius) and, for
// a point with fewer than five map points inside the gate, the generalised hopeless marker: its 5th-nearest map
// point is sqrt(d5) > 1 m away (or beyond the extended gate), so as long as the point has moved less than
// sqrt(d5) - 1 m (minus 1 mm for rounding) since then it still cannot have five neighbours within the gate and
// surfOptimization drops it (:1641) — no search needed.  Exact (triangle inequality), not heuristic.
__device__ __forceinline__ void fz_store_leftover(const FusedArgs& A, const int mine, const float4 sel, const Top5& t,
                                                  const float r2, const bool found) {
  A.prev_nn[mine] = found ? t.i(t.k0) : -1;
  A.prev_nn[(size_t)A.nq + mine] = t.i(t.k1);
  A.prev_nn[2 * (size_t)A.nq + mine] = t.i(t.k2);
  A.prev_nn[3 * (size_t)A.nq + mine] = t.i(t.k3);
  A.prev_nn[4 * (size_t)A.nq + mine] = t.i(t.k4);
#pragma unroll
  for (int j = 5; j < FZ_K; ++j) A.prev_nn[(size_t)j * A.nq + mine] = -1;
  A.prev_lb[mine] = sqrtf(fminf(t.rej, r2)) * (1.f - FZ_REL);
  // d(k4) = the 5th-nearest distance^2 if five points lie inside the enumerated ball, else the ball's radius^2
  const float margin = found ? 0.f : sqrtf(t.d(t.k4)) * (1.f - FZ_REL) - sqrtf(A.g.gate_d2) - 1e-3f;
  A.hopeless[mine] = make_float4(sel.x, sel.y, sel.z, margin > 0.f ? margin : 0.f);
}

// sum of `nrows` partial rows (S2M_SUMS doubles each) in a fixed order: warp w takes rows w, w+8, ... with sixteen
// independent accumulators (sixteen 256-byte loads in flight per warp: the pass is L2-latency bound), added pairwise,
// then the warps are added in order.
// Result: lane l of warp 0 returns sum[l]; every thread must call it.
__device__ __forceinline__ double fz_reduce_rows(const double* __restrict__ rows, const int nrows, double (*red)[S2M_SUMS],
                                                 const int warp, const int lane) {
  constexpr int W = FZ_WARPS, U = 16;
  double a[U];
#pragma unroll
  for (int k = 0; k < U; ++k) a[k] = 0.0;
  int b = warp;
  for (; b + (U - 1) * W < nrows; b += U * W) {
    double v[U];
#pragma unroll
    for (int k = 0; k < U; ++k) v[k] = __ldcg(rows + (size_t)(b + k * W) * S2M_SUMS + lane);
#pragma unroll
    for (int k = 0; k < U; ++k) a[k] += v[k];
  }
  {
    double v[U];
#pragma unroll
    for (int k = 0; k < U; ++k) v[k] = (b + k * W < nrows) ? __ldcg(rows + (size_t)(b + k * W) * S2M_SUMS + lane) : 0.0;
#pragma unroll
    for (int k = 0; k < U; ++k) a[k] += v[k];
  }
#pragma unroll
  for (int o = U / 2; o > 0; o >>= 1) {
#pragma unroll
    for (int k = 0; k < o; ++k) a[k] += a[k + o];
  }
  __syncthreads();
  red[warp][lane] = a[0];
  __syncthreads();
  double sum = 0.0;
  if (warp == 0) {
#pragma unroll
    for (int k = 0; k < FZ_WARPS; ++k) sum += red[k][lane];
  }
  return sum;
}

__global__ void __launch_bounds__(FZ_THREADS, FZ_MINBLOCKS_CFG)
s2m_fused_kernel(const FusedArgs A) {
  __shared__ float sT[12], sTp[12];
  __shared__ LmTrig sTrig;
  __shared__ __align__(16) FzSmem sm;
  __shared__ double red[FZ_WARPS][S2M_SUMS];
  __shared__ double s_sum[S2M_SUMS];
  __shared__ FinSmem s_fin;
  __shared__ int s_chunk, s_wcnt[FZ_WARPS], s_misc[4];
  __shared__ bool s_last;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  LmDevState* const st = A.st;
  const int G = (int)gridDim.x - 1;  // compute CTAs

  if ((int)blockIdx.x == G) {
    // ---- service CTA: iteration 0's eigen-decomposition + matP while iterations 1.. run ----
    if (tid < 32) {
      if (lane == 0) { while (fz_ld_acquire(&st->fz_phase) < 2u) { } __threadfence(); }
      __syncwarp();
      if (__ldcg(&st->eig_pending)) fz_matp_warp(st, s_fin, lane);
    }
    return;
  }

  const bool can_phase1 = A.g.gate1_d2 < A.g.gate_d2;  // dense map: cheap first phase inside a small gate
  const int max_iter = st->max_iter;
  const RowAcc ra = row_acc_of(lane);
  const float ge = sqrtf(A.g.gate_d2) + HOPELESS_MARGIN;  // extended gate of the leftover search
  const float ge2 = ge * ge;
  const unsigned lt_mask = (1u << lane) - 1u;

  for (int it = 0; it < max_iter; ++it) {
    unsigned long long* const probe = A.probe ? A.probe + it * FZ_PROBES : nullptr;
    // ---- this iteration's transform (updatePointAssociateToMap, :1613-1616) ----
    if (it == 0) {
      if (tid < 32) {
        const float pose_l = lane < 6 ? st->pose[lane] : 0.f;
        fz_warp_transform(lane, pose_l, sT, &sTrig.srx);
      }
    } else {
      if (tid < 12) { sT[tid] = __ldcg(st->T + tid); sTp[tid] = __ldcg(st->T_prev + tid); }
      if (tid == 32) {
        sTrig.srx = __ldcg(st->trig + 0); sTrig.crx = __ldcg(st->trig + 1); sTrig.sry = __ldcg(st->trig + 2);
        sTrig.cry = __ldcg(st->trig + 3); sTrig.srz = __ldcg(st->trig + 4); sTrig.crz = __ldcg(st->trig + 5);
      }
    }
    __syncthreads();
    if (probe && blockIdx.x == 0 && tid == 0) probe[0] = fz_globaltimer();
    int cta_deferred = 0;  // meaningful in thread 0

    // =========================== main phase: dynamic queue of 256-point chunks ===========================
    for (;;) {
      if (tid == 0) s_chunk = (int)atomicAdd(&st->fz_queue[it], 1u);
      __syncthreads();
      const int c = s_chunk;
      if (c >= A.nchunks) break;
      const int base = c * FZ_THREADS;
      const int i = base + tid;
      const bool in = i < A.nq;
      // ---- step 1: classify (lane = point) ----
      float4 ori = make_float4(0.f, 0.f, 0.f, 0.f), sel = ori;
      float req = -2.f;  // > 0 seeded bound, 0 phase-1 gate, -1 straight to the leftovers, -2 nothing to search
      int n0 = -1, n1 = -1, n2 = -1, n3 = -1, n4 = -1;  // the five neighbours, ascending (d2, index)
      bool found = false, tie = false, seeded = false, cert = false;
      if (in) {
        ori = A.scan[i];
        sel = apply_T(sT, ori);
        req = can_phase1 ? 0.f : -1.f;
        if (it > 0) {
          const int p0 = __ldcg(A.prev_nn + i);
          if (p0 < 0) {
            const float4 hr = __ldcg(A.hopeless + i);
            if (hr.w > 0.f) {
              const float dx = sel.x - hr.x, dy = sel.y - hr.y, dz = sel.z - hr.z;
              if ((dx * dx + dy * dy + dz * dz) * (1.f + FZ_REL) < hr.w * hr.w) req = -2.f;  // still cannot have 5 neighbours within the gate
            }
          } else {
            u64 key[8];
            int id[8];
            id[0] = p0;
#pragma unroll
            for (int j = 1; j < FZ_K; ++j) id[j] = __ldcg(A.prev_nn + (size_t)j * A.nq + i);
#pragma unroll
            for (int j = 0; j < FZ_K; ++j) {
              key[j] = ~0ull;
              if (id[j] >= 0) {
                const float d = l2_simple(sel, __ldg(A.map4 + id[j]));
                key[j] = (((u64)__float_as_uint(d)) << 32) | (u64)(unsigned)id[j];
              }
            }
            sort8(key);
            const float D5 = __uint_as_float((unsigned)(key[4] >> 32));
            const float bound = __uint_as_float(__float_as_uint(D5) + 1u);  // next float above: the seeds stay inside
            if (bound <= A.g.gate_d2) {
              seeded = true;
              req = bound;
              // certificate: every map point outside the set was >= lb away from where this point stood when the
              // set was built (or last certified); it has moved by |sel - prev|
              const float4 pv = apply_T(sTp, ori);
              const float move = sqrtf(l2_simple(sel, pv));
              const float L = __ldcg(A.prev_lb + i) - move * (1.f + FZ_REL) - 1e-7f;
              if (A.use_cert && L > 0.f && L * L * (1.f - FZ_REL) > D5) {
                cert = true;
                req = -2.f;
                found = true;
                n0 = (int)(unsigned)key[0]; n1 = (int)(unsigned)key[1]; n2 = (int)(unsigned)key[2];
                n3 = (int)(unsigned)key[3]; n4 = (int)(unsigned)key[4];
                const float d0 = __uint_as_float((unsigned)(key[0] >> 32)), d1 = __uint_as_float((unsigned)(key[1] >> 32));
                const float d2 = __uint_as_float((unsigned)(key[2] >> 32)), d3 = __uint_as_float((unsigned)(key[3] >> 32));
                const float d5 = __uint_as_float((unsigned)(key[5] >> 32));
                tie = d0 == d1 || d1 == d2 || d2 == d3 || d3 == D5 || (key[5] != ~0ull && D5 == d5);
                A.prev_lb[i] = L * (1.f - FZ_REL);
              }
            }
          }
        }
      }
      // ---- step 2: search ----
      bool need2 = req == -1.f;
      const bool want = req >= 0.f;
      const unsigned wm = __ballot_sync(FULL, want);
      if (wm) {
        if (it == 0) {
          // no candidate sets yet, and none built here would survive the first (large) step: the plain 5-nearest walk
          if (want) {
            Top5 t;
            grid_knn5(sel, A.g, A.g.gate1_d2, A.map_sorted, A.cell_start, t);
            need2 = !(t.d(t.k4) < A.g.gate1_d2);
            if (!need2) {
              found = true; tie = t.tie();
              n0 = t.i(t.k0); n1 = t.i(t.k1); n2 = t.i(t.k2); n3 = t.i(t.k3); n4 = t.i(t.k4);
              A.prev_nn[i] = n0; A.prev_nn[(size_t)A.nq + i] = n1; A.prev_nn[2 * (size_t)A.nq + i] = n2;
              A.prev_nn[3 * (size_t)A.nq + i] = n3; A.prev_nn[4 * (size_t)A.nq + i] = n4;
#pragma unroll
              for (int j = 5; j < FZ_K; ++j) A.prev_nn[(size_t)j * A.nq + i] = -1;
              A.prev_lb[i] = sqrtf(t.d(t.k4)) * (1.f - FZ_REL);  // everything outside the five is at least this far
            }
          }
        } else if (__popc(wm) > FZ_WCOOP_MAX) {
          // many lanes: lane = point, the 9-nearest walk
          if (want) {
            const bool sd = req > 0.f;
            float gate_use = A.g.gate1_d2;
            if (sd) { const float r = sqrtf(req) + FZ_SEED_MARGIN; gate_use = fmaxf(r * r, req); }
            TopN t;
            grid_knn_topn(sel, A.g, gate_use, A.map_sorted, A.cell_start, t);
            need2 = !(t.d(4) < (sd ? req : A.g.gate1_d2));  // a seeded search always finds its five
            if (!need2) {
              found = true;
              tie = t.d(0) == t.d(1) || t.d(1) == t.d(2) || t.d(2) == t.d(3) || t.d(3) == t.d(4) || t.d(4) == t.d(5);
              n0 = t.i(0); n1 = t.i(1); n2 = t.i(2); n3 = t.i(3); n4 = t.i(4);
              const unsigned gbits = __float_as_uint(gate_use);
#pragma unroll
              for (int j = 0; j < FZ_K; ++j) {
                const bool real = !((unsigned)(t.k[j] >> 32) == gbits && (unsigned)t.k[j] == 0u);
                A.prev_nn[(size_t)j * A.nq + i] = real ? t.i(j) : -1;
              }
              A.prev_lb[i] = sqrtf(t.worst()) * (1.f - FZ_REL);
            }
          }
        } else {
          // a few lanes: the warp serves them one by one, cooperatively
          unsigned todo = wm;
          while (todo) {
            const int j = __ffs(todo) - 1;
            todo &= todo - 1;
            float4 q;
            q.x = __shfl_sync(FULL, sel.x, j); q.y = __shfl_sync(FULL, sel.y, j); q.z = __shfl_sync(FULL, sel.z, j); q.w = 0.f;
            const float rq = __shfl_sync(FULL, req, j);
            const bool sd = rq > 0.f;
            float gate_use = A.g.gate1_d2;
            if (sd) { const float r = sqrtf(rq) + FZ_SEED_MARGIN; gate_use = fmaxf(r * r, rq); }
            u64 k[FZ_K];
            float lb2, d6;
            warp_knn_set(q, A.g, gate_use, A.map_sorted, A.cell_start, lane, k, lb2, d6);
            if (lane == j) {
              const float e0 = __uint_as_float((unsigned)(k[0] >> 32)), e1 = __uint_as_float((unsigned)(k[1] >> 32));
              const float e2 = __uint_as_float((unsigned)(k[2] >> 32)), e3 = __uint_as_float((unsigned)(k[3] >> 32));
              const float e4 = __uint_as_float((unsigned)(k[4] >> 32));
              need2 = !(k[4] != ~0ull && e4 < (sd ? rq : A.g.gate1_d2));
              if (!need2) {
                found = true;
                tie = e0 == e1 || e1 == e2 || e2 == e3 || e3 == e4 || e4 == d6;
                n0 = (int)(unsigned)k[0]; n1 = (int)(unsigned)k[1]; n2 = (int)(unsigned)k[2];
                n3 = (int)(unsigned)k[3]; n4 = (int)(unsigned)k[4];
#pragma unroll
                for (int m = 0; m < FZ_K; ++m) A.prev_nn[(size_t)m * A.nq + i] = k[m] != ~0ull ? (int)(unsigned)k[m] : -1;
                A.prev_lb[i] = sqrtf(lb2) * (1.f - FZ_REL);
              }
            }
          }
        }
      }
      // ---- step 3: leftovers (points the phase-1 gate could not settle) ----
      const unsigned lm = __ballot_sync(FULL, need2);
      const int nl = __popc(lm);
      const bool deferred = nl > FZ_INPLACE;
      if (nl > 0) {
        if (!deferred) {
          unsigned todo = lm;
          while (todo) {
            const int j = __ffs(todo) - 1;
            todo &= todo - 1;
            float4 q;
            q.x = __shfl_sync(FULL, sel.x, j); q.y = __shfl_sync(FULL, sel.y, j); q.z = __shfl_sync(FULL, sel.z, j); q.w = 0.f;
            Top5 t;
            float r2;
            leftover_search(q, A.g, ge2, A.map_sorted, A.cell_start, lane, t, r2);
            if (lane == j) {
              found = t.d(t.k4) < A.g.gate_d2;  // :1641
              fz_store_leftover(A, i, sel, t, r2, found);
              if (found) { tie = t.tie(); n0 = t.i(t.k0); n1 = t.i(t.k1); n2 = t.i(t.k2); n3 = t.i(t.k3); n4 = t.i(t.k4); }
            }
          }
        } else if (need2) {
          sm.m.llist[warp][__popc(lm & lt_mask)] = (unsigned char)tid;
        }
      }
      if (lane == 0) sm.m.nl[warp] = deferred ? nl : 0;
      // ---- step 4: plane fit + Jacobian row ----
      float row[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      float rhs = 0.f;
      bool flag = false;
      if (in) {
        float4 coeff = make_float4(0.f, 0.f, 0.f, 0.f);
        float nd2[5] = {A.g.gate_d2, A.g.gate_d2, A.g.gate_d2, A.g.gate_d2, A.g.gate_d2};
        if (found) {
          float4 nbr[5];
          nbr[0] = __ldg(A.map4 + n0); nbr[1] = __ldg(A.map4 + n1); nbr[2] = __ldg(A.map4 + n2);
          nbr[3] = __ldg(A.map4 + n3); nbr[4] = __ldg(A.map4 + n4);
          flag = plane_residual(ori, sel, nbr, coeff);
          if (!flag) coeff = make_float4(0.f, 0.f, 0.f, 0.f);
          if (flag) jacobian_row(sTrig, ori, coeff, row, rhs);
          if (A.dbg.nn_d2) {
#pragma unroll
            for (int j = 0; j < 5; ++j) nd2[j] = l2_simple(sel, nbr[j]);
          }
        } else {
          tie = false;
        }
        if (!(deferred && need2)) {  // deferred points are written by the leftover phase
          if (A.dbg.nn_idx) { int* o = A.dbg.nn_idx + (size_t)i * 5; o[0] = n0; o[1] = n1; o[2] = n2; o[3] = n3; o[4] = n4; }
          if (A.dbg.nn_d2) { float* o = A.dbg.nn_d2 + (size_t)i * 5; for (int j = 0; j < 5; ++j) o[j] = nd2[j]; }
          if (A.dbg.coeff) A.dbg.coeff[i] = coeff;
          if (A.dbg.flag) A.dbg.flag[i] = flag ? 1 : 0;
          if (A.dbg.tie) A.dbg.tie[i] = tie ? 1 : 0;
        }
      }
#pragma unroll
      for (int k = 0; k < 6; ++k) sm.m.rows[tid][k] = row[k];
      sm.m.rows[tid][6] = rhs;
      sm.m.rows[tid][7] = flag ? 1.f : 0.f;
      const int w_ties = __popc(__ballot_sync(FULL, flag && tie));
      const int w_seed = __popc(__ballot_sync(FULL, seeded));
      const int w_cert = __popc(__ballot_sync(FULL, cert));
      __syncwarp();
      {
        double acc = 0.0;
        if (ra.live) {
#pragma unroll 8
          for (int r = 0; r < 32; ++r) {
            const float* rr = sm.m.rows[warp * 32 + r];
            acc += (double)rr[ra.a] * (double)rr[ra.b];
          }
        }
        if (lane == 28) acc = (double)w_ties;
        if (lane == 29) acc = (double)w_seed;
        if (lane == 30) acc = (double)w_cert;
        if (lane == 31) acc = (double)nl;
        red[warp][lane] = acc;
      }
      __syncthreads();
      if (tid < S2M_SUMS) {
        double sum = 0.0;
#pragma unroll
        for (int k = 0; k < FZ_WARPS; ++k) sum += red[k][tid];
        A.chunk_rows[(size_t)c * S2M_SUMS + tid] = sum;
      }
      {  // the chunk's deferred leftovers, warp by warp, into its segment of the global list
        int off = 0, tot = 0;
#pragma unroll
        for (int w = 0; w < FZ_WARPS; ++w) { if (w < warp) off += sm.m.nl[w]; tot += sm.m.nl[w]; }
        if (lane < sm.m.nl[warp]) A.left_list[(size_t)base + off + lane] = base + sm.m.llist[warp][lane];
        if (tid == 0) { A.chunk_nleft[c] = tot; cta_deferred += tot; }
      }
      __syncthreads();
    }

    // =========================== ticket A: the last CTA out of the main phase decides ===========================
    if (probe && blockIdx.x == 0 && tid == 0) probe[1] = fz_globaltimer();
    if (tid == 0) {
      if (cta_deferred) atomicAdd(&st->fz_deferred[it], (unsigned)cta_deferred);
      __threadfence();
      s_last = (atomicAdd(&st->fz_ticket_a[it], 1u) == (unsigned)(G - 1));
    }
    __syncthreads();
    bool left_phase = false;
    if (s_last) {
      __threadfence();
      if (tid == 0) {
        s_misc[2] = (int)__ldcg(&st->fz_deferred[it]);
        if (probe) probe[2] = fz_globaltimer();
      }
      __syncthreads();
      left_phase = s_misc[2] > 0;
      if (left_phase) {
        if (tid == 0) { __threadfence(); atomicExch(&st->fz_phase, (unsigned)(2 * it + 1)); }
      } else {
        const double sum = fz_reduce_rows(A.chunk_rows, A.nchunks, red, warp, lane);
        if (tid < S2M_SUMS) s_sum[tid] = sum;
        if (probe && tid == 0) probe[6] = fz_globaltimer();
        __syncthreads();
        if (tid < 32) {
          if (tid < 12) st->T_prev[tid] = sT[tid];  // where the points stood in this iteration
          if (tid == 0) {
            st->certified = (int)s_sum[30]; st->leftovers = (int)s_sum[31];
            st->cert_hist[it] = (int)s_sum[30]; st->left_hist[it] = (int)s_sum[31]; st->seed_hist[it] = (int)s_sum[29];
          }
          __syncwarp();
          lm_finalize_warp(st, s_sum, s_fin, tid);
          __syncwarp();
          if (tid == 0) {
            if (probe) probe[7] = fz_globaltimer();
            __threadfence();
            atomicExch(&st->fz_phase, (unsigned)(2 * it + 2));
          }
        }
      }
    }
    // everybody: wait for the decision
    if (tid == 0) {
      unsigned ph;
      while ((ph = fz_ld_acquire(&st->fz_phase)) < (unsigned)(2 * it + 1)) { }
      __threadfence();
      s_misc[3] = (int)ph;
    }
    __syncthreads();

    if (s_misc[3] == 2 * it + 1) {
      // =========================== deferred-leftover phase (whole grid) ===========================
      {
        // exclusive scan of the per-chunk deferred counts (every CTA builds its own copy)
        constexpr int PER = FZ_MAXCHUNKS / FZ_THREADS;  // 16
        int cnt[PER];
        int local = 0;
#pragma unroll
        for (int k = 0; k < PER; ++k) {
          const int cidx = tid * PER + k;
          cnt[k] = cidx < A.nchunks ? __ldcg(A.chunk_nleft + cidx) : 0;
          local += cnt[k];
        }
        int incl = local;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int v = __shfl_up_sync(FULL, incl, o);
          if (lane >= o) incl += v;
        }
        if (lane == 31) s_wcnt[warp] = incl;
        __syncthreads();
        int run = incl - local;
        for (int w = 0; w < warp; ++w) run += s_wcnt[w];
#pragma unroll
        for (int k = 0; k < PER; ++k) {
          const int cidx = tid * PER + k;
          if (cidx < A.nchunks) sm.l.off[cidx] = run;
          run += cnt[k];
        }
        if (tid == FZ_THREADS - 1) s_misc[0] = run;
        __syncthreads();
        if (tid == 0) sm.l.off[A.nchunks] = s_misc[0];
        __syncthreads();
      }
      const int total = s_misc[0];
      const int warps_per_grid = G * FZ_WARPS;
      const int per_warp = min(32, max(1, (total + warps_per_grid - 1) / warps_per_grid));
      const int nbatch = (total + per_warp - 1) / per_warp;
      double acc = 0.0;
      int ties = 0;
      for (int r0 = 0; r0 < nbatch; r0 += warps_per_grid) {
        const int batch = r0 + (int)blockIdx.x * FZ_WARPS + warp;
        float row[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        float rhs = 0.f;
        bool flag = false, tie = false;
        if (batch < nbatch) {
          const int e0 = batch * per_warp;
          const int cnt = min(per_warp, total - e0);
          int mine = -1;
          if (lane < cnt) {
            const int e = e0 + lane;
            int lo = 0, hi = A.nchunks;  // invariant: off[lo] <= e < off[hi]
            while (hi - lo > 1) {
              const int mid = (lo + hi) >> 1;
              if (sm.l.off[mid] <= e) lo = mid; else hi = mid;
            }
            mine = __ldcg(A.left_list + (size_t)lo * FZ_THREADS + (e - sm.l.off[lo]));
          }
          float4 ori = make_float4(0.f, 0.f, 0.f, 0.f), sel = ori;
          if (mine >= 0) { ori = A.scan[mine]; sel = apply_T(sT, ori); }
          Top5 t;
          t.init(A.g.gate_d2);
          float my_r2 = ge2;
          for (int j = 0; j < cnt; ++j) {  // the warp searches for point j; lane j keeps the answer
            float4 q;
            q.x = __shfl_sync(FULL, sel.x, j); q.y = __shfl_sync(FULL, sel.y, j);
            q.z = __shfl_sync(FULL, sel.z, j); q.w = 0.f;
            Top5 tj;
            float r2;
            leftover_search(q, A.g, ge2, A.map_sorted, A.cell_start, lane, tj, r2);
            if (lane == j) { t = tj; my_r2 = r2; }
          }
          if (mine >= 0) {
            const bool found = t.d(t.k4) < A.g.gate_d2;  // :1641
            float4 coeff = make_float4(0.f, 0.f, 0.f, 0.f);
            float4 nbr[5];
            if (found) {
              nbr[0] = __ldg(A.map4 + t.i(t.k0)); nbr[1] = __ldg(A.map4 + t.i(t.k1)); nbr[2] = __ldg(A.map4 + t.i(t.k2));
              nbr[3] = __ldg(A.map4 + t.i(t.k3)); nbr[4] = __ldg(A.map4 + t.i(t.k4));
              flag = plane_residual(ori, sel, nbr, coeff);
              tie = t.tie();
              if (!flag) coeff = make_float4(0.f, 0.f, 0.f, 0.f);
            }
            if (flag) jacobian_row(sTrig, ori, coeff, row, rhs);
            fz_store_leftover(A, mine, sel, t, my_r2, found);
            if (A.dbg.nn_idx) {
              int* o = A.dbg.nn_idx + (size_t)mine * 5;
              o[0] = found ? t.i(t.k0) : -1; o[1] = found ? t.i(t.k1) : -1; o[2] = found ? t.i(t.k2) : -1;
              o[3] = found ? t.i(t.k3) : -1; o[4] = found ? t.i(t.k4) : -1;
            }
            if (A.dbg.nn_d2) {
              float* o = A.dbg.nn_d2 + (size_t)mine * 5;
              o[0] = t.d(t.k0); o[1] = t.d(t.k1); o[2] = t.d(t.k2); o[3] = t.d(t.k3); o[4] = t.d(t.k4);
            }
            if (A.dbg.coeff) A.dbg.coeff[mine] = coeff;
            if (A.dbg.flag) A.dbg.flag[mine] = flag ? 1 : 0;
            if (A.dbg.tie) A.dbg.tie[mine] = tie ? 1 : 0;
          }
        }
#pragma unroll
        for (int k = 0; k < 6; ++k) sm.l.rows[tid][k] = row[k];
        sm.l.rows[tid][6] = rhs;
        sm.l.rows[tid][7] = flag ? 1.f : 0.f;
        if (flag && tie) ++ties;
        __syncwarp();
        if (ra.live) {  // every warp owns the slice of rows its own lanes staged
#pragma unroll 8
          for (int r = 0; r < 32; ++r) {
            const float* rr = sm.l.rows[warp * 32 + r];
            acc += (double)rr[ra.a] * (double)rr[ra.b];
          }
        }
        __syncwarp();
      }
      {
        int wt = ties;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) wt += __shfl_xor_sync(FULL, wt, o);
        if (lane == 28) acc += (double)wt;
      }
      red[warp][lane] = acc;
      __syncthreads();
      if (tid < S2M_SUMS) {
        double sum = 0.0;
#pragma unroll
        for (int k = 0; k < FZ_WARPS; ++k) sum += red[k][tid];
        if (tid == 31 && blockIdx.x == 0) sum += (double)total;
        A.cta_rows[(size_t)blockIdx.x * S2M_SUMS + tid] = sum;
      }
      if (probe && blockIdx.x == 0 && tid == 0) probe[4] = fz_globaltimer();
      // ---- ticket B: the last CTA adds everything in a fixed order and runs the 6x6 tail ----
      __threadfence();
      __syncthreads();
      if (tid == 0) s_last = (atomicAdd(&st->fz_ticket_b[it], 1u) == (unsigned)(G - 1));
      __syncthreads();
      if (s_last) {
        __threadfence();
        if (probe && tid == 0) probe[5] = fz_globaltimer();
        const double sum_a = fz_reduce_rows(A.chunk_rows, A.nchunks, red, warp, lane);
        const double sum_b = fz_reduce_rows(A.cta_rows, G, red, warp, lane);
        if (tid < S2M_SUMS) s_sum[tid] = sum_a + sum_b;
        if (probe && tid == 0) probe[6] = fz_globaltimer();
        __syncthreads();
        if (tid < 32) {
          if (tid < 12) st->T_prev[tid] = sT[tid];
          if (tid == 0) {
            st->certified = (int)s_sum[30]; st->leftovers = (int)s_sum[31];
            st->cert_hist[it] = (int)s_sum[30]; st->left_hist[it] = (int)s_sum[31]; st->seed_hist[it] = (int)s_sum[29];
          }
          __syncwarp();
          lm_finalize_warp(st, s_sum, s_fin, tid);
          __syncwarp();
          if (tid == 0) {
            if (probe) probe[7] = fz_globaltimer();
            __threadfence();
            atomicExch(&st->fz_phase, (unsigned)(2 * it + 2));
          }
        }
      }
      if (tid == 0) {
        while (fz_ld_acquire(&st->fz_phase) < (unsigned)(2 * it + 2)) { }
        __threadfence();
      }
      __syncthreads();
    }
    if (tid == 0) s_misc[1] = __ldcg(&st->done);
    __syncthreads();
    if (s_misc[1]) break;
  }
}

}  // namespace liogpu
