// icp.cu — the loop-closure registration: pcl::IterativeClosestPoint<PointXYZI, PointXYZI>::align as
// configured at mapOptmization.cpp:1111-1121 (also :1203-1213) and icp.getFitnessScore() (:1123); SURVEY §8 row f3.
//
// Per ICP iteration (PCL registration/impl/icp.hpp), all on device, no host round trip inside a chunk:
//   icp_nn_kernel      thread per source point: move it by the previous iteration's transformation_, exact
//                      nearest target point on the sorted grid, shells 0..2 (ties: lower target index)
//   icp_left_kernel    warp per point that needs shells 3..5
//   icp_brute_kernel   block per isolated point: one pass over the target
//   icp_reduce_kernel  f64 sums over the correspondences (d^2 <= max^2): source / target centroids, cross
//                      products, squared distances; the last block runs Eigen::umeyama (3x3 SVD by one-sided
//                      Jacobi in f64), final_transformation_ = transformation_ * final_transformation_ and
//                      DefaultConvergenceCriteria::hasConverged.
// The search stops growing once every uninspected cell is farther than the correspondence distance (such a point
// has no correspondence).  getFitnessScore: the same search with no distance limit on the source moved by the final
// transformation, f64 mean of the squared distances.
//
// liogpu_loop_closure_icp_batch runs many pairs with three launches per iteration (icpb_*).  Both launch structures
// are built from the same device functions: nn_thread_walk (shells 0..2 by one thread), nn_warp_walk (the next shells
// by one warp), nn_brute_block (one pass over the target) and icp_reduce_block (a pair's sums and fold), so a pair's
// result is bit-equal whichever call computed it.
#include "common.cuh"
#include "pose_math.cuh"

#include <stdlib.h>
#include "shell_search.cuh"

namespace liogpu {

namespace {

constexpr int ICP_SUMS = 17;  // 3 src + 3 tgt + 9 cross + mse + count

struct IcpDevState {
  float T_inc[16];   // transformation_ of the last finished iteration (row-major 4x4)
  float finalT[16];  // final_transformation_
  double prev_mse, last_mse, fitness;
  double max_d2, rot_thr, trans_thr, rel_thr, abs_thr;
  int iter, done, state, n_corr, max_iter, fit_nr;
  unsigned n_left, n_brute, ticket, pad;
};

struct IcpArgs {
  const float4* src;        // original source
  float4* cur;              // input_transformed
  int ns;
  const float4* tgt;        // target, original order
  const float4* sorted;     // target in grid order, w = bits(original index)
  const uint32_t* cs;
  const GridParams* gp;
  IcpDevState* st;
  int* nn_idx;
  float* nn_d2;
  uint32_t* left_list;      // [ns] shells 3.., then [ns] exhaustive
  double* partials;         // [reduce blocks][ICP_SUMS]
  int fitness;              // 1: getFitnessScore pass (source moved by finalT, no distance limit)
  int all_warp;             // 1: every source point goes straight to the warp-per-point search (small sources: a
                            //    thread-per-point pass would leave most of the GPU idle and is latency bound)
};

// nearest point: (bits(d^2) << 32 | target index), so that min() also breaks ties toward the lower index
struct Best1 {
  unsigned long long key;
  __device__ __forceinline__ void init() { key = (0x7f800000ULL << 32) | 0xffffffffULL; }  // +inf, index -1
  __device__ __forceinline__ void push(float d2, float w) {
    const unsigned long long k = ((unsigned long long)__float_as_uint(d2) << 32) | (unsigned)__float_as_int(w);
    key = k < key ? k : key;
  }
  __device__ __forceinline__ float d2() const { return __uint_as_float((unsigned)(key >> 32)); }
  __device__ __forceinline__ int idx() const { return (int)(unsigned)(key & 0xffffffffULL); }
};

// pcl::transformPointCloud with a Matrix4f (PCL >= 1.10 detail::Transformer<float>::se3)
__device__ __forceinline__ float4 se3(const float* T, const float4 p) {
  float4 q;
  q.x = p.x * T[0] + (p.y * T[1] + (p.z * T[2] + T[3]));
  q.y = p.x * T[4] + (p.y * T[5] + (p.z * T[6] + T[7]));
  q.z = p.x * T[8] + (p.y * T[9] + (p.z * T[10] + T[11]));
  q.w = p.w;
  return q;
}

// 0: keep growing, 1: nearest point certified, 2: nothing within the correspondence distance
__device__ __forceinline__ int nn_verdict(const Best1& b, float cov2, double max_d2) {
  if (b.d2() <= cov2) return 1;
  if ((double)cov2 > max_d2) return 2;
  return 0;
}

constexpr int NN_THREADS = 128;
constexpr int NN_THREAD_SHELLS = 3;  // shells 0..2 per thread
constexpr int NN_WARP_SHELLS = 6;    // shells 0..5 per warp

__device__ __forceinline__ unsigned long long warp_min_u64(unsigned long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long u = __shfl_xor_sync(0xffffffffu, v, o);
    v = u < v ? u : v;
  }
  return v;
}

// One thread searches shells 0..NN_THREAD_SHELLS-1 around the home cell of p (finite) and returns the verdict of the
// last shell it inspected; `best` is the nearest point found in them.  max_d2 is a reference so that icp_nn_kernel
// reads it from shared memory at each verdict rather than holding it in two more registers.
__device__ __forceinline__ int nn_thread_walk(const float4* sorted, const uint32_t* cs, const GridParams& g,
                                              const float4 p, const double& max_d2, Best1& best) {
  const HomeCell hc = home_cell(g, p);
  best.init();
  int verdict = 0;
  for (int R = 0; R < NN_THREAD_SHELLS && verdict == 0; ++R) {
    const int z0 = max(hc.cz - R, 0), z1 = min(hc.cz + R, g.nz - 1);
    const int y0 = max(hc.cy - R, 0), y1 = min(hc.cy + R, g.ny - 1);
    for (int z = z0; z <= z1; ++z)
      for (int y = y0; y <= y1; ++y) scan_shell_row(sorted, cs, g, hc, R, y, z, p, best);
    verdict = nn_verdict(best, covered_d2(g, hc, R), max_d2);
  }
  return verdict;
}

// The whole warp searches shells R0..NN_WARP_SHELLS-1 around the home cell of p (finite, the same on every lane), each
// lane's rows starting from `best` (what shells 0..R0-1 found, or empty).  Returns the verdict of the last shell
// inspected; `all` is the warp's nearest point.
__device__ __forceinline__ int nn_warp_walk(const float4* sorted, const uint32_t* cs, const GridParams& g,
                                            const float4 p, double max_d2, int R0, Best1 best, Best1& all) {
  const HomeCell hc = home_cell(g, p);
  const int lane = threadIdx.x & 31;
  all.init();
  int verdict = 0;
  for (int R = R0; R < NN_WARP_SHELLS && verdict == 0; ++R) {
    const int side = 2 * R + 1, rows = side * side;
    for (int r = lane; r < rows; r += 32) {
      const int z = hc.cz + r / side - R, y = hc.cy + r % side - R;
      if (z < 0 || z >= g.nz || y < 0 || y >= g.ny) continue;
      scan_shell_row(sorted, cs, g, hc, R, y, z, p, best);
    }
    all.key = warp_min_u64(best.key);
    verdict = nn_verdict(all, covered_d2(g, hc, R), max_d2);
  }
  return verdict;
}

__global__ void __launch_bounds__(NN_THREADS)
icp_nn_kernel(const IcpArgs A) {
  __shared__ GridParams g;
  __shared__ float sT[12];
  __shared__ int s_skip, s_move;
  __shared__ double s_max_d2;
  if (threadIdx.x == 0) {
    g = *A.gp;
    s_skip = A.fitness ? 0 : A.st->done;
    s_move = A.fitness ? 1 : (A.st->iter > 0);
    s_max_d2 = A.fitness ? CUDART_INF : A.st->max_d2;
  }
  if (threadIdx.x < 12) sT[threadIdx.x] = A.fitness ? A.st->finalT[threadIdx.x] : A.st->T_inc[threadIdx.x];
  __syncthreads();
  if (s_skip) return;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= A.ns) return;
  float4 p = A.fitness ? A.src[i] : A.cur[i];
  if (s_move) {
    p = se3(sT, p);
    A.cur[i] = p;
  }
  if (!(isfinite(p.x) && isfinite(p.y) && isfinite(p.z))) { A.nn_idx[i] = -1; A.nn_d2[i] = CUDART_INF_F; return; }
  Best1 best;
  const int verdict = nn_thread_walk(A.sorted, A.cs, g, p, s_max_d2, best);
  if (verdict == 0) {
    A.left_list[atomicAdd(&A.st->n_left, 1u)] = (uint32_t)i;
  } else {
    A.nn_idx[i] = verdict == 1 ? best.idx() : -1;
    A.nn_d2[i] = best.d2();
  }
}

__global__ void __launch_bounds__(256)
icp_left_kernel(const IcpArgs A) {
  __shared__ GridParams g;
  __shared__ float sT[12];
  if (threadIdx.x == 0) g = *A.gp;
  if (threadIdx.x < 12) sT[threadIdx.x] = A.fitness ? A.st->finalT[threadIdx.x] : A.st->T_inc[threadIdx.x];
  __syncthreads();
  if (!A.fitness && A.st->done) return;
  const double max_d2 = A.fitness ? CUDART_INF : A.st->max_d2;
  const bool move = A.all_warp && (A.fitness || A.st->iter > 0);
  const int lane = threadIdx.x & 31;
  const unsigned warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
  const unsigned n_left = A.all_warp ? (unsigned)A.ns : A.st->n_left;
  for (unsigned w = warp; w < n_left; w += n_warps) {
    const uint32_t i = A.all_warp ? w : A.left_list[w];
    float4 p = (A.all_warp && A.fitness) ? A.src[i] : A.cur[i];
    if (move) {
      p = se3(sT, p);
      if (lane == 0) A.cur[i] = p;
    }
    if (!(isfinite(p.x) && isfinite(p.y) && isfinite(p.z))) {
      if (lane == 0) { A.nn_idx[i] = -1; A.nn_d2[i] = CUDART_INF_F; }
      continue;
    }
    Best1 seed, all;
    seed.init();
    const int verdict = nn_warp_walk(A.sorted, A.cs, g, p, max_d2, 0, seed, all);
    if (lane == 0) {
      if (verdict == 0) {
        A.left_list[A.ns + atomicAdd(&A.st->n_brute, 1u)] = i;
      } else {
        A.nn_idx[i] = verdict == 1 ? all.idx() : -1;
        A.nn_d2[i] = all.d2();
      }
    }
  }
}

// The whole block finds the nearest of the n_points sorted targets to point i at p in one pass (eight loads in flight
// per thread), then the block minimum, and writes nn_idx[i] / nn_d2[i]
constexpr int BRT = 512;
__device__ __forceinline__ void nn_brute_block(const float4* sorted, int n_points, const float4 p, double max_d2,
                                               uint32_t i, int* nn_idx, float* nn_d2) {
  __shared__ unsigned long long sh[BRT / 32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  Best1 best;
  best.init();
  for (int base = 0; base < n_points; base += BRT * 8) {
    float4 q[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int t = base + u * BRT + (int)threadIdx.x;
      q[u] = t < n_points ? __ldg(sorted + t) : make_float4(CUDART_INF_F, 0.f, 0.f, __int_as_float(-1));
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) best.push(sor_d2(p, q[u]), q[u].w);
  }
  const unsigned long long wm = warp_min_u64(best.key);
  if (lane == 0) sh[w] = wm;
  __syncthreads();
  if (w == 0) {
    unsigned long long v = lane < BRT / 32 ? sh[lane] : ~0ULL;
    v = warp_min_u64(v);
    if (lane == 0) {
      Best1 b;
      b.key = v;
      const bool ok = (double)b.d2() <= max_d2;  // exhaustive: always the true nearest point
      nn_idx[i] = ok ? b.idx() : -1;
      nn_d2[i] = b.d2();
    }
  }
  __syncthreads();
}

__global__ void __launch_bounds__(BRT)
icp_brute_kernel(const IcpArgs A) {
  if (!A.fitness && A.st->done) return;
  const double max_d2 = A.fitness ? CUDART_INF : A.st->max_d2;
  const int n_points = A.gp->n_points;
  const unsigned n_brute = A.st->n_brute;
  for (unsigned e = blockIdx.x; e < n_brute; e += gridDim.x) {
    const uint32_t i = A.left_list[A.ns + e];
    nn_brute_block(A.sorted, n_points, A.cur[i], max_d2, i, A.nn_idx, A.nn_d2);
  }
}

__device__ void icp_finalize(IcpDevState* st, const double* S) {
  const int cnt = (int)S[16];
  st->n_corr = cnt;
  if (cnt < 3) {  // min_number_correspondences_
    st->state = 5;
    st->done = 1;
    return;
  }
  const double inv_n = 1.0 / (double)cnt;
  const double mse = S[15] / (double)cnt;
  st->last_mse = mse;
  float src_mean[3], dst_mean[3], sigma[9], R[9], T[16];
  for (int a = 0; a < 3; ++a) { src_mean[a] = (float)(S[a] * inv_n); dst_mean[a] = (float)(S[3 + a] * inv_n); }
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) sigma[3 * i + j] = (float)((S[6 + 3 * i + j] - S[3 + i] * S[j] * inv_n) * inv_n);
  umeyama_rotation_dev(sigma, R);
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) T[4 * i + j] = R[3 * i + j];
    T[4 * i + 3] = dst_mean[i] - (R[3 * i] * src_mean[0] + R[3 * i + 1] * src_mean[1] + R[3 * i + 2] * src_mean[2]);
  }
  T[12] = T[13] = T[14] = 0.f; T[15] = 1.f;
  float F[16];
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < 4; ++j)
      F[4 * i + j] = T[4 * i] * st->finalT[j] + T[4 * i + 1] * st->finalT[4 + j] + T[4 * i + 2] * st->finalT[8 + j] +
                     T[4 * i + 3] * st->finalT[12 + j];
  for (int q = 0; q < 16; ++q) { st->finalT[q] = F[q]; st->T_inc[q] = T[q]; }
  const int it = ++st->iter;
  // DefaultConvergenceCriteria::hasConverged
  int state = 0;
  if (it >= st->max_iter) {
    state = 1;
  } else {
    const float tr = T[0] + T[5] + T[10] - 1;
    const double cos_angle = 0.5 * tr;
    const float tsq = T[3] * T[3] + T[7] * T[7] + T[11] * T[11];
    const double translation_sqr = tsq;
    if (cos_angle >= st->rot_thr && translation_sqr <= st->trans_thr) state = 2;
    else if (fabs(mse - st->prev_mse) < st->abs_thr) state = 3;
    else if (fabs(mse - st->prev_mse) / st->prev_mse < st->rel_thr) state = 4;
    else st->prev_mse = mse;
  }
  st->state = state;
  if (state != 0) st->done = 1;
}

// One block's part of the reduction of a pair of ns source points over nblk blocks (lb = this block's index among
// them): the f64 sums of its grid-stride share of the correspondences (d^2 <= max^2; only the squared distances and
// the count for the fitness score), a shuffle tree, the block's row of `partials`; then the block that takes the last
// ticket folds the pair's rows in a fixed order.  Returns the pair's ICP_SUMS sums (shared memory) in that block,
// nullptr in the others.
constexpr int RD_THREADS = 256;
__device__ __forceinline__ const double* icp_reduce_block(const int* nn_idx, const float* nn_d2, const float4* cur,
                                                          const float4* tgt, int ns, int lb, int nblk, double* partials,
                                                          IcpDevState* st, int fitness) {
  __shared__ double sh[RD_THREADS / 32][ICP_SUMS];
  __shared__ bool s_last;
  const double max_d2 = fitness ? CUDART_INF : st->max_d2;
  double acc[ICP_SUMS];
#pragma unroll
  for (int q = 0; q < ICP_SUMS; ++q) acc[q] = 0.0;
  for (int i = lb * blockDim.x + threadIdx.x; i < ns; i += nblk * blockDim.x) {
    const int j = nn_idx[i];
    const float d2 = nn_d2[i];
    if (j < 0 || (double)d2 > max_d2) continue;
    acc[15] += (double)d2;
    acc[16] += 1.0;
    if (!fitness) {
      const float4 s = cur[i], t = tgt[j];
      const double sv[3] = {s.x, s.y, s.z}, tv[3] = {t.x, t.y, t.z};
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        acc[a] += sv[a];
        acc[3 + a] += tv[a];
#pragma unroll
        for (int b = 0; b < 3; ++b) acc[6 + 3 * a + b] += tv[a] * sv[b];
      }
    }
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int q = 0; q < ICP_SUMS; ++q) {
    double v = acc[q];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if (lane == 0) sh[w][q] = v;
  }
  __syncthreads();
  if (threadIdx.x < ICP_SUMS) {
    double v = 0.0;
    for (int k = 0; k < RD_THREADS / 32; ++k) v += sh[k][threadIdx.x];
    partials[(size_t)lb * ICP_SUMS + threadIdx.x] = v;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(&st->ticket, 1u) == (unsigned)nblk - 1;
  __syncthreads();
  if (!s_last) return nullptr;
  __threadfence();
  {  // fixed order: eight interleaved slices of the blocks (their loads in flight together), then the slices
    const int q = threadIdx.x & 31, slice = threadIdx.x >> 5;
    double v = 0.0;
    if (q < ICP_SUMS) {
      for (int b = slice; b < nblk; b += RD_THREADS / 32) v += partials[(size_t)b * ICP_SUMS + q];
      sh[slice][q] = v;
    }
  }
  __syncthreads();
  if (threadIdx.x < ICP_SUMS) {
    double v = 0.0;
    for (int k = 0; k < RD_THREADS / 32; ++k) v += sh[k][threadIdx.x];
    sh[0][threadIdx.x] = v;
  }
  __syncthreads();
  return sh[0];
}

__global__ void __launch_bounds__(RD_THREADS)
icp_reduce_kernel(const IcpArgs A) {
  IcpDevState* st = A.st;
  if (!A.fitness && st->done) return;
  const double* S = icp_reduce_block(A.nn_idx, A.nn_d2, A.cur, A.tgt, A.ns, (int)blockIdx.x, (int)gridDim.x, A.partials,
                                     st, A.fitness);
  if (S && threadIdx.x == 0) {
    if (A.fitness) {
      st->fit_nr = (int)S[16];
      st->fitness = S[16] > 0.0 ? S[15] / S[16] : DBL_MAX;
    } else {
      icp_finalize(st, S);
    }
    st->ticket = 0;
    st->n_left = 0;
    st->n_brute = 0;
  }
}

// ---- many pairs at once (liogpu_loop_closure_icp_batch) ----
// Every pair keeps its own IcpDevState and its own grid; the search is exact (ties go to the lower target index,
// whatever the grid) and each pair is reduced over as many blocks as icp_align_dev launches for it, so every pair's
// result is bit-equal to icp_align_dev.
// The targets of all pairs share one sorted array: key = cell_base[pair] + the cell inside the pair's grid, so a pair's
// points form one contiguous run and cell_start + cell_base[pair] is that pair's cell_start.

struct IcpbCounters {
  unsigned n_brute[2];  // exhaustive-search list of the current launch (parity), the other one is cleared for the next
  int live;             // pairs not yet done
  int pad;
};

struct IcpbArgs {
  const float4* src;        // sources of all pairs, concatenated
  float4* cur;              // input_transformed, same indexing
  const float4* tgt;        // targets of all pairs, concatenated
  const float4* sorted;     // targets in (pair, cell) order, w = bits(index inside the pair's target)
  const uint32_t* cs;       // cell_start over the concatenated cells
  const int* sp;            // [n + 1] source offsets
  const int* tp;            // [n + 1] target offsets
  const int* rp;            // [n + 1] reduce-block offsets
  const unsigned* cell_base;
  const GridParams* gp;
  IcpDevState* st;
  IcpbCounters* cnt;
  int* nn_idx;
  float* nn_d2;
  uint32_t* brute;          // [ns] points left to the exhaustive search
  double* partials;         // [rp[n]][ICP_SUMS]
  int n, ns;
  int fitness;
  int par;                  // launch parity: which n_brute counter this launch uses
};

// segment of element i: the last p with off[p] <= i (segments are non-empty)
__device__ __forceinline__ int find_seg(const int* __restrict__ off, int n, int i) {
  int lo = 0, hi = n - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(off + mid) <= i) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// block per pair: bounding box and finite count of its target, then its grid
constexpr int BB_THREADS = 256;
__global__ void __launch_bounds__(BB_THREADS)
icpb_grid_kernel(const float4* __restrict__ tgt, const int* __restrict__ tp, float cell, unsigned max_cells,
                 GridParams* __restrict__ gp) {
  __shared__ float s_mn[3][BB_THREADS / 32], s_mx[3][BB_THREADS / 32];
  __shared__ int s_cnt[BB_THREADS / 32];
  const int p = blockIdx.x;
  float mn[3] = {CUDART_INF_F, CUDART_INF_F, CUDART_INF_F}, mx[3] = {-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F};
  int cnt = 0;
  for (int t = tp[p] + (int)threadIdx.x; t < tp[p + 1]; t += BB_THREADS) {
    const float4 q = tgt[t];
    if (!(isfinite(q.x) && isfinite(q.y) && isfinite(q.z))) continue;
    mn[0] = fminf(mn[0], q.x); mn[1] = fminf(mn[1], q.y); mn[2] = fminf(mn[2], q.z);
    mx[0] = fmaxf(mx[0], q.x); mx[1] = fmaxf(mx[1], q.y); mx[2] = fmaxf(mx[2], q.z);
    ++cnt;
  }
  for (int o = 16; o > 0; o >>= 1) {
    for (int a = 0; a < 3; ++a) {
      mn[a] = fminf(mn[a], __shfl_xor_sync(0xffffffffu, mn[a], o));
      mx[a] = fmaxf(mx[a], __shfl_xor_sync(0xffffffffu, mx[a], o));
    }
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) {
    for (int a = 0; a < 3; ++a) { s_mn[a][w] = mn[a]; s_mx[a][w] = mx[a]; }
    s_cnt[w] = cnt;
  }
  __syncthreads();
  if (threadIdx.x != 0) return;
  int n_points = 0;
  for (int k = 0; k < BB_THREADS / 32; ++k) {
    for (int a = 0; a < 3; ++a) { mn[a] = fminf(mn[a], s_mn[a][k]); mx[a] = fmaxf(mx[a], s_mx[a][k]); }
    n_points += s_cnt[k];
  }
  gp[p] = grid_setup_compute(mn, mx, n_points, cell, max_cells, 1.0f, 1.0f);
}

__global__ void __launch_bounds__(256)
icpb_key_kernel(const float4* __restrict__ tgt, int nt, const int* __restrict__ tp, int n, const GridParams* __restrict__ gp,
                const unsigned* __restrict__ cell_base, unsigned total_cells, uint32_t* __restrict__ keys,
                uint32_t* __restrict__ cell_count) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nt) return;
  const float4 q = tgt[i];
  uint32_t key = total_cells;  // non-finite points sort last and are never referenced
  if (isfinite(q.x) && isfinite(q.y) && isfinite(q.z)) {
    const int p = find_seg(tp, n, i);
    const GridParams g = gp[p];
    const int cx = cell_coord(q.x, g.ox, g.inv_h, g.nx);
    const int cy = cell_coord(q.y, g.oy, g.inv_h, g.ny);
    const int cz = cell_coord(q.z, g.oz, g.inv_h, g.nz);
    key = cell_base[p] + ((uint32_t)cz * (uint32_t)g.ny + (uint32_t)cy) * (uint32_t)g.nx + (uint32_t)cx;
    atomicAdd(&cell_count[key], 1u);
  }
  keys[i] = key;
}

__global__ void __launch_bounds__(256)
icpb_gather_kernel(const float4* __restrict__ tgt, const uint32_t* __restrict__ perm, int n_valid, const int* __restrict__ tp,
                   int n, float4* __restrict__ sorted) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_valid) return;
  const int src = (int)perm[j];
  const float4 q = tgt[src];
  sorted[j] = make_float4(q.x, q.y, q.z, __int_as_float(src - tp[find_seg(tp, n, src)]));
}

// thread per source point of every live pair: shells 0..NN_THREAD_SHELLS-1; the block's points that need more are
// then taken warp per point for the remaining shells, starting from the nearest point the thread already found
constexpr int NB_THREADS = 128;
__global__ void __launch_bounds__(NB_THREADS)
icpb_nn_kernel(const IcpbArgs A) {
  __shared__ int s_n;
  __shared__ int s_i[NB_THREADS], s_p[NB_THREADS];
  __shared__ unsigned long long s_key[NB_THREADS];
  __shared__ float4 s_pt[NB_THREADS];
  if (threadIdx.x == 0) {
    s_n = 0;
    if (blockIdx.x == 0) A.cnt->n_brute[A.par ^ 1] = 0;  // the next launch's list (this launch's was cleared by the last)
  }
  __syncthreads();
  const int i = blockIdx.x * NB_THREADS + threadIdx.x;
  if (i < A.ns) {
    const int p = find_seg(A.sp, A.n, i);
    const IcpDevState* st = A.st + p;
    if (A.fitness || !st->done) {
      float4 q = A.fitness ? A.src[i] : A.cur[i];
      if (A.fitness || st->iter > 0) {
        q = se3(A.fitness ? st->finalT : st->T_inc, q);
        A.cur[i] = q;
      }
      if (!(isfinite(q.x) && isfinite(q.y) && isfinite(q.z))) {
        A.nn_idx[i] = -1;
        A.nn_d2[i] = CUDART_INF_F;
      } else {
        const GridParams g = A.gp[p];
        const double max_d2 = A.fitness ? CUDART_INF : st->max_d2;
        Best1 best;
        const int verdict = nn_thread_walk(A.sorted, A.cs + A.cell_base[p], g, q, max_d2, best);
        if (verdict == 0) {
          const int slot = atomicAdd(&s_n, 1);
          s_i[slot] = i; s_p[slot] = p; s_key[slot] = best.key; s_pt[slot] = q;
        } else {
          A.nn_idx[i] = verdict == 1 ? best.idx() : -1;
          A.nn_d2[i] = best.d2();
        }
      }
    }
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  for (int e = threadIdx.x >> 5; e < s_n; e += NB_THREADS / 32) {
    const int i = s_i[e], p = s_p[e];
    const float4 q = s_pt[e];
    const GridParams g = A.gp[p];
    const double max_d2 = A.fitness ? CUDART_INF : A.st[p].max_d2;
    Best1 seed, all;
    seed.init();
    if (lane == 0) seed.key = s_key[e];
    const int verdict = nn_warp_walk(A.sorted, A.cs + A.cell_base[p], g, q, max_d2, NN_THREAD_SHELLS, seed, all);
    if (lane == 0) {
      if (verdict == 0) {
        A.brute[atomicAdd(&A.cnt->n_brute[A.par], 1u)] = (uint32_t)i;
      } else {
        A.nn_idx[i] = verdict == 1 ? all.idx() : -1;
        A.nn_d2[i] = all.d2();
      }
    }
  }
}

// block per isolated point: one pass over its pair's finite targets
__global__ void __launch_bounds__(BRT)
icpb_brute_kernel(const IcpbArgs A) {
  const unsigned n_brute = A.cnt->n_brute[A.par];
  for (unsigned e = blockIdx.x; e < n_brute; e += gridDim.x) {
    const uint32_t i = A.brute[e];
    const int p = find_seg(A.sp, A.n, (int)i);
    const double max_d2 = A.fitness ? CUDART_INF : A.st[p].max_d2;
    nn_brute_block(A.sorted + A.cs[A.cell_base[p]], A.gp[p].n_points, A.cur[i], max_d2, i, A.nn_idx, A.nn_d2);
  }
}

// every live pair's reduction: pair p owns blocks rp[p] .. rp[p+1], icp_reduce_blocks of them as for the pair alone
__global__ void __launch_bounds__(RD_THREADS)
icpb_reduce_kernel(const IcpbArgs A) {
  const int p = find_seg(A.rp, A.n, (int)blockIdx.x);
  IcpDevState* st = A.st + p;
  if (!A.fitness && st->done) return;
  const int rb0 = A.rp[p], s0 = A.sp[p], t0 = A.tp[p];
  const double* S = icp_reduce_block(A.nn_idx + s0, A.nn_d2 + s0, A.cur + s0, A.tgt + t0, A.sp[p + 1] - s0,
                                     (int)blockIdx.x - rb0, A.rp[p + 1] - rb0, A.partials + (size_t)rb0 * ICP_SUMS, st,
                                     A.fitness);
  if (S && threadIdx.x == 0) {
    if (A.fitness) {
      st->fit_nr = (int)S[16];
      st->fitness = S[16] > 0.0 ? S[15] / S[16] : DBL_MAX;
    } else {
      icp_finalize(st, S);
      if (st->done) atomicSub(&A.cnt->live, 1);
    }
    st->ticket = 0;
  }
}

// Iterations enqueued between two host checks of convergence.  Both drivers enqueue the same number of iterations, so
// a batch does no more iterations for a pair than icp_align_dev would for it alone.
constexpr int ICP_CHUNK = 10;

// grid cell edge; tuning only (the search is exact).  Measured: 0.5 m 1.33 ms, 1 m 1.58 ms, 1.5 m 1.96 ms
float icp_cell_size(const liogpu_icp_params* prm) { return prm->cell_size > 0.f ? prm->cell_size : 0.5f; }

// reduce blocks of a pair of ns source points
int icp_reduce_blocks(int ns) { return div_up(ns, RD_THREADS) < 256 ? div_up(ns, RD_THREADS) : 256; }

// IcpDevState before the first iteration
void icp_state_init(IcpDevState& s, const liogpu_icp_params* prm) {
  memset(&s, 0, sizeof(IcpDevState));
  for (int q = 0; q < 16; ++q) s.T_inc[q] = s.finalT[q] = (q % 5 == 0) ? 1.f : 0.f;
  s.prev_mse = DBL_MAX;
  s.max_d2 = (double)prm->max_correspondence_distance * (double)prm->max_correspondence_distance;
  s.rot_thr = 1.0 - prm->transformation_epsilon;   // transformation_rotation_epsilon_ unset (icp.hpp)
  s.trans_thr = prm->transformation_epsilon;
  s.rel_thr = prm->euclidean_fitness_epsilon;
  s.abs_thr = 1e-12;
  s.max_iter = prm->max_iterations;
}

// the caller's result from the final IcpDevState
void icp_result(const IcpDevState& s, float gpu_ms, float final_T[16], liogpu_icp_info* info) {
  for (int q = 0; q < 16; ++q) final_T[q] = s.finalT[q];
  info->iterations = s.iter;
  info->convergence_state = s.state;
  info->converged = (s.state >= 1 && s.state <= 4) ? 1 : 0;
  info->n_correspondences = s.n_corr;
  info->fitness_score = s.fitness;
  info->last_mse = s.last_mse;
  info->gpu_ms = gpu_ms;
}

}  // namespace

// source / target: packed float4 on device.  The target's grid index is built into the outlier filter's buffers
// (publishLocalMap and the loop closure never run concurrently on one context).
int icp_align_dev(Ctx* c, const float4* src, int ns, const float4* tgt, int nt, const liogpu_icp_params* prm,
                  float final_T[16], liogpu_icp_info* info) {
  GridParams g;
  int rc = grid_build_core(c, tgt, nt, icp_cell_size(prm), 1.0f, 1.0f, c->sor_setup, c->sor_sorted, c->sor_cell_start, g);
  if (rc) return rc;
  LIOGPU_CUDA_OK(c, c->lm_a.reserve((size_t)ns * sizeof(float4)));
  LIOGPU_CUDA_OK(c, c->lm_flag.reserve((size_t)ns * sizeof(int)));
  LIOGPU_CUDA_OK(c, c->lm_md.reserve((size_t)ns * sizeof(float)));
  LIOGPU_CUDA_OK(c, c->lm_left.reserve((size_t)ns * 2 * sizeof(uint32_t)));
  LIOGPU_CUDA_OK(c, c->lm_stats.reserve(4096 + (size_t)256 * ICP_SUMS * sizeof(double)));
  IcpArgs A;
  A.src = src; A.cur = c->lm_a.as<float4>(); A.ns = ns;
  A.tgt = tgt; A.sorted = c->sor_sorted.as<float4>(); A.cs = c->sor_cell_start.as<uint32_t>();
  A.gp = c->sor_setup.as<GridParams>();
  A.st = reinterpret_cast<IcpDevState*>((char*)c->lm_stats.p + 1024);
  A.nn_idx = c->lm_flag.as<int>(); A.nn_d2 = c->lm_md.as<float>();
  A.left_list = c->lm_left.as<uint32_t>();
  A.partials = reinterpret_cast<double*>((char*)c->lm_stats.p + 4096);
  A.fitness = 0;
  A.all_warp = (ns <= 65536 && !getenv("LIOGPU_ICP_THREAD_PASS")) ? 1 : 0;
  IcpDevState* h = reinterpret_cast<IcpDevState*>((char*)c->h_pinned + 12288);
  icp_state_init(*h, prm);
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(A.st, h, sizeof(IcpDevState), cudaMemcpyHostToDevice, c->stream));
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(A.cur, src, (size_t)ns * sizeof(float4), cudaMemcpyDeviceToDevice, c->stream));
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
  int launched = 0;
  auto enqueue_iteration = [&](const IcpArgs& a) {
    if (!a.all_warp) icp_nn_kernel<<<div_up(ns, NN_THREADS), NN_THREADS, 0, c->stream>>>(a);
    icp_left_kernel<<<a.all_warp ? c->sm_count * 8 : c->sm_count * 2, 256, 0, c->stream>>>(a);
    icp_brute_kernel<<<c->sm_count, BRT, 0, c->stream>>>(a);
    icp_reduce_kernel<<<icp_reduce_blocks(ns), RD_THREADS, 0, c->stream>>>(a);
    c->launches += a.all_warp ? 3 : 4;
  };
  for (;;) {
    const int todo = (prm->max_iterations - launched) < ICP_CHUNK ? (prm->max_iterations - launched) : ICP_CHUNK;
    for (int it = 0; it < todo; ++it) enqueue_iteration(A);
    launched += todo;
    LIOGPU_CUDA_OK(c, cudaGetLastError());
    LIOGPU_CUDA_OK(c, cudaMemcpyAsync(h, A.st, sizeof(IcpDevState), cudaMemcpyDeviceToHost, c->stream));
    LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
    if (h->done || launched >= prm->max_iterations) break;
  }
  // getFitnessScore
  IcpArgs F = A;
  F.fitness = 1;
  enqueue_iteration(F);
  LIOGPU_CUDA_OK(c, cudaGetLastError());
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(h, A.st, sizeof(IcpDevState), cudaMemcpyDeviceToHost, c->stream));
  LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1);
  icp_result(*h, c->last_ms, final_T, info);
  return LIOGPU_OK;
}

int icp_batch_dev(Ctx* c, const float4* src, const int* so, const float4* tgt, const int* to, int n,
                  const liogpu_icp_params* prm, float (*final_T)[16], liogpu_icp_info* info) {
  if (n <= 0) return LIOGPU_OK;
  const int ns = so[n], nt = to[n];
  std::vector<int> rp(n + 1, 0);
  for (int p = 0; p < n; ++p) rp[p + 1] = rp[p] + icp_reduce_blocks(so[p + 1] - so[p]);
  // device tables: sp | tp | rp | cell_base | gp | st | counters | partials
  auto up256 = [](size_t b) { return (b + 255) & ~(size_t)255; };
  const size_t o_tp = up256((size_t)(n + 1) * sizeof(int)), o_rp = o_tp + o_tp, o_cb = o_rp + o_tp;
  const size_t o_gp = o_cb + up256((size_t)n * sizeof(unsigned)), o_st = o_gp + up256((size_t)n * sizeof(GridParams));
  const size_t o_cnt = o_st + up256((size_t)n * sizeof(IcpDevState)), o_part = o_cnt + 256;
  LIOGPU_CUDA_OK(c, c->lc_tab.reserve(o_part + (size_t)rp[n] * ICP_SUMS * sizeof(double)));
  char* d = (char*)c->lc_tab.p;
  std::vector<char> h(o_part, 0);
  memcpy(h.data(), so, (size_t)(n + 1) * sizeof(int));
  memcpy(h.data() + o_tp, to, (size_t)(n + 1) * sizeof(int));
  memcpy(h.data() + o_rp, rp.data(), (size_t)(n + 1) * sizeof(int));
  IcpDevState* hs = reinterpret_cast<IcpDevState*>(h.data() + o_st);
  for (int p = 0; p < n; ++p) icp_state_init(hs[p], prm);
  reinterpret_cast<IcpbCounters*>(h.data() + o_cnt)->live = n;
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(d, h.data(), o_part, cudaMemcpyHostToDevice, c->stream));
  IcpbArgs A;
  A.src = src; A.tgt = tgt; A.n = n; A.ns = ns;
  A.sp = reinterpret_cast<const int*>(d); A.tp = reinterpret_cast<const int*>(d + o_tp);
  A.rp = reinterpret_cast<const int*>(d + o_rp);
  unsigned* d_cb = reinterpret_cast<unsigned*>(d + o_cb);
  A.cell_base = d_cb;
  GridParams* d_gp = reinterpret_cast<GridParams*>(d + o_gp);
  A.gp = d_gp;
  A.st = reinterpret_cast<IcpDevState*>(d + o_st);
  A.cnt = reinterpret_cast<IcpbCounters*>(d + o_cnt);
  A.partials = reinterpret_cast<double*>(d + o_part);

  // one segmented grid index over all targets.  The cell count per pair is capped so that the concatenated cells stay
  // within 2^28 (the grid's cell size never changes a result)
  const unsigned max_cells = (unsigned)((1u << 28) / (unsigned)n) < (1u << 25) ? (unsigned)((1u << 28) / (unsigned)n) : (1u << 25);
  icpb_grid_kernel<<<n, BB_THREADS, 0, c->stream>>>(tgt, A.tp, icp_cell_size(prm), max_cells, d_gp);
  c->launches++;
  LIOGPU_CUDA_OK(c, cudaGetLastError());
  std::vector<GridParams> hg(n);
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(hg.data(), d_gp, (size_t)n * sizeof(GridParams), cudaMemcpyDeviceToHost, c->stream));
  LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  std::vector<unsigned> cb(n);
  unsigned long long total_cells = 0;
  int n_valid = 0;
  for (int p = 0; p < n; ++p) {
    cb[p] = (unsigned)total_cells;
    total_cells += hg[p].n_cells;
    n_valid += hg[p].n_points;
  }
  if (total_cells > (1ull << 30)) { c->err = "icp batch: grid too large"; return LIOGPU_E_INVALID; }
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(d_cb, cb.data(), (size_t)n * sizeof(unsigned), cudaMemcpyHostToDevice, c->stream));
  LIOGPU_CUDA_OK(c, c->keys0.reserve((size_t)nt * 4));
  LIOGPU_CUDA_OK(c, c->keys1.reserve((size_t)nt * 4));
  LIOGPU_CUDA_OK(c, c->vals0.reserve((size_t)nt * 4));
  LIOGPU_CUDA_OK(c, c->vals1.reserve((size_t)nt * 4));
  LIOGPU_CUDA_OK(c, c->sor_sorted.reserve((size_t)nt * sizeof(float4)));
  LIOGPU_CUDA_OK(c, c->sor_cell_start.reserve((size_t)(total_cells + 2) * sizeof(uint32_t)));
  uint32_t* cell_start = c->sor_cell_start.as<uint32_t>();
  LIOGPU_CUDA_OK(c, cudaMemsetAsync(cell_start, 0, (size_t)(total_cells + 2) * sizeof(uint32_t), c->stream));
  icpb_key_kernel<<<div_up(nt, 256), 256, 0, c->stream>>>(tgt, nt, A.tp, n, d_gp, d_cb, (unsigned)total_cells,
                                                         c->keys0.as<uint32_t>(), cell_start);
  c->launches++;
  LIOGPU_CUDA_OK(c, exclusive_scan_u32(c, cell_start, cell_start, (int)total_cells + 1, nullptr));
  int bits = 0;
  while (bits < 32 && (total_cells >> bits) != 0ull) ++bits;
  uint32_t *skeys = nullptr, *sperm = nullptr;
  LIOGPU_CUDA_OK(c, radix_sort_pairs(c, nt, bits, nullptr, &skeys, &sperm));
  if (n_valid > 0) {
    icpb_gather_kernel<<<div_up(n_valid, 256), 256, 0, c->stream>>>(tgt, sperm, n_valid, A.tp, n, c->sor_sorted.as<float4>());
    c->launches++;
  }
  A.sorted = c->sor_sorted.as<float4>();
  A.cs = cell_start;

  LIOGPU_CUDA_OK(c, c->lm_a.reserve((size_t)ns * sizeof(float4)));
  LIOGPU_CUDA_OK(c, c->lm_flag.reserve((size_t)ns * sizeof(int)));
  LIOGPU_CUDA_OK(c, c->lm_md.reserve((size_t)ns * sizeof(float)));
  LIOGPU_CUDA_OK(c, c->lm_left.reserve((size_t)ns * sizeof(uint32_t)));
  A.cur = c->lm_a.as<float4>();
  A.nn_idx = c->lm_flag.as<int>(); A.nn_d2 = c->lm_md.as<float>();
  A.brute = c->lm_left.as<uint32_t>();
  A.fitness = 0;
  A.par = 0;
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(A.cur, src, (size_t)ns * sizeof(float4), cudaMemcpyDeviceToDevice, c->stream));
  int launched = 0;
  int* h_live = reinterpret_cast<int*>((char*)c->h_pinned + 12800);
  auto enqueue_iteration = [&](IcpbArgs& a) {
    icpb_nn_kernel<<<div_up(ns, NB_THREADS), NB_THREADS, 0, c->stream>>>(a);
    icpb_brute_kernel<<<c->sm_count, BRT, 0, c->stream>>>(a);
    icpb_reduce_kernel<<<rp[n], RD_THREADS, 0, c->stream>>>(a);
    c->launches += 3;
    a.par ^= 1;
  };
  for (;;) {
    const int todo = (prm->max_iterations - launched) < ICP_CHUNK ? (prm->max_iterations - launched) : ICP_CHUNK;
    for (int it = 0; it < todo; ++it) enqueue_iteration(A);
    launched += todo;
    LIOGPU_CUDA_OK(c, cudaGetLastError());
    LIOGPU_CUDA_OK(c, cudaMemcpyAsync(h_live, &A.cnt->live, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
    if (*h_live == 0 || launched >= prm->max_iterations) break;
  }
  A.fitness = 1;  // getFitnessScore
  enqueue_iteration(A);
  LIOGPU_CUDA_OK(c, cudaGetLastError());
  std::vector<IcpDevState> hst(n);
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(hst.data(), A.st, (size_t)n * sizeof(IcpDevState), cudaMemcpyDeviceToHost, c->stream));
  LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  for (int p = 0; p < n; ++p) icp_result(hst[p], 0.f, final_T[p], info + p);
  return LIOGPU_OK;
}

}  // namespace liogpu
