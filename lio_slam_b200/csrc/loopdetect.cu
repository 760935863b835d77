// loopdetect.cu — loop-closure detection on the device (SURVEY §8 row f3, detection half):
//   * SCManager::detectLoopClosureID (include/Scancontext.cpp) over a descriptor store kept in the context
//     (polarcontexts_ / polarcontext_invkeys_ / polarcontext_vkeys_, makeAndSaveScancontextAndKeys :228-243);
//   * detectLoopClosureDistance (mapOptmization.cpp ~1271-1300), the radius detector over the key poses.
//
// The reference rebuilds a nanoflann KD-tree over the ring keys every TREE_MAKING_PERIOD_ calls.  The store only grows,
// so that tree is a prefix of the stored keys: the host computes the prefix length of every call (the snapshot
// schedule, O(calls) integers) and the device searches the prefix exhaustively, which returns the tree's k nearest.
//
//   sc_store_kernel      block per added descriptor: ring key (-> f32, eig2stdvec), sector key (scancontext.cuh, the
//                        code of liogpu_make_scancontext) and the 60 column norms (shift-invariant: circshift moves
//                        whole columns) in the oracle's Eigen order.  For liogpu_sc_add_keyframes it first turns the
//                        u32 image that the binning left in the first half of the slot into the f64 descriptor
//                        (scancontext.cu's header)
//   sc_knn_chunk_kernel  block per (query, 1024 prefix keys): nanoflann L2_Adaptor<float> distances as 64-bit
//                        (d2 bits << 32 | index) keys, bitonic sort in shared memory, the k+1 smallest out
//   sc_knn_merge_kernel  block per query: merges its chunks' lists -> k candidates in (d2, index) order, ties counted
//                        (the (k+1)-th key detects a tie across the boundary)
//   sc_score_kernel      warp per (query, candidate), f64: fastAlignUsingVkey over the 60 shifts (lanes over shifts),
//                        then distDirectSC for the search window's shifts (lanes over columns, ordered column sum)
//   sc_final_kernel      thread per query: best candidate in kNN order, threshold, yaw
// The online call (liogpu_sc_detect_loop) is a batch of one query.
//
// The radius detector: loop_distance_kernel answers one call (thread per key pose, atomicMin of a (d2, index) key);
// loop_distance_batch_kernel answers many calls against one sorted-grid index of all key poses (warp per call).
#include "scancontext.cuh"

#include <algorithm>

#include <math_constants.h>

namespace liogpu {

namespace {

constexpr int KNN_CHUNK = 1024;     // prefix keys per block of the chunk kernel
constexpr int KNN_THREADS = 256;
constexpr int MERGE_BUF = 2048;     // entries the merge kernel sorts at a time
constexpr int SCORE_WARPS = 4;      // warps per block of the scoring kernel
constexpr size_t PART_BUDGET = (size_t)256 << 20;  // bytes of per-chunk partial lists per slice of queries
typedef unsigned long long u64;

// Eigen's linear-vectorised redux over 20 column entries (SSE2 doubles: partial sums of j = k mod 4, combined as
// (s0 + s2) + (s1 + s3)): the order DESIGN.md records for this [3P] arithmetic, not pinned against Eigen.
__device__ __forceinline__ double sc_col_sqnorm(const double* d, int c) {
  double s0 = d[c] * d[c], s1 = d[SC_SECTOR + c] * d[SC_SECTOR + c];
  double s2 = d[2 * SC_SECTOR + c] * d[2 * SC_SECTOR + c], s3 = d[3 * SC_SECTOR + c] * d[3 * SC_SECTOR + c];
  for (int r = 4; r < SC_RING; r += 4) {
    s0 += d[r * SC_SECTOR + c] * d[r * SC_SECTOR + c];
    s1 += d[(r + 1) * SC_SECTOR + c] * d[(r + 1) * SC_SECTOR + c];
    s2 += d[(r + 2) * SC_SECTOR + c] * d[(r + 2) * SC_SECTOR + c];
    s3 += d[(r + 3) * SC_SECTOR + c] * d[(r + 3) * SC_SECTOR + c];
  }
  return (s0 + s2) + (s1 + s3);
}

__device__ __forceinline__ float sc_ringkey_d2(const float* q, const float4* __restrict__ k) {  // nanoflann L2_Adaptor<float>
  float result = 0.f;
#pragma unroll
  for (int g = 0; g < SC_RING / 4; ++g) {
    const float4 b = k[g];
    const float d0 = q[4 * g] - b.x, d1 = q[4 * g + 1] - b.y, d2 = q[4 * g + 2] - b.z, d3 = q[4 * g + 3] - b.w;
    result += d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3;
  }
  return result;
}

// ascending bitonic sort of n (a power of two) keys in shared memory by the whole block
__device__ __forceinline__ void bitonic_sort(u64* s, int n) {
  for (int size = 2; size <= n; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      __syncthreads();
      for (int t = threadIdx.x; t < n / 2; t += blockDim.x) {
        const int i = 2 * t - (t & (stride - 1)), j = i + stride;
        const u64 a = s[i], b = s[j];
        if ((a > b) == ((i & size) == 0)) { s[i] = b; s[j] = a; }
      }
    }
  }
  __syncthreads();
}

template <bool FROM_IMAGE>
__global__ void __launch_bounds__(256)
sc_store_kernel(double* __restrict__ desc, float* __restrict__ rkey, double* __restrict__ vkey, double* __restrict__ cnorm) {
  __shared__ double d[SC_BINS];
  const size_t e = blockIdx.x;
  if (FROM_IMAGE) {
    const unsigned* img = reinterpret_cast<const unsigned*>(desc + e * SC_BINS);
    for (int k = threadIdx.x; k < SC_BINS; k += blockDim.x) d[k] = sc_bin_value(img[k]);
    __syncthreads();  // the doubles overwrite the image
    for (int k = threadIdx.x; k < SC_BINS; k += blockDim.x) desc[e * SC_BINS + k] = d[k];
  } else {
    for (int k = threadIdx.x; k < SC_BINS; k += blockDim.x) d[k] = desc[e * SC_BINS + k];
  }
  __syncthreads();
  const int k = threadIdx.x;
  if (k < SC_RING) {
    rkey[e * SC_RING + k] = (float)sc_key(d, k);
  } else if (k < SC_RING + SC_SECTOR) {
    vkey[e * SC_SECTOR + (k - SC_RING)] = sc_key(d, k);
  } else if (k < SC_RING + 2 * SC_SECTOR) {
    const int c = k - SC_RING - SC_SECTOR;
    cnorm[e * SC_SECTOR + c] = sqrt(sc_col_sqnorm(d, c));
  }
}

// qm[q] = (store index of the query, prefix length m).  Blocks past the query's prefix write nothing.
__global__ void __launch_bounds__(KNN_THREADS)
sc_knn_chunk_kernel(const float* __restrict__ rkey, const int2* __restrict__ qm, int n_chunks, int kk, u64* __restrict__ part) {
  __shared__ u64 s[KNN_CHUNK];
  __shared__ float qk[SC_RING];
  const int q = blockIdx.x;
  const int2 a = qm[q];
  const int base = blockIdx.y * KNN_CHUNK;
  if (base >= a.y) return;
  if (threadIdx.x < SC_RING) qk[threadIdx.x] = rkey[(size_t)a.x * SC_RING + threadIdx.x];
  __syncthreads();
  float qr[SC_RING];
#pragma unroll
  for (int r = 0; r < SC_RING; ++r) qr[r] = qk[r];
  for (int i = threadIdx.x; i < KNN_CHUNK; i += KNN_THREADS) {
    const int g = base + i;
    u64 key = ~0ULL;
    if (g < a.y) {
      const float d2 = sc_ringkey_d2(qr, reinterpret_cast<const float4*>(rkey + (size_t)g * SC_RING));
      key = ((u64)__float_as_uint(d2) << 32) | (unsigned)g;
    }
    s[i] = key;
  }
  bitonic_sort(s, KNN_CHUNK);
  for (int r = threadIdx.x; r < kk; r += KNN_THREADS) part[((size_t)q * n_chunks + blockIdx.y) * kk + r] = s[r];
}

// out[q].n_cand / .ties; cand / cd2 [q * k + j]
__global__ void __launch_bounds__(KNN_THREADS)
sc_knn_merge_kernel(const u64* __restrict__ part, const int2* __restrict__ qm, int n_chunks, int kk, int k,
                    int* __restrict__ cand, float* __restrict__ cd2, ScQueryOut* __restrict__ out) {
  __shared__ u64 s[MERGE_BUF];
  const int q = blockIdx.x;
  const int m = qm[q].y;
  const int nch = (m + KNN_CHUNK - 1) / KNN_CHUNK;
  const long long total = (long long)nch * kk;
  const u64* src = part + (size_t)q * n_chunks * kk;  // the query's chunks are contiguous
  for (int i = threadIdx.x; i < kk; i += KNN_THREADS) s[i] = ~0ULL;
  for (long long pos = 0; pos < total; pos += MERGE_BUF - kk) {
    __syncthreads();
    for (int i = kk + threadIdx.x; i < MERGE_BUF; i += KNN_THREADS) {
      const long long p = pos + (i - kk);
      s[i] = p < total ? src[p] : ~0ULL;
    }
    bitonic_sort(s, MERGE_BUF);
  }
  const int n_cand = min(k, m), L = min(kk, m);
  for (int j = threadIdx.x; j < n_cand; j += KNN_THREADS) {
    cand[(size_t)q * k + j] = (int)(unsigned)(s[j] & 0xffffffffULL);
    cd2[(size_t)q * k + j] = __uint_as_float((unsigned)(s[j] >> 32));
  }
  if (threadIdx.x == 0) {
    int ties = 0;
    for (int j = 1; j < L; ++j) ties += (s[j] >> 32) == (s[j - 1] >> 32);
    out[q].n_cand = n_cand;
    out[q].ties = ties;
  }
}

__global__ void __launch_bounds__(SCORE_WARPS * 32)
sc_score_kernel(const double* __restrict__ desc, const double* __restrict__ vkey, const double* __restrict__ cnorm,
                const int2* __restrict__ qm, const int* __restrict__ cand, const ScQueryOut* __restrict__ out, int nq, int k,
                int R, double* __restrict__ cdist, int* __restrict__ cshift) {
  __shared__ double sv[SCORE_WARPS][2][SC_SECTOR];
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long w = (long long)blockIdx.x * SCORE_WARPS + wib;
  const int q = (int)(w / k), j = (int)(w % k);
  if (q >= nq || j >= out[q].n_cand) return;  // warp-uniform
  const size_t qi = (size_t)qm[q].x, ci = (size_t)cand[(size_t)q * k + j];
  double* vq = sv[wib][0];
  double* vc = sv[wib][1];
  for (int t = lane; t < SC_SECTOR; t += 32) { vq[t] = vkey[qi * SC_SECTOR + t]; vc[t] = vkey[ci * SC_SECTOR + t]; }
  __syncwarp();
  // fastAlignUsingVkey: smallest shift with the strictly smallest norm (from 1e7); lanes over shifts
  double bn = CUDART_INF;
  int bs = 0;
  for (int s = lane; s < SC_SECTOR; s += 32) {
    double p[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) { const double d = vq[t] - vc[(t - s + SC_SECTOR) % SC_SECTOR]; p[t] = d * d; }
    for (int t = 4; t < SC_SECTOR; t += 4) {
#pragma unroll
      for (int u = 0; u < 4; ++u) { const double d = vq[t + u] - vc[(t + u - s + SC_SECTOR) % SC_SECTOR]; p[u] += d * d; }
    }
    double nrm = sqrt((p[0] + p[2]) + (p[1] + p[3]));
    if (!(nrm < 10000000.0)) nrm = CUDART_INF;
    if (nrm < bn || (nrm == bn && s < bs)) { bn = nrm; bs = s; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double on = __shfl_xor_sync(0xffffffffu, bn, o);
    const int os = __shfl_xor_sync(0xffffffffu, bs, o);
    if (on < bn || (on == bn && os < bs)) { bn = on; bs = os; }
  }
  const int align = isinf(bn) ? 0 : bs;
  // distDirectSC for the window {align, align +- 1..R} (distinct shifts; order is immaterial with the tie rule below)
  const double* dq = desc + qi * SC_BINS;
  const double* dc = desc + ci * SC_BINS;
  const int c0 = lane, c1 = lane + 32;
  const bool has1 = c1 < SC_SECTOR;
  double q0[SC_RING], q1[SC_RING];
#pragma unroll
  for (int r = 0; r < SC_RING; ++r) { q0[r] = dq[r * SC_SECTOR + c0]; q1[r] = has1 ? dq[r * SC_SECTOR + c1] : 0.0; }
  const double nq0 = cnorm[qi * SC_SECTOR + c0], nq1 = has1 ? cnorm[qi * SC_SECTOR + c1] : 0.0;
  const int W = min(2 * R + 1, SC_SECTOR);
  double best = 10000000.0;
  int best_s = 0;
  for (int wi = 0; wi < W; ++wi) {
    const int s = ((align - R + wi) % SC_SECTOR + SC_SECTOR) % SC_SECTOR;
    double sim0 = 0.0, sim1 = 0.0;
    bool ok0, ok1;
    {
      const int cc = (c0 - s + SC_SECTOR) % SC_SECTOR;
      const double nc = cnorm[ci * SC_SECTOR + cc];
      ok0 = !((nq0 == 0) | (nc == 0));
      if (ok0) {
        double p[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) p[u] = q0[u] * dc[u * SC_SECTOR + cc];
#pragma unroll
        for (int r = 4; r < SC_RING; r += 4)
#pragma unroll
          for (int u = 0; u < 4; ++u) p[u] += q0[r + u] * dc[(r + u) * SC_SECTOR + cc];
        sim0 = ((p[0] + p[2]) + (p[1] + p[3])) / (nq0 * nc);
      }
    }
    ok1 = false;
    if (has1) {
      const int cc = (c1 - s + SC_SECTOR) % SC_SECTOR;
      const double nc = cnorm[ci * SC_SECTOR + cc];
      ok1 = !((nq1 == 0) | (nc == 0));
      if (ok1) {
        double p[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) p[u] = q1[u] * dc[u * SC_SECTOR + cc];
#pragma unroll
        for (int r = 4; r < SC_RING; r += 4)
#pragma unroll
          for (int u = 0; u < 4; ++u) p[u] += q1[r + u] * dc[(r + u) * SC_SECTOR + cc];
        sim1 = ((p[0] + p[2]) + (p[1] + p[3])) / (nq1 * nc);
      }
    }
    // sum_sector_similarity in column order (every lane forms the same sum)
    const unsigned m0 = __ballot_sync(0xffffffffu, ok0), m1 = __ballot_sync(0xffffffffu, ok1);
    double sum = 0.0;
    int n_eff = 0;
#pragma unroll
    for (int l = 0; l < 32; ++l) {
      const double v = __shfl_sync(0xffffffffu, sim0, l);
      if ((m0 >> l) & 1u) { sum = sum + v; ++n_eff; }
    }
#pragma unroll
    for (int l = 0; l < SC_SECTOR - 32; ++l) {
      const double v = __shfl_sync(0xffffffffu, sim1, l);
      if ((m1 >> l) & 1u) { sum = sum + v; ++n_eff; }
    }
    const double dist = 1.0 - sum / n_eff;
    if (dist < best || (dist == best && s < best_s)) { best = dist; best_s = s; }
  }
  if (lane == 0) {
    cdist[(size_t)q * k + j] = best;
    cshift[(size_t)q * k + j] = best_s;
  }
}

__global__ void __launch_bounds__(128)
sc_final_kernel(const int* __restrict__ cand, const double* __restrict__ cdist, const int* __restrict__ cshift, int nq, int k,
                double thres, ScQueryOut* __restrict__ out) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nq) return;
  double min_dist = 10000000.0;
  int nn_align = 0, nn_idx = 0;
  const int n = out[q].n_cand;
  for (int j = 0; j < n; ++j) {
    const double d = cdist[(size_t)q * k + j];
    if (d < min_dist) { min_dist = d; nn_align = cshift[(size_t)q * k + j]; nn_idx = cand[(size_t)q * k + j]; }
  }
  out[q].min_dist = min_dist;
  out[q].nn_idx = nn_idx;
  out[q].nn_align = nn_align;
  out[q].loop_id = min_dist < thres ? nn_idx : -1;
  const float deg = (float)(nn_align * (360.0 / (double)SC_SECTOR));  // deg2rad(float) of Scancontext.cpp
  out[q].yaw = (float)((double)deg * 3.14159265358979323846 / 180.0);
}

// FLANN L2_Simple between the query key pose a and key pose b (nearby.cu: nb_d2).  Both radius detectors take their
// d2 from here, so the per-call and the batched answers cannot drift apart.
__device__ __forceinline__ float key_pose_d2(const float4 a, const float4 b) {
  float d2 = 0.f;
  float d = a.x - b.x; d2 += d * d;
  d = a.y - b.y;       d2 += d * d;
  d = a.z - b.z;       d2 += d * d;
  return d2;
}

__global__ void __launch_bounds__(256)
loop_distance_kernel(const float4* __restrict__ key3d, const double* __restrict__ key_time, int n, double time_cur, float r2,
                     double time_diff, u64* __restrict__ best) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float d2 = key_pose_d2(key3d[n - 1], key3d[i]);
  if (d2 < r2 && fabs(key_time[i] - time_cur) > time_diff) atomicMin(best, ((u64)__float_as_uint(d2) << 32) | (unsigned)i);
}

// key times in the order of the sorted index (the .w of a sorted entry is the key-pose index)
__global__ void __launch_bounds__(256)
loop_time_gather_kernel(const float4* __restrict__ sorted, const double* __restrict__ key_time, int n_valid,
                        double* __restrict__ time_sorted) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < n_valid) time_sorted[j] = key_time[__float_as_int(sorted[j].w)];
}

constexpr int LD_WARPS = 8;  // calls per block of the batched radius detector

// Warp per call j: the minimum (bits(d2) << 32 | i) over the key poses i < m = n_key_at[j] within the radius and old
// enough, i.e. loop_distance_kernel's answer on that prefix.  The minimum does not depend on the order in which the
// candidates are offered, so any cell walk and lane split give the same answer.  The cell range per axis comes from
// q +- (r + slack) as in grid_knn5 (s2m.cu), clamped in float before the conversion so that a huge or infinite radius
// scans the whole grid without overflow.  The stable sort keeps a cell's members in ascending key-pose index, so the
// walk of a cell stops at its first member >= m.
__global__ void __launch_bounds__(LD_WARPS * 32)
loop_distance_batch_kernel(const float4* __restrict__ key3d, const float4* __restrict__ sorted,
                           const double* __restrict__ time_sorted, const uint32_t* __restrict__ cell_start, const GridParams g,
                           const int* __restrict__ n_key_at, const double* __restrict__ time_cur, int n_calls, float radius,
                           float r2, double time_diff, int* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int j = blockIdx.x * LD_WARPS + (threadIdx.x >> 5);
  if (j >= n_calls) return;  // warp-uniform
  const int m = n_key_at[j];
  const float4 q = key3d[m - 1];
  const double tc = time_cur[j];
  u64 best = ~0ULL;
  // a non-finite query has d2 NaN or inf to every pose, never < r2: no candidate (and it is not in the grid)
  if (isfinite(q.x) && isfinite(q.y) && isfinite(q.z)) {
    const float reach = radius * 1.000001f + 2.0f * g.slack;
    const float qc[3] = {q.x, q.y, q.z}, o[3] = {g.ox, g.oy, g.oz};
    const int nc[3] = {g.nx, g.ny, g.nz};
    int lo[3], hi[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const float top = (float)(nc[a] - 1);
      lo[a] = (int)fminf(fmaxf(floorf((qc[a] - reach - o[a]) * g.inv_h), 0.f), top);
      hi[a] = (int)fminf(fmaxf(floorf((qc[a] + reach - o[a]) * g.inv_h), 0.f), top);
    }
    for (int z = lo[2]; z <= hi[2]; ++z)
      for (int y = lo[1]; y <= hi[1]; ++y) {
        const uint32_t row = ((uint32_t)z * (uint32_t)g.ny + (uint32_t)y) * (uint32_t)g.nx;
        for (int x = lo[0]; x <= hi[0]; ++x) {
          const uint32_t s = __ldg(cell_start + row + x), e = __ldg(cell_start + row + x + 1);
          for (uint32_t b = s; b < e; b += 32) {
            const uint32_t k = b + lane;
            bool past = false;
            if (k < e) {
              const float4 p = __ldg(sorted + k);
              const int i = __float_as_int(p.w);
              past = i >= m;
              if (!past) {
                const float d2 = key_pose_d2(q, p);
                if (d2 < r2 && fabs(__ldg(time_sorted + k) - tc) > time_diff) {
                  const u64 key = ((u64)__float_as_uint(d2) << 32) | (unsigned)i;
                  best = key < best ? key : best;
                }
              }
            }
            if (__any_sync(0xffffffffu, past)) break;  // the rest of the cell lies past the prefix
          }
        }
      }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    const u64 ob = __shfl_xor_sync(0xffffffffu, best, off);
    best = ob < best ? ob : best;
  }
  if (lane == 0) {
    const int w = best == ~0ULL ? -1 : (int)(unsigned)(best & 0xffffffffULL);
    out[j] = w == m - 1 ? -1 : w;
  }
}

cudaError_t sc_grow_array(Ctx* c, void** p, size_t old_bytes, size_t new_bytes) {
  void* np_ = nullptr;
  cudaError_t e = cudaMallocAsync(&np_, new_bytes, c->stream);
  if (e != cudaSuccess) return e;
  if (*p) {
    if (old_bytes) e = cudaMemcpyAsync(np_, *p, old_bytes, cudaMemcpyDeviceToDevice, c->stream);
    cudaFreeAsync(*p, c->stream);
  }
  *p = np_;
  return e;
}

// Room for `need` entries: geometric growth, contents carried over on the stream (stream-ordered: no device-wide sync).
int sc_reserve(Ctx* c, int need) {
  ScStore& st = c->sc;
  if (need <= st.cap) return LIOGPU_OK;
  int cap = st.cap > 0 ? st.cap : 1024;
  while (cap < need) cap = cap > (1 << 29) ? need : cap * 2;
  const size_t o = (size_t)st.count, nw = (size_t)cap;
  LIOGPU_CUDA_OK(c, sc_grow_array(c, (void**)&st.desc, o * SC_BINS * 8, nw * SC_BINS * 8));
  LIOGPU_CUDA_OK(c, sc_grow_array(c, (void**)&st.rkey, o * SC_RING * 4, nw * SC_RING * 4));
  LIOGPU_CUDA_OK(c, sc_grow_array(c, (void**)&st.vkey, o * SC_SECTOR * 8, nw * SC_SECTOR * 8));
  LIOGPU_CUDA_OK(c, sc_grow_array(c, (void**)&st.cnorm, o * SC_SECTOR * 8, nw * SC_SECTOR * 8));
  st.cap = cap;
  return LIOGPU_OK;
}

}  // namespace

// Appends n descriptors (host or device memory, row-major [ring][sector] f64) to the store and derives their keys.
int sc_add_dev(Ctx* c, const double* descs, int n) {
  ScStore& st = c->sc;
  const int need = st.count + n;
  int rc = sc_reserve(c, need);
  if (rc) return rc;
  const size_t e0 = (size_t)st.count;
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(st.desc + e0 * SC_BINS, descs, (size_t)n * SC_BINS * sizeof(double), cudaMemcpyDefault,
                                    c->stream));
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
  sc_store_kernel<false><<<n, 256, 0, c->stream>>>(st.desc + e0 * SC_BINS, st.rkey + e0 * SC_RING, st.vkey + e0 * SC_SECTOR,
                                                   st.cnorm + e0 * SC_SECTOR);
  c->launches++;
  LIOGPU_CUDA_OK(c, cudaGetLastError());
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
  LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1);
  st.count = need;
  return LIOGPU_OK;
}

// Points of a pass: the stage_keyframes tables address a pass's clouds with 32-bit offsets.  LIOGPU_SC_PASS_POINTS
// lowers the cap (tests use it to split small batches).
static long long sc_pass_points() {
  long long cap = 0x7fffffffLL;
  if (const char* e = getenv("LIOGPU_SC_PASS_POINTS")) {
    const long long v = atoll(e);
    if (v > 0 && v < cap) cap = v;
  }
  return cap;
}

// The new entries' slots hold the binning's u32 images until sc_store_kernel<true> replaces them with the doubles, so
// the batch needs no table memory of its own.  A pass takes consecutive keyframes up to sc_pass_points() points (a
// larger keyframe runs alone) and costs two launches (slot init, binning) and, before the next pass restages the
// tables, one sync; one store launch for all entries follows.  Up to 2^31 - 1 points in all: one pass.
int sc_add_keyframes_dev(Ctx* c, const int* ids, const std::vector<int>& n_pts, double lidar_height, double max_radius,
                         double* descs_out) {
  ScStore& st = c->sc;
  const int k = (int)n_pts.size();
  const long long cap = sc_pass_points();
  // pass p = keyframes [pass[p], pass[p + 1]); its block-offset table (relative to its first block, one entry past
  // its last keyframe) at tab[pass[p] + p ...]
  std::vector<int> pass{0}, tab;
  tab.reserve((size_t)k + 8);
  long long acc = 0, nb = 0;
  for (int f = 0; f < k; ++f) {
    if (f > pass.back() && acc + n_pts[f] > cap) {
      tab.push_back((int)nb);
      pass.push_back(f);
      acc = nb = 0;
    }
    acc += n_pts[f];
    tab.push_back((int)nb);
    nb += (n_pts[f] + (long long)SC_CHUNK - 1) / SC_CHUNK;  // < cap / SC_CHUNK + k per pass
  }
  tab.push_back((int)nb);
  pass.push_back(k);
  const int need = st.count + k;
  int rc = sc_reserve(c, need);
  if (rc) return rc;
  LIOGPU_CUDA_OK(c, c->sc_q.reserve(tab.size() * sizeof(int)));
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(c->sc_q.p, tab.data(), tab.size() * sizeof(int), cudaMemcpyHostToDevice, c->stream));
  const size_t e0 = (size_t)st.count;
  double* slots = st.desc + e0 * SC_BINS;
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
  for (int p = 0; p + 1 < (int)pass.size(); ++p) {
    const int f0 = pass[p], kp = pass[p + 1] - f0;
    if (p > 0) LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));  // the previous pass's tables were uploaded
    KfTables t{};
    rc = stage_keyframes(c, "liogpu_sc_add_keyframes", ids + f0, nullptr, kp, t);
    if (rc) return rc;
    LIOGPU_CUDA_OK(c, launch_sc_bin_keyframes(c, t.srcs, t.offs, c->sc_q.as<int>() + f0 + p, kp, tab[f0 + p + kp],
                                              lidar_height, max_radius, slots + (size_t)f0 * SC_BINS));
  }
  sc_store_kernel<true><<<k, 256, 0, c->stream>>>(slots, st.rkey + e0 * SC_RING, st.vkey + e0 * SC_SECTOR,
                                                  st.cnorm + e0 * SC_SECTOR);
  c->launches++;
  LIOGPU_CUDA_OK(c, cudaGetLastError());
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
  st.count = need;
  if (descs_out)
    LIOGPU_CUDA_OK(c, cudaMemcpyAsync(descs_out, slots, (size_t)k * SC_BINS * sizeof(double), cudaMemcpyDefault, c->stream));
  LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1);
  return LIOGPU_OK;
}

void sc_release(Ctx* c) {
  ScStore& st = c->sc;
  void* arrays[] = {st.desc, st.rkey, st.vkey, st.cnorm};
  for (void* p : arrays)
    if (p) cudaFreeAsync(p, c->stream);
  st = ScStore();
}

// The queries qm[q] = (store index, prefix length >= 1) with num_candidates = k: results per query in h_out (host).
// With info != NULL (one query) its candidate lists are copied out as well.
int sc_detect_dev(Ctx* c, const std::vector<int2>& qm, int k, int R, double thres, ScQueryOut* h_out, liogpu_sc_info* info) {
  const int nq = (int)qm.size();
  const int kk = k + 1;
  int max_m = 1;
  for (const int2& a : qm) max_m = a.y > max_m ? a.y : max_m;
  const int n_chunks = div_up(max_m, KNN_CHUNK);
  const size_t per_q = (size_t)n_chunks * kk * sizeof(u64);
  const int slice = (int)std::max<size_t>(1, std::min<size_t>((size_t)nq, PART_BUDGET / per_q));
  const size_t nk = (size_t)nq * k;
  LIOGPU_CUDA_OK(c, c->sc_q.reserve((size_t)nq * sizeof(int2)));
  LIOGPU_CUDA_OK(c, c->sc_out.reserve((size_t)nq * sizeof(ScQueryOut)));
  LIOGPU_CUDA_OK(c, c->sc_cand.reserve(nk * (8 + 4 + 4 + 4)));
  LIOGPU_CUDA_OK(c, c->sc_part.reserve((size_t)slice * per_q));
  int2* d_qm = c->sc_q.as<int2>();
  ScQueryOut* d_out = c->sc_out.as<ScQueryOut>();
  double* d_cdist = c->sc_cand.as<double>();
  int* d_cand = reinterpret_cast<int*>(d_cdist + nk);
  float* d_cd2 = reinterpret_cast<float*>(d_cand + nk);
  int* d_cshift = reinterpret_cast<int*>(d_cd2 + nk);
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(d_qm, qm.data(), (size_t)nq * sizeof(int2), cudaMemcpyHostToDevice, c->stream));
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
  for (int q0 = 0; q0 < nq; q0 += slice) {
    const int ns = std::min(slice, nq - q0);
    sc_knn_chunk_kernel<<<dim3(ns, n_chunks), KNN_THREADS, 0, c->stream>>>(c->sc.rkey, d_qm + q0, n_chunks, kk,
                                                                           c->sc_part.as<u64>());
    sc_knn_merge_kernel<<<ns, KNN_THREADS, 0, c->stream>>>(c->sc_part.as<u64>(), d_qm + q0, n_chunks, kk, k,
                                                           d_cand + (size_t)q0 * k, d_cd2 + (size_t)q0 * k, d_out + q0);
    c->launches += 2;
  }
  sc_score_kernel<<<div_up((long long)nq * k, SCORE_WARPS), SCORE_WARPS * 32, 0, c->stream>>>(
      c->sc.desc, c->sc.vkey, c->sc.cnorm, d_qm, d_cand, d_out, nq, k, R, d_cdist, d_cshift);
  sc_final_kernel<<<div_up(nq, 128), 128, 0, c->stream>>>(d_cand, d_cdist, d_cshift, nq, k, thres, d_out);
  c->launches += 2;
  LIOGPU_CUDA_OK(c, cudaGetLastError());
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(h_out, d_out, (size_t)nq * sizeof(ScQueryOut), cudaMemcpyDeviceToHost, c->stream));
  char* h = (char*)c->h_pinned + 32768;  // candidate lists of an online call (k <= 32: 640 bytes)
  if (info) {
    LIOGPU_CUDA_OK(c, cudaMemcpyAsync(h, d_cdist, k * 8, cudaMemcpyDeviceToHost, c->stream));
    LIOGPU_CUDA_OK(c, cudaMemcpyAsync(h + 256, d_cand, k * 4, cudaMemcpyDeviceToHost, c->stream));
    LIOGPU_CUDA_OK(c, cudaMemcpyAsync(h + 384, d_cd2, k * 4, cudaMemcpyDeviceToHost, c->stream));
    LIOGPU_CUDA_OK(c, cudaMemcpyAsync(h + 512, d_cshift, k * 4, cudaMemcpyDeviceToHost, c->stream));
  }
  LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1);
  if (info) {
    const int n = h_out[0].n_cand;
    memcpy(info->candidate_dist, h, n * 8);
    memcpy(info->candidates, h + 256, n * 4);
    memcpy(info->candidate_key_d2, h + 384, n * 4);
    memcpy(info->candidate_shift, h + 512, n * 4);
  }
  return LIOGPU_OK;
}

// key3d: device, packed float4; h_times: host.  *loop_key_pre = the winner or -1.
int detect_loop_distance_dev(Ctx* c, const float4* key3d, int n, const double* h_times, double time_cur, float radius,
                             float time_diff, int* loop_key_pre) {
  LIOGPU_CUDA_OK(c, c->lm_md.reserve((size_t)n * sizeof(double)));
  LIOGPU_CUDA_OK(c, c->lm_stats.reserve(4096));
  u64* d_best = reinterpret_cast<u64*>((char*)c->lm_stats.p + 1024);
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(c->lm_md.p, h_times, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
  LIOGPU_CUDA_OK(c, cudaMemsetAsync(d_best, 0xff, sizeof(u64), c->stream));
  const float r2 = (float)((double)radius * (double)radius);  // pcl::KdTreeFLANN::radiusSearch narrows radius^2 to f32
  loop_distance_kernel<<<div_up(n, 256), 256, 0, c->stream>>>(key3d, c->lm_md.as<double>(), n, time_cur, r2,
                                                              (double)time_diff, d_best);
  c->launches++;
  LIOGPU_CUDA_OK(c, cudaGetLastError());
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
  u64* h = reinterpret_cast<u64*>((char*)c->h_pinned + 36864);
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(h, d_best, sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
  LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1);
  const int best = *h == ~0ULL ? -1 : (int)(unsigned)(*h & 0xffffffffULL);
  *loop_key_pre = best == n - 1 ? -1 : best;
  return LIOGPU_OK;
}

// One sorted-grid index over all n key poses (cell edge = radius, doubled by grid_setup_compute while the grid is over
// its cap), then every call answered against it by loop_distance_batch_kernel.  The index goes to sor_setup /
// sor_sorted / sor_cell_start, the per-call scratch of the secondary grids: the registration's local map and index are
// not touched.  Launches do not depend on n_calls; one sync inside grid_build_core, one for the answers.  The caller
// records ev0 before it uploads the key poses, so that liogpu_last_gpu_ms covers the whole call.
int detect_loops_distance_dev(Ctx* c, const float4* key3d, int n, const double* h_times, const int* n_key_at,
                              const double* time_cur, int n_calls, float radius, float time_diff, int* loop_key_pre) {
  // ld_tab: time_cur [n_calls] f64 | key times [n] f64 | key times in index order [n] f64 | n_key_at [n_calls] i32 |
  // answers [n_calls] i32
  const size_t nc = (size_t)n_calls, nk = (size_t)n;
  LIOGPU_CUDA_OK(c, c->ld_tab.reserve((nc + 2 * nk) * sizeof(double) + 2 * nc * sizeof(int)));
  double* d_tcur = c->ld_tab.as<double>();
  double* d_time = d_tcur + nc;
  double* d_time_sorted = d_time + nk;
  int* d_m = reinterpret_cast<int*>(d_time_sorted + nk);
  int* d_out = d_m + nc;
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(d_tcur, time_cur, nc * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(d_time, h_times, nk * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(d_m, n_key_at, nc * sizeof(int), cudaMemcpyHostToDevice, c->stream));
  GridParams g{};
  int rc = grid_build_core(c, key3d, n, radius, 1.0f, 1.0f, c->sor_setup, c->sor_sorted, c->sor_cell_start, g);
  if (rc) return rc;
  if (g.n_points <= 0) {  // no finite key pose: no call has a candidate
    std::fill(loop_key_pre, loop_key_pre + n_calls, -1);
    LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
    LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
    cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1);
    return LIOGPU_OK;
  }
  const float4* sorted = c->sor_sorted.as<float4>();
  loop_time_gather_kernel<<<div_up(g.n_points, 256), 256, 0, c->stream>>>(sorted, d_time, g.n_points, d_time_sorted);
  const float r2 = (float)((double)radius * (double)radius);  // as detect_loop_distance_dev
  loop_distance_batch_kernel<<<div_up(n_calls, LD_WARPS), LD_WARPS * 32, 0, c->stream>>>(
      key3d, sorted, d_time_sorted, c->sor_cell_start.as<uint32_t>(), g, d_m, d_tcur, n_calls, radius, r2,
      (double)time_diff, d_out);
  c->launches += 2;
  LIOGPU_CUDA_OK(c, cudaGetLastError());
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(loop_key_pre, d_out, nc * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1);
  return LIOGPU_OK;
}

}  // namespace liogpu
