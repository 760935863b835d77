// voxel.cu — sort-based replacement of pcl::VoxelGrid<PointXYZI>::filter as called by liorf at
// mapOptmization.cpp:1536 (key poses), :1582 (local map, leaf surroundingKeyframeMapLeafSize) and
// :1609 (current scan, leaf mappingSurfLeafSize).  Semantics: SURVEY.md Appendix A.1 —
//   min/max (f32, non-finite skipped) -> overflow guard -> int32 voxel index per point -> stable sort
//   by index -> per voxel SEQUENTIAL f32 sums of x,y,z,intensity in ascending input order -> /n.
//
// Kernels (all HBM-bound streaming passes; float4 = one 16-byte coalesced load per point):
//   vox_minmax_kernel   16n B read;  grid = multiple of the SM count, block reduce + ordered-int atomics
//   vox_setup_kernel    1 thread: steps 2-4 of A.1 on device
//   vox_key_kernel      16n read, 4n write
//   radix sort          (sort.cu)  ~3 x 20n per 8-bit pass
//   vox_head_kernel     8n read/write (segment head flags) + exclusive scan
//   vox_segstart_kernel scatter segment starts
//   vox_centroid_kernel one thread per voxel, members gathered through the sorted permutation
#include "common.cuh"
#include <stdlib.h>

namespace liogpu {

__device__ __forceinline__ unsigned f2ord(float f) {
  const unsigned u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(unsigned o) {
  const unsigned u = (o & 0x80000000u) ? (o & 0x7fffffffu) : ~o;
  return __uint_as_float(u);
}
__device__ __forceinline__ bool finite3(const float4 p) { return isfinite(p.x) && isfinite(p.y) && isfinite(p.z); }

// mm[0..2] = min (ordered uint), mm[3..5] = max, mm[6] = finite count
__global__ void vox_minmax_init_kernel(unsigned* mm) {
  if (threadIdx.x < 3) mm[threadIdx.x] = 0xffffffffu;
  else if (threadIdx.x < 6) mm[threadIdx.x] = 0u;
  else if (threadIdx.x == 6) mm[6] = 0u;
}

__global__ void __launch_bounds__(256)
vox_minmax_kernel(const float4* __restrict__ pts, int n, unsigned* __restrict__ mm) {
  float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
  unsigned cnt = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 p = pts[i];
    if (finite3(p)) {
      mn[0] = fminf(mn[0], p.x); mn[1] = fminf(mn[1], p.y); mn[2] = fminf(mn[2], p.z);
      mx[0] = fmaxf(mx[0], p.x); mx[1] = fmaxf(mx[1], p.y); mx[2] = fmaxf(mx[2], p.z);
      ++cnt;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      mn[a] = fminf(mn[a], __shfl_xor_sync(0xffffffffu, mn[a], o));
      mx[a] = fmaxf(mx[a], __shfl_xor_sync(0xffffffffu, mx[a], o));
    }
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  }
  __shared__ float smn[8][3], smx[8][3];
  __shared__ unsigned scnt[8];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) {
#pragma unroll
    for (int a = 0; a < 3; ++a) { smn[w][a] = mn[a]; smx[w][a] = mx[a]; }
    scnt[w] = cnt;
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    const int a = threadIdx.x;
    float lo = smn[0][a], hi = smx[0][a];
    for (int k = 1; k < 8; ++k) { lo = fminf(lo, smn[k][a]); hi = fmaxf(hi, smx[k][a]); }
    atomicMin(&mm[a], f2ord(lo));
    atomicMax(&mm[3 + a], f2ord(hi));
  } else if (threadIdx.x == 3) {
    unsigned c = 0;
    for (int k = 0; k < 8; ++k) c += scnt[k];
    atomicAdd(&mm[6], c);
  }
}

// A.1 steps 2-4 from the f32 bounding box and the finite count
__device__ __forceinline__ void vox_setup_compute(const float mn[3], const float mx[3], int n_valid, float leaf,
                                                  VoxelSetup& v) {
  v.n_valid = n_valid;
  const float inv = 1.0f / leaf;
  v.inv_leaf = inv;
  long long d[3];
  for (int a = 0; a < 3; ++a) {
    v.min_p[a] = mn[a];
    v.max_p[a] = mx[a];
    d[a] = (long long)((v.max_p[a] - v.min_p[a]) * inv) + 1;  // A.1 step 3
  }
  v.overflow = (v.n_valid > 0 && d[0] * d[1] * d[2] > 2147483647LL) ? 1 : 0;
  for (int a = 0; a < 3; ++a) {
    v.min_b[a] = (int)floorf(v.min_p[a] * inv);
    const int max_b = (int)floorf(v.max_p[a] * inv);
    v.div_b[a] = max_b - v.min_b[a] + 1;
  }
  v.mul1 = v.div_b[0];
  v.mul2 = v.div_b[0] * v.div_b[1];
  v.n_cells = 0;
  v.key_bits = 0;
  v.n_vox = 0;
  if (!v.overflow && v.n_valid > 0) {
    v.n_cells = (unsigned)v.div_b[0] * (unsigned)v.div_b[1] * (unsigned)v.div_b[2];
    // keys live in [0, n_cells]; n_cells itself marks non-finite points (sorted last, then dropped)
    const unsigned maxkey = v.n_cells;
    int b = 0;
    while (b < 32 && (maxkey >> b) != 0u) ++b;
    v.key_bits = b;
  }
}

__global__ void vox_setup_kernel(const unsigned* __restrict__ mm, float leaf, VoxelSetup* __restrict__ s) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  VoxelSetup v;
  float mn[3], mx[3];
  for (int a = 0; a < 3; ++a) { mn[a] = ord2f(mm[a]); mx[a] = ord2f(mm[3 + a]); }
  vox_setup_compute(mn, mx, (int)mm[6], leaf, v);
  *s = v;
}

__device__ __forceinline__ uint32_t vox_key_of(const float4 p, const VoxelSetup& s) {
  if (!finite3(p)) return s.n_cells;
  const int ix = (int)(floorf(p.x * s.inv_leaf) - (float)s.min_b[0]);  // A.1 step 5
  const int iy = (int)(floorf(p.y * s.inv_leaf) - (float)s.min_b[1]);
  const int iz = (int)(floorf(p.z * s.inv_leaf) - (float)s.min_b[2]);
  return (uint32_t)(ix + iy * s.mul1 + iz * s.mul2);
}

__global__ void __launch_bounds__(256)
vox_key_kernel(const float4* __restrict__ pts, int n, const VoxelSetup* __restrict__ sp, uint32_t* __restrict__ keys) {
  __shared__ VoxelSetup s;
  if (threadIdx.x == 0) s = *sp;
  __syncthreads();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  keys[i] = vox_key_of(pts[i], s);
}

// head[i] = 1 at the first sorted position of every occupied voxel (finite points only), else 0
__global__ void __launch_bounds__(256)
vox_head_kernel(const uint32_t* __restrict__ keys, int n, const VoxelSetup* __restrict__ sp, uint32_t* __restrict__ head) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int n_valid = sp->overflow ? 0 : sp->n_valid;
  head[i] = (i < n_valid && (i == 0 || keys[i] != keys[i - 1])) ? 1u : 0u;
}

// seg_start[v] = first sorted position of voxel v; seg_start[n_vox] = n_valid
__global__ void __launch_bounds__(256)
vox_segstart_kernel(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ rank, int n,
                    VoxelSetup* __restrict__ sp, uint32_t* __restrict__ seg_start, const uint32_t* __restrict__ n_vox) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int n_valid = sp->overflow ? 0 : sp->n_valid;
  if (i == 0) { seg_start[*n_vox] = (uint32_t)n_valid; sp->n_vox = *n_vox; }
  if (i >= n_valid) return;
  if (i == 0 || keys[i] != keys[i - 1]) seg_start[rank[i]] = (uint32_t)i;
}

// Per-voxel centroid: SEQUENTIAL f32 sums in ascending input index (the sort is stable), true division by
// (float)n — bit-identical to the canonical VoxelGrid (A.1 step 7).  The additions of one voxel cannot be
// reordered, but the LOADS can.
//   vox_centroid_kernel       one thread per voxel; a voxel with <= 8 members is finished here (all member
//                             loads issued before the adds); a longer one is appended to `long_list`.
//   vox_centroid_long_kernel  persistent warps, one long voxel at a time (dynamic: the sizes are heavy
//                             tailed — thousands of members near the sensor when 50 keyframes overlap): the
//                             warp gathers 128 members per step (next step prefetched), stages them in
//                             shared memory, and four lanes — one per component x, y, z, intensity — run the
//                             sequential sums from there (~5 cycles per member instead of one L2 round trip).
constexpr unsigned VOX_SHORT = 8;
constexpr int VOX_LONG_K = 4;                    // 32-member loads per lane and step
constexpr int VOX_LONG_CHUNK = 32 * VOX_LONG_K;  // 128 members per step
constexpr int VOX_LONG_WARPS = 4;

__global__ void __launch_bounds__(256)
vox_centroid_kernel(const float4* __restrict__ pts, const uint32_t* __restrict__ perm,
                    const uint32_t* __restrict__ seg_start, const uint32_t* __restrict__ n_vox_p,
                    float4* __restrict__ out, uint32_t* __restrict__ long_list, uint32_t* __restrict__ long_count) {
  const unsigned nv = *n_vox_p;
  const unsigned v = blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned lane = threadIdx.x & 31;
  if ((v & ~31u) >= nv) return;  // whole warp beyond the last voxel
  uint32_t s = 0, e = 0;
  if (v < nv) { s = seg_start[v]; e = seg_start[v + 1]; }
  const uint32_t cnt = e - s;
  const bool is_long = v < nv && cnt > VOX_SHORT;
  if (v < nv && !is_long) {
    float4 p[VOX_SHORT];
#pragma unroll
    for (unsigned k = 0; k < VOX_SHORT; ++k) p[k] = pts[perm[s + (k < cnt ? k : 0)]];
    float sx = 0.f, sy = 0.f, sz = 0.f, si = 0.f;
#pragma unroll
    for (unsigned k = 0; k < VOX_SHORT; ++k)
      if (k < cnt) { sx += p[k].x; sy += p[k].y; sz += p[k].z; si += p[k].w; }
    const float c = (float)cnt;
    out[v] = make_float4(sx / c, sy / c, sz / c, si / c);
  }
  const unsigned lm = __ballot_sync(0xffffffffu, is_long);
  if (lm) {  // one atomic per warp reserves slots for its long voxels (order in the list is irrelevant)
    uint32_t base = 0;
    if (lane == 0) base = atomicAdd(long_count, (uint32_t)__popc(lm));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (is_long) long_list[base + __popc(lm & ((1u << lane) - 1u))] = v;
  }
}

__global__ void __launch_bounds__(32 * VOX_LONG_WARPS)
vox_centroid_long_kernel(const float4* __restrict__ pts, const uint32_t* __restrict__ perm,
                         const uint32_t* __restrict__ seg_start, const uint32_t* __restrict__ long_list,
                         const uint32_t* __restrict__ long_count, uint32_t* __restrict__ work_counter,
                         float4* __restrict__ out) {
  __shared__ float4 stage[VOX_LONG_WARPS][VOX_LONG_CHUNK];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t total = *long_count;
  float4* st = stage[warp];
  for (;;) {
    uint32_t item = 0;
    if (lane == 0) item = atomicAdd(work_counter, 1u);
    item = __shfl_sync(0xffffffffu, item, 0);
    if (item >= total) break;
    const uint32_t v = long_list[item];
    const uint32_t s = seg_start[v], e = seg_start[v + 1];
    float4 cur[VOX_LONG_K], nxt[VOX_LONG_K];
#pragma unroll
    for (int k = 0; k < VOX_LONG_K; ++k) {
      const uint32_t j = s + k * 32 + lane;
      cur[k] = j < e ? pts[perm[j]] : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    float acc = 0.f;  // lane c < 4 accumulates component c
    for (uint32_t base = s; base < e; base += VOX_LONG_CHUNK) {
      const uint32_t nb = base + VOX_LONG_CHUNK;
#pragma unroll
      for (int k = 0; k < VOX_LONG_K; ++k) {  // prefetch the next step while this one is consumed
        const uint32_t j = nb + k * 32 + lane;
        nxt[k] = j < e ? pts[perm[j]] : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int k = 0; k < VOX_LONG_K; ++k) st[k * 32 + lane] = cur[k];
      __syncwarp();
      if (lane < 4) {
        const int m = (int)min((uint32_t)VOX_LONG_CHUNK, e - base);
        const float* f = reinterpret_cast<const float*>(st) + lane;
#pragma unroll 8
        for (int i = 0; i < m; ++i) acc += f[4 * i];
      }
      __syncwarp();
#pragma unroll
      for (int k = 0; k < VOX_LONG_K; ++k) cur[k] = nxt[k];
    }
    const float c = (float)(e - s);
    const float r = acc / c;
    const float rx = __shfl_sync(0xffffffffu, r, 0), ry = __shfl_sync(0xffffffffu, r, 1);
    const float rz = __shfl_sync(0xffffffffu, r, 2), ri = __shfl_sync(0xffffffffu, r, 3);
    if (lane == 0) out[v] = make_float4(rx, ry, rz, ri);
  }
}

// ---- small clouds (the key-pose filter downSizeFilterSurroundingKeyPoses, MO:1535-1536, runs on a few hundred
// poses every scan): the whole filter in ONE block — bounding box, keys, a shared-memory sort of (key, input
// index) pairs (the index makes the order of equal keys the input order), head flags + scan, per-voxel sequential
// sums.  Same arithmetic as the multi-kernel pipeline, one launch instead of twenty.
constexpr int VS_MAX = 2048;
constexpr int VS_THREADS = 1024;
__global__ void __launch_bounds__(VS_THREADS)
vox_small_kernel(const float4* __restrict__ pts, int n, float leaf, VoxelSetup* __restrict__ sp, float4* __restrict__ out) {
  __shared__ unsigned long long comp[VS_MAX];
  __shared__ uint32_t seg[VS_MAX + 1];
  __shared__ float smn[VS_THREADS / 32][3], smx[VS_THREADS / 32][3];
  __shared__ uint32_t swsum[VS_THREADS / 32];
  __shared__ VoxelSetup s;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  // bounding box of the finite points
  float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
  unsigned cnt = 0;
  for (int i = tid; i < n; i += VS_THREADS) {
    const float4 p = pts[i];
    if (finite3(p)) {
      mn[0] = fminf(mn[0], p.x); mn[1] = fminf(mn[1], p.y); mn[2] = fminf(mn[2], p.z);
      mx[0] = fmaxf(mx[0], p.x); mx[1] = fmaxf(mx[1], p.y); mx[2] = fmaxf(mx[2], p.z);
      ++cnt;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      mn[a] = fminf(mn[a], __shfl_xor_sync(0xffffffffu, mn[a], o));
      mx[a] = fmaxf(mx[a], __shfl_xor_sync(0xffffffffu, mx[a], o));
    }
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  }
  if (lane == 0) {
#pragma unroll
    for (int a = 0; a < 3; ++a) { smn[w][a] = mn[a]; smx[w][a] = mx[a]; }
    swsum[w] = cnt;
  }
  __syncthreads();
  if (tid == 0) {
    unsigned total = 0;
    for (int k = 0; k < VS_THREADS / 32; ++k) {
      total += swsum[k];
      for (int a = 0; a < 3; ++a) { mn[a] = fminf(mn[a], smn[k][a]); mx[a] = fmaxf(mx[a], smx[k][a]); }
    }
    if (total == 0) {  // same encoding the ordered-uint path decodes for an all-non-finite cloud
      for (int a = 0; a < 3; ++a) { mn[a] = ord2f(0xffffffffu); mx[a] = ord2f(0u); }
    }
    VoxelSetup v;
    vox_setup_compute(mn, mx, (int)total, leaf, v);
    s = v;
  }
  __syncthreads();
  if (s.overflow || s.n_valid == 0) {
    if (tid == 0) *sp = s;
    return;
  }
  int m = 2;
  while (m < n) m <<= 1;  // sort size: next power of two
  for (int i = tid; i < m; i += VS_THREADS)
    comp[i] = i < n ? (((unsigned long long)vox_key_of(pts[i], s) << 32) | (unsigned)i) : ~0ULL;
  for (int k = 2; k <= m; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      __syncthreads();
      for (int i = tid; i < m; i += VS_THREADS) {
        const int p = i ^ j;
        if (p > i) {
          const unsigned long long a = comp[i], b = comp[p];
          const bool up = (i & k) == 0;
          if ((a > b) == up) { comp[i] = b; comp[p] = a; }
        }
      }
    }
  }
  __syncthreads();
  // head flags of the occupied voxels (finite points occupy the first n_valid sorted positions) + exclusive scan;
  // thread t owns positions 2t and 2t+1
  const int n_valid = s.n_valid;
  uint32_t h0 = 0, h1 = 0;
  {
    const int i0 = 2 * tid, i1 = 2 * tid + 1;
    if (i0 < n_valid) h0 = (i0 == 0 || (uint32_t)(comp[i0] >> 32) != (uint32_t)(comp[i0 - 1] >> 32)) ? 1u : 0u;
    if (i1 < n_valid) h1 = ((uint32_t)(comp[i1] >> 32) != (uint32_t)(comp[i1 - 1] >> 32)) ? 1u : 0u;
  }
  uint32_t x = h0 + h1;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) swsum[w] = x;
  __syncthreads();
  uint32_t wb = 0, total_vox = 0;
  for (int k = 0; k < VS_THREADS / 32; ++k) {
    if (k < w) wb += swsum[k];
    total_vox += swsum[k];
  }
  const uint32_t r0 = wb + x - (h0 + h1);
  if (h0) seg[r0] = 2 * tid;
  if (h1) seg[r0 + h0] = 2 * tid + 1;
  if (tid == 0) seg[total_vox] = (uint32_t)n_valid;
  __syncthreads();
  for (uint32_t v = tid; v < total_vox; v += VS_THREADS) {
    const uint32_t b = seg[v], e = seg[v + 1];
    float sx = 0.f, sy = 0.f, sz = 0.f, si = 0.f;
    for (uint32_t t = b; t < e; ++t) {  // ascending input index: sequential f32 sums (A.1 step 7)
      const float4 p = pts[(uint32_t)comp[t]];
      sx += p.x; sy += p.y; sz += p.z; si += p.w;
    }
    const float c = (float)(e - b);
    out[v] = make_float4(sx / c, sy / c, sz / c, si / c);
  }
  if (tid == 0) {
    s.n_vox = total_vox;
    *sp = s;
  }
}

// f32 min/max + finite count of a cloud into mm[7] (ordered-uint encoding); shared with grid.cu
cudaError_t launch_minmax(Ctx* c, const float4* pts, int n, unsigned* mm) {
  vox_minmax_init_kernel<<<1, 32, 0, c->stream>>>(mm);
  int grid = div_up(n, 256);
  const int cap = c->sm_count * 8;
  if (grid > cap) grid = cap;
  if (grid < 1) grid = 1;
  vox_minmax_kernel<<<grid, 256, 0, c->stream>>>(pts, n, mm);
  c->launches += 2;
  return cudaGetLastError();
}

// Device-resident VoxelGrid: in (n float4) -> out (n_out float4).  Everything is enqueued without waiting
// for the host: the key width, the finite count and the overflow flag stay on the device (the radix sort
// runs a fixed four passes, the unneeded ones degrade to a copy); ONE read-back at the end returns the voxel
// count and the guard flag.
int voxel_downsample_dev(Ctx* c, const float4* in, int n, float leaf, DevBuf& out, int* n_out, bool* overflow) {
  *n_out = 0;
  *overflow = false;
  if (n <= 0) return LIOGPU_OK;
  if (!(leaf > 0.f)) { c->err = "voxel leaf must be > 0"; return LIOGPU_E_INVALID; }
  LIOGPU_CUDA_OK(c, c->minmax.reserve(64));
  LIOGPU_CUDA_OK(c, c->vox_setup.reserve(sizeof(VoxelSetup)));
  LIOGPU_CUDA_OK(c, c->keys0.reserve((size_t)n * 4));
  LIOGPU_CUDA_OK(c, c->keys1.reserve((size_t)n * 4));
  LIOGPU_CUDA_OK(c, c->vals0.reserve((size_t)n * 4));
  LIOGPU_CUDA_OK(c, c->vals1.reserve((size_t)n * 4));
  LIOGPU_CUDA_OK(c, c->seg_flag.reserve((size_t)n * 4 + 16));
  LIOGPU_CUDA_OK(c, c->seg_start.reserve((size_t)n * 4 + 16));
  LIOGPU_CUDA_OK(c, c->misc.reserve(256));
  LIOGPU_CUDA_OK(c, out.reserve((size_t)n * sizeof(float4)));
  unsigned* mm = c->minmax.as<unsigned>();
  VoxelSetup* d_setup = c->vox_setup.as<VoxelSetup>();
  VoxelSetup* h_setup = reinterpret_cast<VoxelSetup*>(c->h_pinned);
  if (n <= VS_MAX) {  // small cloud: one block does everything
    vox_small_kernel<<<1, VS_THREADS, 0, c->stream>>>(in, n, leaf, d_setup, out.as<float4>());
    c->launches++;
    LIOGPU_CUDA_OK(c, cudaGetLastError());
    LIOGPU_CUDA_OK(c, cudaMemcpyAsync(h_setup, d_setup, sizeof(VoxelSetup), cudaMemcpyDeviceToHost, c->stream));
    LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
    if (h_setup->overflow) {  // q4
      LIOGPU_CUDA_OK(c, cudaMemcpyAsync(out.p, in, (size_t)n * sizeof(float4), cudaMemcpyDeviceToDevice, c->stream));
      *n_out = n;
      *overflow = true;
      return LIOGPU_OK;
    }
    *n_out = (int)h_setup->n_vox;
    return LIOGPU_OK;
  }
  LIOGPU_CUDA_OK(c, launch_minmax(c, in, n, mm));
  vox_setup_kernel<<<1, 32, 0, c->stream>>>(mm, leaf, d_setup);
  vox_key_kernel<<<div_up(n, 256), 256, 0, c->stream>>>(in, n, d_setup, c->keys0.as<uint32_t>());
  c->launches += 2;
  uint32_t *skeys = nullptr, *sperm = nullptr;
  LIOGPU_CUDA_OK(c, radix_sort_pairs(c, n, -1, &d_setup->key_bits, &skeys, &sperm));
  uint32_t* head = c->seg_flag.as<uint32_t>();
  uint32_t* d_nvox = c->misc.as<uint32_t>();
  vox_head_kernel<<<div_up(n, 256), 256, 0, c->stream>>>(skeys, n, d_setup, head);
  c->launches++;
  LIOGPU_CUDA_OK(c, exclusive_scan_u32(c, head, head, n, d_nvox));
  vox_segstart_kernel<<<div_up(n, 256), 256, 0, c->stream>>>(skeys, head, n, d_setup, c->seg_start.as<uint32_t>(), d_nvox);
  // long-voxel list: reuses the (now dead) unsorted-key ping-pong buffer; two counters in misc
  uint32_t* long_list = (skeys == c->keys0.as<uint32_t>()) ? c->keys1.as<uint32_t>() : c->keys0.as<uint32_t>();
  uint32_t* d_long = c->misc.as<uint32_t>() + 2;  // [0] long count, [1] work counter
  LIOGPU_CUDA_OK(c, cudaMemsetAsync(d_long, 0, 2 * sizeof(uint32_t), c->stream));
  vox_centroid_kernel<<<div_up(n, 256), 256, 0, c->stream>>>(in, sperm, c->seg_start.as<uint32_t>(), d_nvox,
                                                             out.as<float4>(), long_list, d_long);
  vox_centroid_long_kernel<<<c->sm_count * 8, 32 * VOX_LONG_WARPS, 0, c->stream>>>(
      in, sperm, c->seg_start.as<uint32_t>(), long_list, d_long, d_long + 1, out.as<float4>());
  c->launches += 3;
  LIOGPU_CUDA_OK(c, cudaGetLastError());
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(h_setup, d_setup, sizeof(VoxelSetup), cudaMemcpyDeviceToHost, c->stream));
  LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  if (h_setup->overflow) {  // q4: PCL warns and returns the input unchanged
    LIOGPU_CUDA_OK(c, cudaMemcpyAsync(out.p, in, (size_t)n * sizeof(float4), cudaMemcpyDeviceToDevice, c->stream));
    *n_out = n;
    *overflow = true;
    return LIOGPU_OK;
  }
  *n_out = (int)h_setup->n_vox;
  return LIOGPU_OK;
}

// ---- segmented VoxelGrid: many keyframe windows per pass (liogpu_merge_keyframes_batch, the loop-closure submaps).
// A pass holds the transformed concatenation of consecutive windows.  Each window gets the single-cloud setup of its
// own points (same bounds, same vox_setup_compute); window w's keys are base_w + its single-cloud key, base_w = the
// cells of the pass's earlier windows, and every point that the single-cloud pipeline drops (non-finite, or in a
// window whose guard fired) gets the pass's sentinel key above every base.  The stable sort keeps each window's
// points in their concatenation order, so the head / scan / centroid kernels above, run unchanged on the pass, sum
// every voxel's members in the order the single-cloud pipeline does (DESIGN.md §7a).

// the window of point i: the last w in [lo, hi) with off[w] <= i (empty windows are skipped)
__device__ __forceinline__ int mw_window_of(const int* __restrict__ off, int lo, int hi, int i) {
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(off + mid) <= i) lo = mid; else hi = mid;
  }
  return lo;
}

// per-window bounds in vox_minmax_kernel's encoding: mn[3w+a] / mx[3w+a] ordered uint, cnt[w] finite points.  A block
// covers MW_TILE consecutive points: one reduction when they lie in one window, else per-point atomics.
constexpr int MW_ITEMS = 4;
constexpr int MW_TILE = 256 * MW_ITEMS;
__global__ void __launch_bounds__(256)
mw_minmax_kernel(const float4* __restrict__ pts, int n, const int* __restrict__ off, int nw, unsigned* __restrict__ mn_o,
                 unsigned* __restrict__ mx_o, unsigned* __restrict__ cnt_o) {
  const int b0 = blockIdx.x * MW_TILE;
  const int b1 = min(b0 + MW_TILE, n);
  const int w0 = mw_window_of(off, 0, nw, b0), w1 = mw_window_of(off, 0, nw, b1 - 1);
  if (w0 != w1) {
    for (int i = b0 + threadIdx.x; i < b1; i += 256) {
      const float4 p = pts[i];
      if (!finite3(p)) continue;
      const int w = mw_window_of(off, w0, w1 + 1, i);
      atomicMin(&mn_o[3 * w], f2ord(p.x)); atomicMin(&mn_o[3 * w + 1], f2ord(p.y)); atomicMin(&mn_o[3 * w + 2], f2ord(p.z));
      atomicMax(&mx_o[3 * w], f2ord(p.x)); atomicMax(&mx_o[3 * w + 1], f2ord(p.y)); atomicMax(&mx_o[3 * w + 2], f2ord(p.z));
      atomicAdd(&cnt_o[w], 1u);
    }
    return;
  }
  float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
  unsigned cnt = 0;
#pragma unroll
  for (int k = 0; k < MW_ITEMS; ++k) {
    const int i = b0 + k * 256 + threadIdx.x;
    if (i < b1) {
      const float4 p = pts[i];
      if (finite3(p)) {
        mn[0] = fminf(mn[0], p.x); mn[1] = fminf(mn[1], p.y); mn[2] = fminf(mn[2], p.z);
        mx[0] = fmaxf(mx[0], p.x); mx[1] = fmaxf(mx[1], p.y); mx[2] = fmaxf(mx[2], p.z);
        ++cnt;
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      mn[a] = fminf(mn[a], __shfl_xor_sync(0xffffffffu, mn[a], o));
      mx[a] = fmaxf(mx[a], __shfl_xor_sync(0xffffffffu, mx[a], o));
    }
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  }
  __shared__ float smn[8][3], smx[8][3];
  __shared__ unsigned scnt[8];
  const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
  if (lane == 0) {
#pragma unroll
    for (int a = 0; a < 3; ++a) { smn[wp][a] = mn[a]; smx[wp][a] = mx[a]; }
    scnt[wp] = cnt;
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    const int a = threadIdx.x;
    float lo = smn[0][a], hi = smx[0][a];
    for (int k = 1; k < 8; ++k) { lo = fminf(lo, smn[k][a]); hi = fmaxf(hi, smx[k][a]); }
    unsigned c = 0;
    for (int k = 0; k < 8; ++k) c += scnt[k];
    if (c) {  // a block of non-finite points leaves the window's bounds at their initial values
      atomicMin(&mn_o[3 * w0 + a], f2ord(lo));
      atomicMax(&mx_o[3 * w0 + a], f2ord(hi));
    }
  } else if (threadIdx.x == 3) {
    unsigned c = 0;
    for (int k = 0; k < 8; ++k) c += scnt[k];
    atomicAdd(&cnt_o[w0], c);
  }
}

// one thread per window: vox_setup_kernel on the window's bounds
__global__ void mw_setup_kernel(const unsigned* __restrict__ mn_o, const unsigned* __restrict__ mx_o,
                                const unsigned* __restrict__ cnt_o, int nw, float leaf, VoxelSetup* __restrict__ s) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= nw) return;
  VoxelSetup v;
  float mn[3], mx[3];
  for (int a = 0; a < 3; ++a) { mn[a] = ord2f(mn_o[3 * w + a]); mx[a] = ord2f(mx_o[3 * w + a]); }
  vox_setup_compute(mn, mx, (int)cnt_o[w], leaf, v);
  s[w] = v;
}

// keys of the pass's points [p0, p0 + n) (windows [wa, wb)); keys[i - p0]
__global__ void __launch_bounds__(256)
mw_key_kernel(const float4* __restrict__ pts, int p0, int n, const int* __restrict__ off, int wa, int wb,
              const VoxelSetup* __restrict__ setups, const unsigned* __restrict__ base, unsigned sentinel,
              uint32_t* __restrict__ keys) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const int i = p0 + t;
  const int w = mw_window_of(off, wa, wb, i);
  const float4 p = pts[i];
  const VoxelSetup& s = setups[w];
  keys[t] = (s.overflow || !finite3(p)) ? sentinel : __ldg(base + w) + vox_key_of(p, s);
}

// voxels of each window of the pass: the scanned head flags at its first and past its last sorted position
__global__ void mw_count_kernel(const uint32_t* __restrict__ rank, int n, const uint32_t* __restrict__ n_vox,
                                const int2* __restrict__ vrange, int wa, int wb, uint32_t* __restrict__ vcount) {
  const int w = wa + blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= wb) return;
  const int2 r = vrange[w];
  const uint32_t s = r.x < n ? rank[r.x] : *n_vox, e = r.y < n ? rank[r.y] : *n_vox;
  vcount[w] = e - s;
}

__global__ void __launch_bounds__(256)
mw_gather_kernel(const float4* const* __restrict__ srcs, const int* __restrict__ off, int nseg, int total,
                 float4* __restrict__ dst) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int s = mw_window_of(off, 0, nseg, i);
  dst[i] = srcs[s][i - __ldg(off + s)];
}

int gather_segments(Ctx* c, const std::vector<const float4*>& srcs, const std::vector<int>& off, float4* dst) {
  const int nseg = (int)srcs.size();
  if (nseg == 0 || off[nseg] == 0) return LIOGPU_OK;
  const size_t b_srcs = (size_t)nseg * sizeof(void*), b_off = ((size_t)nseg + 1) * sizeof(int);
  LIOGPU_CUDA_OK(c, c->mw_seg.reserve(b_srcs + b_off));
  char* d = (char*)c->mw_seg.p;
  // pageable sources: cudaMemcpyAsync has copied them out when it returns
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(d, srcs.data(), b_srcs, cudaMemcpyHostToDevice, c->stream));
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(d + b_srcs, off.data(), b_off, cudaMemcpyHostToDevice, c->stream));
  mw_gather_kernel<<<div_up(off[nseg], 256), 256, 0, c->stream>>>(reinterpret_cast<const float4* const*>(d),
                                                                 reinterpret_cast<const int*>(d + b_srcs), nseg, off[nseg], dst);
  c->launches++;
  LIOGPU_CUDA_OK(c, cudaGetLastError());
  return LIOGPU_OK;
}

// Input points of a pass (all its windows' transformed points).  A window larger than this runs alone.  The pass
// scratch is about 56 bytes a point: the transformed points and the centroids (16 + 16), the sort's keys and values
// (4 x 4) and the head flags and segment starts (2 x 4).  LIOGPU_MERGE_PASS_POINTS lowers it (tests use it to split
// small batches).
static long long merge_pass_points() {
  long long cap = 1ll << 25;
  if (const char* e = getenv("LIOGPU_MERGE_PASS_POINTS")) {
    const long long v = atoll(e);
    if (v > 0 && v < cap) cap = v;
  }
  return cap;
}

// One pass: windows [0, nw) of ids / poses (entries [win_off[0], win_off[nw]) of the caller's arrays, n_in[w] points
// each), appended to `out` at record `out_base`; out_off / overflow are the pass's own nw + 1 / nw entries.
static int merge_pass(Ctx* c, const int* ids, const float* pose6s, const int* win_off, const long long* n_in, int nw,
                      float leaf, DevBuf& out, int* out_off, int* overflow) {
  const int out_base = out_off[0];
  for (int w = 0; w < nw; ++w) overflow[w] = 0;
  const int k = win_off[nw] - win_off[0];
  KfTables t;
  int rc = stage_keyframes(c, "liogpu_merge_keyframes_batch", ids + win_off[0], pose6s + 6 * (size_t)win_off[0], k, t);
  if (rc) return rc;
  const int total = (int)t.total;
  if (!(leaf > 0.f)) {  // no VoxelGrid: the transformed concatenation, which is already in window order
    for (int w = 0; w < nw; ++w) out_off[w + 1] = out_off[w] + (int)n_in[w];
    if (total == 0) return LIOGPU_OK;
    rc = reserve_keep(c, out, ((size_t)out_base + total) * sizeof(float4), (size_t)out_base * sizeof(float4));
    if (rc) return rc;
    LIOGPU_CUDA_OK(c, launch_transform_multi(c, t.srcs, t.offs, k, t.poses, t.T12, (long long)total,
                                             out.as<float4>() + out_base));
    LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));  // the next pass restages the keyframe tables
    return LIOGPU_OK;
  }
  if (total == 0) {
    for (int w = 0; w < nw; ++w) out_off[w + 1] = out_off[w];
    return LIOGPU_OK;
  }
  std::vector<int> off(nw + 1, 0);
  for (int w = 0; w < nw; ++w) off[w + 1] = off[w] + (int)n_in[w];
  // device tables: off | mn | mx | cnt | vcount | setups | base | vrange | pass setups (<= nw)
  auto up256 = [](size_t b) { return (b + 255) & ~(size_t)255; };
  const size_t o_mn = up256(((size_t)nw + 1) * 4), o_mx = o_mn + up256((size_t)nw * 12), o_cnt = o_mx + up256((size_t)nw * 12);
  const size_t o_vc = o_cnt + up256((size_t)nw * 4), o_set = o_vc + up256((size_t)nw * 4);
  const size_t o_base = o_set + up256((size_t)nw * sizeof(VoxelSetup)), o_vr = o_base + up256((size_t)nw * 4);
  const size_t o_ps = o_vr + up256((size_t)nw * 8), tab_bytes = o_ps + (size_t)nw * sizeof(VoxelSetup);
  LIOGPU_CUDA_OK(c, c->mw_tab.reserve(tab_bytes));
  char* d = (char*)c->mw_tab.p;
  const int* d_off = reinterpret_cast<const int*>(d);
  unsigned *d_mn = reinterpret_cast<unsigned*>(d + o_mn), *d_mx = reinterpret_cast<unsigned*>(d + o_mx);
  unsigned *d_cnt = reinterpret_cast<unsigned*>(d + o_cnt), *d_vc = reinterpret_cast<unsigned*>(d + o_vc);
  VoxelSetup* d_set = reinterpret_cast<VoxelSetup*>(d + o_set);
  VoxelSetup* d_ps = reinterpret_cast<VoxelSetup*>(d + o_ps);
  const unsigned* d_base = reinterpret_cast<const unsigned*>(d + o_base);
  const int2* d_vr = reinterpret_cast<const int2*>(d + o_vr);
  LIOGPU_CUDA_OK(c, c->lm_a.reserve((size_t)total * sizeof(float4)));
  LIOGPU_CUDA_OK(c, c->lm_out.reserve((size_t)total * sizeof(float4)));
  LIOGPU_CUDA_OK(c, c->keys0.reserve((size_t)total * 4));
  LIOGPU_CUDA_OK(c, c->keys1.reserve((size_t)total * 4));
  LIOGPU_CUDA_OK(c, c->vals0.reserve((size_t)total * 4));
  LIOGPU_CUDA_OK(c, c->vals1.reserve((size_t)total * 4));
  LIOGPU_CUDA_OK(c, c->seg_flag.reserve((size_t)total * 4 + 16));
  LIOGPU_CUDA_OK(c, c->seg_start.reserve((size_t)total * 4 + 16));
  LIOGPU_CUDA_OK(c, c->misc.reserve(256));
  float4* pts = c->lm_a.as<float4>();
  float4* cent = c->lm_out.as<float4>();
  LIOGPU_CUDA_OK(c, launch_transform_multi(c, t.srcs, t.offs, k, t.poses, t.T12, (long long)total, pts));
  // bounds and setups of every window, read back once
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(d, off.data(), ((size_t)nw + 1) * 4, cudaMemcpyHostToDevice, c->stream));
  LIOGPU_CUDA_OK(c, cudaMemsetAsync(d_mn, 0xff, (size_t)nw * 12, c->stream));
  LIOGPU_CUDA_OK(c, cudaMemsetAsync(d_mx, 0, o_set - o_mx, c->stream));  // mx, cnt and vcount
  mw_minmax_kernel<<<div_up(total, MW_TILE), 256, 0, c->stream>>>(pts, total, d_off, nw, d_mn, d_mx, d_cnt);
  mw_setup_kernel<<<div_up(nw, 128), 128, 0, c->stream>>>(d_mn, d_mx, d_cnt, nw, leaf, d_set);
  c->launches += 2;
  LIOGPU_CUDA_OK(c, cudaGetLastError());
  std::vector<VoxelSetup> set(nw);
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(set.data(), d_set, (size_t)nw * sizeof(VoxelSetup), cudaMemcpyDeviceToHost, c->stream));
  LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  // key space: windows share it while their cells fit 32 bits next to the sentinel; a window that needs all of it
  // keys alone, with exactly the single-cloud keys and sentinel
  std::vector<unsigned> base(nw);
  std::vector<int2> vr(nw);
  std::vector<VoxelSetup> ps;
  std::vector<int> seg_w{0};  // key segments: windows [seg_w[s], seg_w[s+1])
  unsigned long long cells_sum = 0;
  int valid = 0;
  bool alone = false;
  auto close = [&]() {
    VoxelSetup v{};
    v.n_valid = valid;
    v.n_cells = (unsigned)cells_sum;
    int b = 0;
    while (b < 32 && (v.n_cells >> b) != 0u) ++b;
    v.key_bits = b;
    ps.push_back(v);
  };
  for (int w = 0; w < nw; ++w) {
    const VoxelSetup& s = set[w];
    const bool used = !s.overflow && s.n_valid > 0;
    const unsigned long long cells =
        used ? (unsigned long long)s.div_b[0] * (unsigned long long)s.div_b[1] * (unsigned long long)s.div_b[2] : 0ull;
    const bool big = cells > 0xffffffffull;
    if (w > seg_w.back() && (alone || big || cells_sum + cells > 0xffffffffull)) {
      close();
      seg_w.push_back(w);
      cells_sum = 0;
      valid = 0;
    }
    alone = big;
    base[w] = (unsigned)cells_sum;
    const int nv = used ? s.n_valid : 0;
    vr[w] = make_int2(valid, valid + nv);
    cells_sum += cells;
    valid += nv;
    overflow[w] = s.overflow ? 1 : 0;
  }
  close();
  seg_w.push_back(nw);
  const int n_seg = (int)ps.size();
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(d + o_base, base.data(), (size_t)nw * 4, cudaMemcpyHostToDevice, c->stream));
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(d + o_vr, vr.data(), (size_t)nw * 8, cudaMemcpyHostToDevice, c->stream));
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(d_ps, ps.data(), (size_t)n_seg * sizeof(VoxelSetup), cudaMemcpyHostToDevice, c->stream));
  uint32_t* d_nvox = c->misc.as<uint32_t>();
  uint32_t* d_long = c->misc.as<uint32_t>() + 2;  // [0] long count, [1] work counter
  for (int sg = 0; sg < n_seg; ++sg) {
    if (ps[sg].n_valid == 0) continue;  // nothing but dropped points: every window of it keeps vcount 0
    const int wa = seg_w[sg], wb = seg_w[sg + 1];
    const int p0 = off[wa], n = off[wb] - off[wa];
    mw_key_kernel<<<div_up(n, 256), 256, 0, c->stream>>>(pts, p0, n, d_off, wa, wb, d_set, d_base, ps[sg].n_cells,
                                                         c->keys0.as<uint32_t>());
    c->launches++;
    uint32_t *skeys = nullptr, *sperm = nullptr;
    LIOGPU_CUDA_OK(c, radix_sort_pairs(c, n, ps[sg].key_bits, nullptr, &skeys, &sperm));
    uint32_t* head = c->seg_flag.as<uint32_t>();
    vox_head_kernel<<<div_up(n, 256), 256, 0, c->stream>>>(skeys, n, d_ps + sg, head);
    c->launches++;
    LIOGPU_CUDA_OK(c, exclusive_scan_u32(c, head, head, n, d_nvox));
    vox_segstart_kernel<<<div_up(n, 256), 256, 0, c->stream>>>(skeys, head, n, d_ps + sg, c->seg_start.as<uint32_t>(), d_nvox);
    uint32_t* long_list = (skeys == c->keys0.as<uint32_t>()) ? c->keys1.as<uint32_t>() : c->keys0.as<uint32_t>();
    LIOGPU_CUDA_OK(c, cudaMemsetAsync(d_long, 0, 2 * sizeof(uint32_t), c->stream));
    vox_centroid_kernel<<<div_up(n, 256), 256, 0, c->stream>>>(pts + p0, sperm, c->seg_start.as<uint32_t>(), d_nvox,
                                                               cent + p0, long_list, d_long);
    vox_centroid_long_kernel<<<c->sm_count * 8, 32 * VOX_LONG_WARPS, 0, c->stream>>>(
        pts + p0, sperm, c->seg_start.as<uint32_t>(), long_list, d_long, d_long + 1, cent + p0);
    mw_count_kernel<<<div_up(wb - wa, 128), 128, 0, c->stream>>>(head, n, d_nvox, d_vr, wa, wb, d_vc);
    c->launches += 4;
    LIOGPU_CUDA_OK(c, cudaGetLastError());
  }
  std::vector<unsigned> vc(nw);
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(vc.data(), d_vc, (size_t)nw * 4, cudaMemcpyDeviceToHost, c->stream));
  LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  // placement: window w's centroids start at its key segment's first point plus the voxels of the segment's earlier
  // windows; a window whose guard fired is its transformed input (q4)
  std::vector<const float4*> srcs(nw);
  std::vector<int> dst(nw + 1, 0);
  for (int sg = 0; sg < n_seg; ++sg) {
    long long v = 0;
    for (int w = seg_w[sg]; w < seg_w[sg + 1]; ++w) {
      const int m = overflow[w] ? (int)n_in[w] : (int)vc[w];
      srcs[w] = overflow[w] ? pts + off[w] : cent + off[seg_w[sg]] + v;
      if (!overflow[w]) v += vc[w];
      dst[w + 1] = dst[w] + m;
      out_off[w + 1] = out_off[w] + m;
    }
  }
  if (dst[nw] == 0) return LIOGPU_OK;
  rc = reserve_keep(c, out, ((size_t)out_base + dst[nw]) * sizeof(float4), (size_t)out_base * sizeof(float4));
  if (rc) return rc;
  return gather_segments(c, srcs, dst, out.as<float4>() + out_base);
}

int merge_windows_dev(Ctx* c, const int* ids, const float* pose6s, const int* win_off, int n_windows, float leaf,
                      DevBuf& out, int* out_off, int* overflow) {
  out_off[0] = 0;
  std::vector<long long> n_in(n_windows);
  for (int w = 0; w < n_windows; ++w) {
    long long n = 0;
    for (int j = win_off[w]; j < win_off[w + 1]; ++j) n += c->keyframes.at(ids[j]).second;
    n_in[w] = n;
  }
  const long long cap = merge_pass_points();
  for (int w0 = 0; w0 < n_windows;) {
    long long pts = n_in[w0];
    int w1 = w0 + 1;
    while (w1 < n_windows && pts + n_in[w1] <= cap) pts += n_in[w1++];
    const int rc = merge_pass(c, ids, pose6s, win_off + w0, n_in.data() + w0, w1 - w0, leaf, out, out_off + w0, overflow + w0);
    if (rc) return rc;
    w0 = w1;
  }
  return LIOGPU_OK;
}

}  // namespace liogpu
