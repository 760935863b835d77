// api.cu — the C ABI of libliogpu.so (include/liogpu.h).  Thin: argument checks, host<->device
// staging, and calls into the kernel drivers.  No CPU implementation of any operator lives here:
// without a usable CUDA device every entry point fails with LIOGPU_E_CUDA.
#include "common.cuh"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>

#include <nvtx3/nvToolsExt.h>  // header-only: ranges cost nothing unless a profiler is attached

using namespace liogpu;

struct liogpu_ctx {
  Ctx c;
};

namespace {

thread_local std::string g_create_err;

// one NVTX range per ABI entry point (SURVEY §5: the reference's commented-out per-stage timers, MO:461-501)
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

bool is_device_ptr(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

bool stride_ok(int stride) { return stride == 16 || (stride >= 32 && (stride % 4) == 0); }

// caller cloud (host or device, `stride` bytes per record) -> packed float4 in dst
int load_cloud(Ctx* c, const void* src, int& n, int stride, DevBuf& dst) {
  if (src == LIOGPU_DEVICE_RESIDENT) {  // the cloud this context kept in HBM
    if (!c->resident) { c->err = "LIOGPU_DEVICE_RESIDENT: no resident cloud"; return LIOGPU_E_INVALID; }
    n = c->resident_n;
    if (c->resident == &dst || n == 0) return LIOGPU_OK;
    LIOGPU_CUDA_OK(c, dst.reserve((size_t)n * sizeof(float4)));
    LIOGPU_CUDA_OK(c, cudaMemcpyAsync(dst.p, c->resident->p, (size_t)n * sizeof(float4), cudaMemcpyDeviceToDevice, c->stream));
    return LIOGPU_OK;
  }
  if (src == LIOGPU_UPLOADED_SCAN) {  // the sweep liogpu_upload_scan_async put on its way
    if (c->upload_count <= 0) { c->err = "LIOGPU_UPLOADED_SCAN: no upload pending"; return LIOGPU_E_INVALID; }
    Ctx::Upload& u = c->upload[c->upload_head];  // first in, first out
    u.valid = false;
    c->upload_head ^= 1;
    c->upload_count--;
    n = u.n;
    LIOGPU_CUDA_OK(c, dst.reserve((size_t)(n > 0 ? n : 1) * sizeof(float4)));
    if (n == 0) return LIOGPU_OK;
    LIOGPU_CUDA_OK(c, cudaStreamWaitEvent(c->stream, u.ev, 0));
    if (u.stride == 16) {
      LIOGPU_CUDA_OK(c, cudaMemcpyAsync(dst.p, u.raw.p, (size_t)n * 16, cudaMemcpyDeviceToDevice, c->stream));
    } else {
      LIOGPU_CUDA_OK(c, launch_unpack(c, u.raw.p, n, u.stride, dst.as<float4>()));
    }
    return LIOGPU_OK;
  }
  if (n < 0 || (n > 0 && !src) || !stride_ok(stride)) { c->err = "bad cloud pointer / size / stride"; return LIOGPU_E_INVALID; }
  LIOGPU_CUDA_OK(c, dst.reserve((size_t)(n > 0 ? n : 1) * sizeof(float4)));
  if (n == 0) return LIOGPU_OK;
  const bool dev = is_device_ptr(src);
  if (stride == 16) {
    LIOGPU_CUDA_OK(c, cudaMemcpyAsync(dst.p, src, (size_t)n * 16, dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, c->stream));
    return LIOGPU_OK;
  }
  const void* d_raw = src;
  if (!dev) {
    LIOGPU_CUDA_OK(c, c->raw_in.reserve((size_t)n * stride));
    LIOGPU_CUDA_OK(c, cudaMemcpyAsync(c->raw_in.p, src, (size_t)n * stride, cudaMemcpyHostToDevice, c->stream));
    d_raw = c->raw_in.p;
  }
  LIOGPU_CUDA_OK(c, launch_unpack(c, d_raw, n, stride, dst.as<float4>()));
  return LIOGPU_OK;
}

// packed float4 -> caller cloud (host or device)
int store_cloud(Ctx* c, const float4* src, int n, void* dst, int stride) {
  if (n <= 0) return LIOGPU_OK;
  if (!dst || !stride_ok(stride)) { c->err = "bad output pointer / stride"; return LIOGPU_E_INVALID; }
  const bool dev = is_device_ptr(dst);
  if (stride == 16) {
    LIOGPU_CUDA_OK(c, cudaMemcpyAsync(dst, src, (size_t)n * 16, dev ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, c->stream));
  } else if (dev) {
    LIOGPU_CUDA_OK(c, launch_pack(c, src, n, dst, stride));
  } else {
    LIOGPU_CUDA_OK(c, c->raw_out.reserve((size_t)n * stride));
    LIOGPU_CUDA_OK(c, launch_pack(c, src, n, c->raw_out.p, stride));
    LIOGPU_CUDA_OK(c, cudaMemcpyAsync(dst, c->raw_out.p, (size_t)n * stride, cudaMemcpyDeviceToHost, c->stream));
  }
  LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  return LIOGPU_OK;
}

// A call that is about to overwrite `buf` without declaring it the new resident cloud invalidates a resident
// cloud that lives there: a later LIOGPU_DEVICE_RESIDENT use then fails loudly instead of reading other data.
void clobber(Ctx* c, DevBuf* buf) {
  if (c->resident == buf) { c->resident = nullptr; c->resident_n = 0; }
}

}  // namespace

// The k named keyframes as device tables for the multi-keyframe transform kernels: validates the ids, stages
// poses [k*6 f32] | offsets [k+1 i32] | source pointers [k u64] in pinned memory (second half of h_pinned) and
// uploads them in one copy.  Concatenation order = argument order (the reference's "+=" loops).
int liogpu::stage_keyframes(Ctx* c, const char* who, const int* ids, const float* pose6s, int k, KfTables& t) {
  t.total = 0;
  for (int f = 0; f < k; ++f) {
    auto it = c->keyframes.find(ids[f]);
    if (it == c->keyframes.end()) { c->err = std::string(who) + ": unknown keyframe id"; return LIOGPU_E_NO_KEYFRAME; }
    t.total += (size_t)it->second.second;
  }
  if (t.total > 0x7fffffffULL) { c->err = std::string(who) + ": cloud too large"; return LIOGPU_E_INVALID; }
  if (t.total == 0) return LIOGPU_OK;
  // tables sized from k (saveMapService merges EVERY keyframe of a run, mapOptmization.cpp:936-941): poses | offsets | pointers
  auto up256 = [](size_t b) { return (b + 255) & ~(size_t)255; };
  const size_t off_offs = up256((size_t)k * 6 * sizeof(float));
  const size_t off_srcs = off_offs + up256(((size_t)k + 1) * sizeof(int));
  const size_t tab_bytes = off_srcs + up256((size_t)k * sizeof(void*));
  if (tab_bytes > c->h_kf_cap) {  // nothing of this context is in flight here: every call ends with a stream sync
    if (c->h_kf_tab) cudaFreeHost(c->h_kf_tab);
    c->h_kf_tab = nullptr;
    c->h_kf_cap = 0;
    const size_t want = tab_bytes + tab_bytes / 2 + 4096;
    LIOGPU_CUDA_OK(c, cudaHostAlloc(&c->h_kf_tab, want, cudaHostAllocDefault));
    c->h_kf_cap = want;
  }
  char* hp = (char*)c->h_kf_tab;
  float* hposes = reinterpret_cast<float*>(hp);
  int* hoffs = reinterpret_cast<int*>(hp + off_offs);
  const float4** hsrcs = reinterpret_cast<const float4**>(hp + off_srcs);
  std::memcpy(hposes, pose6s, (size_t)k * 6 * sizeof(float));
  size_t off = 0;
  for (int f = 0; f < k; ++f) {
    auto& kf = c->keyframes[ids[f]];
    hoffs[f] = (int)off;
    hsrcs[f] = kf.first.as<float4>();
    off += (size_t)kf.second;
  }
  hoffs[k] = (int)off;
  LIOGPU_CUDA_OK(c, c->kf_tab.reserve(tab_bytes + (size_t)k * 12 * sizeof(float)));  // tables + k transforms
  char* dp = (char*)c->kf_tab.p;
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(dp, hp, tab_bytes, cudaMemcpyHostToDevice, c->stream));
  t.srcs = reinterpret_cast<const float4* const*>(dp + off_srcs);
  t.offs = reinterpret_cast<const int*>(dp + off_offs);
  t.poses = reinterpret_cast<const float*>(dp);
  t.T12 = reinterpret_cast<float*>(dp + tab_bytes);
  return LIOGPU_OK;
}

int liogpu::reserve_keep(Ctx* c, DevBuf& b, size_t need, size_t used) {
  if (need <= b.cap) return LIOGPU_OK;
  const size_t want = need + need / 2 + 4096;
  void* np_ = nullptr;
  LIOGPU_CUDA_OK(c, cudaMallocAsync(&np_, want, c->stream));
  if (used) LIOGPU_CUDA_OK(c, cudaMemcpyAsync(np_, b.p, used, cudaMemcpyDeviceToDevice, c->stream));
  if (b.p) LIOGPU_CUDA_OK(c, cudaFreeAsync(b.p, c->stream));
  b.p = np_;
  b.cap = want;
  return LIOGPU_OK;
}

namespace {

int enter(liogpu_ctx* ctx) {
  if (!ctx) return LIOGPU_E_INVALID;
  ctx->c.err.clear();
  ctx->c.last_result = nullptr;  // liogpu_fetch_result serves only the call right before it
  if (cudaSetDevice(ctx->c.device) != cudaSuccess) {
    ctx->c.err = std::string("cudaSetDevice: ") + cudaGetErrorString(cudaGetLastError());
    return LIOGPU_E_CUDA;
  }
  return LIOGPU_OK;
}

}  // namespace

extern "C" {

int liogpu_abi_version(void) { return LIOGPU_ABI_VERSION; }

void liogpu_default_params(liogpu_params* p) {
  if (!p) return;
  std::memset(p, 0, sizeof(*p));
  p->device = 0;
  p->n_scan = 16;                                   // utility.h:275
  p->horizon_scan = 1800;                           // :276
  p->mapping_surf_leaf_size = 0.2f;                 // :303
  p->surrounding_keyframe_map_leaf_size = 0.2f;     // :304
  p->downsample_rate = 1;                           // :277
  p->point_filter_num = 3;                          // :278
  p->lidar_min_front = 1.0f;                        // :280
  p->lidar_min_back = 5.0f;                         // :281
  p->lidar_min_left = 2.0f;                         // :282
  p->lidar_min_right = 2.0f;                        // :283
  p->lidar_max_range = 1000.0f;                     // :284
  p->lidar_max_intensity = 100.0f;                  // :285
  p->knn_cell_size = 0.0f;
}

int liogpu_create(liogpu_ctx** out, const liogpu_params* params) {
  if (!out || !params) return LIOGPU_E_INVALID;
  *out = nullptr;
  if (params->downsample_rate < 1 || params->point_filter_num < 1 || params->n_scan < 1) return LIOGPU_E_INVALID;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || params->device < 0 || params->device >= ndev) {
    cudaGetLastError();
    return LIOGPU_E_CUDA;  // no CPU fallback by design
  }
  if (cudaSetDevice(params->device) != cudaSuccess) return LIOGPU_E_CUDA;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, params->device) != cudaSuccess) return LIOGPU_E_CUDA;
  if (prop.major < 10) return LIOGPU_E_CUDA;  // built for sm_100a only
  liogpu_ctx* ctx = new (std::nothrow) liogpu_ctx();
  if (!ctx) return LIOGPU_E_INVALID;
  Ctx& c = ctx->c;
  c.prm = *params;
  c.device = params->device;
  c.sm_count = prop.multiProcessorCount;
  int prio_lo = 0, prio_hi = 0;
  cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
  if (cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithPriority(&c.side_stream, cudaStreamNonBlocking, prio_hi) != cudaSuccess ||
      cudaEventCreateWithFlags(&c.ev_it0, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&c.ev_side, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreate(&c.ev0) != cudaSuccess || cudaEventCreate(&c.ev1) != cudaSuccess ||
      cudaStreamCreateWithFlags(&c.copy_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&c.upload[0].ev, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&c.upload[1].ev, cudaEventDisableTiming) != cudaSuccess ||
      cudaHostAlloc(&c.h_pinned, 262144, cudaHostAllocDefault) != cudaSuccess) {
    liogpu_destroy(ctx);
    return LIOGPU_E_CUDA;
  }
  {
    DevBuf* bufs[] = {&c.raw_in, &c.raw_out, &c.scan4, &c.scan_ds4, &c.map_raw4, &c.map4, &c.map_sorted, &c.cell_start,
                      &c.keys0, &c.keys1, &c.vals0, &c.vals1, &c.counters, &c.scan_tmp, &c.seg_flag, &c.seg_start,
                      &c.vox_setup, &c.grid_setup, &c.minmax, &c.lm_state, &c.partials, &c.block_counter, &c.misc,
                      &c.fail_buf, &c.prev_nn, &c.hopeless, &c.fz_rows, &c.fz_left, &c.fz_lb, &c.fz_probe, &c.tile_plan,
                      &c.tile_hist, &c.tile_pts, &c.tile_out, &c.dbg_idx, &c.dbg_d2, &c.dbg_coeff, &c.dbg_flag, &c.dbg_tie,
                      &c.imu_tab, &c.dsk_flags, &c.dsk_scan, &c.lm_flag, &c.lm_pos, &c.lm_a, &c.lm_b, &c.lm_md, &c.lm_left,
                      &c.lm_out, &c.lm_stats, &c.sor_setup, &c.sor_sorted, &c.sor_cell_start, &c.kf_tab,
                      &c.sc_q, &c.sc_part, &c.sc_cand, &c.sc_out, &c.lc_src, &c.lc_tgt, &c.lc_tab, &c.mw_tab, &c.mw_seg};
    for (DevBuf* b : bufs) { b->stream = c.stream; b->async = true; }
  }
  // scratch hint of allocateMemory (mapOptmization.cpp:333-335)
  const size_t hint = (size_t)params->n_scan * (size_t)(params->horizon_scan > 0 ? params->horizon_scan : 1);
  c.scan4.reserve(hint * sizeof(float4));
  c.scan_ds4.reserve(hint * sizeof(float4));
  *out = ctx;
  return LIOGPU_OK;
}

void liogpu_destroy(liogpu_ctx* ctx) {
  if (!ctx) return;
  Ctx& c = ctx->c;
  cudaSetDevice(c.device);
  if (c.stream) cudaStreamSynchronize(c.stream);
  if (c.side_stream) cudaStreamSynchronize(c.side_stream);
  if (c.copy_stream) cudaStreamSynchronize(c.copy_stream);
  for (auto& u : c.upload) { u.raw.release(); if (u.ev) cudaEventDestroy(u.ev); }
  if (c.copy_stream) cudaStreamDestroy(c.copy_stream);
  if (c.h_kf_tab) cudaFreeHost(c.h_kf_tab);
  c.kf_tab.release();
  DevBuf* bufs[] = {&c.raw_in, &c.raw_out, &c.scan4, &c.scan_ds4, &c.map_raw4, &c.map4, &c.map_sorted, &c.cell_start,
                    &c.keys0, &c.keys1, &c.vals0, &c.vals1, &c.counters, &c.scan_tmp, &c.seg_flag, &c.seg_start,
                    &c.vox_setup, &c.grid_setup, &c.minmax, &c.lm_state, &c.partials, &c.block_counter, &c.misc,
                    &c.fail_buf, &c.prev_nn, &c.hopeless, &c.fz_rows, &c.fz_left, &c.fz_lb, &c.fz_probe, &c.tile_plan, &c.tile_hist, &c.tile_pts, &c.tile_out, &c.dbg_idx, &c.dbg_d2, &c.dbg_coeff, &c.dbg_flag, &c.dbg_tie, &c.imu_tab, &c.dsk_flags, &c.dsk_scan,
                    &c.lm_flag, &c.lm_pos, &c.lm_a, &c.lm_b, &c.lm_md, &c.lm_left, &c.lm_out, &c.lm_stats, &c.sor_setup,
                    &c.sor_sorted, &c.sor_cell_start, &c.sc_q, &c.sc_part, &c.sc_cand, &c.sc_out, &c.lc_src, &c.lc_tgt,
                    &c.lc_tab, &c.mw_tab, &c.mw_seg};
  for (DevBuf* b : bufs) b->release();
  sc_release(&c);
  for (auto& kv : c.keyframes) kv.second.first.release();
  for (void* slab : c.kf_slabs) cudaFree(slab);
  if (c.h_pinned) cudaFreeHost(c.h_pinned);
  if (c.ev0) cudaEventDestroy(c.ev0);
  if (c.ev1) cudaEventDestroy(c.ev1);
  for (cudaEvent_t e : c.prof_ev) cudaEventDestroy(e);
  if (c.ev_mid) cudaEventDestroy(c.ev_mid);
  if (c.ev_it0) cudaEventDestroy(c.ev_it0);
  if (c.ev_side) cudaEventDestroy(c.ev_side);
  if (c.side_stream) cudaStreamDestroy(c.side_stream);
  if (c.stream) cudaStreamDestroy(c.stream);
  delete ctx;
}

const char* liogpu_last_error(const liogpu_ctx* ctx) { return ctx ? ctx->c.err.c_str() : "null context"; }

void* liogpu_host_alloc(unsigned long long bytes) {
  void* p = nullptr;
  if (cudaHostAlloc(&p, (size_t)bytes, cudaHostAllocDefault) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return p;
}
void liogpu_host_free(void* p) {
  if (p) cudaFreeHost(p);
}

int liogpu_deskew(liogpu_ctx* ctx, const void* xyzirt, int n, int stride, double time_scan_cur, const double* imu_time,
                  const double* imu_rot_x, const double* imu_rot_y, const double* imu_rot_z, int n_imu,
                  int deskew_enabled, void* xyzi_out, int out_stride, int cap_out, int* n_out) {
  NvtxRange nvtx_range_(__func__);
  int rc = enter(ctx);
  if (rc) return rc;
  Ctx* c = &ctx->c;
  if (!n_out || n < 0 || (n > 0 && !xyzirt) || stride < 28 || (stride % 4) != 0 || n_imu < 0 || n_imu > 2000 ||
      (n_imu > 0 && (!imu_time || !imu_rot_x || !imu_rot_y || !imu_rot_z))) {
    c->err = "liogpu_deskew: bad arguments";
    return LIOGPU_E_INVALID;
  }
  *n_out = 0;
  if (n == 0) return LIOGPU_OK;
  const void* d_raw = xyzirt;
  if (!is_device_ptr(xyzirt)) {
    LIOGPU_CUDA_OK(c, c->raw_in.reserve((size_t)n * stride));
    LIOGPU_CUDA_OK(c, cudaMemcpyAsync(c->raw_in.p, xyzirt, (size_t)n * stride, cudaMemcpyHostToDevice, c->stream));
    d_raw = c->raw_in.p;
  }
  double* tab = reinterpret_cast<double*>((char*)c->h_pinned + 65536);  // 4 x 2000 doubles = 64000 B
  for (int k = 0; k < n_imu; ++k) {
    tab[k] = imu_time[k];
    tab[n_imu + k] = imu_rot_x[k];
    tab[2 * n_imu + k] = imu_rot_y[k];
    tab[3 * n_imu + k] = imu_rot_z[k];
  }
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
  int m = 0;
  clobber(c, &c->dsk_scan);
  rc = deskew_dev(c, d_raw, n, stride, time_scan_cur, tab, n_imu, deskew_enabled, c->dsk_scan, &m);
  if (rc) return rc;
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
  *n_out = m;
  if (xyzi_out == LIOGPU_DEVICE_RESIDENT) {
    c->resident = &c->dsk_scan;
    c->resident_n = m;
  } else if (xyzi_out) {
    if (m > cap_out) { c->err = "liogpu_deskew: output capacity too small"; return LIOGPU_E_CAPACITY; }
    rc = store_cloud(c, c->dsk_scan.as<float4>(), m, xyzi_out, out_stride);
    if (rc) return rc;
  }
  LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1);
  return LIOGPU_OK;
}

int liogpu_transform_cloud(liogpu_ctx* ctx, const void* xyzi, int n, int stride, const float pose6[6], void* xyzi_out,
                           int out_stride) {
  NvtxRange nvtx_range_(__func__);
  int rc = enter(ctx);
  if (rc) return rc;
  Ctx* c = &ctx->c;
  if (!pose6) { c->err = "null pose"; return LIOGPU_E_INVALID; }
  rc = load_cloud(c, xyzi, n, stride, c->scan4);
  if (rc) return rc;
  if (n == 0) return LIOGPU_OK;
  clobber(c, &c->scan4);
  clobber(c, &c->scan_ds4);
  LIOGPU_CUDA_OK(c, c->misc.reserve(256));
  LIOGPU_CUDA_OK(c, c->scan_ds4.reserve((size_t)n * sizeof(float4)));
  float* hp = reinterpret_cast<float*>((char*)c->h_pinned + 3200);
  for (int k = 0; k < 6; ++k) hp[k] = pose6[k];
  float* d_pose = c->misc.as<float>() + 32;
  LIOGPU_CUDA_OK(c, cudaMemcpyAsync(d_pose, hp, 6 * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
  LIOGPU_CUDA_OK(c, launch_transform(c, c->scan4.as<float4>(), n, d_pose, c->scan_ds4.as<float4>()));
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
  rc = store_cloud(c, c->scan_ds4.as<float4>(), n, xyzi_out, out_stride);
  if (rc) return rc;
  cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1);
  return LIOGPU_OK;
}

int liogpu_voxel_downsample(liogpu_ctx* ctx, const void* xyzi, int n, int stride, float leaf, void* xyzi_out,
                            int out_stride, int cap_out, int* n_out) {
  NvtxRange nvtx_range_(__func__);
  int rc = enter(ctx);
  if (rc) return rc;
  Ctx* c = &ctx->c;
  if (!n_out) { c->err = "null n_out"; return LIOGPU_E_INVALID; }
  *n_out = 0;
  rc = load_cloud(c, xyzi, n, stride, c->scan4);
  if (rc) return rc;
  if (n == 0) return LIOGPU_OK;
  clobber(c, &c->scan4);
  clobber(c, &c->scan_ds4);
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
  int m = 0;
  bool overflow = false;
  rc = voxel_downsample_dev(c, c->scan4.as<float4>(), n, leaf, c->scan_ds4, &m, &overflow);
  if (rc) return rc;
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
  *n_out = m;
  if (xyzi_out == LIOGPU_DEVICE_RESIDENT) {
    c->resident = &c->scan_ds4;
    c->resident_n = m;
  } else if (xyzi_out) {
    if (m > cap_out) { c->err = "liogpu_voxel_downsample: output capacity too small"; return LIOGPU_E_CAPACITY; }
    rc = store_cloud(c, c->scan_ds4.as<float4>(), m, xyzi_out, out_stride);
    if (rc) return rc;
  }
  LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1);
  return overflow ? LIOGPU_W_LEAF_OVERFLOW : LIOGPU_OK;
}

int liogpu_keyframe_put(liogpu_ctx* ctx, int id, const void* xyzi, int n, int stride) {
  NvtxRange nvtx_range_(__func__);
  int rc = enter(ctx);
  if (rc) return rc;
  Ctx* c = &ctx->c;
  // arguments are checked BEFORE the table is touched, and the cloud is loaded into a buffer of its own that replaces
  // the old one only on success: a failed overwrite keeps the previous keyframe and nothing leaks
  const bool special = xyzi == LIOGPU_DEVICE_RESIDENT || xyzi == LIOGPU_UPLOADED_SCAN;
  if (!special && (n < 0 || (n > 0 && !xyzi) || !stride_ok(stride))) { c->err = "liogpu_keyframe_put: bad cloud pointer / size / stride"; return LIOGPU_E_INVALID; }
  int n_in = n;
  if (xyzi == LIOGPU_DEVICE_RESIDENT) { if (!c->resident) { c->err = "LIOGPU_DEVICE_RESIDENT: no resident cloud"; return LIOGPU_E_INVALID; } n_in = c->resident_n; }
  if (xyzi == LIOGPU_UPLOADED_SCAN) { if (c->upload_count <= 0) { c->err = "LIOGPU_UPLOADED_SCAN: no upload pending"; return LIOGPU_E_INVALID; } n_in = c->upload[c->upload_head].n; }
  DevBuf fresh;
  {
    auto old = c->keyframes.find(id);
    const size_t need = ((size_t)(n_in > 0 ? n_in : 1) * sizeof(float4) + 255) & ~(size_t)255;
    if (old != c->keyframes.end() && old->second.first.cap >= need) {
      fresh = old->second.first;  // overwrite in place (same id, fits): nothing can fail between here and the copy
    } else {
      constexpr size_t SLAB = 32u << 20;
      // current slab, else the next one kept from before liogpu_keyframe_clear, else a new one (cudaMalloc synchronises the
      // whole device, i.e. every other context on it: slabs are therefore never given back before the context is destroyed)
      for (;;) {
        if (c->kf_slab_cur < c->kf_slabs.size() && c->kf_slab_used + need <= c->kf_slab_sizes[c->kf_slab_cur]) break;
        if (c->kf_slab_cur + 1 < c->kf_slabs.size()) { ++c->kf_slab_cur; c->kf_slab_used = 0; continue; }
        const size_t sz = need > SLAB ? need : SLAB;
        void* slab = nullptr;
        LIOGPU_CUDA_OK(c, cudaMalloc(&slab, sz));
        c->kf_slabs.push_back(slab);
        c->kf_slab_sizes.push_back(sz);
        c->kf_slab_cur = c->kf_slabs.size() - 1;
        c->kf_slab_used = 0;
        break;
      }
      fresh.p = (char*)c->kf_slabs[c->kf_slab_cur] + c->kf_slab_used;
      fresh.cap = need;
      fresh.pooled = true;
      c->kf_slab_used += need;  // an overwritten, smaller keyframe's bytes stay in their slab until liogpu_keyframe_clear
    }
  }
  rc = load_cloud(c, xyzi, n, stride, fresh);
  if (rc == LIOGPU_OK && cudaStreamSynchronize(c->stream) != cudaSuccess) {  // raw_in staging is reused by the next call
    c->err = std::string("liogpu_keyframe_put: ") + cudaGetErrorString(cudaGetLastError());
    rc = LIOGPU_E_CUDA;
  }
  if (rc) return rc;
  auto& slot = c->keyframes[id];
  slot.first = fresh;
  slot.second = n;
  return LIOGPU_OK;
}

int liogpu_keyframe_clear(liogpu_ctx* ctx) {
  NvtxRange nvtx_range_(__func__);
  int rc = enter(ctx);
  if (rc) return rc;
  Ctx* c = &ctx->c;
  cudaStreamSynchronize(c->stream);
  for (auto& kv : c->keyframes) kv.second.first.release();
  c->keyframes.clear();
  c->kf_slab_cur = 0;  // the slabs stay with the context and are filled again from the first one (no cudaFree / cudaMalloc:
  c->kf_slab_used = 0; // both synchronise the device); liogpu_destroy releases them
  return LIOGPU_OK;
}

int liogpu_keyframe_count(const liogpu_ctx* ctx) { return ctx ? (int)ctx->c.keyframes.size() : 0; }

int liogpu_build_local_map(liogpu_ctx* ctx, const int* ids, const float* pose6s, int k, float leaf, int* n_map,
                           void* xyzi_out, int out_stride, int cap_out) {
  NvtxRange nvtx_range_(__func__);
  int rc = enter(ctx);
  if (rc) return rc;
  Ctx* c = &ctx->c;
  if (k < 0 || (k > 0 && (!ids || !pose6s)) || !n_map) { c->err = "liogpu_build_local_map: bad arguments"; return LIOGPU_E_INVALID; }
  *n_map = 0;
  KfTables t;
  rc = stage_keyframes(c, "liogpu_build_local_map", ids, pose6s, k, t);
  if (rc) return rc;
  const size_t total = t.total;
  c->grid_valid = false;
  c->n_map = 0;
  if (total == 0) return LIOGPU_W_NO_KEYFRAMES;
  LIOGPU_CUDA_OK(c, c->map_raw4.reserve(total * sizeof(float4)));
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
  // transformPointCloud + "+=" concatenation (mapOptmization.cpp:1566-1576) in one launch
  LIOGPU_CUDA_OK(c, launch_transform_multi(c, t.srcs, t.offs, k, t.poses, t.T12, (long long)total, c->map_raw4.as<float4>()));
  int m = 0;
  bool overflow = false;
  rc = voxel_downsample_dev(c, c->map_raw4.as<float4>(), (int)total, leaf, c->map4, &m, &overflow);
  if (rc) return rc;
  rc = grid_build_dev(c, c->map4.as<float4>(), m, leaf);
  if (rc) return rc;
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
  *n_map = m;
  c->last_result = c->map4.as<float4>(); c->last_result_n = m; c->last_result_status = overflow ? LIOGPU_W_LEAF_OVERFLOW : LIOGPU_OK;
  if (xyzi_out) {
    if (m > cap_out) { c->err = "liogpu_build_local_map: output capacity too small"; return LIOGPU_E_CAPACITY; }
    rc = store_cloud(c, c->map4.as<float4>(), m, xyzi_out, out_stride);
    if (rc) return rc;
  }
  LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1);
  return overflow ? LIOGPU_W_LEAF_OVERFLOW : LIOGPU_OK;
}

int liogpu_voxel_tile(liogpu_ctx* ctx, const int* ids, const float* pose6s, int k, float leaf, int tile, int n_tiles,
                      void* xyzi_out, int out_stride, int cap_out, int* n_out, liogpu_tile_info* info) {
  NvtxRange nvtx_range_(__func__);
  int rc = enter(ctx);
  if (rc) return rc;
  Ctx* c = &ctx->c;
  liogpu_tile_info local_info;
  if (!info) info = &local_info;
  std::memset(info, 0, sizeof(*info));
  if (k < 0 || (k > 0 && (!ids || !pose6s)) || !n_out || n_tiles < 1 || tile < 0 || tile >= n_tiles || !(leaf > 0.f)) {
    c->err = "liogpu_voxel_tile: bad arguments";
    return LIOGPU_E_INVALID;
  }
  *n_out = 0;
  KfTables t;
  rc = stage_keyframes(c, "liogpu_voxel_tile", ids, pose6s, k, t);
  if (rc) return rc;
  if (t.total == 0) return LIOGPU_W_NO_KEYFRAMES;
  const int total = (int)t.total;
  if (!c->ev_mid) LIOGPU_CUDA_OK(c, cudaEventCreate(&c->ev_mid));
  // scratch of publishLocalMap: the registration's local map / index and a resident sweep are not touched
  LIOGPU_CUDA_OK(c, c->lm_a.reserve(t.total * sizeof(float4)));
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
  LIOGPU_CUDA_OK(c, launch_transform_multi(c, t.srcs, t.offs, k, t.poses, t.T12, (long long)total, c->lm_a.as<float4>()));
  int m = 0;
  bool overflow = false;
  rc = voxel_tile_dev(c, c->lm_a.as<float4>(), total, leaf, tile, n_tiles, c->tile_out, &m, &overflow, info);
  if (rc) return rc;
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
  *n_out = m;
  c->last_result = c->tile_out.as<float4>(); c->last_result_n = m; c->last_result_status = overflow ? LIOGPU_W_LEAF_OVERFLOW : LIOGPU_OK;
  if (xyzi_out && m > 0) {
    if (m > cap_out) { c->err = "liogpu_voxel_tile: output capacity too small"; return LIOGPU_E_CAPACITY; }
    rc = store_cloud(c, c->tile_out.as<float4>(), m, xyzi_out, out_stride);
    if (rc) return rc;
  }
  LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1);
  info->gpu_ms = c->last_ms;
  cudaEventElapsedTime(&info->plan_ms, c->ev0, c->ev_mid);
  return overflow ? LIOGPU_W_LEAF_OVERFLOW : LIOGPU_OK;
}

void liogpu_default_local_map_params(liogpu_local_map_params* p) {
  if (!p) return;
  std::memset(p, 0, sizeof(*p));
  p->local_map_front = 70.0f;             // utility.h:220
  p->local_map_left = 40.0f;              // :221
  p->local_map_back = 20.0f;              // :222
  p->local_map_right = 40.0f;             // :223
  p->use_down_sampling = 1;               // :224
  p->local_mapping_surf_leaf_size = 0.01f; // :226
  p->use_removing_outliers = 1;           // :227
  p->mean_k = 10;                         // :228
  p->stddev_threshold = 1.0f;             // :229
}

int liogpu_publish_local_map(liogpu_ctx* ctx, const int* ids, const float* pose6s, int k, const float pose_now[6],
                             const liogpu_local_map_params* params, void* xyzi_out, int out_stride, int cap_out,
                             int* n_out, liogpu_local_map_info* info) {
  NvtxRange nvtx_range_(__func__);
  int rc = enter(ctx);
  if (rc) return rc;
  Ctx* c = &ctx->c;
  liogpu_local_map_info local_info;
  if (!info) info = &local_info;
  std::memset(info, 0, sizeof(*info));
  if (k < 0 || (k > 0 && (!ids || !pose6s)) || !pose_now || !params || !n_out) {
    c->err = "liogpu_publish_local_map: bad arguments";
    return LIOGPU_E_INVALID;
  }
  *n_out = 0;
  if (params->use_removing_outliers && (params->mean_k < 1 || params->mean_k > 31)) {
    c->err = "liogpu_publish_local_map: mean_k must be in 1..31";
    return LIOGPU_E_INVALID;
  }
  if (params->use_down_sampling && !(params->local_mapping_surf_leaf_size > 0.f)) {
    c->err = "liogpu_publish_local_map: leaf must be > 0";
    return LIOGPU_E_INVALID;
  }
  if (k == 0) return LIOGPU_W_NO_KEYFRAMES;  // cloudKeyPoses3D->points.empty(), mapOptmization.cpp:2444
  KfTables t;
  rc = stage_keyframes(c, "liogpu_publish_local_map", ids, pose6s, k, t);   // "+=" order of mapOptmization.cpp:2463-2466
  if (rc) return rc;
  const size_t total = t.total;
  if (total == 0) return LIOGPU_OK;
  // The yaw-aligned vehicle frame (mapOptmization.cpp:2474-2488), f32 like the reference; canonical trig = f64
  // sin/cos rounded to f32 as everywhere in this library.  Rotation = Eigen::AngleAxisf(-yaw, UnitZ)
  // .toRotationMatrix(): its zz entry is (1 - c) + c, which is not always exactly 1.
  float yw[16];
  {
    const float yaw = pose_now[2], X = pose_now[3], Y = pose_now[4], Z = pose_now[5];
    const float nyaw = -yaw;
    const float cs = (float)cos((double)nyaw), sn = (float)sin((double)nyaw);
    const float px = X * cs, py = Y * sn, qx = Y * cs, qy = X * sn;
    const float tX = px - py;  // :2474
    const float tY = qx + qy;  // :2475
    const float tZ = Z;        // :2476
    const float zz = (1.0f - cs) + cs;
    const float m[12] = {cs, -sn, 0.f, -tX, sn, cs, 0.f, -tY, 0.f, 0.f, zz, -tZ};
    for (int q = 0; q < 12; ++q) yw[q] = m[q];
    yw[12] = -params->local_map_left;   // :297
    yw[13] = params->local_map_right;
    yw[14] = -params->local_map_back;   // :301
    yw[15] = params->local_map_front;
  }
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
  const float4* result = nullptr;
  int m = 0;
  rc = publish_local_map_dev(c, t.srcs, t.offs, k, t.poses, t.T12, (long long)total, yw, params, &result, &m, info);
  if (rc) return rc;
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
  *n_out = m;
  c->last_result = result; c->last_result_n = m; c->last_result_status = info->leaf_overflow ? LIOGPU_W_LEAF_OVERFLOW : LIOGPU_OK;
  if (xyzi_out && m > 0) {
    if (m > cap_out) { c->err = "liogpu_publish_local_map: output capacity too small"; return LIOGPU_E_CAPACITY; }
    rc = store_cloud(c, result, m, xyzi_out, out_stride);
    if (rc) return rc;
  }
  LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1);
  info->gpu_ms = c->last_ms;
  return info->leaf_overflow ? LIOGPU_W_LEAF_OVERFLOW : LIOGPU_OK;
}

int liogpu_merge_keyframes(liogpu_ctx* ctx, const int* ids, const float* pose6s, int k, float leaf, void* xyzi_out,
                           int out_stride, int cap_out, int* n_out) {
  NvtxRange nvtx_range_(__func__);
  int rc = enter(ctx);
  if (rc) return rc;
  Ctx* c = &ctx->c;
  if (k < 0 || (k > 0 && (!ids || !pose6s)) || !n_out) { c->err = "liogpu_merge_keyframes: bad arguments"; return LIOGPU_E_INVALID; }
  *n_out = 0;
  KfTables t;
  rc = stage_keyframes(c, "liogpu_merge_keyframes", ids, pose6s, k, t);
  if (rc) return rc;
  if (t.total == 0) return LIOGPU_OK;
  const int total = (int)t.total;
  // scratch of publishLocalMap: neither the registration's local map / index nor a resident sweep is touched
  LIOGPU_CUDA_OK(c, c->lm_a.reserve(t.total * sizeof(float4)));
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
  LIOGPU_CUDA_OK(c, launch_transform_multi(c, t.srcs, t.offs, k, t.poses, t.T12, (long long)total, c->lm_a.as<float4>()));
  const float4* result = c->lm_a.as<float4>();
  int m = total;
  bool overflow = false;
  if (leaf > 0.f) {  // req.resolution != 0 (mapOptmization.cpp:943) / the visualisation leaf (:1037-1039)
    rc = voxel_downsample_dev(c, result, total, leaf, c->lm_out, &m, &overflow);
    if (rc) return rc;
    result = c->lm_out.as<float4>();
  }
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
  *n_out = m;
  c->last_result = result; c->last_result_n = m; c->last_result_status = overflow ? LIOGPU_W_LEAF_OVERFLOW : LIOGPU_OK;
  if (xyzi_out && m > 0) {
    if (m > cap_out) { c->err = "liogpu_merge_keyframes: output capacity too small"; return LIOGPU_E_CAPACITY; }
    rc = store_cloud(c, result, m, xyzi_out, out_stride);
    if (rc) return rc;
  }
  LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1);
  return overflow ? LIOGPU_W_LEAF_OVERFLOW : LIOGPU_OK;
}

int liogpu_merge_keyframes_batch(liogpu_ctx* ctx, const int* ids, const float* pose6s, const int* win_off, int n_windows,
                                 float leaf, void* xyzi_out, int out_stride, int cap_out, int* out_off, int* overflow) {
  NvtxRange nvtx_range_(__func__);
  int rc = enter(ctx);
  if (rc) return rc;
  Ctx* c = &ctx->c;
  bool ok = n_windows >= 0 && win_off && out_off && win_off[0] == 0 && (!xyzi_out || stride_ok(out_stride));
  for (int w = 0; ok && w < n_windows; ++w) ok = win_off[w + 1] >= win_off[w];
  if (ok && win_off[n_windows] > 0 && (!ids || !pose6s)) ok = false;
  if (!ok) { c->err = "liogpu_merge_keyframes_batch: bad arguments"; return LIOGPU_E_INVALID; }
  const int k = win_off[n_windows];
  long long total = 0;
  for (int j = 0; j < k; ++j) {
    auto it = c->keyframes.find(ids[j]);
    if (it == c->keyframes.end()) { c->err = "liogpu_merge_keyframes_batch: unknown keyframe id"; return LIOGPU_E_NO_KEYFRAME; }
    total += it->second.second;
  }
  if (total > 0x7fffffffLL) { c->err = "liogpu_merge_keyframes_batch: windows too large"; return LIOGPU_E_INVALID; }
  std::vector<int> ovf(n_windows);
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
  // lm_b: neither the registration's local map / index nor a resident sweep lives there
  rc = merge_windows_dev(c, ids, pose6s, win_off, n_windows, leaf, c->lm_b, out_off, ovf.data());
  if (rc) return rc;
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
  bool any = false;
  for (int w = 0; w < n_windows; ++w) {
    any = any || ovf[w];
    if (overflow) overflow[w] = ovf[w];
  }
  const int m = out_off[n_windows];
  if (m > 0) {
    c->last_result = c->lm_b.as<float4>(); c->last_result_n = m; c->last_result_status = any ? LIOGPU_W_LEAF_OVERFLOW : LIOGPU_OK;
  }
  if (xyzi_out && m > 0) {
    if (m > cap_out) { c->err = "liogpu_merge_keyframes_batch: output capacity too small"; return LIOGPU_E_CAPACITY; }
    rc = store_cloud(c, c->lm_b.as<float4>(), m, xyzi_out, out_stride);
    if (rc) return rc;
  }
  LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1);
  return any ? LIOGPU_W_LEAF_OVERFLOW : LIOGPU_OK;
}

void liogpu_default_icp_params(liogpu_icp_params* p, float history_keyframe_search_radius) {
  if (!p) return;
  std::memset(p, 0, sizeof(*p));
  p->max_correspondence_distance = history_keyframe_search_radius * 2;  // mapOptmization.cpp:1112
  p->max_iterations = 100;                                              // :1113
  p->transformation_epsilon = 1e-6;                                     // :1114
  p->euclidean_fitness_epsilon = 1e-6;                                  // :1115
}

int liogpu_icp_align(liogpu_ctx* ctx, const void* source_xyzi, int n_source, int source_stride, const void* target_xyzi,
                     int n_target, int target_stride, const liogpu_icp_params* params, float final_transformation[16],
                     liogpu_icp_info* info) {
  NvtxRange nvtx_range_(__func__);
  int rc = enter(ctx);
  if (rc) return rc;
  Ctx* c = &ctx->c;
  liogpu_icp_info local_info;
  if (!info) info = &local_info;
  std::memset(info, 0, sizeof(*info));
  if (!params || !final_transformation || n_source <= 0 || n_target <= 0 || params->max_iterations < 1 ||
      !(params->max_correspondence_distance > 0.f) || source_xyzi == LIOGPU_DEVICE_RESIDENT ||
      target_xyzi == LIOGPU_DEVICE_RESIDENT) {
    c->err = "liogpu_icp_align: bad arguments";
    return LIOGPU_E_INVALID;
  }
  rc = load_cloud(c, source_xyzi, n_source, source_stride, c->lm_b);
  if (rc) return rc;
  rc = load_cloud(c, target_xyzi, n_target, target_stride, c->lm_out);
  if (rc) return rc;
  return icp_align_dev(c, c->lm_b.as<float4>(), n_source, c->lm_out.as<float4>(), n_target, params, final_transformation, info);
}

}  // extern "C"

extern "C" {

int liogpu_loop_closure_icp_batch(liogpu_ctx* ctx, const int* key_cur, const int* key_pre, int n_pairs,
                                  const float* key_pose6s, int n_key, int search_num, float icp_leaf,
                                  const liogpu_icp_params* params, liogpu_loop_icp_result* results) {
  NvtxRange nvtx_range_(__func__);
  int rc = enter(ctx);
  if (rc) return rc;
  Ctx* c = &ctx->c;
  if (n_pairs < 0 || (n_pairs > 0 && (!key_cur || !key_pre || !key_pose6s || !results)) || n_key < 0 || search_num < 0 ||
      !(icp_leaf > 0.f) || !params || params->max_iterations < 1 || !(params->max_correspondence_distance > 0.f)) {
    c->err = "liogpu_loop_closure_icp_batch: bad arguments";
    return LIOGPU_E_INVALID;
  }
  for (int j = 0; j < n_pairs; ++j) {
    if (key_cur[j] < 0 || key_cur[j] >= n_key || key_pre[j] < 0 || key_pre[j] >= n_key) {
      c->err = "liogpu_loop_closure_icp_batch: key outside [0, n_key)";
      return LIOGPU_E_INVALID;
    }
    const long long lo = (long long)key_pre[j] - search_num, hi = (long long)key_pre[j] + search_num;
    bool ok = c->keyframes.count(key_cur[j]) != 0;
    for (long long k = lo < 0 ? 0 : lo; ok && k <= hi && k < n_key; ++k) ok = c->keyframes.count((int)k) != 0;
    if (!ok) { c->err = "liogpu_loop_closure_icp_batch: unknown keyframe id"; return LIOGPU_E_NO_KEYFRAME; }
  }
  for (int j = 0; j < n_pairs; ++j) {
    std::memset(&results[j], 0, sizeof(results[j]));
    for (int q = 0; q < 16; ++q) results[j].final_transformation[q] = (q % 5 == 0) ? 1.f : 0.f;
  }
  // Submaps: loopFindNearKeyframes (MO:1360-1383) of both ends of every pair, window [key - n, key + n] ∩ [0, n_key)
  // (MO:1102-1103), built by merge_windows_dev for a batch of pairs at a time (the batch's inputs stay under 2^25
  // points, so the submaps are bounded too).  The pairs that pass the size guard (MO:1104) are copied into the
  // contiguous lc_src / lc_tgt layout and go to the ICP in groups that keep the submaps (and with them the index and
  // per-point buffers) under a fixed size; every pair's result is independent of the batch and group it lands in.
  // LIOGPU_LOOP_ICP_GROUP caps the pairs of a group (tests use it to split small batches).
  constexpr long long GROUP_POINTS = 1ll << 25, BATCH_POINTS = 1ll << 25;
  int group_pairs = 1024;
  if (const char* e = getenv("LIOGPU_LOOP_ICP_GROUP")) {
    const int v = atoi(e);
    if (v > 0 && v < group_pairs) group_pairs = v;
  }
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
  auto kf_points = [&](int key, int s) {
    long long n = 0;
    for (long long k = std::max(0ll, (long long)key - s); k <= (long long)key + s && k < n_key; ++k)
      n += c->keyframes.at((int)k).second;
    return n;
  };
  std::vector<int> members, so{0}, to{0}, ids, win_off, out_off, ovf;
  std::vector<const float4*> src_seg, tgt_seg;  // submaps of the group's members not yet copied to lc_src / lc_tgt
  std::vector<float> T, poses;
  std::vector<liogpu_icp_info> info;
  int copied = 0;  // members already in lc_src / lc_tgt
  auto gather = [&]() -> int {
    const int n = (int)members.size();
    if (n == copied) return LIOGPU_OK;
    for (auto* v : {&so, &to}) {
      std::vector<int> off(v->begin() + copied, v->end());
      for (int& o : off) o -= (*v)[copied];
      DevBuf& dst = v == &so ? c->lc_src : c->lc_tgt;
      int r = reserve_keep(c, dst, (size_t)v->back() * sizeof(float4), (size_t)(*v)[copied] * sizeof(float4));
      if (!r) r = gather_segments(c, v == &so ? src_seg : tgt_seg, off, dst.as<float4>() + (*v)[copied]);
      if (r) return r;
    }
    src_seg.clear();
    tgt_seg.clear();
    copied = n;
    return LIOGPU_OK;
  };
  auto flush = [&]() -> int {
    const int n = (int)members.size();
    if (n == 0) return LIOGPU_OK;
    int r = gather();
    if (r) return r;
    T.resize((size_t)n * 16);
    info.assign(n, liogpu_icp_info{});
    r = icp_batch_dev(c, c->lc_src.as<float4>(), so.data(), c->lc_tgt.as<float4>(), to.data(), n, params,
                      reinterpret_cast<float(*)[16]>(T.data()), info.data());
    if (r) return r;
    for (int g = 0; g < n; ++g) {
      liogpu_loop_icp_result& res = results[members[g]];
      std::memcpy(res.final_transformation, &T[(size_t)g * 16], 16 * sizeof(float));
      res.icp = info[g];
    }
    members.clear();
    so.assign(1, 0);
    to.assign(1, 0);
    copied = 0;
    return LIOGPU_OK;
  };
  for (int j0 = 0; j0 < n_pairs;) {
    // a batch of pairs, windows in the order (source, target) of each pair
    ids.clear();
    poses.clear();
    win_off.assign(1, 0);
    long long pts = 0;
    int j1 = j0;
    for (; j1 < n_pairs; ++j1) {
      const long long add = kf_points(key_cur[j1], 0) + kf_points(key_pre[j1], search_num);
      if (j1 > j0 && pts + add > BATCH_POINTS) break;
      pts += add;
      for (int e = 0; e < 2; ++e) {
        const int key = e ? key_pre[j1] : key_cur[j1], s = e ? search_num : 0;
        for (long long k = std::max(0ll, (long long)key - s); k <= (long long)key + s && k < n_key; ++k) {
          ids.push_back((int)k);
          poses.insert(poses.end(), key_pose6s + 6 * k, key_pose6s + 6 * k + 6);
        }
        win_off.push_back((int)ids.size());
      }
    }
    const int nw = 2 * (j1 - j0);
    out_off.assign(nw + 1, 0);
    ovf.assign(nw, 0);
    rc = merge_windows_dev(c, ids.data(), poses.data(), win_off.data(), nw, icp_leaf, c->lm_b, out_off.data(), ovf.data());
    if (rc) return rc;
    const float4* arena = c->lm_b.as<float4>();
    for (int j = j0; j < j1; ++j) {
      liogpu_loop_icp_result& res = results[j];
      const int ws = 2 * (j - j0), wt = ws + 1;
      const int ms = out_off[ws + 1] - out_off[ws], mt = out_off[wt + 1] - out_off[wt];
      res.n_source = ms;
      res.n_target = mt;
      res.source_overflow = ovf[ws];
      res.target_overflow = ovf[wt];
      if (ms < 300 || mt < 1000) {  // MO:1104
        res.rejected_by_size = 1;
        continue;
      }
      members.push_back(j);
      src_seg.push_back(arena + out_off[ws]);
      tgt_seg.push_back(arena + out_off[wt]);
      so.push_back(so.back() + ms);
      to.push_back(to.back() + mt);
      if ((int)members.size() >= group_pairs || (long long)so.back() + to.back() >= GROUP_POINTS) {
        rc = flush();
        if (rc) return rc;
      }
    }
    rc = gather();  // the next batch reuses the arena
    if (rc) return rc;
    j0 = j1;
  }
  rc = flush();
  if (rc) return rc;
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
  LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1);
  return LIOGPU_OK;
}

int liogpu_make_scancontext(liogpu_ctx* ctx, const void* xyzi, int n, int stride, double lidar_height, double max_radius,
                            double* desc, double* ringkey, double* sectorkey) {
  NvtxRange nvtx_range_(__func__);
  int rc = enter(ctx);
  if (rc) return rc;
  Ctx* c = &ctx->c;
  if (!desc || !ringkey || !sectorkey || !(max_radius > 0.0)) { c->err = "liogpu_make_scancontext: bad arguments"; return LIOGPU_E_INVALID; }
  const float4* pts = nullptr;
  if (xyzi == LIOGPU_DEVICE_RESIDENT) {  // read in place, the resident cloud stays valid
    if (!c->resident) { c->err = "LIOGPU_DEVICE_RESIDENT: no resident cloud"; return LIOGPU_E_INVALID; }
    n = c->resident_n;
    pts = c->resident->as<float4>();
  } else {
    rc = load_cloud(c, xyzi, n, stride, c->lm_b);
    if (rc) return rc;
    pts = c->lm_b.as<float4>();
  }
  double out[LIOGPU_SC_NUM_RING * LIOGPU_SC_NUM_SECTOR + LIOGPU_SC_NUM_RING + LIOGPU_SC_NUM_SECTOR];
  rc = scancontext_dev(c, pts, n, lidar_height, max_radius, out);
  if (rc) return rc;
  const int bins = LIOGPU_SC_NUM_RING * LIOGPU_SC_NUM_SECTOR;
  std::memcpy(desc, out, bins * sizeof(double));
  std::memcpy(ringkey, out + bins, LIOGPU_SC_NUM_RING * sizeof(double));
  std::memcpy(sectorkey, out + bins + LIOGPU_SC_NUM_RING, LIOGPU_SC_NUM_SECTOR * sizeof(double));
  return LIOGPU_OK;
}

int liogpu_extract_nearby(liogpu_ctx* ctx, const void* key_poses3d, int n_key, int stride3d, const void* key_times,
                          int time_stride, double time_laser_info_cur, float search_radius, float density_leaf, int* ids_out,
                          int cap_ids, int* n_ids) {
  NvtxRange nvtx_range_(__func__);
  int rc = enter(ctx);
  if (rc) return rc;
  Ctx* c = &ctx->c;
  if (!n_ids || n_key < 0 || (n_key > 0 && (!key_poses3d || !key_times)) || time_stride < 8 || cap_ids < 0 ||
      (cap_ids > 0 && !ids_out) || !(search_radius > 0.f) || !(density_leaf > 0.f) || key_poses3d == LIOGPU_DEVICE_RESIDENT) {
    c->err = "liogpu_extract_nearby: bad arguments";
    return LIOGPU_E_INVALID;
  }
  *n_ids = 0;
  if (n_key == 0) return LIOGPU_W_NO_KEYFRAMES;  // extractSurroundingKeyFrames returns at once (mapOptmization.cpp:1592)
  rc = load_cloud(c, key_poses3d, n_key, stride3d, c->lm_a);
  if (rc) return rc;
  std::vector<double> times((size_t)n_key);
  for (int i = 0; i < n_key; ++i) std::memcpy(&times[i], (const char*)key_times + (size_t)i * time_stride, sizeof(double));
  return extract_nearby_dev(c, c->lm_a.as<float4>(), n_key, times.data(), time_laser_info_cur, search_radius, density_leaf,
                            ids_out, cap_ids, n_ids);
}

void liogpu_default_sc_params(liogpu_sc_params* p) {
  if (!p) return;
  std::memset(p, 0, sizeof(*p));
  p->num_exclude_recent = 30;        // Scancontext.h: NUM_EXCLUDE_RECENT
  p->num_candidates_from_tree = 3;   // NUM_CANDIDATES_FROM_TREE
  p->tree_making_period = 30;        // TREE_MAKING_PERIOD_
  p->search_ratio = 0.1;             // SEARCH_RATIO
  p->sc_dist_thres = 0.2;            // SC_DIST_THRES
}

int liogpu_sc_add(liogpu_ctx* ctx, const double* descs, int n) {
  NvtxRange nvtx_range_(__func__);
  int rc = enter(ctx);
  if (rc) return rc;
  Ctx* c = &ctx->c;
  if (!descs || n <= 0 || (long long)c->sc.count + n > 0x7fffffffLL) { c->err = "liogpu_sc_add: bad arguments"; return LIOGPU_E_INVALID; }
  return sc_add_dev(c, descs, n);
}

int liogpu_sc_clear(liogpu_ctx* ctx) {
  NvtxRange nvtx_range_(__func__);
  int rc = enter(ctx);
  if (rc) return rc;
  Ctx* c = &ctx->c;
  c->sc.count = 0;  // the arrays stay with the context and are filled again (freeing would synchronise the device)
  c->sc.counter = 0;
  c->sc.snap = 0;
  c->last_ms = 0.f;
  return LIOGPU_OK;
}

static bool sc_params_ok(const liogpu_sc_params* p) {
  return p && p->num_exclude_recent >= 0 && p->num_candidates_from_tree >= 1 &&
         p->num_candidates_from_tree <= LIOGPU_SC_MAX_CANDIDATES && p->tree_making_period >= 1 && p->search_ratio > 0.0 &&
         p->search_ratio <= 1.0 && !std::isnan(p->sc_dist_thres);
}
static int sc_search_radius(const liogpu_sc_params* p) {  // SEARCH_RADIUS = round(0.5 * SEARCH_RATIO * cols)
  return (int)std::round(0.5 * p->search_ratio * LIOGPU_SC_NUM_SECTOR);
}

int liogpu_sc_detect_loop(liogpu_ctx* ctx, const liogpu_sc_params* p, int* loop_id, float* yaw_diff_rad, liogpu_sc_info* info) {
  NvtxRange nvtx_range_(__func__);
  int rc = enter(ctx);
  if (rc) return rc;
  Ctx* c = &ctx->c;
  if (!sc_params_ok(p) || !loop_id || !yaw_diff_rad) { c->err = "liogpu_sc_detect_loop: bad arguments"; return LIOGPU_E_INVALID; }
  liogpu_sc_info local_info;
  if (!info) info = &local_info;
  std::memset(info, 0, sizeof(*info));
  ScStore& st = c->sc;
  info->n_stored = st.count;
  info->nn_idx = -1;
  info->min_dist = 10000000.0;
  *loop_id = -1;
  *yaw_diff_rad = 0.f;
  c->last_ms = 0.f;
  if (st.count < p->num_exclude_recent + 1) {  // early return: the counter does not advance
    info->n_searchable = st.snap;
    return LIOGPU_OK;
  }
  const bool rebuild = st.counter % p->tree_making_period == 0;
  const int snap = rebuild ? st.count - p->num_exclude_recent : st.snap;
  std::vector<int2> qm(1, make_int2(st.count - 1, snap));
  ScQueryOut out;
  rc = sc_detect_dev(c, qm, p->num_candidates_from_tree, sc_search_radius(p), p->sc_dist_thres, &out, info);
  if (rc) return rc;
  st.snap = snap;
  st.counter++;
  info->n_searchable = snap;
  info->tree_rebuilt = rebuild ? 1 : 0;
  info->n_candidates = out.n_cand;
  info->nn_idx = out.nn_idx;
  info->nn_align = out.nn_align;
  info->min_dist = out.min_dist;
  info->knn_ties = out.ties;
  info->gpu_ms = c->last_ms;
  *loop_id = out.loop_id;
  *yaw_diff_rad = out.yaw;
  return LIOGPU_OK;
}

int liogpu_sc_detect_loops(liogpu_ctx* ctx, const liogpu_sc_params* p, const int* store_sizes, int n_calls, int* loop_ids,
                           float* yaw_diff_rad, double* min_dist) {
  NvtxRange nvtx_range_(__func__);
  int rc = enter(ctx);
  if (rc) return rc;
  Ctx* c = &ctx->c;
  bool ok = sc_params_ok(p) && store_sizes && loop_ids && n_calls > 0;
  for (int j = 0; ok && j < n_calls; ++j)
    ok = store_sizes[j] >= 0 && store_sizes[j] <= c->sc.count && (j == 0 || store_sizes[j] >= store_sizes[j - 1]);
  if (!ok) { c->err = "liogpu_sc_detect_loops: bad arguments"; return LIOGPU_E_INVALID; }
  // the snapshot schedule of a fresh SCManager: which calls search, and over which prefix
  std::vector<int2> qm;
  std::vector<int> slot((size_t)n_calls, -1);
  long long counter = 0;
  int snap = 0;
  for (int j = 0; j < n_calls; ++j) {
    const int size = store_sizes[j];
    if (size < p->num_exclude_recent + 1) continue;  // early return, counter untouched
    if (counter % p->tree_making_period == 0) snap = size - p->num_exclude_recent;
    ++counter;
    slot[j] = (int)qm.size();
    qm.push_back(make_int2(size - 1, snap));
  }
  std::vector<ScQueryOut> out(qm.size());
  c->last_ms = 0.f;
  if (!qm.empty()) {
    rc = sc_detect_dev(c, qm, p->num_candidates_from_tree, sc_search_radius(p), p->sc_dist_thres, out.data(), nullptr);
    if (rc) return rc;
  }
  for (int j = 0; j < n_calls; ++j) {
    const int s = slot[j];
    loop_ids[j] = s < 0 ? -1 : out[s].loop_id;
    if (yaw_diff_rad) yaw_diff_rad[j] = s < 0 ? 0.f : out[s].yaw;
    if (min_dist) min_dist[j] = s < 0 ? 10000000.0 : out[s].min_dist;
  }
  return LIOGPU_OK;
}

int liogpu_detect_loop_distance(liogpu_ctx* ctx, const void* key_poses3d, int n_key, int stride3d, const void* key_times,
                                int time_stride, double time_laser_info_cur, float search_radius, float time_diff,
                                int* loop_key_pre) {
  NvtxRange nvtx_range_(__func__);
  int rc = enter(ctx);
  if (rc) return rc;
  Ctx* c = &ctx->c;
  if (!loop_key_pre || n_key <= 0 || !key_poses3d || !key_times || time_stride < 8 || !(search_radius > 0.f) ||
      std::isnan(time_diff) || key_poses3d == LIOGPU_DEVICE_RESIDENT || key_poses3d == LIOGPU_UPLOADED_SCAN || !stride_ok(stride3d)) {
    c->err = "liogpu_detect_loop_distance: bad arguments";
    return LIOGPU_E_INVALID;
  }
  *loop_key_pre = -1;
  rc = load_cloud(c, key_poses3d, n_key, stride3d, c->lm_a);  // the key-pose upload of liogpu_extract_nearby
  if (rc) return rc;
  std::vector<double> times((size_t)n_key);
  for (int i = 0; i < n_key; ++i) std::memcpy(&times[i], (const char*)key_times + (size_t)i * time_stride, sizeof(double));
  return detect_loop_distance_dev(c, c->lm_a.as<float4>(), n_key, times.data(), time_laser_info_cur, search_radius, time_diff,
                                  loop_key_pre);
}

int liogpu_set_local_map(liogpu_ctx* ctx, const void* xyzi, int n, int stride) {
  NvtxRange nvtx_range_(__func__);
  int rc = enter(ctx);
  if (rc) return rc;
  Ctx* c = &ctx->c;
  c->grid_valid = false;
  rc = load_cloud(c, xyzi, n, stride, c->map4);
  if (rc) return rc;
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
  rc = grid_build_dev(c, c->map4.as<float4>(), n, c->prm.surrounding_keyframe_map_leaf_size);
  if (rc) return rc;
  LIOGPU_CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
  LIOGPU_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1);
  if (n == 0) { c->grid_valid = true; c->n_map = 0; }
  return LIOGPU_OK;
}

int liogpu_local_map_size(const liogpu_ctx* ctx) { return ctx ? ctx->c.n_map : 0; }
int liogpu_resident_size(const liogpu_ctx* ctx) { return (ctx && ctx->c.resident) ? ctx->c.resident_n : 0; }

static int s2m_guards(Ctx* c, int n, liogpu_s2m_info* info) {
  if (info) {
    std::memset(info, 0, sizeof(*info));
    info->n_query = n;
  }
  if (!c->grid_valid) { c->err = "no local map installed"; return LIOGPU_E_NO_MAP; }
  if (c->n_map <= 0) return LIOGPU_W_NO_KEYFRAMES;  // mapOptmization.cpp:1841
  if (!(n > 30)) return LIOGPU_W_FEW_FEATURES;      // :1844
  return LIOGPU_OK;
}

int liogpu_scan2map(liogpu_ctx* ctx, const void* scan_ds, int n, int stride, float pose_io[6], float matP_io[36],
                    int* degenerate_io, int max_iter, liogpu_s2m_info* info) {
  NvtxRange nvtx_range_(__func__);
  int rc = enter(ctx);
  if (rc) return rc;
  Ctx* c = &ctx->c;
  if (!pose_io || !matP_io || !degenerate_io) { c->err = "liogpu_scan2map: null state pointer"; return LIOGPU_E_INVALID; }
  if (scan_ds == LIOGPU_DEVICE_RESIDENT) {
    if (!c->resident) { c->err = "LIOGPU_DEVICE_RESIDENT: no resident cloud"; return LIOGPU_E_INVALID; }
    n = c->resident_n;
  }
  if (scan_ds == LIOGPU_UPLOADED_SCAN) {
    if (c->upload_count <= 0) { c->err = "LIOGPU_UPLOADED_SCAN: no upload pending"; return LIOGPU_E_INVALID; }
    n = c->upload[c->upload_head].n;
  }
  rc = s2m_guards(c, n, info);
  if (rc) {
    if (info) info->is_degenerate = *degenerate_io;
    return rc;
  }
  rc = load_cloud(c, scan_ds, n, stride, c->scan_ds4);
  if (rc) return rc;
  if (scan_ds != LIOGPU_DEVICE_RESIDENT) clobber(c, &c->scan_ds4);
  return scan2map_dev(c, c->scan_ds4.as<float4>(), n, pose_io, matP_io, degenerate_io, max_iter, info);
}

int liogpu_scan2map_trace(liogpu_ctx* ctx, const void* scan_ds, int n, int stride, float pose_io[6], float matP_io[36],
                          int* degenerate_io, int max_iter, liogpu_s2m_info* info, int* nn_idx, float* nn_d2, float* coeff,
                          unsigned char* flag, unsigned char* tie) {
  NvtxRange nvtx_range_(__func__);
  int rc = enter(ctx);
  if (rc) return rc;
  Ctx* c = &ctx->c;
  if (!pose_io || !matP_io || !degenerate_io) { c->err = "liogpu_scan2map_trace: null state pointer"; return LIOGPU_E_INVALID; }
  if (scan_ds == LIOGPU_DEVICE_RESIDENT) {
    if (!c->resident) { c->err = "LIOGPU_DEVICE_RESIDENT: no resident cloud"; return LIOGPU_E_INVALID; }
    n = c->resident_n;
  }
  if (scan_ds == LIOGPU_UPLOADED_SCAN) {
    if (c->upload_count <= 0) { c->err = "LIOGPU_UPLOADED_SCAN: no upload pending"; return LIOGPU_E_INVALID; }
    n = c->upload[c->upload_head].n;
  }
  rc = s2m_guards(c, n, info);
  if (rc) {
    if (info) info->is_degenerate = *degenerate_io;
    return rc;
  }
  rc = load_cloud(c, scan_ds, n, stride, c->scan_ds4);
  if (rc) return rc;
  if (scan_ds != LIOGPU_DEVICE_RESIDENT) clobber(c, &c->scan_ds4);
  return scan2map_trace_dev(c, c->scan_ds4.as<float4>(), n, pose_io, matP_io, degenerate_io, max_iter, info, nn_idx, nn_d2,
                            coeff, flag, tie);
}

int liogpu_downsample_scan2map(liogpu_ctx* ctx, const void* scan, int n, int stride, float pose_io[6],
                               float matP_io[36], int* degenerate_io, int max_iter, liogpu_s2m_info* info, int* n_ds,
                               void* scan_ds_out, int out_stride, int cap_out) {
  NvtxRange nvtx_range_(__func__);
  int rc = enter(ctx);
  if (rc) return rc;
  Ctx* c = &ctx->c;
  if (!pose_io || !matP_io || !degenerate_io || !n_ds) { c->err = "liogpu_downsample_scan2map: null pointer"; return LIOGPU_E_INVALID; }
  *n_ds = 0;
  rc = load_cloud(c, scan, n, stride, c->scan4);
  if (rc) return rc;
  clobber(c, &c->scan4);
  clobber(c, &c->scan_ds4);
  int m = 0;
  bool overflow = false;
  rc = voxel_downsample_dev(c, c->scan4.as<float4>(), n, c->prm.mapping_surf_leaf_size, c->scan_ds4, &m, &overflow);
  if (rc) return rc;
  *n_ds = m;
  if (scan_ds_out == LIOGPU_DEVICE_RESIDENT) {
    c->resident = &c->scan_ds4;
    c->resident_n = m;
  } else if (scan_ds_out) {
    if (m > cap_out) { c->err = "liogpu_downsample_scan2map: output capacity too small"; return LIOGPU_E_CAPACITY; }
    rc = store_cloud(c, c->scan_ds4.as<float4>(), m, scan_ds_out, out_stride);
    if (rc) return rc;
  }
  rc = s2m_guards(c, m, info);
  if (rc) {
    if (info) info->is_degenerate = *degenerate_io;
    return rc;
  }
  rc = scan2map_dev(c, c->scan_ds4.as<float4>(), m, pose_io, matP_io, degenerate_io, max_iter, info);
  if (rc) return rc;
  return overflow ? LIOGPU_W_LEAF_OVERFLOW : LIOGPU_OK;
}

int liogpu_surf_optimization(liogpu_ctx* ctx, const void* scan_ds, int n, int stride, const float* pose6,
                             const float* T12, int* nn_idx, float* nn_d2, float* coeff, unsigned char* flag,
                             unsigned char* tie) {
  NvtxRange nvtx_range_(__func__);
  int rc = enter(ctx);
  if (rc) return rc;
  Ctx* c = &ctx->c;
  if (!c->grid_valid) { c->err = "no local map installed"; return LIOGPU_E_NO_MAP; }
  if (scan_ds == LIOGPU_DEVICE_RESIDENT) {
    if (!c->resident) { c->err = "LIOGPU_DEVICE_RESIDENT: no resident cloud"; return LIOGPU_E_INVALID; }
    n = c->resident_n;
  }
  if (c->n_map <= 0 || c->grid.n_points <= 0) {  // empty map: no neighbours, nothing accepted
    for (int i = 0; i < n; ++i) {
      for (int j = 0; j < 5; ++j) {
        if (nn_idx) nn_idx[i * 5 + j] = -1;
        if (nn_d2) nn_d2[i * 5 + j] = 1.0f;
      }
      if (coeff) coeff[i * 4] = coeff[i * 4 + 1] = coeff[i * 4 + 2] = coeff[i * 4 + 3] = 0.f;
      if (flag) flag[i] = 0;
      if (tie) tie[i] = 0;
    }
    return LIOGPU_OK;
  }
  rc = load_cloud(c, scan_ds, n, stride, c->scan_ds4);
  if (rc) return rc;
  if (scan_ds != LIOGPU_DEVICE_RESIDENT) clobber(c, &c->scan_ds4);
  return surf_optimization_dev(c, c->scan_ds4.as<float4>(), n, pose6, T12, nn_idx, nn_d2, coeff, flag, tie);
}

int liogpu_fetch_result(liogpu_ctx* ctx, void* xyzi_out, int out_stride, int cap_out, int* n_out) {
  NvtxRange nvtx_range_(__func__);
  if (!ctx) return LIOGPU_E_INVALID;
  Ctx* c = &ctx->c;
  c->err.clear();
  if (cudaSetDevice(c->device) != cudaSuccess) { c->err = "cudaSetDevice failed"; return LIOGPU_E_CUDA; }
  if (!n_out) { c->err = "liogpu_fetch_result: null n_out"; return LIOGPU_E_INVALID; }
  if (!c->last_result) { c->err = "liogpu_fetch_result: no result pending (it serves only the call right before it)"; return LIOGPU_E_INVALID; }
  *n_out = c->last_result_n;
  if (c->last_result_n > cap_out) { c->err = "liogpu_fetch_result: output capacity too small"; return LIOGPU_E_CAPACITY; }
  const int rc = store_cloud(c, c->last_result, c->last_result_n, xyzi_out, out_stride);
  return rc ? rc : c->last_result_status;  // the producing call's warning travels with its result
}

int liogpu_upload_scan_async(liogpu_ctx* ctx, const void* xyzi, int n, int stride) {
  NvtxRange nvtx_range_(__func__);
  if (!ctx) return LIOGPU_E_INVALID;
  Ctx* c = &ctx->c;
  // touches only the upload slots and the copy stream, so it may overlap ONE other call on the context (the node
  // starts the copy when the message arrives, before it takes mtx)
  if (cudaSetDevice(c->device) != cudaSuccess) return LIOGPU_E_CUDA;
  if (n < 0 || (n > 0 && !xyzi) || !stride_ok(stride)) return LIOGPU_E_INVALID;
  if (c->upload_count >= 2) return LIOGPU_E_CAPACITY;  // two sweeps already on their way
  Ctx::Upload& u = c->upload[(c->upload_head + c->upload_count) & 1];
  if (u.raw.reserve((size_t)(n > 0 ? n : 1) * stride) != cudaSuccess) return LIOGPU_E_CUDA;
  if (n > 0 && cudaMemcpyAsync(u.raw.p, xyzi, (size_t)n * stride,
                               is_device_ptr(xyzi) ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, c->copy_stream) != cudaSuccess)
    return LIOGPU_E_CUDA;
  if (cudaEventRecord(u.ev, c->copy_stream) != cudaSuccess) return LIOGPU_E_CUDA;
  u.n = n; u.stride = stride; u.valid = true;
  c->upload_count++;
  return LIOGPU_OK;
}

float liogpu_last_gpu_ms(const liogpu_ctx* ctx) { return ctx ? ctx->c.last_ms : 0.f; }
unsigned long long liogpu_launch_count(const liogpu_ctx* ctx) { return ctx ? ctx->c.launches : 0ULL; }
void* liogpu_stream(const liogpu_ctx* ctx) { return ctx ? (void*)ctx->c.stream : nullptr; }

}  // extern "C"
