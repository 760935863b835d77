// common.cuh — shared definitions of libliogpu (sm_100a).  Product code: never includes oracle/.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <float.h>
#include <string.h>
#include <string>
#include <vector>
#include <map>

#include "../../include/liogpu.h"

namespace liogpu {

// ---- device buffer that grows on demand (steady state: no allocation on the per-scan path) ----
// Context buffers are allocated STREAM-ORDERED on the context's stream (cudaMallocAsync / cudaFreeAsync): growing one
// never synchronises the device, so several contexts sharing a GPU (batch offline mapping, one sequence per context)
// do not stall each other while their buffers find their size.
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaStream_t stream = nullptr;
  bool async = false;   // stream-ordered allocation on `stream`
  bool pooled = false;  // carved out of a slab (keyframe pool): never freed individually
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (pooled) return cudaErrorMemoryAllocation;
    size_t want = bytes + bytes / 2 + 4096;
    void* np_ = nullptr;
    cudaError_t e = async ? cudaMallocAsync(&np_, want, stream) : cudaMalloc(&np_, want);
    if (e != cudaSuccess) return e;
    if (p) { if (async) cudaFreeAsync(p, stream); else cudaFree(p); }
    p = np_;
    cap = want;
    return cudaSuccess;
  }
  void release() {
    if (p && !pooled) { if (async) cudaFreeAsync(p, stream); else cudaFree(p); }
    p = nullptr;
    cap = 0;
    pooled = false;
  }
  template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

// ---- voxel grid parameters computed on device by voxel_setup_kernel (SURVEY A.1 steps 1-4) ----
struct VoxelSetup {
  float min_p[3], max_p[3];
  float inv_leaf;
  int min_b[3];
  int div_b[3];
  int mul1, mul2;
  int overflow;       // 1 = guard fired (output = input)
  unsigned n_cells;   // div.x*div.y*div.z (valid when !overflow)
  int n_valid;        // finite points
  int key_bits;       // bits needed to sort keys in [0, n_cells]
  unsigned n_vox;     // number of occupied voxels (written by the last stage)
};

// ---- sorted-grid 5-NN index over the local map ----
struct GridParams {
  float ox, oy, oz;   // origin = per-axis minimum of the map
  float h, inv_h;     // cell edge
  float slack;        // positional slack covering f32 rounding of the cell assignment
  int nx, ny, nz;
  int n_points;
  unsigned n_cells;
  float gate_d2;      // squared search radius (1.0 for surfOptimization, MO:1641)
  float gate1_d2;     // squared radius of the cheap first search phase (>= gate_d2 disables it)
};

#define LIOGPU_FZ_K 8  // members of a point's candidate set (s2m_fused.cuh)

// ---- state of the LM loop kept on device between iterations (MO:171,176,177) ----
struct LmDevState {
  float T[12];     // transPointAssociateToMap of `pose` (MO:1615), refreshed after every pose update
  float trig[6];   // srx, crx, sry, cry, srz, crz of `pose` (MO:1714-1719)
  float pose[6];
  float matP[36];
  int degenerate;
  int iter;        // iterations executed so far
  int done;        // converged or max_iter reached
  int converged;
  int max_iter;
  int n_sel;
  int tie_queries;
  float delta_r, delta_t;
  double JtJ[36];
  double Jtr[6];
  float pose_hist[LIOGPU_MAX_ITER][6];
  int nsel_hist[LIOGPU_MAX_ITER];
  // iteration-0 eigen analysis moved off the critical path (s2m.cu: lm_matp_kernel)
  float AtA0[36];     // AtA of iteration 0 (f32, as cv::eigen sees it)
  int eig_pending;    // 1: matP still has to be computed from AtA0 by lm_matp_kernel
  int cert_mismatch;  // must stay 0: the side computation contradicted the non-degeneracy certificate
  int seeded;         // points of the last executed iteration that started from the previous neighbours
  // ---- fused persistent loop (s2m_fused.cuh); zeroed with the rest of the block at every registration ----
  float T_prev[12];   // transform of the previous iteration: where every point stood when its candidate set was certified
  unsigned fz_ticket_a[LIOGPU_MAX_ITER];  // CTAs that finished the main phase, per iteration
  unsigned fz_ticket_b[LIOGPU_MAX_ITER];  // CTAs that finished the deferred-leftover phase, per iteration
  unsigned fz_phase;                      // 2*it+1: iteration it needs the deferred-leftover phase; 2*it+2: iteration it done
  unsigned fz_queue[LIOGPU_MAX_ITER];     // chunk queue head, one per iteration
  unsigned fz_deferred[LIOGPU_MAX_ITER];  // leftovers deferred to the grid-wide phase, per iteration
  int certified;      // last executed iteration: points whose five neighbours came from the certificate (no grid walk)
  int leftovers;      // last executed iteration: points finished by the warp-cooperative full-gate search
  int cert_hist[LIOGPU_MAX_ITER], left_hist[LIOGPU_MAX_ITER], seed_hist[LIOGPU_MAX_ITER];
  int main_finalized_iter;  // two-kernel path: value of `iter` after the main kernel's last block ran the tail itself
};

// ---- loop-closure detection (loopdetect.cu) ----
// SCManager's descriptor store (polarcontexts_ and its keys), one entry per liogpu_sc_add-ed descriptor: the f64
// descriptor [SC_BINS], the f32 ring key [20], the f64 sector key [60] and the f64 column norms [60], in four arrays of
// `cap` entries.  Grows geometrically (stream-ordered, contents carried over); emptied but kept by liogpu_sc_clear.
struct ScStore {
  double* desc = nullptr;
  float* rkey = nullptr;
  double* vkey = nullptr;
  double* cnorm = nullptr;
  int count = 0, cap = 0;
  long long counter = 0;  // tree_making_period_conter
  int snap = 0;           // size of the tree's snapshot (a prefix of the store)
};
// result of one detectLoopClosureID query, as the device leaves it
struct ScQueryOut {
  int n_cand, ties, nn_idx, nn_align, loop_id;
  float yaw;
  double min_dist;
};

// host-visible context
struct Ctx {
  liogpu_params prm;
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  cudaStream_t side_stream = nullptr;  // iteration-0 eigen analysis, overlapped with iterations 1..
  cudaEvent_t ev_it0 = nullptr, ev_side = nullptr;
  std::vector<cudaEvent_t> prof_ev;  // params.profile_kernels: 3 events per iteration of a chunk
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  std::string err;
  unsigned long long launches = 0;
  float last_ms = 0.f;

  // staging
  DevBuf raw_in, raw_out;
  // scan / queries
  DevBuf scan4, scan_ds4;
  // local map + grid
  DevBuf map_raw4, map4, map_sorted, cell_start;
  int n_map = 0;
  bool grid_valid = false;
  GridParams grid{};
  // sort + scan scratch
  DevBuf keys0, keys1, vals0, vals1, counters, scan_tmp, seg_flag, seg_start;
  // small device structs
  DevBuf vox_setup, grid_setup, minmax, lm_state, partials, block_counter, misc, fail_buf, prev_nn, hopeless;
  // fused persistent loop: per-chunk / per-CTA partial rows, leftover segments, candidate-set bounds, probes
  DevBuf fz_rows, fz_left, fz_lb, fz_probe;
  // tile-sharded rebuild (tile.cu)
  DevBuf tile_plan, tile_hist, tile_pts, tile_out;
  cudaEvent_t ev_mid = nullptr;
  int fz_grid = 0;        // CTAs of the cooperative launch (0 = not yet queried, < 0 = unavailable)
  // per-point debug outputs of surf_optimization
  DevBuf dbg_idx, dbg_d2, dbg_coeff, dbg_flag, dbg_tie;
  // pinned host mirrors
  void* h_pinned = nullptr;  // 128 KiB: small readbacks in the first 64 KiB, IMU table in the second
  // keyframes (lidar frame, packed float4), carved out of 32 MiB slabs: surfCloudKeyFrames.push_back (MO:2142) costs
  // no cudaMalloc (which would synchronise the whole device, i.e. every other context on it)
  std::map<int, std::pair<DevBuf, int>> keyframes;
  std::vector<void*> kf_slabs;
  std::vector<size_t> kf_slab_sizes;
  size_t kf_slab_cur = 0, kf_slab_used = 0;  // slab being filled, bytes used in it
  // deskew
  DevBuf imu_tab, dsk_flags, dsk_scan;
  // publishLocalMap (localmap.cu): crop / outlier-filter scratch and the filter's own neighbour grid
  DevBuf lm_flag, lm_pos, lm_a, lm_b, lm_md, lm_left, lm_out, lm_stats, sor_setup, sor_sorted, sor_cell_start;
  // device-resident hand-off (LIOGPU_DEVICE_RESIDENT)
  DevBuf* resident = nullptr;
  int resident_n = 0;
  // keyframe tables of the multi-keyframe calls (poses | offsets | source pointers), sized from k
  void* h_kf_tab = nullptr;
  size_t h_kf_cap = 0;
  DevBuf kf_tab;
  // result of the last build_local_map / merge_keyframes / publish_local_map / voxel_tile, for liogpu_fetch_result
  const float4* last_result = nullptr;
  int last_result_n = 0;
  int last_result_status = 0;  // the warning the producing call would have returned (LIOGPU_W_LEAF_OVERFLOW)
  // liogpu_upload_scan_async: two staging slots filled on a copy stream
  cudaStream_t copy_stream = nullptr;
  struct Upload { DevBuf raw; cudaEvent_t ev = nullptr; int n = 0, stride = 0; bool valid = false; } upload[2];
  int upload_head = 0, upload_count = 0;  // FIFO: a consumer takes the OLDEST pending upload
  // loop-closure detection: the descriptor store and the per-call scratch (queries, partial top-k lists, candidates)
  ScStore sc;
  DevBuf sc_q, sc_part, sc_cand, sc_out;
  // batched loop-closure ICP: the group's source / target submaps (packed float4, one segment per pair) and its
  // device tables (per-pair offsets, grids, ICP states, reduce partials)
  DevBuf lc_src, lc_tgt, lc_tab;
  // segmented VoxelGrid over many keyframe windows (voxel.cu merge_windows_dev): per-window tables of a pass, and the
  // segment table of the copy that places the windows' clouds
  DevBuf mw_tab, mw_seg;
};

#define LIOGPU_CUDA_OK(ctx, expr)                                                        \
  do {                                                                                   \
    cudaError_t e__ = (expr);                                                            \
    if (e__ != cudaSuccess) {                                                            \
      (ctx)->err = std::string(#expr) + ": " + cudaGetErrorString(e__);                  \
      return LIOGPU_E_CUDA;                                                              \
    }                                                                                    \
  } while (0)

// kernels' launch wrappers (each returns cudaError_t from cudaGetLastError)
// --- layout.cu
cudaError_t launch_unpack(Ctx* c, const void* d_raw, int n, int stride, float4* out);
cudaError_t launch_pack(Ctx* c, const float4* in, int n, void* d_raw, int stride);
cudaError_t launch_transform(Ctx* c, const float4* in, int n, const float* d_pose6, float4* out);
cudaError_t launch_pose_table(Ctx* c, const float* d_poses6, int k, float* d_T12);
cudaError_t launch_transform_multi(Ctx* c, const float4* const* d_srcs, const int* d_offs, int k, const float* d_poses6,
                                   float* d_T12, long long total, float4* out);
// --- sort.cu
cudaError_t radix_sort_pairs(Ctx* c, int n, int key_bits, const int* d_key_bits, uint32_t** keys_out,
                             uint32_t** vals_out);
cudaError_t exclusive_scan_u32(Ctx* c, const uint32_t* in, uint32_t* out, int n, uint32_t* d_total);
// --- api.cu
// The k named keyframes as device tables for launch_transform_multi (ids must have been validated by the caller or
// are refused here with LIOGPU_E_NO_KEYFRAME).  The tables are staged in pinned memory that the next call reuses, so
// the stream must have passed the upload before stage_keyframes runs again.
struct KfTables {
  const float4* const* srcs;
  const int* offs;
  const float* poses;
  float* T12;
  size_t total;
};
int stage_keyframes(Ctx* c, const char* who, const int* ids, const float* pose6s, int k, KfTables& t);
// grows `b` to `need` bytes keeping its first `used` bytes (stream-ordered, like DevBuf::reserve)
int reserve_keep(Ctx* c, DevBuf& b, size_t need, size_t used);
// --- voxel.cu
cudaError_t launch_minmax(Ctx* c, const float4* pts, int n, unsigned* mm);
int voxel_downsample_dev(Ctx* c, const float4* in, int n, float leaf, DevBuf& out, int* n_out, bool* overflow);
// liogpu_merge_keyframes of n_windows windows (window w = ids / pose6s entries [win_off[w], win_off[w+1]), host
// arrays, ids validated, input total <= INT32_MAX): the clouds go to `out` one after another in window order, window w
// at records [out_off[w], out_off[w+1]); overflow[w] = its VoxelGrid guard fired.  Each window's cloud is bit-equal
// to the single-window call whatever windows surround it.  `out` must not be lm_a, lm_out or mw_seg.
int merge_windows_dev(Ctx* c, const int* ids, const float* pose6s, const int* win_off, int n_windows, float leaf,
                      DevBuf& out, int* out_off, int* overflow);
// dst[off[s] .. off[s+1]) = srcs[s][0 .. off[s+1] - off[s]) for every segment s, in one launch (off[0] = 0)
int gather_segments(Ctx* c, const std::vector<const float4*>& srcs, const std::vector<int>& off, float4* dst);
// --- tile.cu
int voxel_tile_dev(Ctx* c, const float4* pts, int n, float leaf, int tile, int n_tiles, DevBuf& out, int* n_out,
                   bool* overflow, liogpu_tile_info* info);
// --- grid.cu
int grid_build_dev(Ctx* c, const float4* map4, int n, float leaf_hint);
int grid_build_core(Ctx* c, const float4* pts, int n, float cell, float gate_d2, float gate1_d2, DevBuf& setup,
                    DevBuf& sorted, DevBuf& cell_start_buf, GridParams& host_gp);
// --- localmap.cu
int publish_local_map_dev(Ctx* c, const float4* const* d_srcs, const int* d_offs, int k, const float* d_poses6,
                          float* d_T12, long long total, const float* h_yaw16, const liogpu_local_map_params* prm,
                          const float4** result, int* n_result, liogpu_local_map_info* info);
// --- nearby.cu
int extract_nearby_dev(Ctx* c, const float4* key3d, int n, const double* h_times, double time_cur, float radius,
                       float density, int* ids, int cap, int* n_ids);
// --- scancontext.cu
int scancontext_dev(Ctx* c, const float4* pts, int n, double lidar_height, double max_radius, double* h_out);
// --- loopdetect.cu
int sc_add_dev(Ctx* c, const double* descs, int n);
void sc_release(Ctx* c);
int sc_detect_dev(Ctx* c, const std::vector<int2>& qm, int k, int R, double thres, ScQueryOut* h_out, liogpu_sc_info* info);
int detect_loop_distance_dev(Ctx* c, const float4* key3d, int n, const double* h_times, double time_cur, float radius,
                             float time_diff, int* loop_key_pre);
// --- icp.cu
int icp_align_dev(Ctx* c, const float4* src, int ns, const float4* tgt, int nt, const liogpu_icp_params* prm,
                  float final_T[16], liogpu_icp_info* info);
// n pairs at once: pair p's source is src[src_off[p] .. src_off[p+1]), its target tgt[tgt_off[p] .. tgt_off[p+1])
// (offsets in records, n + 1 entries each, every segment non-empty).  Each pair's result is bit-equal to icp_align_dev
// on its two segments.
int icp_batch_dev(Ctx* c, const float4* src, const int* src_off, const float4* tgt, const int* tgt_off, int n,
                  const liogpu_icp_params* prm, float (*final_T)[16], liogpu_icp_info* info);
// --- s2m.cu
int scan2map_dev(Ctx* c, const float4* scan4, int n, float pose_io[6], float matP_io[36], int* degenerate_io,
                 int max_iter, liogpu_s2m_info* info);
int scan2map_trace_dev(Ctx* c, const float4* scan4, int n, float pose_io[6], float matP_io[36], int* degenerate_io,
                       int max_iter, liogpu_s2m_info* info, int* nn_idx, float* nn_d2, float* coeff, unsigned char* flag,
                       unsigned char* tie);
int surf_optimization_dev(Ctx* c, const float4* scan4, int n, const float* pose6, const float* T12, int* nn_idx,
                          float* nn_d2, float* coeff, unsigned char* flag, unsigned char* tie);
// --- deskew.cu
int deskew_dev(Ctx* c, const void* d_raw, int n, int stride, double t_scan, const double* imu4_host, int n_imu,
               int enabled, DevBuf& out, int* n_out);

static inline int div_up(long long a, long long b) { return (int)((a + b - 1) / b); }

}  // namespace liogpu
