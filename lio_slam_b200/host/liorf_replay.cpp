// liorf_replay.cpp — see liorf_replay.h.  The loop body follows laserCloudInfoHandler (mapOptmization.cpp:432-506)
// and cloudHandler (imageProjection.cpp:206) line by line; everything device-side goes through the mirrored member
// functions of map_optimization_gpu.h.
#include "liorf_replay.h"

#include <chrono>
#include <cstdio>
#include <cstring>
#include <exception>
#include <memory>

#include "map_optimization_gpu.h"

using namespace liorf_gpu;
typedef std::chrono::steady_clock Clock;
static inline double ms_since(const Clock::time_point& t0) { return std::chrono::duration<double, std::milli>(Clock::now() - t0).count(); }

struct liorf_worker {
  liogpu_params params;
  liogpu_ctx* ctx;
};

static int replay_impl(const liogpu_params* params, liogpu_ctx* borrowed, const liorf_replay_options* options, const liorf_sweep* sweeps,
                       int n, float* poses_out, int* iters_out, int* nds_out, liorf_replay_stats* stats, char* err, int err_len);

extern "C" liorf_worker* liorf_worker_create(const liogpu_params* params, char* err, int err_len) {
  if (err && err_len > 0) err[0] = 0;
  if (!params) return nullptr;
  liorf_worker* w = new liorf_worker();
  w->params = *params;
  w->ctx = nullptr;
  if (liogpu_create(&w->ctx, params) != LIOGPU_OK) {
    if (err && err_len > 0) std::snprintf(err, (size_t)err_len, "liogpu_create failed (no sm_100 GPU? there is no CPU fallback)");
    delete w;
    return nullptr;
  }
  return w;
}
extern "C" void liorf_worker_destroy(liorf_worker* w) {
  if (!w) return;
  liogpu_destroy(w->ctx);
  delete w;
}
extern "C" int liorf_worker_replay(liorf_worker* w, const liorf_replay_options* options, const liorf_sweep* sweeps, int n,
                                   float* poses_out, int* iters_out, int* nds_out, liorf_replay_stats* stats, char* err, int err_len) {
  if (!w) return LIOGPU_E_INVALID;
  int rc = liogpu_keyframe_clear(w->ctx);  // a new sequence starts with an empty map
  if (rc < 0) return rc;
  rc = liogpu_sc_clear(w->ctx);            // ... and a fresh SCManager
  if (rc < 0) return rc;
  return replay_impl(&w->params, w->ctx, options, sweeps, n, poses_out, iters_out, nds_out, stats, err, err_len);
}
extern "C" int liorf_replay_sequence(const liogpu_params* params, const liorf_replay_options* options, const liorf_sweep* sweeps,
                                     int n, float* poses_out, int* iters_out, int* nds_out, liorf_replay_stats* stats, char* err,
                                     int err_len) {
  return replay_impl(params, nullptr, options, sweeps, n, poses_out, iters_out, nds_out, stats, err, err_len);
}

static int replay_impl(const liogpu_params* params, liogpu_ctx* borrowed, const liorf_replay_options* options, const liorf_sweep* sweeps,
                       int n, float* poses_out, int* iters_out, int* nds_out, liorf_replay_stats* stats, char* err, int err_len) {
  if (err && err_len > 0) err[0] = 0;
  if (!params || !sweeps || n < 0) return LIOGPU_E_INVALID;
  liorf_replay_stats st;
  std::memset(&st, 0, sizeof(st));
  liorf_replay_options opt;
  std::memset(&opt, 0, sizeof(opt));
  if (options) opt = *options;
  int rc = LIOGPU_OK;
  try {
    std::unique_ptr<mapOptimization> mo(borrowed ? new mapOptimization(*params, borrowed) : new mapOptimization(*params));
    mapOptimization& MO = *mo;
    ImageProjection IP(MO.context());   // co-located nodes: one context, the deskewed sweep never leaves HBM
    MO.selectKeyPosesOnDevice = opt.select_key_poses_on_device != 0;
    if (opt.keyframe_dist > 0.f) MO.surroundingkeyframeAddingDistThreshold = opt.keyframe_dist;
    if (opt.keyframe_angle > 0.f) MO.surroundingkeyframeAddingAngleThreshold = opt.keyframe_angle;
    if (opt.search_radius > 0.f) MO.surroundingKeyframeSearchRadius = opt.search_radius;
    if (opt.density > 0.f) MO.surroundingKeyframeDensity = opt.density;
    MO.detectLoopDistanceOnDevice = true;  // the replay runs both detectors through the library
    const unsigned long long launches0 = liogpu_launch_count(MO.context());
    const Clock::time_point t_all = Clock::now();
    int last_map_n = -1;
    for (int s = 0; s < n && rc >= 0; ++s) {
      const liorf_sweep& sw = sweeps[s];
      // ---- ImageProjection::cloudHandler: imuDeskewInfo stays host (tables given), projectPointCloud on device ----
      Clock::time_point t0 = Clock::now();
      IP.timeScanCur = sw.time_scan_cur;
      IP.imuAvailable = sw.n_imu > 0;
      IP.imuPointerCur = sw.n_imu - 1;
      IP.imuTime.assign(sw.imu, sw.imu + sw.n_imu);
      IP.imuRotX.assign(sw.imu + sw.n_imu, sw.imu + 2 * sw.n_imu);
      IP.imuRotY.assign(sw.imu + 2 * sw.n_imu, sw.imu + 3 * sw.n_imu);
      IP.imuRotZ.assign(sw.imu + 3 * sw.n_imu, sw.imu + 4 * sw.n_imu);
      int n_deskewed = 0;
      rc = IP.projectPointCloudResident(static_cast<const PointXYZIRT*>(sw.raw), sw.n_raw, &n_deskewed);
      if (rc < 0) break;
      st.h2d_bytes += (long long)sw.n_raw * (long long)sizeof(PointXYZIRT) + (long long)sw.n_imu * 32;
      st.deskew_ms += ms_since(t0);
      // ---- mapOptimization::laserCloudInfoHandler (:432-506) ----
      MO.timeLaserInfoCur = sw.time_scan_cur;
      std::memcpy(MO.transformTobeMapped, sw.guess, sizeof(sw.guess));  // updateInitialGuess (:1438-1502) stays host
      t0 = Clock::now();
      MO.extractSurroundingKeyFrames();                                  // :469
      if (MO.lastStatus < 0) { rc = MO.lastStatus; break; }
      if (MO.laserCloudSurfFromMapDSNum != last_map_n) { ++st.map_rebuilds; last_map_n = MO.laserCloudSurfFromMapDSNum; }
      st.nearby_ms += ms_since(t0);
      t0 = Clock::now();
      const bool had_keyframes = !MO.cloudKeyPoses3D.empty();
      MO.downsampleAndScan2MapResident();                                // :474 + :479
      if (MO.lastStatus < 0) { rc = MO.lastStatus; break; }
      if (had_keyframes) {
        ++st.registered;
        st.lm_iterations += MO.lastInfo.iterations;
        st.loop_gpu_ms += MO.lastInfo.gpu_ms;
        st.d2h_bytes += 2520;  // sizeof(LmDevState): the one read-back of a registration
        st.h2d_bytes += 2520;
      }
      st.register_ms += ms_since(t0);
      t0 = Clock::now();
      if (MO.saveFrame()) {                                              // saveKeyFramesAndFactor (:2085), gate :1909-1928
        MO.saveKeyFrameResident();
        if (MO.lastStatus < 0) { rc = MO.lastStatus; break; }
        if (opt.loop_detection_every > 0) {                              // :2151-2166
          MO.makeAndSaveScancontextAndKeys();
          if (MO.lastStatus < 0) { rc = MO.lastStatus; break; }
        }
      }
      if (opt.loop_detection_every > 0 && (s + 1) % opt.loop_detection_every == 0 && !MO.cloudKeyPoses3D.empty()) {
        int cur = -1, pre = -1;                                          // loopClosureThread: RS, then SC
        if (MO.detectLoopClosureDistance(&cur, &pre)) ++st.loops_rs;
        if (MO.lastStatus < 0) { rc = MO.lastStatus; break; }
        if (MO.detectLoopClosureID().first != -1) ++st.loops_sc;
        if (MO.lastStatus < 0) { rc = MO.lastStatus; break; }
      }
      if (opt.publish_local_map) {
        MO.publishLocalMap();                                            // :504
        if (MO.lastStatus < 0) { rc = MO.lastStatus; break; }
        st.d2h_bytes += (long long)MO.localMapCloud.size() * (long long)sizeof(PointType);
      }
      st.keyframe_ms += ms_since(t0);
      if (poses_out) std::memcpy(poses_out + 6 * (size_t)s, MO.transformTobeMapped, 6 * sizeof(float));
      if (iters_out) iters_out[s] = had_keyframes ? MO.lastInfo.iterations : 0;
      if (nds_out) nds_out[s] = MO.laserCloudSurfLastDSNum;
      ++st.scans;
    }
    st.wall_ms = ms_since(t_all);
    st.keyframes = (int)MO.cloudKeyPoses3D.size();
    st.map_points_last = MO.laserCloudSurfFromMapDSNum;
    st.gpu_launches = liogpu_launch_count(MO.context()) - launches0;
    if (rc < 0 && err && err_len > 0) std::snprintf(err, (size_t)err_len, "%s", MO.lastError());
  } catch (const std::exception& e) {
    if (err && err_len > 0) std::snprintf(err, (size_t)err_len, "%s", e.what());
    rc = LIOGPU_E_CUDA;
  }
  if (stats) *stats = st;
  return rc < 0 ? rc : 0;
}
