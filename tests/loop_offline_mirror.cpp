// mapOptimization::performLoopClosuresOffline against the loop thread run tick by tick (performRSLoopClosure, then
// performSCLoopClosure) on a node whose key poses and Scan Context descriptors grow as the keyframes arrive.
// Built and run by tests/test_gpu_loop_distance_batch.py and tests/perf/bench_loop_distance_batch.py.
//
// Input (little-endian): int n_key, int n_pool, int search_num, int num_exclude_recent, float radius, float time_diff;
// n_pool clouds (int n, n * 4 f32 xyzi); n_key pool indices (i32); n_key poses (6 f32: roll pitch yaw x y z);
// n_key times (f64); int n_ticks; n_ticks x (int n_key, f64 time).
// Output: one line of "name value" pairs; exit code 1 when any tick differs.
#include <chrono>
#include <cstdio>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "map_optimization_gpu.h"
using namespace liorf_gpu;

template <class T> static bool rd(FILE* f, T* p, size_t n) { return std::fread(p, sizeof(T), n, f) == n; }

static void configure(mapOptimization& mo, int search_num, int exclude, float radius, float time_diff) {
  mo.historyKeyframeSearchNum = search_num;
  mo.historyKeyframeSearchRadius = radius;
  mo.historyKeyframeSearchTimeDiff = time_diff;
  mo.scParams.num_exclude_recent = exclude;
}

static bool same_half(const mapOptimization::LoopHalfOutcome& a, const mapOptimization::LoopHalfOutcome& b) {
  return a.loopKeyCur == b.loopKeyCur && a.loopKeyPre == b.loopKeyPre && a.accepted == b.accepted &&
         std::memcmp(a.correctionLidarFrame, b.correctionLidarFrame, sizeof(a.correctionLidarFrame)) == 0 &&
         std::memcmp(&a.noiseScore, &b.noiseScore, sizeof(float)) == 0;
}

int main(int argc, char** argv) {
  FILE* f = std::fopen(argv[1], "rb");
  if (!f) return 2;
  int n_key = 0, n_pool = 0, search_num = 0, exclude = 0, n_ticks = 0;
  float radius = 0.f, time_diff = 0.f;
  if (!rd(f, &n_key, 1) || !rd(f, &n_pool, 1) || !rd(f, &search_num, 1) || !rd(f, &exclude, 1) || !rd(f, &radius, 1) ||
      !rd(f, &time_diff, 1))
    return 2;
  std::vector<Cloud> pool(n_pool);
  for (Cloud& c : pool) {
    int n = 0;
    if (!rd(f, &n, 1)) return 2;
    std::vector<float> xyzi((size_t)n * 4);
    if (!rd(f, xyzi.data(), xyzi.size())) return 2;
    c.resize(n);
    for (int i = 0; i < n; ++i) {
      PointType p{};
      p.x = xyzi[4 * i]; p.y = xyzi[4 * i + 1]; p.z = xyzi[4 * i + 2]; p.intensity = xyzi[4 * i + 3];
      c[i] = p;
    }
  }
  std::vector<int> which(n_key);
  std::vector<float> p6((size_t)n_key * 6);
  std::vector<double> times(n_key);
  if (!rd(f, which.data(), which.size()) || !rd(f, p6.data(), p6.size()) || !rd(f, times.data(), times.size()) ||
      !rd(f, &n_ticks, 1))
    return 2;
  std::vector<mapOptimization::LoopTick> ticks(n_ticks);
  for (auto& t : ticks)
    if (!rd(f, &t.n_key, 1) || !rd(f, &t.timeLaserInfoCur, 1)) return 2;
  std::fclose(f);
  std::vector<PointType> k3(n_key);
  std::vector<PointTypePose> k6(n_key);
  for (int k = 0; k < n_key; ++k) {
    const float* q = &p6[(size_t)k * 6];
    PointType a{};
    a.x = q[3]; a.y = q[4]; a.z = q[5]; a.data3 = 1.f; a.intensity = (float)k;
    PointTypePose b{};
    b.x = a.x; b.y = a.y; b.z = a.z; b.intensity = a.intensity; b.roll = q[0]; b.pitch = q[1]; b.yaw = q[2];
    b.time = times[k];
    k3[k] = a;
    k6[k] = b;
  }
  liogpu_params prm;
  liogpu_default_params(&prm);
  mapOptimization online(prm), offline(prm);
  for (mapOptimization* mo : {&online, &offline}) {
    configure(*mo, search_num, exclude, radius, time_diff);
    for (int k = 0; k < n_key; ++k) {
      const Cloud& c = pool[which[k]];
      if (liogpu_keyframe_put(mo->context(), k, c.data(), (int)c.size(), sizeof(PointType)) != LIOGPU_OK) return 3;
    }
  }

  // the loop thread, one tick at a time; the descriptors are appended as the keyframes arrive
  std::vector<mapOptimization::LoopTickOutcome> want(n_ticks);
  std::map<int, char> closedBy;  // cur -> the half that recorded it last
  int online_icp = 0, rs_suppressed = 0, rs_suppressed_after_sc = 0, repeated_ticks = 0, below_exclude = 0;
  double online_ms = 0;
  for (int j = 0; j < n_ticks; ++j) {
    const int n = ticks[j].n_key;
    while ((int)online.cloudKeyPoses3D.size() < n) {
      const int k = (int)online.cloudKeyPoses3D.size();
      online.cloudKeyPoses3D.push_back(k3[k]);
      online.cloudKeyPoses6D.push_back(k6[k]);
      if (liogpu_sc_add_keyframes(online.context(), &k, 1, 2.0, 80.0, nullptr) != LIOGPU_OK) return 3;
    }
    online.timeLaserInfoCur = ticks[j].timeLaserInfoCur;
    if (j > 0 && n == ticks[j - 1].n_key) ++repeated_ticks;
    if (n > 0 && n < exclude + 1) ++below_exclude;
    if (n > 0 && online.loopIndexContainer.count(n - 1)) {
      ++rs_suppressed;
      if (closedBy[n - 1] == 's') ++rs_suppressed_after_sc;
    }
    mapOptimization::LoopTickOutcome& o = want[j];
    const auto t0 = std::chrono::steady_clock::now();
    o.rs.accepted = online.performRSLoopClosure(&o.rs.loopKeyCur, &o.rs.loopKeyPre, o.rs.correctionLidarFrame, &o.rs.noiseScore);
    if (o.rs.accepted) closedBy[o.rs.loopKeyCur] = 'r';
    o.sc.accepted = online.performSCLoopClosure(&o.sc.loopKeyCur, &o.sc.loopKeyPre, o.sc.correctionLidarFrame, &o.sc.noiseScore);
    if (o.sc.accepted) closedBy[o.sc.loopKeyCur] = 's';
    online_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    online_icp += (o.rs.loopKeyPre >= 0) + (o.sc.loopKeyPre >= 0);
  }

  // the whole sequence in one pass
  offline.cloudKeyPoses3D = k3;
  offline.cloudKeyPoses6D = k6;
  std::vector<mapOptimization::LoopTickOutcome> got;
  int offline_icp = 0;
  const auto t0 = std::chrono::steady_clock::now();
  const int st = offline.performLoopClosuresOffline(ticks, got, &offline_icp);
  const double offline_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  if (st != LIOGPU_OK) { std::printf("offline pass failed (%d): %s\n", st, offline.lastError()); return 4; }

  int bad = 0, rs_det = 0, rs_acc = 0, sc_det = 0, sc_acc = 0, rs_clamped = 0, sc_clamped = 0;
  for (int j = 0; j < n_ticks; ++j) {
    const bool ok = same_half(want[j].rs, got[j].rs) && same_half(want[j].sc, got[j].sc);
    if (!ok && bad++ < 10)
      std::fprintf(stderr, "tick %d (n_key %d): rs %d/%d/%d vs %d/%d/%d, sc %d/%d/%d vs %d/%d/%d\n", j, ticks[j].n_key,
                   want[j].rs.loopKeyCur, want[j].rs.loopKeyPre, want[j].rs.accepted, got[j].rs.loopKeyCur,
                   got[j].rs.loopKeyPre, got[j].rs.accepted, want[j].sc.loopKeyCur, want[j].sc.loopKeyPre,
                   want[j].sc.accepted, got[j].sc.loopKeyCur, got[j].sc.loopKeyPre, got[j].sc.accepted);
    const int n = ticks[j].n_key;
    if (want[j].rs.loopKeyPre >= 0) {
      ++rs_det;
      rs_acc += want[j].rs.accepted;
      rs_clamped += want[j].rs.loopKeyPre + search_num >= n;
    }
    if (want[j].sc.loopKeyPre >= 0) {
      ++sc_det;
      sc_acc += want[j].sc.accepted;
      sc_clamped += want[j].sc.loopKeyPre + search_num >= n;
    }
  }
  if (online.loopIndexContainer != offline.loopIndexContainer) ++bad;
  std::printf("mismatched %d ticks %d rs_detected %d rs_accepted %d sc_detected %d sc_accepted %d rs_clamped %d "
              "sc_clamped %d rs_suppressed %d rs_suppressed_after_sc %d repeated_ticks %d below_exclude %d "
              "online_icp %d offline_icp %d online_ms %.3f offline_ms %.3f\n",
              bad, n_ticks, rs_det, rs_acc, sc_det, sc_acc, rs_clamped, sc_clamped, rs_suppressed, rs_suppressed_after_sc,
              repeated_ticks, below_exclude, online_icp, offline_icp, online_ms, offline_ms);
  return bad ? 1 : 0;
}
