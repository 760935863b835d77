// map_optimization_gpu.cpp — bodies of the mirrored member functions: thin calls into the C ABI.
#include "map_optimization_gpu.h"

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <stdexcept>

namespace liorf_gpu {

int ImageProjection::projectPointCloud() {
  fullCloud.resize(laserCloudIn.size());
  int n_out = 0;
  const int enabled = (deskewFlag != -1 && imuAvailable) ? 1 : 0;  // imageProjection.cpp:547
  const int st = liogpu_deskew(ctx_, laserCloudIn.data(), (int)laserCloudIn.size(), sizeof(PointXYZIRT), timeScanCur,
                               imuTime.data(), imuRotX.data(), imuRotY.data(), imuRotZ.data(), imuPointerCur + 1, enabled,
                               fullCloud.data(), sizeof(PointType), (int)fullCloud.size(), &n_out);
  fullCloud.resize(st < 0 ? 0 : n_out);
  return st;
}

int ImageProjection::projectPointCloudResident(const PointXYZIRT* raw, int n, int* n_out) {
  const int enabled = (deskewFlag != -1 && imuAvailable) ? 1 : 0;  // imageProjection.cpp:547
  return liogpu_deskew(ctx_, raw, n, sizeof(PointXYZIRT), timeScanCur, imuTime.data(), imuRotX.data(), imuRotY.data(),
                       imuRotZ.data(), imuPointerCur + 1, enabled, LIOGPU_DEVICE_RESIDENT, sizeof(PointType), 0, n_out);
}

mapOptimization::mapOptimization(const liogpu_params& params) : params_(params) {
  const int st = liogpu_create(&ctx_, &params_);  // allocateMemory (mapOptmization.cpp:316-349)
  if (st != LIOGPU_OK) throw std::runtime_error("liogpu_create failed (no sm_100 GPU? there is no CPU fallback)");
  liogpu_default_local_map_params(&localMapParams);  // utility.h:219-229
  liogpu_default_sc_params(&scParams);
}
mapOptimization::mapOptimization(const liogpu_params& params, liogpu_ctx* borrowed) : ctx_(borrowed), owns_ctx_(false), params_(params) {
  if (!ctx_) throw std::runtime_error("mapOptimization: null context");
  liogpu_default_local_map_params(&localMapParams);
  liogpu_default_sc_params(&scParams);
}
mapOptimization::~mapOptimization() { if (owns_ctx_) liogpu_destroy(ctx_); }
const char* mapOptimization::lastError() const { return liogpu_last_error(ctx_); }

static inline float pointDistance(const PointType& a, const PointType& b) {  // common_lib.cpp:33-37
  return std::sqrt((a.x - b.x) * (a.x - b.x) + (a.y - b.y) * (a.y - b.y) + (a.z - b.z) * (a.z - b.z));
}

void mapOptimization::extractSurroundingKeyFrames() {
  if (cloudKeyPoses3D.empty()) return;  // :1592
  extractNearby();
}

// Host logic, as in the reference (mapOptmization.cpp:1519-1554): which keyframes form the local map.
//   1. radiusSearch around the last key pose (PCL returns the hits sorted by distance);
//   2. downSizeFilterSurroundingKeyPoses (VoxelGrid, leaf surroundingKeyframeDensity) on those poses — here through
//      liogpu_voxel_downsample, the same routine the path uses everywhere;
//   3. each centroid is snapped to its nearest key pose (nearestKSearch(pt, 1), :1538-1542);
//   4. every keyframe younger than 10 s is appended WITHOUT de-duplication (:1545-1551) — a keyframe listed twice
//      is concatenated twice by extractCloud, exactly as in the reference.
void mapOptimization::extractNearby() {
  // the same selection in one library call (SURVEY §8 f4): 0.15-0.18 ms whatever the number of key poses, against
  // 0.06 ms (1,000 poses) / 0.48 ms (10,000 poses) for the host loops below -> automatic above the measured crossover
  if (selectKeyPosesOnDevice || (int)cloudKeyPoses3D.size() > selectKeyPosesOnDeviceAbove) {
    std::vector<double> times(cloudKeyPoses6D.size());
    for (size_t i = 0; i < times.size(); ++i) times[i] = cloudKeyPoses6D[i].time;
    std::vector<int> ids(2 * cloudKeyPoses3D.size() + 1);
    int n_ids = 0;
    const auto t_dbg0 = std::chrono::steady_clock::now();
    lastStatus = liogpu_extract_nearby(ctx_, cloudKeyPoses3D.data(), (int)cloudKeyPoses3D.size(), sizeof(PointType), times.data(),
                                       sizeof(double), timeLaserInfoCur, surroundingKeyframeSearchRadius, surroundingKeyframeDensity,
                                       ids.data(), (int)ids.size(), &n_ids);
    ids.resize(lastStatus < 0 ? 0 : n_ids);
    if (std::getenv("LIORF_DEBUG_TIMING"))
      std::fprintf(stderr, "[liorf] extract_nearby on device: %d key poses -> %d ids, %.3f ms (device %.3f ms)\n", (int)cloudKeyPoses3D.size(),
                   n_ids, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_dbg0).count(), (double)liogpu_last_gpu_ms(ctx_));
    surroundingKeyPosesDS = ids;
    extractCloudFromIds(ids);
    return;
  }
  const PointType& last = cloudKeyPoses3D.back();
  std::vector<std::pair<float, int>> hits;
  for (int i = 0; i < (int)cloudKeyPoses3D.size(); ++i) {
    const PointType& p = cloudKeyPoses3D[i];
    const float d2 = (p.x - last.x) * (p.x - last.x) + (p.y - last.y) * (p.y - last.y) + (p.z - last.z) * (p.z - last.z);
    // FLANN's radius result set keeps dist < radius^2 (strict), the squared radius narrowed to f32 by PCL
    if (d2 < (float)((double)surroundingKeyframeSearchRadius * (double)surroundingKeyframeSearchRadius)) hits.emplace_back(d2, i);
  }
  std::sort(hits.begin(), hits.end());  // by distance, equal distances by index
  Cloud surroundingKeyPoses, ds(hits.size());
  for (const auto& h : hits) surroundingKeyPoses.push_back(cloudKeyPoses3D[h.second]);
  int n_ds = 0;
  lastStatus = liogpu_voxel_downsample(ctx_, surroundingKeyPoses.data(), (int)surroundingKeyPoses.size(), sizeof(PointType),
                                       surroundingKeyframeDensity, ds.data(), sizeof(PointType), (int)ds.size(), &n_ds);
  if (lastStatus < 0) n_ds = 0;
  std::vector<int> ids;
  for (int k = 0; k < n_ds; ++k) {
    int best = 0;
    float bd = 3.4e38f;
    for (int i = 0; i < (int)cloudKeyPoses3D.size(); ++i) {
      const PointType& p = cloudKeyPoses3D[i];
      const float d2 = (p.x - ds[k].x) * (p.x - ds[k].x) + (p.y - ds[k].y) * (p.y - ds[k].y) + (p.z - ds[k].z) * (p.z - ds[k].z);
      if (d2 < bd) { bd = d2; best = i; }
    }
    // extractCloud's guard (:1562) tests the CENTROID's position, not the pose it was snapped to
    if (pointDistance(ds[k], last) > surroundingKeyframeSearchRadius) continue;
    ids.push_back((int)cloudKeyPoses3D[best].intensity);
  }
  for (int i = (int)cloudKeyPoses3D.size() - 1; i >= 0; --i) {
    if (timeLaserInfoCur - cloudKeyPoses6D[i].time < 10.0) {
      if (pointDistance(cloudKeyPoses3D[i], last) > surroundingKeyframeSearchRadius) continue;
      ids.push_back((int)cloudKeyPoses3D[i].intensity);
    } else break;
  }
  surroundingKeyPosesDS = ids;
  extractCloudFromIds(ids);
}

void mapOptimization::extractCloud(const std::vector<int>& ids) {
  std::vector<int> use;
  for (int id : ids) {
    if (pointDistance(cloudKeyPoses3D[id], cloudKeyPoses3D.back()) > surroundingKeyframeSearchRadius) continue;  // :1562
    use.push_back(id);
  }
  extractCloudFromIds(use);
}

void mapOptimization::extractCloudFromIds(const std::vector<int>& use) {
  std::vector<float> poses;
  for (int id : use) {
    const PointTypePose& p = cloudKeyPoses6D[id];
    const float pose6[6] = {p.roll, p.pitch, p.yaw, p.x, p.y, p.z};
    poses.insert(poses.end(), pose6, pose6 + 6);
  }
  // quirk q1: the reference rebuilds the KD-tree every scan; the device index is rebuilt only when the
  // keyframe set or a pose in it changed
  if (use == mapKeyIds_ && poses == mapKeyPoses_) return;
  int n_map = 0;
  if (fetchLocalMap) {
    laserCloudSurfFromMapDS.resize(1);
    int st = liogpu_build_local_map(ctx_, use.data(), poses.data(), (int)use.size(), params_.surrounding_keyframe_map_leaf_size,
                                    &n_map, laserCloudSurfFromMapDS.data(), sizeof(PointType), 0);
    if (st == LIOGPU_E_CAPACITY) {  // the map is built and installed; copy it out without rebuilding it
      laserCloudSurfFromMapDS.resize(n_map);
      st = liogpu_fetch_result(ctx_, laserCloudSurfFromMapDS.data(), sizeof(PointType), n_map, &n_map);
    }
    lastStatus = st;
    laserCloudSurfFromMapDS.resize(st < 0 ? 0 : n_map);
  } else {
    lastStatus = liogpu_build_local_map(ctx_, use.data(), poses.data(), (int)use.size(),
                                        params_.surrounding_keyframe_map_leaf_size, &n_map, nullptr, 0, 0);
  }
  laserCloudSurfFromMapDSNum = n_map;
  mapKeyIds_ = use;
  mapKeyPoses_ = poses;
}

void mapOptimization::downsampleCurrentScan() {
  laserCloudSurfLastDS.resize(laserCloudSurfLast.size());
  int n = 0;
  lastStatus = liogpu_voxel_downsample(ctx_, laserCloudSurfLast.data(), (int)laserCloudSurfLast.size(), sizeof(PointType),
                                       params_.mapping_surf_leaf_size, laserCloudSurfLastDS.data(), sizeof(PointType),
                                       (int)laserCloudSurfLastDS.size(), &n);
  laserCloudSurfLastDS.resize(lastStatus < 0 ? 0 : n);
  laserCloudSurfLastDSNum = (int)laserCloudSurfLastDS.size();
}

void mapOptimization::scan2MapOptimization() {
  if (cloudKeyPoses3D.empty()) return;  // :1841
  int deg = isDegenerate ? 1 : 0;
  lastStatus = liogpu_scan2map(ctx_, laserCloudSurfLastDS.data(), laserCloudSurfLastDSNum, sizeof(PointType), transformTobeMapped,
                               matP, &deg, LIOGPU_MAX_ITER, &lastInfo);
  isDegenerate = deg != 0;
  // transformUpdate() (:1861, IMU roll/pitch slerp + clamps) stays with the caller, as in the reference
}

void mapOptimization::downsampleAndScan2Map() {
  if (cloudKeyPoses3D.empty()) { downsampleCurrentScan(); return; }
  int deg = isDegenerate ? 1 : 0, n_ds = 0;
  laserCloudSurfLastDS.resize(laserCloudSurfLast.size());
  lastStatus = liogpu_downsample_scan2map(ctx_, laserCloudSurfLast.data(), (int)laserCloudSurfLast.size(), sizeof(PointType),
                                          transformTobeMapped, matP, &deg, LIOGPU_MAX_ITER, &lastInfo, &n_ds,
                                          laserCloudSurfLastDS.data(), sizeof(PointType), (int)laserCloudSurfLastDS.size());
  isDegenerate = deg != 0;
  laserCloudSurfLastDS.resize(lastStatus < 0 ? 0 : n_ds);
  laserCloudSurfLastDSNum = n_ds;
}

void mapOptimization::downsampleAndScan2MapResident() {
  int n_ds = 0;
  if (cloudKeyPoses3D.empty()) {  // scan2MapOptimization returns at once (:1841); downsampleCurrentScan still runs
    lastStatus = liogpu_voxel_downsample(ctx_, LIOGPU_DEVICE_RESIDENT, 0, 16, params_.mapping_surf_leaf_size,
                                         LIOGPU_DEVICE_RESIDENT, 16, 0, &n_ds);
    laserCloudSurfLastDSNum = lastStatus < 0 ? 0 : n_ds;
    return;
  }
  int deg = isDegenerate ? 1 : 0;
  lastStatus = liogpu_downsample_scan2map(ctx_, LIOGPU_DEVICE_RESIDENT, 0, 16, transformTobeMapped, matP, &deg,
                                          LIOGPU_MAX_ITER, &lastInfo, &n_ds, LIOGPU_DEVICE_RESIDENT, 16, 0);
  isDegenerate = deg != 0;
  laserCloudSurfLastDSNum = n_ds;
}

void mapOptimization::saveKeyFrameResident() {  // :2128-2142 without the factor graph
  PointType p3{};
  p3.x = transformTobeMapped[3]; p3.y = transformTobeMapped[4]; p3.z = transformTobeMapped[5];
  p3.data3 = 1.0f;
  p3.intensity = (float)cloudKeyPoses3D.size();
  PointTypePose p6{};
  p6.x = p3.x; p6.y = p3.y; p6.z = p3.z; p6.intensity = p3.intensity;
  p6.roll = transformTobeMapped[0]; p6.pitch = transformTobeMapped[1]; p6.yaw = transformTobeMapped[2];
  p6.time = timeLaserInfoCur;
  lastStatus = liogpu_keyframe_put(ctx_, (int)cloudKeyPoses3D.size(), LIOGPU_DEVICE_RESIDENT, 0, 16);
  cloudKeyPoses3D.push_back(p3);
  cloudKeyPoses6D.push_back(p6);
}

Cloud mapOptimization::transformPointCloud(const Cloud& in, const PointTypePose& p) {
  Cloud out(in.size());
  const float pose6[6] = {p.roll, p.pitch, p.yaw, p.x, p.y, p.z};
  lastStatus = liogpu_transform_cloud(ctx_, in.data(), (int)in.size(), sizeof(PointType), pose6, out.data(), sizeof(PointType));
  return out;
}

bool mapOptimization::saveFrame() const {  // :1909-1928 — relative motion since the last keyframe
  if (cloudKeyPoses3D.empty()) return true;
  const PointTypePose& k = cloudKeyPoses6D.back();
  auto rot = [](float r, float p, float y, double R[9]) {
    const double cr = std::cos(r), sr = std::sin(r), cp = std::cos(p), sp = std::sin(p), cy = std::cos(y), sy = std::sin(y);
    R[0] = cy * cp; R[1] = cy * sp * sr - sy * cr; R[2] = sy * sr + cy * sp * cr;
    R[3] = sy * cp; R[4] = cy * cr + sy * sp * sr; R[5] = sy * sp * cr - cy * sr;
    R[6] = -sp;     R[7] = cp * sr;                R[8] = cp * cr;
  };
  double A[9], B[9], D[9];
  rot(k.roll, k.pitch, k.yaw, A);
  rot(transformTobeMapped[0], transformTobeMapped[1], transformTobeMapped[2], B);
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) D[i * 3 + j] = A[0 * 3 + i] * B[0 * 3 + j] + A[1 * 3 + i] * B[1 * 3 + j] + A[2 * 3 + i] * B[2 * 3 + j];
  const double dt[3] = {transformTobeMapped[3] - k.x, transformTobeMapped[4] - k.y, transformTobeMapped[5] - k.z};
  double loc[3];
  for (int i = 0; i < 3; ++i) loc[i] = A[0 * 3 + i] * dt[0] + A[1 * 3 + i] * dt[1] + A[2 * 3 + i] * dt[2];
  const double roll = std::atan2(D[7], D[8]), pitch = std::asin(-D[6]), yaw = std::atan2(D[3], D[0]);
  if (std::fabs(roll) < surroundingkeyframeAddingAngleThreshold && std::fabs(pitch) < surroundingkeyframeAddingAngleThreshold &&
      std::fabs(yaw) < surroundingkeyframeAddingAngleThreshold &&
      std::sqrt(loc[0] * loc[0] + loc[1] * loc[1] + loc[2] * loc[2]) < surroundingkeyframeAddingDistThreshold)
    return false;
  return true;
}

void mapOptimization::saveKeyFrame() {  // :2128-2142 without the factor graph
  PointType p3{};
  p3.x = transformTobeMapped[3]; p3.y = transformTobeMapped[4]; p3.z = transformTobeMapped[5];
  p3.data3 = 1.0f;
  p3.intensity = (float)cloudKeyPoses3D.size();
  PointTypePose p6{};
  p6.x = p3.x; p6.y = p3.y; p6.z = p3.z; p6.intensity = p3.intensity;
  p6.roll = transformTobeMapped[0]; p6.pitch = transformTobeMapped[1]; p6.yaw = transformTobeMapped[2];
  p6.time = timeLaserInfoCur;
  // surfCloudKeyFrames.push_back(thisSurfKeyFrame): the downsampled sweep stays resident on the GPU
  lastStatus = liogpu_keyframe_put(ctx_, (int)cloudKeyPoses3D.size(), laserCloudSurfLastDS.data(), (int)laserCloudSurfLastDS.size(),
                                   sizeof(PointType));
  cloudKeyPoses3D.push_back(p3);
  cloudKeyPoses6D.push_back(p6);
}

void mapOptimization::loopFindNearKeyframes(Cloud& nearKeyframes, int key, int searchNum) {  // :1360-1383
  nearKeyframes.clear();
  const int cloudSize = (int)cloudKeyPoses6D.size();
  std::vector<int> ids;
  std::vector<float> poses;
  for (int i = -searchNum; i <= searchNum; ++i) {
    const int keyNear = key + i;
    if (keyNear < 0 || keyNear >= cloudSize) continue;
    const PointTypePose& p = cloudKeyPoses6D[keyNear];
    const float pose6[6] = {p.roll, p.pitch, p.yaw, p.x, p.y, p.z};
    ids.push_back(keyNear);
    poses.insert(poses.end(), pose6, pose6 + 6);
  }
  if (ids.empty()) return;
  int n = 0;
  nearKeyframes.resize(1);
  int st = liogpu_merge_keyframes(ctx_, ids.data(), poses.data(), (int)ids.size(), loopClosureICPSurfLeafSize,
                                  nearKeyframes.data(), sizeof(PointType), 0, &n);   // downSizeFilterICP (:1378-1381)
  if (st == LIOGPU_E_CAPACITY) {  // size now known: fetch the merged cloud, no second merge
    nearKeyframes.resize(n);
    st = liogpu_fetch_result(ctx_, nearKeyframes.data(), sizeof(PointType), n, &n);
  }
  lastStatus = st;
  nearKeyframes.resize(st < 0 ? 0 : n);
}

int mapOptimization::loopClosureICPBatch(const std::vector<std::pair<int, int>>& pairs,
                                         std::vector<LoopClosureOutcome>& results) {
  results.assign(pairs.size(), LoopClosureOutcome{});
  std::vector<int> cur(pairs.size()), pre(pairs.size());
  for (size_t j = 0; j < pairs.size(); ++j) { cur[j] = pairs[j].first; pre[j] = pairs[j].second; }
  std::vector<float> poses;
  for (const PointTypePose& p : cloudKeyPoses6D) {
    const float pose6[6] = {p.roll, p.pitch, p.yaw, p.x, p.y, p.z};
    poses.insert(poses.end(), pose6, pose6 + 6);
  }
  std::vector<liogpu_loop_icp_result> raw(pairs.size());
  liogpu_icp_params ip;
  liogpu_default_icp_params(&ip, historyKeyframeSearchRadius);                     // :1112-1116
  // loopFindNearKeyframes(cur, 0) / (pre, historyKeyframeSearchNum) with downSizeFilterICP (:1102-1103), icp.align
  lastStatus = liogpu_loop_closure_icp_batch(ctx_, cur.data(), pre.data(), (int)pairs.size(), poses.data(),
                                             (int)cloudKeyPoses6D.size(), historyKeyframeSearchNum,
                                             loopClosureICPSurfLeafSize, &ip, raw.data());
  if (lastStatus < 0) return lastStatus;
  for (size_t j = 0; j < pairs.size(); ++j) {
    LoopClosureOutcome& o = results[j];
    o.result = raw[j];
    std::memcpy(o.correctionLidarFrame, raw[j].final_transformation, sizeof(o.correctionLidarFrame));
    o.noiseScore = (float)raw[j].icp.fitness_score;                                 // :1145
    o.accepted = !raw[j].rejected_by_size && raw[j].icp.converged &&                 // :1104
                 raw[j].icp.fitness_score <= historyKeyframeFitnessScore;            // :1123
  }
  return lastStatus;
}

bool mapOptimization::loopClosureICP(int loopKeyCur, int loopKeyPre, float correctionLidarFrame[16], float* noiseScore) {
  std::vector<LoopClosureOutcome> out;
  if (loopClosureICPBatch({{loopKeyCur, loopKeyPre}}, out) < 0) return false;
  const LoopClosureOutcome& o = out[0];
  if (o.result.rejected_by_size) return false;                                      // :1104
  lastIcpInfo = o.result.icp;
  std::memcpy(correctionLidarFrame, o.correctionLidarFrame, sizeof(o.correctionLidarFrame));
  if (!o.accepted) return false;                                                    // :1123
  if (noiseScore) *noiseScore = o.noiseScore;                                       // :1145
  return true;
}

void mapOptimization::makeAndSaveScancontextAndKeys() {
  double desc[LIOGPU_SC_NUM_RING * LIOGPU_SC_NUM_SECTOR], ringkey[LIOGPU_SC_NUM_RING], sectorkey[LIOGPU_SC_NUM_SECTOR];
  // LIDAR_HEIGHT 2.0, PC_MAX_RADIUS 80.0 (Scancontext.h); the resident cloud is read in place and stays valid
  lastStatus = liogpu_make_scancontext(ctx_, LIOGPU_DEVICE_RESIDENT, 0, 16, 2.0, 80.0, desc, ringkey, sectorkey);
  if (lastStatus < 0) return;
  lastStatus = liogpu_sc_add(ctx_, desc, 1);
}

std::pair<int, float> mapOptimization::detectLoopClosureID() {
  int loop_id = -1;
  float yaw = 0.f;
  lastStatus = liogpu_sc_detect_loop(ctx_, &scParams, &loop_id, &yaw, &lastScInfo);
  if (lastStatus < 0) return {-1, 0.f};
  return {loop_id, yaw};
}

bool mapOptimization::detectLoopClosureDistance(int* latestID, int* closestID) {
  if (cloudKeyPoses3D.empty()) return false;
  const int loopKeyCur = (int)cloudKeyPoses3D.size() - 1;
  if (loopIndexContainer.find(loopKeyCur) != loopIndexContainer.end()) return false;  // :1277-1279
  int loopKeyPre = -1;
  if (detectLoopDistanceOnDevice) {
    lastStatus = liogpu_detect_loop_distance(ctx_, cloudKeyPoses3D.data(), (int)cloudKeyPoses3D.size(), sizeof(PointType),
                                             &cloudKeyPoses6D[0].time, sizeof(PointTypePose), timeLaserInfoCur,
                                             historyKeyframeSearchRadius, historyKeyframeSearchTimeDiff, &loopKeyPre);
    if (lastStatus < 0) return false;
  } else {  // radiusSearch (d2 < (float)(r*r), by distance, ties by index), then the first old enough (:1282-1291)
    const PointType& last = cloudKeyPoses3D.back();
    const float r2 = (float)((double)historyKeyframeSearchRadius * (double)historyKeyframeSearchRadius);
    float best = 0.f;
    for (int i = 0; i < (int)cloudKeyPoses3D.size(); ++i) {
      const PointType& p = cloudKeyPoses3D[i];
      float d2 = 0.f, d = last.x - p.x;
      d2 += d * d; d = last.y - p.y;
      d2 += d * d; d = last.z - p.z;
      d2 += d * d;
      if (!(d2 < r2) || !(std::fabs(cloudKeyPoses6D[i].time - timeLaserInfoCur) > (double)historyKeyframeSearchTimeDiff)) continue;
      if (loopKeyPre < 0 || d2 < best) { loopKeyPre = i; best = d2; }
    }
  }
  if (loopKeyPre == -1 || loopKeyCur == loopKeyPre) return false;
  *latestID = loopKeyCur;
  *closestID = loopKeyPre;
  return true;
}

bool mapOptimization::performSCLoopClosure(int* loopKeyCur, int* loopKeyPre, float correctionLidarFrame[16], float* noiseScore) {
  if (cloudKeyPoses3D.empty()) return false;
  const std::pair<int, float> detectResult = detectLoopClosureID();
  if (detectResult.first == -1) return false;
  *loopKeyCur = (int)cloudKeyPoses3D.size() - 1;
  *loopKeyPre = detectResult.first;
  if (!loopClosureICP(*loopKeyCur, *loopKeyPre, correctionLidarFrame, noiseScore)) return false;
  loopIndexContainer[*loopKeyCur] = *loopKeyPre;
  return true;
}

bool mapOptimization::performRSLoopClosure(int* loopKeyCur, int* loopKeyPre, float correctionLidarFrame[16], float* noiseScore) {
  if (cloudKeyPoses3D.empty()) return false;
  if (!detectLoopClosureDistance(loopKeyCur, loopKeyPre)) return false;
  if (!loopClosureICP(*loopKeyCur, *loopKeyPre, correctionLidarFrame, noiseScore)) return false;
  loopIndexContainer[*loopKeyCur] = *loopKeyPre;
  return true;
}

void mapOptimization::publishLocalMap() {  // :2442-2541; the reference calls it after every registration (:504)
  if (cloudKeyPoses3D.empty()) return;     // :2444
  const int thisPoseNum = (int)cloudKeyPoses3D.size();
  const int startPoseNum = (thisPoseNum < localMapKeyFramesNumber) ? 0 : thisPoseNum - localMapKeyFramesNumber;  // :2462
  std::vector<int> ids;
  std::vector<float> poses;
  for (int i = startPoseNum; i < thisPoseNum; ++i) {
    const PointTypePose& p = cloudKeyPoses6D[i];
    const float pose6[6] = {p.roll, p.pitch, p.yaw, p.x, p.y, p.z};
    ids.push_back(i);
    poses.insert(poses.end(), pose6, pose6 + 6);
  }
  // thisPoseX/Y/Z/Yaw are copies of transformTobeMapped (:2249-2254)
  int n = 0;
  localMapCloud.resize(localMapCloud.capacity() > 0 ? localMapCloud.capacity() : 1);
  int st = liogpu_publish_local_map(ctx_, ids.data(), poses.data(), (int)ids.size(), transformTobeMapped, &localMapParams,
                                    localMapCloud.data(), sizeof(PointType), (int)localMapCloud.size(), &n, &lastLocalMapInfo);
  if (st == LIOGPU_E_CAPACITY) {  // the cloud grew: fetch it, the pipeline is not run twice
    localMapCloud.resize(n);
    st = liogpu_fetch_result(ctx_, localMapCloud.data(), sizeof(PointType), n, &n);
  }
  lastStatus = st;
  localMapCloud.resize(st < 0 ? 0 : n);
}

}  // namespace liorf_gpu
