// map_optimization_gpu.h — host-side mirror of the reference's interface for the scan-to-map path.
//
// The reference has no plugin API: the path is a set of member functions of `class mapOptimization`
// (src/liorf/src/mapOptmization.cpp:74) and `class ImageProjection` (src/liorf/src/imageProjection.cpp:64)
// working on member clouds.  This header keeps the SAME member and method names so that a maintainer can
// paste the bodies into the ROS node (INTEGRATION.md); each body is a call into the C ABI (include/liogpu.h).
// Everything the reference keeps on the host stays on the host here: key-pose selection (extractNearby),
// keyframe gating (saveFrame), transformUpdate, and the pose graph (stubbed in the replay driver — GTSAM is
// out of scope).  C++14, no ROS / PCL / Eigen / OpenCV.
#pragma once
#include <cmath>
#include <cstdint>
#include <map>
#include <string>
#include <utility>
#include <vector>

#include "../../include/liogpu.h"

namespace liorf_gpu {

struct PointType {  // pcl::PointXYZI memory layout (utility.h:65): 32 bytes, 16-byte aligned
  float x, y, z, data3;
  float intensity, pad[3];
};
static_assert(sizeof(PointType) == 32, "pcl::PointXYZI is 32 bytes");

struct PointXYZIRT {  // imageProjection.cpp:4-15
  float x, y, z, data3;
  float intensity;
  uint16_t ring, pad0;
  float time, pad1;
};
static_assert(sizeof(PointXYZIRT) == 32, "PointXYZIRT is 32 bytes");

struct PointTypePose {  // mapOptmization.cpp:48-65
  float x, y, z, intensity, roll, pitch, yaw;
  double time;
};

typedef std::vector<PointType> Cloud;

class ImageProjection {
 public:
  explicit ImageProjection(liogpu_ctx* ctx) : ctx_(ctx) {}
  // members of the reference (imageProjection.cpp:62-100)
  std::vector<double> imuTime, imuRotX, imuRotY, imuRotZ;
  int imuPointerCur = 0;
  double timeScanCur = 0;
  int deskewFlag = 1;
  bool imuAvailable = false;
  std::vector<PointXYZIRT> laserCloudIn;
  Cloud fullCloud;
  // imageProjection.cpp:577-615 (+ deskewPoint, findRotation) -> liogpu_deskew
  int projectPointCloud();
  // the same call with the device-resident hand-off (SURVEY §8 f1): the deskewed cloud stays in HBM for a
  // co-located mapOptimization (same context); `raw` = laserCloudIn->points.data(), nothing is copied on the host
  int projectPointCloudResident(const PointXYZIRT* raw, int n, int* n_out);

 private:
  liogpu_ctx* ctx_;
};

class mapOptimization {
 public:
  explicit mapOptimization(const liogpu_params& params);
  // the same node around a context owned by somebody else (a mapping worker that replays one sequence after another)
  mapOptimization(const liogpu_params& params, liogpu_ctx* borrowed);
  ~mapOptimization();
  mapOptimization(const mapOptimization&) = delete;

  // ---- members with the reference's names (mapOptmization.cpp:137-178) ----
  Cloud laserCloudSurfLast;        // deskewed sweep
  Cloud laserCloudSurfLastDS;      // after downsampleCurrentScan
  Cloud laserCloudSurfFromMapDS;   // voxelised local map (kept for publishing)
  std::vector<PointType> cloudKeyPoses3D;
  std::vector<PointTypePose> cloudKeyPoses6D;
  std::vector<int> surroundingKeyPosesDS;  // ids chosen by extractNearby
  float transformTobeMapped[6] = {0, 0, 0, 0, 0, 0};
  bool isDegenerate = false;
  float matP[36] = {0};
  int laserCloudSurfLastDSNum = 0, laserCloudSurfFromMapDSNum = 0;
  double timeLaserInfoCur = 0;
  // parameters (utility.h:303-316)
  float surroundingKeyframeSearchRadius = 50.0f, surroundingKeyframeDensity = 2.0f;
  float surroundingkeyframeAddingDistThreshold = 1.0f, surroundingkeyframeAddingAngleThreshold = 0.2f;
  bool fetchLocalMap = false;      // copy laserCloudSurfFromMapDS back (it is only needed for publishing)
  bool selectKeyPosesOnDevice = false;  // extractNearby through liogpu_extract_nearby whatever the number of key poses
  int selectKeyPosesOnDeviceAbove = 3000;  // ... and automatically above this many key poses (measured crossover)
  // publishLocalMap settings (utility.h:219-229) and its output cloud (tempCloud, :2541)
  int localMapKeyFramesNumber = 30;
  liogpu_local_map_params localMapParams;
  liogpu_local_map_info lastLocalMapInfo{};
  Cloud localMapCloud;
  // loop closure (utility.h:315, 321-324)
  float historyKeyframeSearchRadius = 10.0f, historyKeyframeFitnessScore = 0.3f, loopClosureICPSurfLeafSize = 0.3f;
  int historyKeyframeSearchNum = 25;
  float historyKeyframeSearchTimeDiff = 30.0f;  // utility.h
  liogpu_sc_params scParams;                    // SCManager's constants (Scancontext.h)
  liogpu_sc_info lastScInfo{};
  std::map<int, int> loopIndexContainer;        // loop closures already made: loopKeyCur -> loopKeyPre
  // detectLoopClosureDistance through liogpu_detect_loop_distance instead of the host loop.  Off by default: on a B200
  // the host loop was faster at every measured size up to 10^5 key poses (profiles/r03_loop_detection.jsonl)
  bool detectLoopDistanceOnDevice = false;
  liogpu_icp_info lastIcpInfo{};
  liogpu_s2m_info lastInfo{};
  int lastStatus = 0;

  // ---- the hot path, same names as the reference ----
  void extractSurroundingKeyFrames();                    // :1590-1603
  void extractNearby();                                  // :1519-1554 (host: radius search + density filter + recency)
  void extractCloud(const std::vector<int>& ids);        // :1556-1588 -> liogpu_build_local_map
  void extractCloudFromIds(const std::vector<int>& ids); // the part of extractCloud after the distance guard of :1562
  void downsampleCurrentScan();                          // :1605-1611 -> liogpu_voxel_downsample
  void scan2MapOptimization();                           // :1839-1865 -> liogpu_scan2map
  void downsampleAndScan2Map();                          // both fused on device -> liogpu_downsample_scan2map
  // device-resident variants (SURVEY §8 f1): the sweep is the context's resident cloud (left there by
  // ImageProjection::projectPointCloudResident); laserCloudSurfLastDS stays in HBM, only its size comes back
  void downsampleAndScan2MapResident();
  void saveKeyFrameResident();                           // saveKeyFrame with thisSurfKeyFrame taken from the resident cloud
  Cloud transformPointCloud(const Cloud& in, const PointTypePose& pose);  // :849-868 -> liogpu_transform_cloud
  bool saveFrame() const;                                // :1909-1928 (host)
  void saveKeyFrame();                                   // the cloud/pose bookkeeping of saveKeyFramesAndFactor (:2128-2142)
  void loopFindNearKeyframes(Cloud& nearKeyframes, int key, int searchNum);  // :1360-1383 -> liogpu_merge_keyframes
  // the cloud / ICP part of performRSLoopClosure (:1098-1125): false when a guard rejects the closure;
  // correctionLidarFrame = icp.getFinalTransformation() (row-major 4x4), noiseScore = icp.getFitnessScore()
  // One pair through liogpu_loop_closure_icp_batch: the submaps stay on the device.
  bool loopClosureICP(int loopKeyCur, int loopKeyPre, float correctionLidarFrame[16], float* noiseScore);
  // loopClosureICP for many (loopKeyCur, loopKeyPre) pairs in one library call (an offline job verifying the loops of a
  // whole sequence).  results[j] holds pair j's verdict; loopIndexContainer is left to the caller, as above.
  struct LoopClosureOutcome {
    bool accepted = false;                 // passed the guards of MO:1104 and MO:1123
    float correctionLidarFrame[16] = {0};  // icp.getFinalTransformation() (identity when the size guard rejected it)
    float noiseScore = 0.f;                // icp.getFitnessScore()
    liogpu_loop_icp_result result{};       // submap sizes, overflow flags and the ICP's own report
  };
  int loopClosureICPBatch(const std::vector<std::pair<int, int>>& pairs, std::vector<LoopClosureOutcome>& results);
  // ---- loop-closure detection (the loop context of INTEGRATION.md); descriptors are stored in this node's context ----
  // scManager.makeAndSaveScancontextAndKeys(*thisSurfKeyFrame) (:2151-2166) on the keyframe's cloud as
  // saveKeyFrameResident leaves it (the downsampled sweep, SCInputType::SINGLE_SCAN_FEAT) -> liogpu_make_scancontext +
  // liogpu_sc_add
  void makeAndSaveScancontextAndKeys();
  // scManager.detectLoopClosureID() -> liogpu_sc_detect_loop: {loop id or -1, yaw difference (rad)}
  std::pair<int, float> detectLoopClosureID();
  // detectLoopClosureDistance (:1271-1300) -> liogpu_detect_loop_distance; false when there is no candidate or the
  // newest key pose already closed a loop (loopIndexContainer)
  bool detectLoopClosureDistance(int* latestID, int* closestID);
  // performSCLoopClosure / performRSLoopClosure (:1187-1268 / :1086-1185): detection -> loopClosureICP.  Instead of
  // queueing a GTSAM factor they return the pair and the correction (icp.getFinalTransformation()); true when a
  // closure passed every guard (it is then recorded in loopIndexContainer).
  bool performSCLoopClosure(int* loopKeyCur, int* loopKeyPre, float correctionLidarFrame[16], float* noiseScore);
  bool performRSLoopClosure(int* loopKeyCur, int* loopKeyPre, float correctionLidarFrame[16], float* noiseScore);
  // ---- offline loop closure: the loop thread's work for every tick of a recorded sequence ----
  // A tick is one wake-up of loopClosureThread (:1050-1084) after the first n_key key poses were saved, at
  // timeLaserInfoCur.  Its outcome is what performRSLoopClosure and then performSCLoopClosure return at that tick on a
  // node whose cloudKeyPoses3D / 6D hold the first n_key entries: each half's pair (written only when a candidate was
  // detected, -1 otherwise), whether the closure was accepted, the correction (written once the ICP passed the size
  // guard, zero otherwise) and the noise score (written when accepted, zero otherwise).  A tick with n_key == 0 gives the
  // empty outcome.  loopIndexContainer is updated in tick order exactly as the online calls would update it.
  struct LoopTick {
    int n_key = 0;
    double timeLaserInfoCur = 0;
  };
  struct LoopHalfOutcome {
    int loopKeyCur = -1, loopKeyPre = -1;
    bool accepted = false;
    float correctionLidarFrame[16] = {0};
    float noiseScore = 0.f;
  };
  struct LoopTickOutcome {
    LoopHalfOutcome rs, sc;
  };
  // The ticks' n_key must not decrease and may not exceed the key poses held here.  The SC half assumes a fresh Scan
  // Context manager that holds one descriptor per keyframe, in keyframe order, and serves no other detection calls
  // (the contract of liogpu_sc_detect_loops): descriptors this node has not stored yet (makeAndSaveScancontextAndKeys
  // or an earlier pass) are added from the resident keyframes.  Library calls: one liogpu_detect_loops_distance, at
  // most one liogpu_sc_add_keyframes, one liogpu_sc_detect_loops and one liogpu_loop_closure_icp_batch per distinct
  // n_key at which a detected pair's window [pre - historyKeyframeSearchNum, pre + historyKeyframeSearchNum] is
  // clamped (every other pair shares one call at the full size).  The ICP runs once per distinct detected pair,
  // including pairs whose tick ends up skipping the RS half; icpPairs (may be NULL) receives that count.
  // Returns LIOGPU_OK or the failing call's status (LIOGPU_E_INVALID for malformed ticks).
  int performLoopClosuresOffline(const std::vector<LoopTick>& ticks, std::vector<LoopTickOutcome>& outcomes,
                                 int* icpPairs = nullptr);
  void publishLocalMap();                                // :2442-2541 -> liogpu_publish_local_map (fills localMapCloud)
  const char* lastError() const;
  liogpu_ctx* context() { return ctx_; }

 private:
  liogpu_ctx* ctx_ = nullptr;
  bool owns_ctx_ = true;
  liogpu_params params_;
  std::vector<int> mapKeyIds_;  // keyframe set the device-resident local map was built from
  int scStored_ = 0;            // descriptors this node added to the context's Scan Context store
  // loopClosureICPBatch on a node that held only the first nKey key poses (windows clamped to [0, nKey))
  int loopClosureICPBatchAt(int nKey, const std::vector<std::pair<int, int>>& pairs,
                            std::vector<LoopClosureOutcome>& results);
  std::vector<float> mapKeyPoses_;
};

}  // namespace liorf_gpu
