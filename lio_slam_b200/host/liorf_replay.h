/* liorf_replay.h — C entry point of the ROS-free host mirror (lio_slam_b200/host): replays one sequence of raw sweeps
 * through the per-scan path of the reference's two nodes,
 *   ImageProjection::cloudHandler  (imageProjection.cpp:206: projectPointCloud + deskew)          -> liogpu_deskew
 *   mapOptimization::laserCloudInfoHandler (mapOptmization.cpp:432-506): extractSurroundingKeyFrames,
 *     downsampleCurrentScan, scan2MapOptimization, saveKeyFramesAndFactor (keyframe gate + bookkeeping)
 * with the device-resident hand-off between them (SURVEY §8 f1).  One call = one sequence = one liogpu context = one
 * GPU; several calls may run concurrently from different host threads (batch offline mapping, BASELINE configs[4]).
 * The pose graph (GTSAM iSAM2) is out of scope: the optimised pose of a keyframe is the registered pose.
 * libliorf_host.so links libliogpu.so; there is no CPU fallback. */
#ifndef LIORF_REPLAY_H_
#define LIORF_REPLAY_H_
#include "../../include/liogpu.h"
#ifdef __cplusplus
extern "C" {
#endif

typedef struct liorf_sweep {
  const void* raw;       /* n_raw PointXYZIRT records (32 bytes: x y z pad intensity ring(u16) time pad), host memory */
  int n_raw;
  double time_scan_cur;  /* header stamp of the sweep (timeScanCur / timeLaserInfoCur) */
  float guess[6];        /* what updateInitialGuess (MO:1438-1502) provides: {roll, pitch, yaw, x, y, z} */
  const double* imu;     /* 4 x n_imu doubles: imuTime | imuRotX | imuRotY | imuRotZ (imuDeskewInfo, IP:359-418) */
  int n_imu;
} liorf_sweep;

typedef struct liorf_replay_options {
  int select_key_poses_on_device; /* extractNearby through liogpu_extract_nearby (0: host loops as in the mirror) */
  int publish_local_map;          /* also run publishLocalMap after every scan (MO:504) */
  float keyframe_dist, keyframe_angle; /* surroundingkeyframeAddingDistThreshold / AngleThreshold (UT:312-313); 0 = 1.0 / 0.2 */
  float search_radius, density;   /* surroundingKeyframeSearchRadius / Density (UT:315-316); 0 = 50 / 2 */
  int loop_detection_every;       /* 0 = off; N = every N sweeps, after the keyframe step, run detectLoopClosureDistance and
                                     detectLoopClosureID (the 1 Hz loopClosureThread at 10 Hz sweeps: N = 10); a Scan
                                     Context descriptor is then saved at every keyframe.  Both run through the library
                                     (liogpu_detect_loop_distance, liogpu_sc_detect_loop).  The registration is unchanged. */
  int reserved[5];
} liorf_replay_options;

typedef struct liorf_replay_stats {
  int scans, registered, keyframes, map_rebuilds;
  int lm_iterations;               /* summed over the registered scans */
  int map_points_last;             /* laserCloudSurfFromMapDSNum of the last rebuild */
  double wall_ms;                  /* whole replay, host clock, uploads and read-backs included */
  double deskew_ms, nearby_ms, register_ms, keyframe_ms;  /* host clock per stage, summed */
  double loop_gpu_ms;              /* device time of the LM loops, summed */
  long long h2d_bytes, d2h_bytes;  /* sweep uploads / pose + state read-backs */
  unsigned long long gpu_launches;
  int loops_sc, loops_rs;          /* loop_detection_every: detections of detectLoopClosureID / detectLoopClosureDistance */
  int reserved[2];
} liorf_replay_stats;

/* poses_out: n x 6 floats (transformTobeMapped after every scan); iters_out, nds_out: n ints (LM iterations,
 * laserCloudSurfLastDSNum), any of them may be NULL.  Returns 0 or the first negative liogpu status; err receives
 * liogpu_last_error. */
int liorf_replay_sequence(const liogpu_params* params, const liorf_replay_options* options, const liorf_sweep* sweeps,
                          int n, float* poses_out, int* iters_out, int* nds_out, liorf_replay_stats* stats, char* err,
                          int err_len);

/* A mapping worker = one liogpu context (one GPU, one stream) that replays sequence after sequence: the context, its
 * pinned staging memory and its device buffers are created once and reused (liogpu_keyframe_clear and liogpu_sc_clear
 * between sequences),
 * as a batch-mapping service would do.  One worker per host thread. */
typedef struct liorf_worker liorf_worker;
liorf_worker* liorf_worker_create(const liogpu_params* params, char* err, int err_len);
void liorf_worker_destroy(liorf_worker* w);
int liorf_worker_replay(liorf_worker* w, const liorf_replay_options* options, const liorf_sweep* sweeps, int n,
                        float* poses_out, int* iters_out, int* nds_out, liorf_replay_stats* stats, char* err, int err_len);

#ifdef __cplusplus
}
#endif
#endif
