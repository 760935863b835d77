/*
 * liogpu.h — C ABI of libliogpu.so: B200-native (sm_100a) scan-to-map registration for liorf.
 *
 * This is the drop-in boundary for ONE hot path of JiLiBIT/LIO-SLAM (liorf): every entry point
 * replaces the body of a member function of the reference's two ROS node classes.  Citations are
 * relative to the reference tree:
 *     MO = src/liorf/src/mapOptmization.cpp      IP = src/liorf/src/imageProjection.cpp
 *     UT = src/liorf/include/utility.h
 *
 * Conventions
 *   - C linkage, plain pointers and sizes only; no C++/torch types cross this boundary.
 *   - Every call returns an int status: 0 = OK, < 0 = error (nothing written), > 0 = warning
 *     (the call completed with the reference's own guard behaviour, see LIOGPU_W_*).
 *   - Point clouds are arrays of records `stride` bytes apart with float x@0, y@4, z@8 and the
 *     intensity at byte 16 when stride >= 32 (the pcl::PointXYZI layout the reference uses, UT:65)
 *     or at byte 12 when stride == 16 (packed float4).  Outputs use the same rule.
 *   - Pointers may be HOST pointers (pageable or pinned) or DEVICE pointers of ctx's GPU; the
 *     library detects which (cudaPointerGetAttributes).  The caller owns them; the library never
 *     keeps a caller pointer after the call returns.
 *   - pose6 = float[6] = {roll, pitch, yaw, x, y, z}: the layout of transformTobeMapped (MO:171).
 *   - One context = one GPU = one CUDA stream; calls on one context must be serialised by the
 *     caller (the reference holds `mtx` around the whole path, MO:449).
 *   - There is no CPU fallback: every entry point fails with LIOGPU_E_CUDA if no sm_100 device
 *     can be used.
 */
#ifndef LIOGPU_H_
#define LIOGPU_H_

#ifdef __cplusplus
extern "C" {
#endif

#define LIOGPU_ABI_VERSION 2

/* status codes */
#define LIOGPU_OK 0
#define LIOGPU_E_INVALID (-1)      /* bad argument                                         */
#define LIOGPU_E_CUDA (-2)         /* CUDA runtime error, see liogpu_last_error            */
#define LIOGPU_E_NO_MAP (-3)       /* scan2map / knn before any local map was installed    */
#define LIOGPU_E_NO_KEYFRAME (-4)  /* build_local_map names an id never put                */
#define LIOGPU_E_CAPACITY (-5)     /* caller's output buffer too small (n_out = needed)    */
#define LIOGPU_W_LEAF_OVERFLOW 1   /* VoxelGrid index overflow guard: output == input      */
#define LIOGPU_W_FEW_FEATURES 2    /* n <= 30 scan points: pose untouched (MO:1844,1863)   */
#define LIOGPU_W_NO_KEYFRAMES 3    /* local map empty: pose untouched (MO:1841)            */

typedef struct liogpu_ctx liogpu_ctx;

/* Device-resident hand-off (SURVEY §8 f1).  Passed as an OUTPUT cloud pointer to liogpu_deskew,
 * liogpu_voxel_downsample or liogpu_downsample_scan2map it means "do not copy the result out, keep it in
 * HBM as this context's resident cloud"; passed as an INPUT cloud pointer (n and stride are then ignored) to
 * liogpu_voxel_downsample, liogpu_scan2map, liogpu_downsample_scan2map, liogpu_surf_optimization or
 * liogpu_keyframe_put it means "use the resident cloud".  A co-located imageProjection + mapOptimization
 * thus moves a sweep over PCIe once (the raw XYZIRT records) and nothing else.  The resident cloud lives in the
 * context's scratch buffers: a later call that reuses its buffer for something else invalidates it (a subsequent
 * LIOGPU_DEVICE_RESIDENT input then fails with LIOGPU_E_INVALID rather than reading other data). */
#define LIOGPU_DEVICE_RESIDENT ((void*)(unsigned long long)1)

/* As an INPUT cloud pointer of liogpu_scan2map, liogpu_downsample_scan2map, liogpu_voxel_downsample or
 * liogpu_keyframe_put (n and stride are then ignored): the sweep a preceding liogpu_upload_scan_async put on its way. */
#define LIOGPU_UPLOADED_SCAN ((void*)(unsigned long long)2)

/* Parameters the hot path reads from ParamServer (UT:199-331); defaults are UT's compiled-in ones.
 * Fill with liogpu_default_params() and override. */
typedef struct liogpu_params {
  int device;                /* CUDA device ordinal                                              */
  int n_scan;                /* N_SCAN        (UT:275)  ring bound in deskew (IP:602)            */
  int horizon_scan;          /* Horizon_SCAN  (UT:276)  n_scan*horizon_scan = scratch hint MO:333 */
  float mapping_surf_leaf_size;              /* mappingSurfLeafSize            (UT:303, MO:286)  */
  float surrounding_keyframe_map_leaf_size;  /* surroundingKeyframeMapLeafSize (UT:304, MO:287)  */
  int downsample_rate;       /* downsampleRate   (UT:277, IP:605)                                */
  int point_filter_num;      /* point_filter_num (UT:278, IP:608)                                */
  float lidar_min_front, lidar_min_back, lidar_min_left, lidar_min_right; /* UT:280-283, IP:596  */
  float lidar_max_range;     /* UT:284, IP:598                                                   */
  float lidar_max_intensity; /* UT:285, IP:598                                                   */
  float knn_cell_size;       /* edge of the sorted-grid cell used for the 5-NN index; 0 = auto   */
  float knn_phase1_radius;   /* radius of the cheap first search phase; 0 = auto (2 x map leaf),
                                < 0 = single phase.  Tuning only: results do not depend on it.   */
  int profile_kernels;       /* 1: time the phases of the LM loop on the device (bench.py)        */
  int s2m_path;              /* how the LM loop of liogpu_scan2map is run.  Tuning only: results do not
                                depend on it.
                                0 = automatic (the faster one for the workload as measured on B200:
                                    currently always 1, see DESIGN.md "A/B of the LM loop");
                                1 = two launches per Gauss-Newton iteration (search + plane fit; leftovers
                                    + fixed-order reduction + 6x6 tail), chained with programmatic launch;
                                2 = the whole loop as ONE persistent cooperative launch with candidate
                                    sets and the exact no-search certificate (s2m_fused.cuh).           */
  int s2m_no_certificate;    /* 1 = never use the exact no-search certificate (A/B runs): every point
                                with a candidate set is searched again.  Results do not depend on it. */
  int reserved[3];
} liogpu_params;

/* Result block of liogpu_scan2map (everything the reference keeps in members after the loop). */
#define LIOGPU_MAX_ITER 30 /* MO:1848 */
typedef struct liogpu_s2m_info {
  int iterations;    /* LM iterations executed (MO:1848-1859)                                      */
  int converged;     /* 1 if LMOptimization returned true (MO:1833)                                */
  int n_query;       /* laserCloudSurfLastDSNum                                                    */
  int n_sel;         /* laserCloudSelNum of the last executed iteration (MO:1721)                  */
  int is_degenerate; /* isDegenerate after the loop (MO:176)                                       */
  int tie_queries;   /* last iteration: accepted queries whose 5-NN set contains / borders an
                        equidistant tie (neighbour parity is "modulo logged ties")                 */
  float delta_r_deg; /* last iteration's deltaR (MO:1824)                                          */
  float delta_t_cm;  /* last iteration's deltaT (MO:1828)                                          */
  double JtJ[36];    /* last iteration's AtA, f64 accumulation before rounding to f32 (MO:1782)    */
  double Jtr[6];     /* last iteration's AtB (MO:1783)                                             */
  float pose_hist[LIOGPU_MAX_ITER][6]; /* transformTobeMapped after each executed iteration        */
  int nsel_hist[LIOGPU_MAX_ITER];
  float gpu_ms;      /* device time of the loop (CUDA events on the context's stream)              */
  int seeded;        /* last iteration: points whose search started from the previous neighbours   */
  /* filled only when params.profile_kernels != 0 (CUDA events around every launch of the first chunk): */
  float main_kernel_ms;   /* summed device time of the search + plane-fit phase over the executed iterations
                             (s2m_path 1: of s2m_main_kernel)                                       */
  float left_kernel_ms;   /* summed device time of the leftover search + reduction + 6x6 tail
                             (s2m_path 1: of s2m_left_kernel)                                       */
  int main_kernel_launches, left_kernel_launches; /* executed iterations timed                     */
  /* s2m_path 2 only: */
  int certified;     /* last iteration: points whose 5 neighbours came from the exact certificate  */
  int leftovers;     /* last iteration: points finished by the warp-cooperative full-gate search   */
  float tail_ms;     /* profile_kernels: summed time between a CTA's partial row and the release of
                        the next iteration (fixed-order reduction + 6x6 tail + barrier)            */
  int kernel_launches; /* kernels launched by this call                                            */
  int certified_hist[LIOGPU_MAX_ITER]; /* per executed iteration: certified / seeded / leftover points      */
  int seeded_hist[LIOGPU_MAX_ITER];
  int leftover_hist[LIOGPU_MAX_ITER];
  float main_us_hist[LIOGPU_MAX_ITER]; /* profile_kernels: search + plane-fit phase of every iteration, us   */
  float rest_us_hist[LIOGPU_MAX_ITER]; /* profile_kernels: everything after it until the next iteration, us  */
} liogpu_s2m_info;

int liogpu_abi_version(void);
void liogpu_default_params(liogpu_params* p);

/* allocateMemory (MO:316-349): one context per mapOptimization / ImageProjection instance. */
int liogpu_create(liogpu_ctx** out, const liogpu_params* params);
void liogpu_destroy(liogpu_ctx* ctx);
const char* liogpu_last_error(const liogpu_ctx* ctx);

/* Pinned host memory for callers that want their clouds DMA-able (optional). */
void* liogpu_host_alloc(unsigned long long bytes);
void liogpu_host_free(void* p);

/* ImageProjection::projectPointCloud + deskewPoint + findRotation (IP:577-615, 545-575, 502-527).
 * xyzirt: n records, `stride` bytes apart: x@0 y@4 z@8 intensity@16 ring(u16)@20 time(f32)@24
 * (PointXYZIRT, IP:4-15).  imu_time/rot_x/rot_y/rot_z: the imuTime/imuRotX/Y/Z tables built by
 * imuDeskewInfo (IP:359-418) with n_imu = imuPointerCur + 1 valid rows (host code, stays host).
 * deskew_enabled = (deskewFlag != -1 && cloudInfo.imuAvailable) (IP:547).
 * Survivors are written in input order to xyzi_out (capacity cap_out records). */
int liogpu_deskew(liogpu_ctx* ctx, const void* xyzirt, int n, int stride, double time_scan_cur,
                  const double* imu_time, const double* imu_rot_x, const double* imu_rot_y,
                  const double* imu_rot_z, int n_imu, int deskew_enabled, void* xyzi_out,
                  int out_stride, int cap_out, int* n_out);

/* mapOptimization::transformPointCloud (MO:849-868). pose6 = keyframe {roll,pitch,yaw,x,y,z}. */
int liogpu_transform_cloud(liogpu_ctx* ctx, const void* xyzi, int n, int stride,
                           const float pose6[6], void* xyzi_out, int out_stride);

/* pcl::VoxelGrid<PointXYZI>::filter as called at MO:1536, 1582, 1609 (semantics: SURVEY A.1).
 * On the overflow guard the input is returned unchanged with LIOGPU_W_LEAF_OVERFLOW. */
int liogpu_voxel_downsample(liogpu_ctx* ctx, const void* xyzi, int n, int stride, float leaf,
                            void* xyzi_out, int out_stride, int cap_out, int* n_out);

/* surfCloudKeyFrames.push_back (MO:2142): keep a lidar-frame keyframe cloud resident on the GPU. */
int liogpu_keyframe_put(liogpu_ctx* ctx, int id, const void* xyzi, int n, int stride);
/* drop all keyframes (node reset).  The device slabs that held them stay with the context and are filled again by the
 * next keyframes (freeing / allocating device memory would synchronise every other context on the GPU); they are
 * released by liogpu_destroy. */
int liogpu_keyframe_clear(liogpu_ctx* ctx);
int liogpu_keyframe_count(const liogpu_ctx* ctx);

/* extractCloud (MO:1556-1588): transform the k named keyframes by their poses, concatenate in the
 * given order, VoxelGrid with `leaf`, install the result as the local map and build its 5-NN grid
 * index.  The host still chooses WHICH keyframes (extractNearby MO:1519-1554 stays host).
 * xyzi_out may be NULL; otherwise the voxelised map (laserCloudSurfFromMapDS) is copied out. */
int liogpu_build_local_map(liogpu_ctx* ctx, const int* ids, const float* pose6s /* k*6 */, int k,
                           float leaf, int* n_map, void* xyzi_out, int out_stride, int cap_out);

/* ---- extractCloud with the VoxelGrid pass sharded by spatial tile over several GPUs (BASELINE configs[3], SURVEY §8e) ----
 * Every GPU holds the keyframes (liogpu_keyframe_put on each context) and calls liogpu_voxel_tile with the same
 * ids / poses / leaf and its own `tile` in [0, n_tiles).  The call transforms and concatenates the k keyframes like
 * liogpu_build_local_map, plans the tiles ON THE DEVICE (coarse histogram of the voxel-row index (iz, iy), tile t =
 * the rows between the t/N and (t+1)/N quantiles of the point count — the same plan on every GPU, nothing is
 * exchanged), selects this tile's points in input order and voxelises them.  The tiles' outputs concatenated in tile
 * order are bit-identical to the cloud liogpu_build_local_map produces (a voxel never spans two tiles and PCL's
 * output order is lexicographic in (iz, iy, ix)); the caller gathers them (rank-ordered copies into disjoint slices,
 * or an NCCL all-gather) and installs the result with liogpu_set_local_map.  xyzi_out may be a device pointer.
 * On the overflow guard of the WHOLE cloud (q4) tile t returns the t-th contiguous slice of the input and the status
 * is LIOGPU_W_LEAF_OVERFLOW, so the concatenation is again what PCL returns.  The registration's installed local
 * map is left untouched. */
typedef struct liogpu_tile_info {
  int n_points;       /* points of the concatenated keyframes */
  int n_rows;         /* voxel rows (iz, iy) of the whole cloud's bounding box */
  int n_bins;         /* histogram bins the rows were grouped into (<= 65,536) */
  int bin_lo, bin_hi; /* this tile's bin range [lo, hi) */
  int n_tile_points;  /* points selected for this tile */
  int leaf_overflow;
  float gpu_ms;       /* device time of the call's kernels */
  float plan_ms;      /* of which: transform + bounding box + histogram + bounds + selection */
  int reserved[3];
} liogpu_tile_info;
int liogpu_voxel_tile(liogpu_ctx* ctx, const int* ids, const float* pose6s /* k*6 */, int k, float leaf, int tile,
                      int n_tiles, void* xyzi_out, int out_stride, int cap_out, int* n_out, liogpu_tile_info* info);

/* ---- publishLocalMap (MO:2442-2541; SURVEY §8 row f2), called after every registration (MO:504) ----
 * Filter settings of the node (utility.h:219-229, set up at MO:293-304). */
typedef struct liogpu_local_map_params {
  float local_map_left;          /* localMapLeft   UT:221: PassThrough x in [-left, right]  (MO:296-297) */
  float local_map_right;         /* localMapRight  UT:223 */
  float local_map_front;         /* localMapFront  UT:220: PassThrough y in [-back, front]  (MO:300-301) */
  float local_map_back;          /* localMapBack   UT:222 */
  int   use_removing_outliers;   /* useRemovingOutliers UT:227 -> pcl::StatisticalOutlierRemoval (MO:2510-2516) */
  int   mean_k;                  /* meanK UT:228 (1..31) */
  float stddev_threshold;        /* stddevThreshold UT:229 */
  int   use_down_sampling;       /* useDownSamplingLocalMap UT:224 -> VoxelGrid (MO:2517-2540) */
  float local_mapping_surf_leaf_size; /* localMappingSurfLeafSize UT:226 */
  float sor_cell_size;           /* tuning only (never changes results): cell edge of the outlier filter's
                                    neighbour grid, <= 0 = automatic */
  int   reserved[6];
} liogpu_local_map_params;

typedef struct liogpu_local_map_info {
  int    n_concat;        /* points of the concatenated keyframes (globalMapCloud, MO:2463-2466) */
  int    n_cropped;       /* after the two PassThrough filters (localMapCloud, MO:2502-2507) */
  int    n_after_sor;     /* after the outlier filter (= n_cropped when it is off) */
  int    n_out;           /* published points */
  int    leaf_overflow;   /* 1: the VoxelGrid overflow guard fired, cloud published un-downsampled (q4) */
  int    sor_borderline;  /* points whose mean distance is within 1e-9 (relative) of the threshold: the only
                             ones a different summation order of the statistics could flip */
  double sor_mean, sor_stddev, sor_threshold; /* statistics of the mean k-NN distances */
  float  gpu_ms;
  int    sor_leftover;    /* points finished by the wide (warp-cooperative) neighbour search */
  int    sor_exhaustive;  /* of those, isolated points that needed the exhaustive search */
  int    reserved[4];
} liogpu_local_map_info;

/* UT:219-229 defaults. */
void liogpu_default_local_map_params(liogpu_local_map_params* p);

/* publishLocalMap (MO:2442-2541): transform the k named keyframes (the host passes the last
 * localMapKeyFramesNumber ids, MO:2462) by their poses and concatenate them, move the cloud into the vehicle's
 * yaw-aligned frame of pose_now = transformTobeMapped (thisPoseX/Y/Z/Yaw, MO:2249-2254, 2474-2489), crop it with
 * PassThrough x then y, optionally remove statistical outliers and VoxelGrid it.  The result (tempCloud,
 * MO:2541) is written to xyzi_out in the reference's order.  info may be NULL. */
int liogpu_publish_local_map(liogpu_ctx* ctx, const int* ids, const float* pose6s /* k*6 */, int k,
                             const float pose_now[6], const liogpu_local_map_params* params,
                             void* xyzi_out, int out_stride, int cap_out, int* n_out,
                             liogpu_local_map_info* info);

/* The keyframe-merging loops outside the registration: saveMapService (MO:936-950: every keyframe, optional
 * VoxelGrid at req.resolution), publishGlobalMap (MO:1031-1039: the key poses chosen by the host, VoxelGrid at
 * globalMapVisualizationLeafSize) and loopFindNearKeyframes (MO:1360-1383).  Transforms the k named keyframes by
 * their poses, concatenates them in the given order and, when leaf > 0, applies pcl::VoxelGrid.  Unlike
 * liogpu_build_local_map it leaves the registration's local map and index untouched. */
int liogpu_merge_keyframes(liogpu_ctx* ctx, const int* ids, const float* pose6s /* k*6 */, int k, float leaf,
                           void* xyzi_out, int out_stride, int cap_out, int* n_out);

/* liogpu_merge_keyframes for n_windows windows in one call (offline loop verification, submap export).  Window w is
 * ids[win_off[w] .. win_off[w+1]) with the poses pose6s[6*j] of the same entries (win_off: n_windows + 1 entries,
 * non-decreasing from 0; ids may repeat, inside a window and across windows).  Its cloud is bit-equal to
 * liogpu_merge_keyframes of that window with the same leaf, whatever windows surround it, and is written to xyzi_out
 * records [out_off[w], out_off[w+1]).  overflow (may be NULL) receives each window's VoxelGrid guard flag (q4; that
 * window's cloud is its transformed concatenation).  Returns LIOGPU_W_LEAF_OVERFLOW if any window's guard fired, and
 * LIOGPU_E_CAPACITY when cap_out < out_off[n_windows], with out_off filled: liogpu_fetch_result then copies the whole
 * concatenation without recomputing it.  Malformed arguments and window inputs of more than INT32_MAX points in all
 * (LIOGPU_E_INVALID) and unknown ids (LIOGPU_E_NO_KEYFRAME) are refused before any work is done.  The registration's
 * local map and index and the resident cloud are left untouched. */
int liogpu_merge_keyframes_batch(liogpu_ctx* ctx, const int* ids, const float* pose6s, const int* win_off,
                                 int n_windows, float leaf, void* xyzi_out, int out_stride, int cap_out,
                                 int* out_off /* n_windows + 1 */, int* overflow /* n_windows or NULL */);

/* ---- loop-closure registration (SURVEY §8 row f3): pcl::IterativeClosestPoint<PointXYZI,PointXYZI> as configured
 * at MO:1111-1121 (performRSLoopClosure) / MO:1203-1213 (performSCLoopClosure). */
typedef struct liogpu_icp_params {
  float  max_correspondence_distance; /* icp.setMaxCorrespondenceDistance(historyKeyframeSearchRadius*2)  MO:1112 */
  int    max_iterations;              /* icp.setMaximumIterations(100)                                   MO:1113 */
  double transformation_epsilon;      /* icp.setTransformationEpsilon(1e-6)                              MO:1114 */
  double euclidean_fitness_epsilon;   /* icp.setEuclideanFitnessEpsilon(1e-6)                            MO:1115 */
  float  cell_size;                   /* tuning only: cell edge of the target's neighbour grid, <= 0 = automatic */
  int    reserved[5];
} liogpu_icp_params;

typedef struct liogpu_icp_info {
  int    iterations;          /* nr_iterations_ */
  int    converged;           /* icp.hasConverged() (MO:1123) */
  int    convergence_state;   /* 1 iterations, 2 transform, 3 absolute MSE, 4 relative MSE, 5 no correspondences */
  int    n_correspondences;   /* of the last iteration */
  double fitness_score;       /* icp.getFitnessScore() (MO:1123, 1145) */
  double last_mse;
  float  gpu_ms;
  int    reserved[5];
} liogpu_icp_info;

/* the settings of MO:1112-1116 for a given historyKeyframeSearchRadius (utility.h:321) */
void liogpu_default_icp_params(liogpu_icp_params* p, float history_keyframe_search_radius);

/* icp.setInputSource(cureKeyframeCloud); icp.setInputTarget(prevKeyframeCloud); icp.align(); (MO:1118-1121):
 * point-to-point ICP with SVD alignment (Eigen::umeyama) and PCL's default convergence criteria.  The clouds are
 * what liogpu_merge_keyframes returns for loopFindNearKeyframes (MO:1102-1103); the size guard of MO:1104 stays with
 * the caller.  final_transformation = icp.getFinalTransformation(), row-major 4x4. */
int liogpu_icp_align(liogpu_ctx* ctx, const void* source_xyzi, int n_source, int source_stride,
                     const void* target_xyzi, int n_target, int target_stride, const liogpu_icp_params* params,
                     float final_transformation[16], liogpu_icp_info* info);

typedef struct liogpu_loop_icp_result {
  int   n_source, n_target;              /* cureKeyframeCloud / prevKeyframeCloud after downSizeFilterICP (MO:1102-1103) */
  int   source_overflow, target_overflow;  /* VoxelGrid overflow guard (q4) fired on that submap */
  int   rejected_by_size;                /* n_source < 300 || n_target < 1000 (MO:1104): ICP not run, icp zeroed, T = I */
  float final_transformation[16];        /* icp.getFinalTransformation(), row-major */
  liogpu_icp_info icp;                   /* as liogpu_icp_align fills it; icp.gpu_ms = 0 (per-pair device time is not
                                            separable) */
  int   reserved[4];
} liogpu_loop_icp_result;

/* loopFindNearKeyframes (MO:1360-1383) for both ends of n_pairs candidate pairs, followed by the ICP of MO:1104-1123 for
 * each pair.  Keyframe ids are indices into key_pose6s (n_key x 6, cloudKeyPoses6D: roll, pitch, yaw, x, y, z).  The
 * window [key - search_num, key + search_num] is clamped to [0, n_key).  key_cur uses search_num 0, key_pre uses
 * search_num, and both submaps are voxelised at icp_leaf (loopClosureICPSurfLeafSize, > 0).  Every key must lie in
 * [0, n_key) (LIOGPU_E_INVALID) and every id of every window must have been put (LIOGPU_E_NO_KEYFRAME); both are checked
 * before any work is done.  The submaps never leave the device.  One params struct for all pairs.  results[j] are
 * bit-equal to liogpu_merge_keyframes of the two windows followed by liogpu_icp_align on the results, whatever the
 * batch around pair j.  The registration's local map and index and the resident cloud are left untouched.
 * The acceptance test of MO:1123 (converged && fitness <= historyKeyframeFitnessScore) stays with the caller.
 * liogpu_last_gpu_ms covers the whole call. */
int liogpu_loop_closure_icp_batch(liogpu_ctx* ctx, const int* key_cur, const int* key_pre, int n_pairs,
                                  const float* key_pose6s, int n_key, int search_num, float icp_leaf,
                                  const liogpu_icp_params* params, liogpu_loop_icp_result* results);

/* SCManager::makeScancontext (include/Scancontext.cpp:151-195) and the ring / sector keys (:198-225) that
 * makeAndSaveScancontextAndKeys stores at every keyframe (MO:2151-2166).  desc is the 20 x 60 MatrixXd, row-major
 * [ring][sector]; lidar_height = LIDAR_HEIGHT (Scancontext.h:80: 2.0), max_radius = PC_MAX_RADIUS (:84: 80.0).
 * The cloud may be LIOGPU_DEVICE_RESIDENT (the deskewed sweep, SCInputType::SINGLE_SCAN_FULL). */
#define LIOGPU_SC_NUM_RING 20
#define LIOGPU_SC_NUM_SECTOR 60
int liogpu_make_scancontext(liogpu_ctx* ctx, const void* xyzi, int n, int stride, double lidar_height,
                            double max_radius, double desc[LIOGPU_SC_NUM_RING * LIOGPU_SC_NUM_SECTOR],
                            double ringkey[LIOGPU_SC_NUM_RING], double sectorkey[LIOGPU_SC_NUM_SECTOR]);

/* ---- loop-closure detection (SURVEY §8 row f3): SCManager::detectLoopClosureID (include/Scancontext.cpp) over a
 * descriptor store kept in the context, and the key-pose radius detector detectLoopClosureDistance (MO ~1271-1300).
 * SCManager's constants (include/Scancontext.h); defaults by liogpu_default_sc_params are SC-LIO-SAM's Scancontext.h,
 * which liorf vendors: NUM_EXCLUDE_RECENT 30, NUM_CANDIDATES_FROM_TREE 3, TREE_MAKING_PERIOD_ 30, SEARCH_RATIO 0.1,
 * SC_DIST_THRES 0.2 (and historyKeyframeSearchTimeDiff 30.0 in utility.h for the radius detector).  They are taken
 * from the public sources as remembered, not checked against the reference tree. */
#define LIOGPU_SC_MAX_CANDIDATES 32
typedef struct liogpu_sc_params {
  int    num_exclude_recent;        /* NUM_EXCLUDE_RECENT        (>= 0)      */
  int    num_candidates_from_tree;  /* NUM_CANDIDATES_FROM_TREE  (1..LIOGPU_SC_MAX_CANDIDATES) */
  int    tree_making_period;        /* TREE_MAKING_PERIOD_       (>= 1)      */
  double search_ratio;              /* SEARCH_RATIO              (0, 1]      */
  double sc_dist_thres;             /* SC_DIST_THRES                         */
  int    reserved[4];
} liogpu_sc_params;

typedef struct liogpu_sc_info {     /* everything detectLoopClosureID computes on the way */
  int    n_stored, n_searchable;    /* polarcontexts_.size(), size of the tree's snapshot */
  int    tree_rebuilt;              /* this call rebuilt the snapshot (counter % period == 0) */
  int    n_candidates;              /* min(num_candidates_from_tree, n_searchable) */
  int    candidates[LIOGPU_SC_MAX_CANDIDATES];        /* kNN order */
  float  candidate_key_d2[LIOGPU_SC_MAX_CANDIDATES];  /* ring-key distance, nanoflann L2 (f32) */
  double candidate_dist[LIOGPU_SC_MAX_CANDIDATES];    /* distanceBtnScanContext().first */
  int    candidate_shift[LIOGPU_SC_MAX_CANDIDATES];   /* ... .second */
  int    nn_idx, nn_align;          /* best candidate and its shift, also when it is not a loop (-1 / 0 when the
                                       call returned early) */
  double min_dist;                  /* 1e7 (the reference's initial value) when nothing was scored */
  int    knn_ties;                  /* ring-key distances equal across the k-th boundary or inside the set */
  float  gpu_ms;
  int    reserved[4];
} liogpu_sc_info;

void liogpu_default_sc_params(liogpu_sc_params* p);
/* polarcontexts_ / invkeys / vkeys .push_back (makeAndSaveScancontextAndKeys, Scancontext.cpp:228-243) for n
 * descriptors as liogpu_make_scancontext returns them (row-major [ring][sector], f64, 1200 each; host or device memory).
 * The keys are derived on the device with the same code as liogpu_make_scancontext, so they are bit-equal to the ones it
 * returns. */
int liogpu_sc_add(liogpu_ctx* ctx, const double* descs, int n);
/* drop every stored descriptor and reset the tree counter (a fresh SCManager); liogpu_keyframe_clear does not touch the
 * store */
int liogpu_sc_clear(liogpu_ctx* ctx);
/* SCManager::detectLoopClosureID on the newest stored descriptor, with the reference's tree-snapshot state kept in the
 * context.  loop_id = -1 when there is no loop; yaw_diff_rad as the reference returns it; info may be NULL.  With fewer
 * than num_exclude_recent + 1 stored descriptors: LIOGPU_OK, loop_id = -1, yaw 0, counter not advanced (the reference's
 * early return).  Candidates are the exact k nearest ring keys of the snapshot in (distance, index) order; the
 * reference's KD-tree may order equal distances differently (counted in knn_ties). */
int liogpu_sc_detect_loop(liogpu_ctx* ctx, const liogpu_sc_params* p, int* loop_id, float* yaw_diff_rad,
                          liogpu_sc_info* info);
/* Offline: the results of n_calls detectLoopClosureID calls of a FRESH SCManager (counter 0) made when it held
 * store_sizes[j] descriptors (non-decreasing, each <= the stored count).  Bit-equal to clearing a store, adding the
 * same descriptors and calling liogpu_sc_detect_loop at those sizes.  Does not change the context's online counter.
 * yaw_diff_rad and min_dist may be NULL. */
int liogpu_sc_detect_loops(liogpu_ctx* ctx, const liogpu_sc_params* p, const int* store_sizes, int n_calls,
                           int* loop_ids, float* yaw_diff_rad, double* min_dist);
/* detectLoopClosureDistance (MO ~1271-1300) minus the loopIndexContainer check, which stays with the caller:
 * among the key poses strictly within search_radius of the newest one (FLANN: d2 < (float)(r*r), sorted by
 * distance, ties by lower index), the first whose |time - time_laser_info_cur| > time_diff; -1 if none or if it
 * is the newest itself.  Same key-pose / time arguments as liogpu_extract_nearby. */
int liogpu_detect_loop_distance(liogpu_ctx* ctx, const void* key_poses3d, int n_key, int stride3d,
                                const void* key_times, int time_stride, double time_laser_info_cur,
                                float search_radius, float time_diff, int* loop_key_pre);

/* ---- key-pose selection (SURVEY §8 row f4): extractNearby (MO:1519-1554) + the guard of extractCloud (MO:1562).
 * key_poses3d = cloudKeyPoses3D->points (x, y, z, intensity = keyframe index; n_key records of stride3d bytes),
 * key_times = the `time` field of cloudKeyPoses6D->points (n_key doubles, time_stride bytes apart: 8 for a plain
 * array, sizeof(PointTypePose) = 48 when pointing at cloudKeyPoses6D->points[0].time).  Radius search around the
 * newest key pose, VoxelGrid(density_leaf) of the hits, each centroid snapped to its nearest key pose, the poses
 * younger than 10 s appended, entries farther than search_radius dropped.  ids_out receives the keyframe indices in
 * the order extractCloud concatenates them (duplicates kept); pass them to liogpu_build_local_map with their poses. */
int liogpu_extract_nearby(liogpu_ctx* ctx, const void* key_poses3d, int n_key, int stride3d, const void* key_times,
                          int time_stride, double time_laser_info_cur, float search_radius, float density_leaf,
                          int* ids_out, int cap_ids, int* n_ids);

/* kdtreeSurfFromMap->setInputCloud(laserCloudSurfFromMapDS) (MO:1846) for a map built elsewhere:
 * install the cloud as the local map and build the grid index. */
int liogpu_set_local_map(liogpu_ctx* ctx, const void* xyzi, int n, int stride);
int liogpu_local_map_size(const liogpu_ctx* ctx);
/* number of points of the resident cloud (0 if none) */
int liogpu_resident_size(const liogpu_ctx* ctx);

/* The loop of scan2MapOptimization (MO:1848-1859): per iteration surfOptimization (MO:1618-1687),
 * combineOptimizationCoeffs (MO:1689-1700) and LMOptimization (MO:1702-1837), entirely on device.
 * scan_ds = laserCloudSurfLastDS (n points).  pose_io = transformTobeMapped, matP_io = matP
 * (row-major 6x6, MO:177) and degenerate_io = isDegenerate (MO:176) persist across scans in the
 * reference, so they are in/out.  max_iter <= LIOGPU_MAX_ITER (the reference uses 30).
 * transformUpdate (MO:1861) stays on the host. */
int liogpu_scan2map(liogpu_ctx* ctx, const void* scan_ds, int n, int stride, float pose_io[6],
                    float matP_io[36], int* degenerate_io, int max_iter, liogpu_s2m_info* info);

/* downsampleCurrentScan (MO:1605-1611) fused with liogpu_scan2map: the deskewed scan is
 * voxelised with params.mapping_surf_leaf_size on device and registered without leaving HBM.
 * n_ds receives laserCloudSurfLastDSNum; scan_ds_out may be NULL. */
int liogpu_downsample_scan2map(liogpu_ctx* ctx, const void* scan, int n, int stride,
                               float pose_io[6], float matP_io[36], int* degenerate_io,
                               int max_iter, liogpu_s2m_info* info, int* n_ds, void* scan_ds_out,
                               int out_stride, int cap_out);

/* One surfOptimization pass (MO:1618-1687) with its per-point results exposed for parity checks:
 * nn_idx[n*5] (indices into the installed local map, ascending distance, -1 when the query has
 * fewer than 5 map points within the gate), nn_d2[n*5] (pointSearchSqDis), coeff[n*4]
 * (coeffSelSurfVec: x,y,z,intensity), flag[n] (laserCloudOriSurfFlag), tie[n] (1 = tie logged).
 * Exactly one of pose6 / T12 (row-major 3x4 transPointAssociateToMap, MO:1615) is non-NULL.
 * Any output pointer may be NULL. */
int liogpu_surf_optimization(liogpu_ctx* ctx, const void* scan_ds, int n, int stride,
                             const float* pose6, const float* T12, int* nn_idx, float* nn_d2,
                             float* coeff, unsigned char* flag, unsigned char* tie);

/* liogpu_scan2map with the per-point results of its LAST EXECUTED iteration exposed (same outputs and meaning as
 * liogpu_surf_optimization; any pointer may be NULL).  Parity tests use it to check every iteration of the
 * on-device loop — including the ones that take the no-search certificate — against a surfOptimization pass of the
 * reference at the pose that iteration started from (info->pose_hist).  Runs the one-launch loop (s2m_path 2). */
int liogpu_scan2map_trace(liogpu_ctx* ctx, const void* scan_ds, int n, int stride, float pose_io[6],
                          float matP_io[36], int* degenerate_io, int max_iter, liogpu_s2m_info* info,
                          int* nn_idx, float* nn_d2, float* coeff, unsigned char* flag, unsigned char* tie);

/* Start copying a sweep to the GPU on the context's copy stream and return at once.  The node calls it when the message
 * arrives (pcl::fromROSMsg, MO:440), BEFORE it takes `mtx` (MO:449): the copy then overlaps the registration of the
 * previous sweep, and the next call that names LIOGPU_UPLOADED_SCAN as its input waits for it on the device.  The
 * caller's buffer must stay valid until that call returns (pinned memory — liogpu_host_alloc — for a truly
 * asynchronous copy).  Two sweeps may be in flight (a third returns LIOGPU_E_CAPACITY); consumers take them first in,
 * first out.  Unlike every other entry point it may overlap ONE other call
 * on the same context. */
int liogpu_upload_scan_async(liogpu_ctx* ctx, const void* xyzi, int n, int stride);

/* Copy out the cloud produced by the call RIGHT BEFORE this one (liogpu_build_local_map, liogpu_merge_keyframes,
 * liogpu_merge_keyframes_batch, liogpu_publish_local_map, liogpu_voxel_tile) without recomputing it: a caller that does not know the size passes
 * cap_out = 0 to the producing call, reads the size from its LIOGPU_E_CAPACITY return, sizes its buffer and fetches.
 * Returns the status the producing call would have returned (LIOGPU_OK or LIOGPU_W_LEAF_OVERFLOW). */
int liogpu_fetch_result(liogpu_ctx* ctx, void* xyzi_out, int out_stride, int cap_out, int* n_out);

/* Timing hook for bench.py: device milliseconds of the last call's kernels (events on ctx's stream). */
float liogpu_last_gpu_ms(const liogpu_ctx* ctx);
/* Kernels launched by this context since creation (bench.py's gpu_launches). */
unsigned long long liogpu_launch_count(const liogpu_ctx* ctx);
/* The context's cudaStream_t, so a caller timing with CUDA events can record on it. */
void* liogpu_stream(const liogpu_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* LIOGPU_H_ */
