// liorf_oracle.cpp — CPU ORACLE (TEST INFRASTRUCTURE, NOT PRODUCT CODE).  PARITY UNPINNED — see the
// header of liorf_oracle_core.h.  extern "C" entry points for ctypes (tests/, smoke(), bench.py's
// cpu_baseline / --impl reference legs).  Clouds are packed float4 arrays (x, y, z, intensity).
//
// When built with -DLIORF_USE_NANOFLANN -I/root/reference/src/liorf/include (oracle/Makefile target
// `_ref`), the KD-tree is the reference's own vendored nanoflann 1.3.2 header (compiled where it
// lies, never copied); the symbols then carry the prefix refnf_ instead of ref_.
#include "liorf_oracle_core.h"

#include <chrono>
#include <cstdio>
#ifdef _OPENMP
#include <omp.h>
#endif

#ifdef LIORF_USE_NANOFLANN
#include <nanoflann.hpp>
#define SYM(name) refnf_##name
#else
#define SYM(name) ref_##name
#endif

using namespace liorf_oracle;

namespace {

#ifdef LIORF_USE_NANOFLANN
// Adaptor over the packed map; nanoflann's L2_Simple_Adaptor evaluates (a-b)^2 summed over x,y,z in
// f32 like FLANN's L2_Simple.  Its KNNResultSet keeps the first-visited point on ties, so results
// are canonical only modulo logged ties.
struct NfCloud {
  const P4* pts; size_t n;
  inline size_t kdtree_get_point_count() const { return n; }
  inline float kdtree_get_pt(const size_t i, const size_t d) const {
    return d == 0 ? pts[i].x : (d == 1 ? pts[i].y : pts[i].z);
  }
  template <class BBOX> bool kdtree_get_bbox(BBOX&) const { return false; }
};
typedef nanoflann::KDTreeSingleIndexAdaptor<nanoflann::L2_Simple_Adaptor<float, NfCloud>, NfCloud, 3, int> NfTree;
struct Index {
  NfCloud cloud;
  NfTree* tree = nullptr;
  const P4* pts; int n;
  void build(const P4* p, int count) {
    pts = p; n = count;
    cloud.pts = p; cloud.n = (size_t)count;
    tree = new NfTree(3, cloud, nanoflann::KDTreeSingleIndexAdaptorParams(15));
    tree->buildIndex();
  }
  ~Index() { delete tree; }
  void knn(const P4& q, Knn6& r) const {
    r.init();
    int idx[6]; float d2[6];
    const float qq[3] = {q.x, q.y, q.z};
    const size_t found = tree->knnSearch(qq, 6, idx, d2);
    for (size_t k = 0; k < found; ++k) { r.d2[k] = d2[k]; r.idx[k] = idx[k]; }
  }
  void knn_dist(const P4& q, KnnDist& r) const {
    r.init();
    int idx[32]; float d2[32];
    const float qq[3] = {q.x, q.y, q.z};
    const size_t found = tree->knnSearch(qq, (size_t)r.k, idx, d2);
    for (size_t k = 0; k < found; ++k) r.d2[k] = d2[k];
    r.found = (int)found;
  }
};
#else
struct Index {
  KdTree tree;
  const P4* pts; int n;
  void build(const P4* p, int count) { pts = p; n = count; tree.build(p, count); }
  void knn(const P4& q, Knn6& r) const { tree.knn(q, r); }
  void knn_dist(const P4& q, KnnDist& r) const { tree.knn(q, r); }
};
#endif

inline double now_ms() {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// surfOptimization (MO:1618-1687) over all queries; index == nullptr -> brute force k-NN.
void surf_optimization(const P4* map, int nm, const Index* index, const P4* scan, int nq, const float T[12],
                       int* nn_idx, float* nn_d2, P4* coeff, unsigned char* flag, unsigned char* tie,
                       int threads) {
#pragma omp parallel for num_threads(threads) schedule(static)
  for (int i = 0; i < nq; ++i) {
    const P4 ori = scan[i];
    const P4 sel = apply_T(T, ori);
    Knn6 r;
    if (index) index->knn(sel, r); else knn_brute(map, nm, sel, r);
    P4 c{0.f, 0.f, 0.f, 0.f};
    bool ok = false, tied = false;
    if (nm >= 5 && r.idx[4] != INT_MAX) {
      P4 nb[5];
      for (int j = 0; j < 5; ++j) nb[j] = map[r.idx[j]];
      ok = plane_residual(ori, sel, nb, r.d2[4], c);
      tied = (r.d2[4] < 1.0) && r.tie();
    }
    if (nn_idx) for (int j = 0; j < 5; ++j) nn_idx[i * 5 + j] = r.idx[j] == INT_MAX ? -1 : r.idx[j];
    if (nn_d2) for (int j = 0; j < 5; ++j) nn_d2[i * 5 + j] = r.d2[j];
    if (coeff) coeff[i] = c;
    if (flag) flag[i] = ok ? 1 : 0;
    if (tie) tie[i] = tied ? 1 : 0;
  }
}

// combineOptimizationCoeffs (MO:1689-1700) + the accumulation half of LMOptimization (MO:1735-1783):
// ordered compaction is implicit (rows are visited in query order), AtA/AtB accumulate in f64.
int accumulate_normal_equations(const P4* scan, const P4* coeff, const unsigned char* flag, int nq,
                                const float pose[6], double JtJ[36], double Jtr[6]) {
  const Trig g = lm_trig(pose);
  for (int i = 0; i < 36; ++i) JtJ[i] = 0;
  for (int i = 0; i < 6; ++i) Jtr[i] = 0;
  int nsel = 0;
  for (int i = 0; i < nq; ++i) {
    if (!flag[i]) continue;
    ++nsel;
    float row[6], rhs;
    jacobian_row(g, scan[i], coeff[i], row, rhs);
    for (int a = 0; a < 6; ++a) {
      for (int b = 0; b < 6; ++b) JtJ[a * 6 + b] += (double)row[a] * (double)row[b];
      Jtr[a] += (double)row[a] * (double)rhs;
    }
  }
  return nsel;
}

}  // namespace

extern "C" {

void SYM(pose_to_T)(const float* pose6, float* T12) { pose_to_T(pose6, T12); }

// transformPointCloud (MO:849-868)
void SYM(transform_cloud)(const float* in4, int n, const float* pose6, float* out4, int threads) {
  float T[12];
  pose_to_T(pose6, T);
  const P4* in = (const P4*)in4;
  P4* out = (P4*)out4;
#pragma omp parallel for num_threads(threads) schedule(static)
  for (int i = 0; i < n; ++i) out[i] = apply_T(T, in[i]);
}

// VoxelGrid::filter (MO:1536,1582,1609).  out4 must hold n points.  Returns 1 on the overflow guard.
int SYM(voxel_grid)(const float* in4, int n, float leaf, float* out4, int* n_out) {
  std::vector<P4> out;
  const int ov = voxel_grid((const P4*)in4, n, leaf, out);
  std::memcpy(out4, out.data(), out.size() * sizeof(P4));
  *n_out = (int)out.size();
  return ov;
}

// extractCloud (MO:1556-1588): transform + concatenate + VoxelGrid.  clouds = concatenated keyframe
// clouds, offsets[k+1] = their boundaries.
int SYM(build_local_map)(const float* clouds4, const int* offsets, const float* pose6s, int k, float leaf,
                         float* out4, int* n_out, int threads) {
  const int total = offsets[k];
  std::vector<P4> raw((size_t)total);
  for (int f = 0; f < k; ++f)
    SYM(transform_cloud)(clouds4 + 4 * (size_t)offsets[f], offsets[f + 1] - offsets[f], pose6s + 6 * f,
                         (float*)(raw.data() + offsets[f]), threads);
  return SYM(voxel_grid)((const float*)raw.data(), total, leaf, out4, n_out);
}

// f2: publishLocalMap (MO:2442-2541).  clouds4/offsets/pose6s = the keyframes to publish (the caller passes the
// last localMapKeyFramesNumber, MO:2462) and their poses; pose_now6 = transformTobeMapped.  brute != 0: the
// outlier filter's (meanK+1)-NN by exhaustive search, else through the KD-tree (the reference's path).
// out4 must hold offsets[k] points.  md_out (optional, n_cropped floats) receives the per-point mean distances.
// Returns 1 when the VoxelGrid overflow guard fired.
int SYM(publish_local_map)(const float* clouds4, const int* offsets, const float* pose6s, int k, const float* pose_now6,
                           const LocalMapParams* prm, int brute, float* out4, int* n_out, LocalMapInfo* info,
                           float* md_out, int threads) {
  std::memset(info, 0, sizeof(*info));
  *n_out = 0;
  if (k <= 0) return 0;  // cloudKeyPoses3D->points.empty(), MO:2444
  const int total = offsets[k];
  std::vector<P4> globalMapCloud((size_t)total);
  for (int f = 0; f < k; ++f)   // MO:2463-2466
    SYM(transform_cloud)(clouds4 + 4 * (size_t)offsets[f], offsets[f + 1] - offsets[f], pose6s + 6 * f,
                         (float*)(globalMapCloud.data() + offsets[f]), threads);
  float m[12];
  yaw_frame_T(pose_now6, m);
  std::vector<P4> transformedGlobalMapCloud((size_t)total);
#pragma omp parallel for num_threads(threads) schedule(static)
  for (int i = 0; i < total; ++i) transformedGlobalMapCloud[i] = pcl_transform_se3(m, globalMapCloud[i]);
  std::vector<P4> tempCloud;
  pass_through_xy(transformedGlobalMapCloud, -prm->left, prm->right, -prm->back, prm->front, tempCloud);
  info->n_concat = total;
  info->n_cropped = (int)tempCloud.size();
  info->n_after_sor = info->n_cropped;
  if (prm->use_removing_outliers && !tempCloud.empty()) {   // MO:2510-2516
    const int n = (int)tempCloud.size();
    const P4* pts = tempCloud.data();
    std::vector<float> distances;
    int valid;
    if (brute) {
      valid = sor_mean_distances(n, prm->mean_k, [&](int i, KnnDist& r) {
        for (int j = 0; j < n; ++j) r.insert(l2_simple(pts[i], pts[j]), j);
      }, distances, threads);
    } else {
      Index ix;
      ix.build(pts, n);
      valid = sor_mean_distances(n, prm->mean_k, [&](int i, KnnDist& r) { ix.knn_dist(pts[i], r); }, distances, threads);
    }
    if (md_out) std::memcpy(md_out, distances.data(), (size_t)n * sizeof(float));
    std::vector<int> kept;
    sor_select(distances, valid, (double)prm->stddev_threshold, kept, info->sor_mean, info->sor_stddev, info->sor_threshold);
    std::vector<P4> filtered(kept.size());
    for (size_t i = 0; i < kept.size(); ++i) filtered[i] = tempCloud[kept[i]];
    tempCloud.swap(filtered);
    info->n_after_sor = (int)tempCloud.size();
  }
  int ov = 0;
  if (prm->use_down_sampling && !tempCloud.empty()) {   // MO:2517-2540
    std::vector<P4> ds;
    ov = voxel_grid(tempCloud.data(), (int)tempCloud.size(), prm->leaf, ds);
    tempCloud.swap(ds);
  }
  info->leaf_overflow = ov;
  info->n_out = (int)tempCloud.size();
  std::memcpy(out4, tempCloud.data(), tempCloud.size() * sizeof(P4));
  *n_out = (int)tempCloud.size();
  return ov;
}
void SYM(yaw_frame_T)(const float* pose_now6, float* m12) { yaw_frame_T(pose_now6, m12); }

// f3: pcl::IterativeClosestPoint::align + getFitnessScore as configured at MO:1111-1123.  brute != 0: exhaustive
// nearest neighbour, else the KD-tree.
int SYM(icp_align)(const float* source4, int ns, const float* target4, int nt, const IcpParams* prm, int brute,
                   IcpResult* res, int threads) {
  const P4* src = (const P4*)source4;
  const P4* tgt = (const P4*)target4;
  Index ix;
  if (!brute) ix.build(tgt, nt);
  auto nn = [&](const P4& q, int& idx, float& d2) {
    Knn6 k;
    if (brute) knn_brute(tgt, nt, q, k); else ix.knn(q, k);
    idx = k.idx[0] == INT_MAX ? -1 : k.idx[0];
    d2 = k.d2[0];
  };
  icp_align(src, ns, tgt, nn, *prm, *res, threads);
  return res->converged;
}

// f3: SCManager::makeScancontext + ring / sector keys (Scancontext.cpp:151-225)
void SYM(make_scancontext)(const float* scan4, int n, double lidar_height, double max_radius, double* desc,
                           double* ringkey, double* sectorkey) {
  make_scancontext((const P4*)scan4, n, lidar_height, max_radius, desc, ringkey, sectorkey);
}

// f4: extractNearby + the selection half of extractCloud (MO:1519-1565).  ids_out must hold 2*n entries.
int SYM(extract_nearby)(const float* key3d4, const double* key_time, int n, double time_cur, float radius, float density,
                        int* ids_out) {
  std::vector<int> ids;
  std::vector<P4> ds;
  extract_nearby((const P4*)key3d4, key_time, n, time_cur, radius, density, ids, ds);
  for (size_t k = 0; k < ids.size(); ++k) ids_out[k] = ids[k];
  return (int)ids.size();
}

// KD-tree handle (kdtreeSurfFromMap->setInputCloud, MO:1846).  The map memory must outlive the handle.
void* SYM(index_build)(const float* map4, int nm) {
  Index* ix = new Index();
  ix->build((const P4*)map4, nm);
  return ix;
}
void SYM(index_free)(void* h) { delete (Index*)h; }

// 5-NN of already-transformed queries: index handle, or brute force when h == NULL.
void SYM(knn5)(const float* map4, int nm, void* h, const float* q4, int nq, int* nn_idx, float* nn_d2,
               unsigned char* tie, int threads) {
  const P4* map = (const P4*)map4;
  const P4* q = (const P4*)q4;
  const Index* ix = (const Index*)h;
#pragma omp parallel for num_threads(threads) schedule(static)
  for (int i = 0; i < nq; ++i) {
    Knn6 r;
    if (ix) ix->knn(q[i], r); else knn_brute(map, nm, q[i], r);
    for (int j = 0; j < 5; ++j) {
      nn_idx[i * 5 + j] = r.idx[j] == INT_MAX ? -1 : r.idx[j];
      nn_d2[i * 5 + j] = r.d2[j];
    }
    if (tie) tie[i] = (r.d2[4] < 1.0 && r.tie()) ? 1 : 0;
  }
}

// One surfOptimization pass (MO:1618-1687).  Exactly one of pose6 / T12 non-NULL.
void SYM(surf_optimization)(const float* map4, int nm, void* h, const float* scan4, int nq, const float* pose6,
                            const float* T12, int* nn_idx, float* nn_d2, float* coeff4, unsigned char* flag,
                            unsigned char* tie, int threads) {
  float T[12];
  if (pose6) pose_to_T(pose6, T); else std::memcpy(T, T12, sizeof(T));
  surf_optimization((const P4*)map4, nm, (const Index*)h, (const P4*)scan4, nq, T, nn_idx, nn_d2, (P4*)coeff4,
                    flag, tie, threads);
}

// combineOptimizationCoeffs + AtA/AtB of LMOptimization (MO:1689-1700, 1735-1783).  Returns Nsel.
int SYM(normal_equations)(const float* scan4, const float* coeff4, const unsigned char* flag, int nq,
                          const float* pose6, double* JtJ, double* Jtr) {
  return accumulate_normal_equations((const P4*)scan4, (const P4*)coeff4, flag, nq, pose6, JtJ, Jtr);
}

// The 6x6 tail of LMOptimization (MO:1784-1835).  Returns 1 when converged.
int SYM(lm_solve_update)(const double* JtJ, const double* Jtr, int iter_count, float* pose_io, float* matP_io,
                         int* degenerate_io, float* delta_r, float* delta_t) {
  LmState st;
  std::memcpy(st.pose, pose_io, sizeof(st.pose));
  std::memcpy(st.matP, matP_io, sizeof(st.matP));
  st.degenerate = *degenerate_io;
  const bool conv = lm_solve_update(JtJ, Jtr, iter_count, st, *delta_r, *delta_t);
  std::memcpy(pose_io, st.pose, sizeof(st.pose));
  std::memcpy(matP_io, st.matP, sizeof(st.matP));
  *degenerate_io = st.degenerate;
  return conv ? 1 : 0;
}

// OpenCV pieces, exposed one by one so tests can pin them against cv2.
int SYM(cv_solve6_qr)(const float* A, const float* b, float* x) { return cv_solve6_qr(A, b, x) ? 1 : 0; }
void SYM(cv_eigen6)(const float* A, float* W, float* V) { cv_eigen6(A, W, V); }
int SYM(cv_inv6)(const float* A, float* inv) { return cv_inv6(A, inv) ? 1 : 0; }
void SYM(cv_gemm6)(const float* A, const float* B, float* C) { cv_gemm6(A, B, C); }
void SYM(qr53_solve)(const float* A15, const float* b5, float* x3) {
  float A[5][3];
  std::memcpy(A, A15, sizeof(A));
  qr53_solve(A, b5, x3);
}
// surfOptimization's per-point plane fit and weight (MO:1641-1684) on given neighbours; returns the accept flag.
int SYM(plane_residual)(const float* ori4, const float* sel4, const float* nbr20, float d2_4, float* coeff4) {
  P4 nb[5], c;
  std::memcpy(nb, nbr20, sizeof(nb));
  const bool ok = plane_residual(*(const P4*)ori4, *(const P4*)sel4, nb, d2_4, c);
  std::memcpy(coeff4, &c, sizeof(c));
  return ok ? 1 : 0;
}
// Eigen::umeyama's rotation (no scaling) from the 3x3 cross-covariance, row-major.
void SYM(umeyama_rotation)(const float* sigma9, float* R9) { umeyama_rotation(sigma9, R9); }

struct s2m_result {
  int iterations, converged, n_sel, is_degenerate, tie_queries;
  float delta_r, delta_t;
  double JtJ[36], Jtr[6];
  float pose_hist[30][6];
  int nsel_hist[30];
  double ms_build, ms_loop;
};

// scan2MapOptimization (MO:1839-1865) without transformUpdate.  Returns 0 OK, 2 few features
// (n <= 30, MO:1844), 3 empty map.  The KD-tree is (re)built inside, as the reference does every scan
// (MO:1846), unless a prebuilt handle is passed; brute != 0 forces brute-force k-NN.
int SYM(scan2map)(const float* map4, int nm, void* h, int brute, const float* scan4, int nq, float* pose_io,
                  float* matP_io, int* degenerate_io, int max_iter, int threads, s2m_result* res) {
  std::memset(res, 0, sizeof(*res));
  res->is_degenerate = *degenerate_io;
  if (nm <= 0) return 3;
  if (!(nq > 30)) return 2;
  const P4* map = (const P4*)map4;
  const P4* scan = (const P4*)scan4;
  Index* own = nullptr;
  const Index* ix = (const Index*)h;
  double t0 = now_ms();
  if (!ix && !brute) { own = new Index(); own->build(map, nm); ix = own; }
  if (brute) ix = nullptr;
  res->ms_build = now_ms() - t0;
  t0 = now_ms();
  std::vector<P4> coeff((size_t)nq);
  std::vector<unsigned char> flag((size_t)nq), tie((size_t)nq);
  LmState st;
  std::memcpy(st.pose, pose_io, sizeof(st.pose));
  std::memcpy(st.matP, matP_io, sizeof(st.matP));
  st.degenerate = *degenerate_io;
  for (int it = 0; it < max_iter; ++it) {
    float T[12];
    pose_to_T(st.pose, T);  // updatePointAssociateToMap (MO:1613-1616)
    surf_optimization(map, nm, ix, scan, nq, T, nullptr, nullptr, coeff.data(), flag.data(), tie.data(), threads);
    const int nsel = accumulate_normal_equations(scan, coeff.data(), flag.data(), nq, st.pose, res->JtJ, res->Jtr);
    int nt = 0;
    for (int i = 0; i < nq; ++i) nt += (tie[i] && flag[i]) ? 1 : 0;
    res->iterations = it + 1;
    res->n_sel = nsel;
    res->tie_queries = nt;
    res->nsel_hist[it] = nsel;
    bool conv = false;
    if (nsel >= 50)  // MO:1721-1724: below 50 the pose is untouched and the loop simply repeats
      conv = lm_solve_update(res->JtJ, res->Jtr, it, st, res->delta_r, res->delta_t);
    std::memcpy(res->pose_hist[it], st.pose, sizeof(st.pose));
    if (conv) { res->converged = 1; break; }
  }
  res->ms_loop = now_ms() - t0;
  res->is_degenerate = st.degenerate;
  std::memcpy(pose_io, st.pose, sizeof(st.pose));
  std::memcpy(matP_io, st.matP, sizeof(st.matP));
  *degenerate_io = st.degenerate;
  delete own;
  return 0;
}

// ---------------------------------------------------------------------------------------------
// a1: ImageProjection::projectPointCloud + deskewPoint + findRotation (IP:577-615, 545-575, 502-527).
// raw = n records of 8 floats: x y z pad intensity (ring u16 | pad) time pad  (PointXYZIRT, IP:4-15).
struct deskew_params {
  int n_scan, downsample_rate, point_filter_num;
  float min_front, min_back, min_left, min_right, max_range, max_intensity;
};

static void rot_from_rpy(float rx, float ry, float rz, float R[9]) {  // getTransformation(0,0,0,rx,ry,rz)
  const float pose[6] = {rx, ry, rz, 0.f, 0.f, 0.f};
  float T[12];
  pose_to_T(pose, T);
  R[0] = T[0]; R[1] = T[1]; R[2] = T[2]; R[3] = T[4]; R[4] = T[5]; R[5] = T[6]; R[6] = T[8]; R[7] = T[9]; R[8] = T[10];
}
static void inv3(const float m[9], float r[9]) {  // Eigen compute_inverse_size3 (cofactors / det)
#define M(i, j) m[(i) * 3 + (j)]
#define COF(i, j) (M(((i) + 1) % 3, ((j) + 1) % 3) * M(((i) + 2) % 3, ((j) + 2) % 3) - M(((i) + 1) % 3, ((j) + 2) % 3) * M(((i) + 2) % 3, ((j) + 1) % 3))
  const float c00 = COF(0, 0), c10 = COF(1, 0), c20 = COF(2, 0);
  const float det = (c00 * M(0, 0) + c10 * M(1, 0)) + c20 * M(2, 0);
  const float invdet = 1.f / det;
  r[0] = c00 * invdet; r[1] = c10 * invdet; r[2] = c20 * invdet;
  r[3] = COF(0, 1) * invdet; r[4] = COF(1, 1) * invdet; r[5] = COF(2, 1) * invdet;
  r[6] = COF(0, 2) * invdet; r[7] = COF(1, 2) * invdet; r[8] = COF(2, 2) * invdet;
#undef COF
#undef M
}
static void find_rotation(double t, const double* imu_t, const double* rx, const double* ry, const double* rz,
                          int ptr_cur, float* ox, float* oy, float* oz) {  // IP:502-527
  int f = 0;
  while (f < ptr_cur) {
    if (t < imu_t[f]) break;
    ++f;
  }
  if (t > imu_t[f] || f == 0) {
    *ox = (float)rx[f]; *oy = (float)ry[f]; *oz = (float)rz[f];
  } else {
    const int b = f - 1;
    const double rf = (t - imu_t[b]) / (imu_t[f] - imu_t[b]);
    const double rb = (imu_t[f] - t) / (imu_t[f] - imu_t[b]);
    *ox = (float)(rx[f] * rf + rx[b] * rb);
    *oy = (float)(ry[f] * rf + ry[b] * rb);
    *oz = (float)(rz[f] * rf + rz[b] * rb);
  }
}

int SYM(deskew)(const float* raw8, int n, const deskew_params* prm, double time_scan_cur, const double* imu_t,
                const double* imu_rx, const double* imu_ry, const double* imu_rz, int n_imu, int deskew_enabled,
                float* out4) {
  P4* out = (P4*)out4;
  int m = 0;
  bool first = true;
  float Rs_inv[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
  const int ptr_cur = n_imu - 1;  // imuPointerCur after the --imuPointerCur at IP:411
  for (int i = 0; i < n; ++i) {
    const float* r = raw8 + (size_t)i * 8;
    P4 p{r[0], r[1], r[2], r[4]};
    uint16_t ring;
    std::memcpy(&ring, r + 5, sizeof(ring));
    const float time = r[6];
    const float range = std::sqrt(p.x * p.x + p.y * p.y + p.z * p.z);  // common_lib pointDistance
    if ((p.y < prm->min_front && -prm->min_back < p.y && p.x < prm->min_left && -prm->min_right < p.x) ||
        range > prm->max_range || p.i > prm->max_intensity)
      continue;
    const int row = ring;
    if (row < 0 || row >= prm->n_scan) continue;
    if (row % prm->downsample_rate != 0) continue;
    if (i % prm->point_filter_num != 0) continue;
    if (deskew_enabled && n_imu > 1) {
      const double pt = time_scan_cur + (double)time;
      float ax, ay, az;
      find_rotation(pt, imu_t, imu_rx, imu_ry, imu_rz, ptr_cur, &ax, &ay, &az);
      float R[9];
      rot_from_rpy(ax, ay, az, R);
      if (first) { inv3(R, Rs_inv); first = false; }
      float B[9];
      for (int a = 0; a < 3; ++a)
        for (int b = 0; b < 3; ++b)
          B[a * 3 + b] = (Rs_inv[a * 3 + 0] * R[0 * 3 + b] + Rs_inv[a * 3 + 1] * R[1 * 3 + b]) + Rs_inv[a * 3 + 2] * R[2 * 3 + b];
      P4 q;
      q.x = B[0] * p.x + B[1] * p.y + B[2] * p.z + 0.f;
      q.y = B[3] * p.x + B[4] * p.y + B[5] * p.z + 0.f;
      q.z = B[6] * p.x + B[7] * p.y + B[8] * p.z + 0.f;
      q.i = p.i;
      p = q;
    }
    out[m++] = p;
  }
  return m;
}

int SYM(omp_max_threads)(void) {
#ifdef _OPENMP
  return omp_get_max_threads();
#else
  return 1;
#endif
}

}  // extern "C"
