// liorf_oracle_loop.h — CPU ORACLE (TEST INFRASTRUCTURE, NOT PRODUCT CODE) for loop-closure detection.
//
// The restatement of SCManager::detectLoopClosureID and detectLoopClosureDistance, kept beside the main restatement
// (liorf_oracle_core.h, whose types and L2_Simple distance it uses) with the same rules: C++14, no dependencies,
// every float expression in the operation order of the cited source, built with -ffp-contract=off.  PARITY UNPINNED.
#pragma once
#include "liorf_oracle_core.h"

#include <string>
#include <utility>

namespace liorf_oracle {

// ---------------------------------------------------------------------------------------------
// f3 (detection): SCManager::detectLoopClosureID (include/Scancontext.cpp) driven call by call, with the state the
// reference keeps between calls (tree_making_period_conter and the snapshot polarcontext_invkeys_to_search_).  The
// store only grows, so the KD-tree's snapshot is a prefix of the stored ring keys; the tree is replaced by an
// exhaustive search that returns the same set.
// Third-party arithmetic restated [3P] (versions unpinned like everything else in the oracle):
//   * nanoflann L2_Adaptor<float> (KDTreeVectorOfVectorsAdaptor over the f32 ring keys, eig2stdvec): per group of
//     four dimensions result += ((d0*d0 + d1*d1) + d2*d2) + d3*d3, five groups, f32.  Exact k nearest; ties are
//     ordered by (d2, index) here (nanoflann keeps the first visited) and counted in knn_ties.
//   * Eigen 3.3.7 linear-vectorised redux for doubles with SSE2 (two doubles a packet, two packets a step) for
//     VectorXd::dot / norm over the 20 rows of a column and MatrixXd(1,60)::norm of the sector-key difference:
//     four partial sums s_k over the elements j = k mod 4 in ascending j, combined as (s0 + s2) + (s1 + s3); the
//     norm is sqrt of that squared sum.  Chosen as the restatement of Redux.h; not pinned against Eigen.
// circshift moves column c to (c + s) % 60; distDirectSC skips a column pair with a zero norm and returns
// 1 - sum / n_eff (NaN for n_eff = 0, which never wins a `<`).
struct ScParams {
  int num_exclude_recent, num_candidates, tree_making_period;
  double search_ratio, sc_dist_thres;
};
constexpr int SC_MAX_CAND = 32;
struct ScResult {
  int loop_id;
  float yaw;
  int n_stored, n_searchable, tree_rebuilt, n_candidates;
  int nn_idx, nn_align, knn_ties;
  double min_dist;
  int cand[SC_MAX_CAND];
  float cand_d2[SC_MAX_CAND];
  double cand_dist[SC_MAX_CAND];
  int cand_shift[SC_MAX_CAND];
};

inline void sc_keys(const double* desc, double* ringkey, double* sectorkey) {  // Scancontext.cpp:198-225
  for (int r = 0; r < SC_NUM_RING; ++r) {
    double sum = 0;
    for (int c = 0; c < SC_NUM_SECTOR; ++c) sum += desc[r * SC_NUM_SECTOR + c];
    ringkey[r] = sum / SC_NUM_SECTOR;
  }
  for (int c = 0; c < SC_NUM_SECTOR; ++c) {
    double sum = 0;
    for (int r = 0; r < SC_NUM_RING; ++r) sum += desc[r * SC_NUM_SECTOR + c];
    sectorkey[c] = sum / SC_NUM_RING;
  }
}

// Eigen redux order [3P]: x_j = f(j) for j < n (n a multiple of 4)
template <class F>
inline double eigen_redux4(int n, F f) {
  double s0 = f(0), s1 = f(1), s2 = f(2), s3 = f(3);
  for (int j = 4; j < n; j += 4) { s0 += f(j); s1 += f(j + 1); s2 += f(j + 2); s3 += f(j + 3); }
  return (s0 + s2) + (s1 + s3);
}
inline double sc_col_norm(const double* desc, int c) {
  return std::sqrt(eigen_redux4(SC_NUM_RING, [&](int r) { const double v = desc[r * SC_NUM_SECTOR + c]; return v * v; }));
}
inline double sc_col_dot(const double* d1, int c1, const double* d2, int c2) {
  return eigen_redux4(SC_NUM_RING, [&](int r) { return d1[r * SC_NUM_SECTOR + c1] * d2[r * SC_NUM_SECTOR + c2]; });
}
inline float sc_ringkey_d2(const float* a, const float* b) {  // nanoflann L2_Adaptor<float>, 20 dims
  float result = 0.f;
  for (int g = 0; g < SC_NUM_RING; g += 4) {
    const float d0 = a[g] - b[g], d1 = a[g + 1] - b[g + 1], d2 = a[g + 2] - b[g + 2], d3 = a[g + 3] - b[g + 3];
    result += d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3;
  }
  return result;
}
inline int sc_search_radius(double search_ratio) {  // SEARCH_RADIUS = round(0.5 * SEARCH_RATIO * cols)
  return (int)std::round(0.5 * search_ratio * SC_NUM_SECTOR);
}
inline float sc_deg2rad(float degrees) { return degrees * M_PI / 180.0; }  // Scancontext.cpp

class ScManager {
 public:
  std::vector<double> descs, vkeys, norms;  // per entry: 1200 / 60 / 60 doubles
  std::vector<float> rkeys;                 // per entry: 20 floats
  int size = 0;
  long long counter = 0;  // tree_making_period_conter
  int snap = 0;           // size of polarcontext_invkeys_to_search_

  void add(const double* desc) {  // makeAndSaveScancontextAndKeys (Scancontext.cpp:228-243)
    double rk[SC_NUM_RING], sk[SC_NUM_SECTOR];
    sc_keys(desc, rk, sk);
    descs.insert(descs.end(), desc, desc + SC_NUM_RING * SC_NUM_SECTOR);
    for (int r = 0; r < SC_NUM_RING; ++r) rkeys.push_back((float)rk[r]);
    vkeys.insert(vkeys.end(), sk, sk + SC_NUM_SECTOR);
    for (int c = 0; c < SC_NUM_SECTOR; ++c) norms.push_back(sc_col_norm(desc, c));
    ++size;
  }

  // distanceBtnScanContext(query q, candidate i) -> (distance, shift)
  void distance(int q, int i, double search_ratio, double& dist, int& shift) const {
    const double* vq = &vkeys[(size_t)q * SC_NUM_SECTOR];
    const double* vc = &vkeys[(size_t)i * SC_NUM_SECTOR];
    int align = 0;  // fastAlignUsingVkey
    double min_norm = 10000000;
    for (int s = 0; s < SC_NUM_SECTOR; ++s) {
      const double nrm = std::sqrt(eigen_redux4(SC_NUM_SECTOR, [&](int j) {
        const double d = vq[j] - vc[(j - s + SC_NUM_SECTOR) % SC_NUM_SECTOR];
        return d * d;
      }));
      if (nrm < min_norm) { align = s; min_norm = nrm; }
    }
    const int R = sc_search_radius(search_ratio);
    std::vector<int> space{align};
    for (int ii = 1; ii < R + 1; ++ii) {
      space.push_back((align + ii + SC_NUM_SECTOR) % SC_NUM_SECTOR);
      space.push_back((align - ii + SC_NUM_SECTOR) % SC_NUM_SECTOR);
    }
    std::sort(space.begin(), space.end());
    const double* dq = &descs[(size_t)q * SC_NUM_RING * SC_NUM_SECTOR];
    const double* dc = &descs[(size_t)i * SC_NUM_RING * SC_NUM_SECTOR];
    const double* nq = &norms[(size_t)q * SC_NUM_SECTOR];
    const double* nc = &norms[(size_t)i * SC_NUM_SECTOR];
    shift = 0;
    dist = 10000000;
    for (int s : space) {  // distDirectSC(query, circshift(candidate, s))
      int n_eff = 0;
      double sum = 0;
      for (int c = 0; c < SC_NUM_SECTOR; ++c) {
        const int cc = (c - s + SC_NUM_SECTOR) % SC_NUM_SECTOR;
        if ((nq[c] == 0) | (nc[cc] == 0)) continue;
        sum = sum + sc_col_dot(dq, c, dc, cc) / (nq[c] * nc[cc]);
        n_eff = n_eff + 1;
      }
      const double d = 1.0 - sum / n_eff;
      if (d < dist) { shift = s; dist = d; }
    }
  }

  // detectLoopClosureID on the newest stored descriptor
  ScResult detect(const ScParams& p, int threads) {
    ScResult r;
    std::memset(&r, 0, sizeof(r));
    r.loop_id = -1;
    r.nn_idx = -1;
    r.min_dist = 10000000;
    r.n_stored = size;
    if (size < p.num_exclude_recent + 1) { r.n_searchable = snap; return r; }  // early return, counter untouched
    if (counter % p.tree_making_period == 0) { snap = size - p.num_exclude_recent; r.tree_rebuilt = 1; }
    counter = counter + 1;
    r.n_searchable = snap;
    const int q = size - 1;
    const float* qk = &rkeys[(size_t)q * SC_NUM_RING];
    std::vector<std::pair<float, int>> d2((size_t)snap);
#pragma omp parallel for num_threads(threads) schedule(static) if (snap > 4096)
    for (int i = 0; i < snap; ++i) d2[i] = std::make_pair(sc_ringkey_d2(qk, &rkeys[(size_t)i * SC_NUM_RING]), i);
    const int L = std::min(p.num_candidates + 1, snap);  // the k nearest and the next one (ties across the boundary)
    std::nth_element(d2.begin(), d2.begin() + (L - 1), d2.end());
    std::sort(d2.begin(), d2.begin() + L);
    for (int j = 1; j < L; ++j) r.knn_ties += d2[j].first == d2[j - 1].first;
    r.n_candidates = std::min(p.num_candidates, snap);
    double min_dist = 10000000;
    int nn_align = 0, nn_idx = 0;
    for (int j = 0; j < r.n_candidates; ++j) {
      r.cand[j] = d2[j].second;
      r.cand_d2[j] = d2[j].first;
      distance(q, r.cand[j], p.search_ratio, r.cand_dist[j], r.cand_shift[j]);
      if (r.cand_dist[j] < min_dist) { min_dist = r.cand_dist[j]; nn_align = r.cand_shift[j]; nn_idx = r.cand[j]; }
    }
    r.min_dist = min_dist;
    r.nn_idx = nn_idx;
    r.nn_align = nn_align;
    if (min_dist < p.sc_dist_thres) r.loop_id = nn_idx;
    r.yaw = sc_deg2rad(nn_align * (360.0 / double(SC_NUM_SECTOR)));
    return r;
  }
};

// detectLoopClosureDistance (MO ~1271-1300) minus the loopIndexContainer check: among the key poses with L2_Simple
// d2 < (float)(r*r) around the newest one (FLANN radiusSearch, sorted by distance; ties by lower index here), the
// first with |time - time_cur| > time_diff; -1 if there is none or it is the newest pose itself.
inline int detect_loop_distance(const P4* key3d, const double* key_time, int n, double time_cur, float radius, float time_diff) {
  if (n <= 0) return -1;
  const P4& last = key3d[n - 1];
  const float r2 = (float)((double)radius * (double)radius);
  float best_d2 = 0.f;
  int best = -1;
  for (int i = 0; i < n; ++i) {
    const float d2 = l2_simple(last, key3d[i]);
    if (!(d2 < r2) || !(std::fabs(key_time[i] - time_cur) > (double)time_diff)) continue;
    if (best < 0 || d2 < best_d2) { best = i; best_d2 = d2; }
  }
  return best == n - 1 ? -1 : best;
}

}  // namespace liorf_oracle
