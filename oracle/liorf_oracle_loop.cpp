// liorf_oracle_loop.cpp — CPU ORACLE (TEST INFRASTRUCTURE, NOT PRODUCT CODE).  PARITY UNPINNED — see the header of
// liorf_oracle_core.h.  extern "C" entry points for ctypes (oracle/loop_oracle.py) of the loop-closure detection
// restatement in liorf_oracle_loop.h.  Built by loop_oracle.build() with the flags of oracle/Makefile.
#include "liorf_oracle_loop.h"

#ifdef _OPENMP
#include <omp.h>
#endif

using namespace liorf_oracle;

extern "C" {

// n_calls detectLoopClosureID calls of a fresh SCManager, call j made after the store has grown to store_sizes[j]
// descriptors (non-decreasing, <= n_desc): descriptors are added one by one and the manager keeps its own counter.
int loop_sc_detect_loops(const double* descs, int n_desc, const int* store_sizes, int n_calls, const ScParams* prm,
                         int threads, ScResult* out) {
  ScManager sc;
  for (int j = 0; j < n_calls; ++j) {
    if (store_sizes[j] > n_desc || (j > 0 && store_sizes[j] < store_sizes[j - 1])) return -1;
    while (sc.size < store_sizes[j]) sc.add(descs + (size_t)sc.size * SC_NUM_RING * SC_NUM_SECTOR);
    out[j] = sc.detect(*prm, threads);
  }
  return 0;
}

// detectLoopClosureDistance (MO ~1271-1300) without the loopIndexContainer check
int loop_detect_loop_distance(const float* key3d4, const double* key_time, int n, double time_cur, float radius,
                              float time_diff) {
  return detect_loop_distance((const P4*)key3d4, key_time, n, time_cur, radius, time_diff);
}

int loop_omp_max_threads(void) {
#ifdef _OPENMP
  return omp_get_max_threads();
#else
  return 1;
#endif
}

}  // extern "C"
