// scancontext.cuh — Scan Context pieces shared by the descriptor (scancontext.cu) and the loop-closure detection
// over the descriptor store (loopdetect.cu), so that both derive a descriptor's keys with the same arithmetic.
#pragma once
#include "common.cuh"

namespace liogpu {

constexpr int SC_RING = LIOGPU_SC_NUM_RING, SC_SECTOR = LIOGPU_SC_NUM_SECTOR, SC_BINS = SC_RING * SC_SECTOR;

// Key k of a descriptor d (row-major [ring][sector], f64, typically in shared memory): k < SC_RING is the ring key
// (row mean, makeRingkeyFromScancontext, Scancontext.cpp:198-210), SC_RING <= k < SC_RING + SC_SECTOR the sector key
// k - SC_RING (column mean, makeSectorkeyFromScancontext, :212-225).  Sequential sums, then / size.
__device__ __forceinline__ double sc_key(const double* d, int k) {
  double s = 0.0;
  if (k < SC_RING) {
    for (int c = 0; c < SC_SECTOR; ++c) s += d[k * SC_SECTOR + c];
    return s / SC_SECTOR;
  }
  const int c = k - SC_RING;
  for (int r = 0; r < SC_RING; ++r) s += d[r * SC_SECTOR + c];
  return s / SC_RING;
}

}  // namespace liogpu
