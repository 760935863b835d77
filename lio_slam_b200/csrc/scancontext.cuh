// scancontext.cuh — Scan Context pieces shared by the descriptor (scancontext.cu) and the loop-closure detection
// over the descriptor store (loopdetect.cu), so that both derive a descriptor's bins and keys with the same arithmetic.
#pragma once
#include "common.cuh"

namespace liogpu {

constexpr int SC_RING = LIOGPU_SC_NUM_RING, SC_SECTOR = LIOGPU_SC_NUM_SECTOR, SC_BINS = SC_RING * SC_SECTOR;
constexpr int SC_CHUNK = 4096;  // points per block when many keyframes are binned at once (16 per thread)

// The images of n keyframes' descriptors (scancontext.cu): entry f's u32 image goes to the first half of its f64 slot
// slots + f * SC_BINS.  blk_off[f] = sum over earlier keyframes of ceil(n_g / SC_CHUNK), n_blocks = blk_off[n];
// srcs / offs as stage_keyframes builds them (not read when n_blocks = 0).  Two launches at most.
cudaError_t launch_sc_bin_keyframes(Ctx* c, const float4* const* srcs, const int* offs, const int* blk_off, int n,
                                    int n_blocks, double lidar_height, double max_radius, double* slots);

// image of NO_POINT (Scancontext.cpp:158), the initial value of every bin
__device__ __forceinline__ unsigned sc_none() { return f2ord(-1000.0f); }
// the descriptor entry of a bin's image: empty bins (still NO_POINT) -> 0 (:186-189)
__device__ __forceinline__ double sc_bin_value(unsigned o) {
  const float v = ord2f(o);
  return v == -1000.0f ? 0.0 : (double)v;
}

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
