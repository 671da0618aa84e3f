// Block-wide exclusive prefix sums shared by the observation compaction kernels (frz_gather.cu, frz_obs.cu).
// Works on int (row offsets) and int2 (row offsets and mask byte offsets of the compact download side by side).
#pragma once

#include "frz_common.cuh"

namespace frz {

constexpr int kScanThreads = 256;
constexpr int kScanItems = 4;  // counts per thread
constexpr int kScanBlock = kScanThreads * kScanItems;

__device__ __forceinline__ int scan_add(int a, int b) { return a + b; }
__device__ __forceinline__ int2 scan_add(int2 a, int2 b) { return make_int2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ int scan_shfl_up(int value, int d) { return __shfl_up_sync(kFullMask, value, d); }
__device__ __forceinline__ int2 scan_shfl_up(int2 value, int d) {
  return make_int2(__shfl_up_sync(kFullMask, value.x, d), __shfl_up_sync(kFullMask, value.y, d));
}
__device__ __forceinline__ int scan_sub(int a, int b) { return a - b; }
__device__ __forceinline__ int2 scan_sub(int2 a, int2 b) { return make_int2(a.x - b.x, a.y - b.y); }

template <class T>
__device__ __forceinline__ T warp_inclusive_scan(T value, int lane) {
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const T below = scan_shfl_up(value, d);
    if (lane >= d) value = scan_add(value, below);
  }
  return value;
}

// exclusive scan of one value per thread over the CTA; returns this thread's prefix, *total = the CTA's sum
template <class T>
__device__ __forceinline__ T cta_exclusive_scan(T value, T* total) {
  __shared__ T warp_sums[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const T inclusive = warp_inclusive_scan(value, lane);
  if (lane == 31) warp_sums[warp] = inclusive;
  __syncthreads();
  if (warp == 0) {
    const int warps = (blockDim.x + 31) >> 5;
    const T sum = lane < warps ? warp_sums[lane] : T{};
    const T scanned = warp_inclusive_scan(sum, lane);
    warp_sums[lane] = scan_sub(scanned, sum);  // exclusive prefix of the warps
    if (lane == 31) *total = scanned;
  }
  __syncthreads();
  const T result = scan_add(scan_sub(inclusive, value), warp_sums[warp]);
  __syncthreads();  // (warp_sums is reused by the next call)
  return result;
}

}  // namespace frz
