// Compaction of the padded per-environment observation arrays for callers that read them on the host
// (frz_gather_live_rows, include/frz.h).
//
// The step kernels publish observations as padded arrays -- task_obs [B, capacity, columns], action masks
// [B, agents, capacity] -- of which only the first count[b] rows of every environment are live.  The reference hands the
// same data to a policy as jagged nested tensors (a value buffer + offsets: wildfire.py:669-717, rideshare.py:398-467).
// A policy on the host needs exactly that value buffer, and the PCIe link is the slowest hop of the whole step, so the
// live rows are packed on the device first: offsets = exclusive prefix sum of the counts, then one warp per
// (environment, row block) segment copies its rows to the packed position.  All of it is plain HBM streaming.
#include <algorithm>

#include "frz_scan.cuh"

namespace frz {
namespace {

// block_sums[i] = sum of counts[i * kScanBlock ... )
__global__ void __launch_bounds__(kScanThreads) gather_block_sums(const int32_t* __restrict__ counts, int B,
                                                                  int32_t* __restrict__ block_sums) {
  __shared__ int total;
  const int base = blockIdx.x * kScanBlock + threadIdx.x * kScanItems;
  int mine = 0;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) mine += base + i < B ? max(counts[base + i], 0) : 0;
  cta_exclusive_scan(mine, &total);
  if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

// in place: block_sums[i] <- sum of block_sums[0 .. i), block_sums[blocks] <- everything (one CTA, any number of blocks)
__global__ void __launch_bounds__(kScanThreads) gather_top_scan(int32_t* __restrict__ block_sums, int blocks) {
  __shared__ int total;
  int carry = 0;
  for (int base = 0; base < blocks; base += kScanThreads) {
    const int at = base + threadIdx.x;
    const int mine = at < blocks ? block_sums[at] : 0;
    const int prefix = cta_exclusive_scan(mine, &total);
    if (at < blocks) block_sums[at] = carry + prefix;
    carry += total;
  }
  if (threadIdx.x == 0) block_sums[blocks] = carry;
}

// offsets[b] = live rows before environment b; offsets[B] = all of them
__global__ void __launch_bounds__(kScanThreads) gather_offsets(const int32_t* __restrict__ counts, int B,
                                                               const int32_t* __restrict__ block_sums, int blocks,
                                                               int32_t* __restrict__ offsets) {
  __shared__ int total;
  const int base = blockIdx.x * kScanBlock + threadIdx.x * kScanItems;
  int item[kScanItems], mine = 0;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    item[i] = base + i < B ? max(counts[base + i], 0) : 0;
    mine += item[i];
  }
  int prefix = block_sums[blockIdx.x] + cta_exclusive_scan(mine, &total);
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    if (base + i < B) offsets[base + i] = prefix;
    prefix += item[i];
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) offsets[B] = block_sums[blocks];
}

// One warp per (environment, row block): count[b] rows of row_bytes bytes from the padded array to the packed one.
__global__ void __launch_bounds__(256) gather_copy(const FrzGatherArray array, const int32_t* __restrict__ counts,
                                                   const int32_t* __restrict__ offsets, const int B) {
  const int lane = threadIdx.x & 31;
  const long long segments = (long long)B * array.groups;
  const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
  const size_t row = size_t(array.row_bytes);
  for (long long s = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); s < segments; s += warps) {
    const int env = int(s / array.groups), group = int(s - (long long)env * array.groups);
    const int count = min(max(counts[env], 0), array.capacity);
    const size_t bytes = size_t(count) * row;
    const char* from = static_cast<const char*>(array.src) + (size_t(env) * array.groups + group) * array.capacity * row;
    char* to = static_cast<char*>(array.dst) + (size_t(offsets[env]) * array.groups + size_t(group) * count) * row;
    const size_t misalignment = reinterpret_cast<size_t>(from) | reinterpret_cast<size_t>(to) | bytes;
    if ((misalignment & 15u) == 0u) {
      for (size_t i = lane; i < (bytes >> 4); i += 32) reinterpret_cast<uint4*>(to)[i] = reinterpret_cast<const uint4*>(from)[i];
    } else if ((misalignment & 3u) == 0u) {
      for (size_t i = lane; i < (bytes >> 2); i += 32) reinterpret_cast<uint32_t*>(to)[i] = reinterpret_cast<const uint32_t*>(from)[i];
    } else {
      for (size_t i = lane; i < bytes; i += 32) to[i] = from[i];
    }
  }
}

}  // namespace
}  // namespace frz

extern "C" {

int frz_gather_live_rows(const int32_t* counts, int32_t parallel_envs, int32_t* offsets, int32_t* scratch,
                         const FrzGatherArray* arrays, int32_t array_count, void* stream) {
  using namespace frz;
  if (counts == nullptr || offsets == nullptr || scratch == nullptr || (array_count > 0 && arrays == nullptr)) {
    set_error("frz_gather_live_rows: NULL counts / offsets / scratch / arrays");
    return FRZ_ERR_NULL;
  }
  if (parallel_envs <= 0 || array_count < 0) {
    set_error("frz_gather_live_rows: unsupported shape B=%d arrays=%d", parallel_envs, array_count);
    return FRZ_ERR_SHAPE;
  }
  for (int i = 0; i < array_count; ++i) {
    const FrzGatherArray& a = arrays[i];
    if (a.src == nullptr || a.dst == nullptr) {
      set_error("frz_gather_live_rows: array %d has a NULL pointer", i);
      return FRZ_ERR_NULL;
    }
    if (a.row_bytes < 1 || a.capacity < 1 || a.groups < 1 ||
        uint64_t(parallel_envs) * uint64_t(a.capacity) >= (1ull << 31)) {  // offsets are int32 row counts
      set_error("frz_gather_live_rows: array %d: unsupported row_bytes=%d capacity=%d groups=%d", i, a.row_bytes, a.capacity,
                a.groups);
      return FRZ_ERR_SHAPE;
    }
  }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int blocks = (parallel_envs + kScanBlock - 1) / kScanBlock;
  gather_block_sums<<<blocks, kScanThreads, 0, s>>>(counts, parallel_envs, scratch);
  gather_top_scan<<<1, kScanThreads, 0, s>>>(scratch, blocks);
  gather_offsets<<<blocks, kScanThreads, 0, s>>>(counts, parallel_envs, scratch, blocks, offsets);
  for (int i = 0; i < array_count; ++i) {
    const long long segments = (long long)parallel_envs * arrays[i].groups;
    const int grid = persistent_grid(int(std::min<long long>((segments + 7) / 8, 1 << 30)), 8);
    gather_copy<<<grid, 256, 0, s>>>(arrays[i], counts, offsets, parallel_envs);
  }
  return check_launch("frz_gather_live_rows");
}

}  // extern "C"
