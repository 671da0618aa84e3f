// Compact observation download (frz_observe_compact, include/frz_obs.h).
//
// The encoders read the padded observation arrays from HBM and write the compact encoding to device staging buffers;
// a flush kernel then moves exactly the live bytes of every array to the caller's page-locked host buffers through
// their device mapping, with aligned 16-byte stores over the whole contiguous range (full lines on the link).  The
// live sizes are read on the device, so the host needs no read-back between compaction and download.  Storing from
// the encoders straight into mapped memory was measured first and rejected: one environment's rows or mask bits are
// 25-100-byte runs written by different warps, partial lines on the link (profiles/README.md).
//
//   obs_block_sums / obs_top_scan / obs_offsets  int2 prefix sum of (counts[b], ceil(groups * counts[b] / 8)): row
//                                                offsets and mask byte offsets
//   obs_dense   one thread per 32-bit word of the output: column selection and narrowing of whole arrays
//   obs_rows    one warp per (environment, row block): the live rows, narrowed, to their packed position
//   obs_mask    one warp per environment: __ballot_sync over the flattened (agent, task) index -> its mask bytes
//   obs_flush   staging -> mapped host memory, the live bytes only
#include <algorithm>
#include <vector>

#include "frz_obs.h"
#include "frz_scan.cuh"

namespace frz {
namespace {

__host__ __device__ __forceinline__ int type_bytes(int type) {
  return (type == FRZ_OBS_I32 || type == FRZ_OBS_F32) ? 4 : (type == FRZ_OBS_I16 ? 2 : 1);
}

// element `index` of a source array as 32 raw bits (float32 as its bit pattern, uint8 zero-extended)
__device__ __forceinline__ int32_t load_element(const void* src, int type, size_t index) {
  if (type == FRZ_OBS_U8) return int32_t(static_cast<const uint8_t*>(src)[index]);
  return static_cast<const int32_t*>(src)[index];
}

// whether `value` is representable in `type`
__device__ __forceinline__ bool fits(int32_t value, int type) {
  switch (type) {
    case FRZ_OBS_I8: return value >= -128 && value <= 127;
    case FRZ_OBS_U8: return value >= 0 && value <= 255;
    case FRZ_OBS_I16: return value >= -32768 && value <= 32767;
    default: return true;
  }
}

// the low type_bytes(type) bytes of the encoded element
__device__ __forceinline__ uint32_t encode(int32_t value, int type) {
  return type_bytes(type) == 4 ? uint32_t(value) : uint32_t(value) & (type_bytes(type) == 2 ? 0xffffu : 0xffu);
}

__device__ __forceinline__ void store_element(char* dst, int type, size_t index, uint32_t bits) {
  switch (type_bytes(type)) {
    case 1: reinterpret_cast<uint8_t*>(dst)[index] = uint8_t(bits); break;
    case 2: reinterpret_cast<uint16_t*>(dst)[index] = uint16_t(bits); break;
    default: reinterpret_cast<uint32_t*>(dst)[index] = bits; break;
  }
}

// n elements of dst (starting at element `first` of dst) <- element(e) for e in [0, n), converted to a.dst_type, by the
// `threads` threads numbered `rank`: whole 32-bit words where the run is word-aligned, single elements at its ends
template <class Element>
__device__ __forceinline__ bool store_run(const FrzObsArray& a, size_t first, size_t n, int rank, int threads,
                                          Element&& element) {
  bool bad = false;
  const int size = type_bytes(a.dst_type), per = 4 / size;
  char* const dst = static_cast<char*>(a.dst);
  // leading elements up to the first word boundary, then whole words, then the tail
  const size_t lead = size_t((per - int(first % per)) % per), head = lead < n ? lead : n;
  for (size_t e = rank; e < head; e += threads) {
    const int32_t value = element(e);
    bad |= !fits(value, a.dst_type);
    store_element(dst, a.dst_type, first + e, encode(value, a.dst_type));
  }
  const size_t words = (n - head) / per;
  uint32_t* const word_dst = reinterpret_cast<uint32_t*>(dst + (first + head) * size);
  for (size_t w = rank; w < words; w += threads) {
    uint32_t word = 0;
#pragma unroll 4
    for (int j = 0; j < per; ++j) {
      const int32_t value = element(head + w * per + j);
      bad |= !fits(value, a.dst_type);
      word |= encode(value, a.dst_type) << (8 * size * j);
    }
    word_dst[w] = word;
  }
  for (size_t e = head + words * per + rank; e < n; e += threads) {
    const int32_t value = element(e);
    bad |= !fits(value, a.dst_type);
    store_element(dst, a.dst_type, first + e, encode(value, a.dst_type));
  }
  return bad;
}

// live rows of environment `env`: counts outside [0, limit] are clamped here and flagged by the row / mask encoders, so
// that the offsets and the encoders agree and nothing is written beyond the buffers (limit <= every array's capacity)
__device__ __forceinline__ int live_rows(const int32_t* counts, int env, int limit) { return min(max(counts[env], 0), limit); }

__device__ __forceinline__ int2 env_sizes(const int32_t* counts, int env, int limit, int mask_groups) {
  const int count = live_rows(counts, env, limit);
  return make_int2(count, (mask_groups * count + 7) >> 3);
}

// block_sums[i] = sums of (rows, mask bytes) of environments [i * kScanBlock, ...)
__global__ void __launch_bounds__(kScanThreads) obs_block_sums(const int32_t* __restrict__ counts, int B, int limit,
                                                               int mask_groups, int2* __restrict__ block_sums) {
  __shared__ int2 total;
  const int base = blockIdx.x * kScanBlock + threadIdx.x * kScanItems;
  int2 mine = make_int2(0, 0);
#pragma unroll
  for (int i = 0; i < kScanItems; ++i)
    if (base + i < B) mine = scan_add(mine, env_sizes(counts, base + i, limit, mask_groups));
  cta_exclusive_scan(mine, &total);
  if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

// in place: block_sums[i] <- sum of block_sums[0 .. i), block_sums[blocks] <- everything (one CTA)
__global__ void __launch_bounds__(kScanThreads) obs_top_scan(int2* __restrict__ block_sums, int blocks) {
  __shared__ int2 total;
  int2 carry = make_int2(0, 0);
  for (int base = 0; base < blocks; base += kScanThreads) {
    const int at = base + threadIdx.x;
    const int2 mine = at < blocks ? block_sums[at] : make_int2(0, 0);
    const int2 prefix = cta_exclusive_scan(mine, &total);
    if (at < blocks) block_sums[at] = scan_add(carry, prefix);
    carry = scan_add(carry, total);
  }
  if (threadIdx.x == 0) block_sums[blocks] = carry;
}

// scan[b] = (rows, mask bytes) before environment b, scan[B] = all of them; offsets <- the row part.  Also writes the
// status block (overflow flag cleared -- the encoders run after this kernel on the same stream -- and the totals).
__global__ void __launch_bounds__(kScanThreads) obs_offsets(const int32_t* __restrict__ counts, int B, int limit,
                                                            int mask_groups,
                                                            const int2* __restrict__ block_sums, int blocks,
                                                            int2* __restrict__ scan, int32_t* __restrict__ offsets,
                                                            uint32_t* __restrict__ overflow) {
  __shared__ int2 total;
  const int base = blockIdx.x * kScanBlock + threadIdx.x * kScanItems;
  int2 item[kScanItems], mine = make_int2(0, 0);
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    item[i] = base + i < B ? env_sizes(counts, base + i, limit, mask_groups) : make_int2(0, 0);
    mine = scan_add(mine, item[i]);
  }
  int2 prefix = scan_add(block_sums[blockIdx.x], cta_exclusive_scan(mine, &total));
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    if (base + i < B) {
      scan[base + i] = prefix;
      offsets[base + i] = prefix.x;
    }
    prefix = scan_add(prefix, item[i]);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    scan[B] = block_sums[blocks];
    offsets[B] = block_sums[blocks].x;
    *reinterpret_cast<uint4*>(overflow) = make_uint4(0u, uint32_t(block_sums[blocks].x), uint32_t(block_sums[blocks].y), 0u);
  }
}

__global__ void __launch_bounds__(256) obs_dense(const FrzObsArray a, const int B, uint32_t* __restrict__ overflow) {
  const size_t n = size_t(B) * a.capacity * a.columns;
  const int threads = gridDim.x * blockDim.x, rank = blockIdx.x * blockDim.x + threadIdx.x;
  const void* const src = a.src;
  const int src_type = a.src_type, columns = a.columns, src_columns = a.src_columns, column_first = a.column_first;
  const bool bad = store_run(a, 0, n, rank, threads, [=](size_t e) {
    // (32-bit index arithmetic: the host side keeps every padded array below 2^31 elements)
    const uint32_t row = uint32_t(e) / uint32_t(columns), column = uint32_t(e) - row * uint32_t(columns);
    return load_element(src, src_type, size_t(row) * src_columns + column_first + column);
  });
  if (bad) *overflow = 1u;
}

__global__ void __launch_bounds__(256) obs_rows(const FrzObsArray a, const int32_t* __restrict__ counts,
                                                const int2* __restrict__ scan, const int B, const int limit,
                                                uint32_t* __restrict__ overflow) {
  const int lane = threadIdx.x & 31;
  const long long segments = (long long)B * a.groups;
  const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
  bool bad = false;
  for (long long s = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); s < segments; s += warps) {
    const int env = int(s / a.groups), group = int(s - (long long)env * a.groups);
    const int count = live_rows(counts, env, limit);
    bad |= count != counts[env];
    const size_t src_row = (size_t(env) * a.groups + group) * a.capacity;
    const size_t first = (size_t(scan[env].x) * a.groups + size_t(group) * count) * a.columns;
    bad |= store_run(a, first, size_t(count) * a.columns, lane, 32, [=](size_t e) {
      const uint32_t row = uint32_t(e) / uint32_t(a.columns), column = uint32_t(e) - row * uint32_t(a.columns);
      return load_element(a.src, a.src_type, (src_row + row) * a.src_columns + a.column_first + column);
    });
  }
  if (bad) *overflow = 1u;
}

__global__ void __launch_bounds__(256) obs_mask(const FrzObsArray a, const int32_t* __restrict__ counts,
                                                const int2* __restrict__ scan, const int B, const int limit,
                                                uint32_t* __restrict__ overflow) {
  const int lane = threadIdx.x & 31;
  const int warps = gridDim.x * (blockDim.x >> 5);
  const uint8_t* const src = static_cast<const uint8_t*>(a.src);
  for (int env = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); env < B; env += warps) {
    const int count = live_rows(counts, env, limit);
    if (count != counts[env]) *overflow = 1u;
    const int bits = a.groups * count, bytes = (bits + 7) >> 3, words = (bits + 31) >> 5;
    uint8_t* const dst = static_cast<uint8_t*>(a.dst) + scan[env].y;
    const uint8_t* const rows = src + size_t(env) * a.groups * a.capacity;
    for (int first = 0; first < words; first += 32) {
      // word first + j of the environment's bit string ends up in lane j
      uint32_t mine = 0;
      for (int j = 0; j < min(32, words - first); ++j) {
        const int k = (first + j) * 32 + lane;
        bool set = false;
        if (k < bits) {
          const int group = k / count;
          set = rows[size_t(group) * a.capacity + (k - group * count)] != 0;
        }
        const uint32_t word = __ballot_sync(kFullMask, set);
        if (lane == j) mine = word;
      }
      const int at = 4 * (first + lane);
      if (at + 4 <= bytes && ((reinterpret_cast<size_t>(dst) + at) & 3u) == 0) {
        *reinterpret_cast<uint32_t*>(dst + at) = mine;
      } else {
        for (int i = 0; i < 4 && at + i < bytes; ++i) dst[at + i] = uint8_t(mine >> (8 * i));
      }
    }
  }
}

// staging -> host: fixed + scale * (pick == 1 ? total rows : pick == 2 ? total mask bytes : 0) bytes, both buffers
// 16-byte aligned
__global__ void __launch_bounds__(256) obs_flush(const uint4* __restrict__ src, uint4* __restrict__ dst,
                                                 const int2* __restrict__ total, const int pick, const long long scale,
                                                 const long long fixed) {
  long long bytes = fixed;
  if (pick != 0) bytes += scale * (pick == 1 ? total->x : total->y);
  const long long chunks = bytes >> 4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < chunks; i += (long long)gridDim.x * blockDim.x)
    dst[i] = src[i];
  if (blockIdx.x == 0 && threadIdx.x < int(bytes & 15))
    reinterpret_cast<char*>(dst + chunks)[threadIdx.x] = reinterpret_cast<const char*>(src + chunks)[threadIdx.x];
}

int flush_grid(long long max_bytes) {
  return persistent_grid(int(std::min<long long>((max_bytes / 16 + 255) / 256 + 1, 1 << 30)), 8);
}

// device address of page-locked host memory, or nullptr (with the error cleared) when it is not mapped for this device
template <class T>
T* mapped(T* host) {
  void* device = nullptr;
  if (cudaHostGetDevicePointer(&device, const_cast<void*>(static_cast<const void*>(host)), 0) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return static_cast<T*>(device);
}

bool valid_types(const FrzObsArray& a) {
  if (a.kind == FRZ_OBS_MASK_BITS) return a.src_type == FRZ_OBS_U8 && a.dst_type == FRZ_OBS_U8;
  if (a.src_type == FRZ_OBS_I32)
    return a.dst_type == FRZ_OBS_I32 || a.dst_type == FRZ_OBS_I16 || a.dst_type == FRZ_OBS_I8 || a.dst_type == FRZ_OBS_U8;
  return (a.src_type == FRZ_OBS_F32 || a.src_type == FRZ_OBS_U8) && a.dst_type == a.src_type;
}

}  // namespace
}  // namespace frz

extern "C" {

int frz_observe_compact(const FrzObsDownload* download, int32_t parallel_envs, void* stream) {
  using namespace frz;
  const char* what = "frz_observe_compact";
  if (download == nullptr || download->counts == nullptr || download->offsets == nullptr || download->scan == nullptr ||
      download->scratch == nullptr || download->status == nullptr ||
      (download->array_count > 0 && download->arrays == nullptr)) {
    set_error("%s: NULL download / counts / offsets / scan / scratch / status / arrays", what);
    return FRZ_ERR_NULL;
  }
  const int B = parallel_envs;
  if (B <= 0 || download->array_count < 0) {
    set_error("%s: unsupported shape B=%d arrays=%d", what, B, download->array_count);
    return FRZ_ERR_SHAPE;
  }
  bool has_mask = false;
  for (int i = 0; i < download->array_count; ++i) {
    const FrzObsArray& a = download->arrays[i];
    if (a.src == nullptr || a.dst == nullptr) {  // (host may be NULL: the caller downloads the staging itself)
      set_error("%s: array %d has a NULL pointer", what, i);
      return FRZ_ERR_NULL;
    }
    const bool mask = a.kind == FRZ_OBS_MASK_BITS;
    has_mask |= mask;
    const uint64_t padded = uint64_t(B) * uint64_t(a.groups > 0 ? a.groups : 0) * uint64_t(a.capacity > 0 ? a.capacity : 0);
    if ((a.kind != FRZ_OBS_DENSE && a.kind != FRZ_OBS_ROWS && !mask) || !valid_types(a) || a.groups < 1 ||
        a.capacity < 1 || a.columns < 1 || a.column_first < 0 || a.column_first + a.columns > a.src_columns ||
        (a.kind == FRZ_OBS_DENSE && a.groups != 1) ||
        (mask && (a.groups != download->mask_groups || a.src_columns != 1 || a.columns != 1)) ||
        (reinterpret_cast<uintptr_t>(a.dst) & 15u) != 0 ||  // (word stores, 16-byte flush)
        (reinterpret_cast<uintptr_t>(a.host) & 15u) != 0 ||
        padded * uint64_t(a.src_columns) >= (1ull << 31)) {  // offsets and mask offsets are int32
      set_error("%s: array %d: unsupported kind=%d types=%d->%d groups=%d capacity=%d columns=[%d, +%d) of %d", what, i,
                a.kind, a.src_type, a.dst_type, a.groups, a.capacity, a.column_first, a.columns, a.src_columns);
      return FRZ_ERR_SHAPE;
    }
  }
  if ((reinterpret_cast<uintptr_t>(download->offsets) & 15u) != 0 ||
      (reinterpret_cast<uintptr_t>(download->host_offsets) & 15u) != 0 ||
      (reinterpret_cast<uintptr_t>(download->status) & 15u) != 0) {
    set_error("%s: offsets / host_offsets / status must be 16-byte aligned", what);
    return FRZ_ERR_SHAPE;
  }
  const int mask_groups = has_mask ? download->mask_groups : 0;
  int limit = INT32_MAX / B;  // (the row offsets are int32; with row / mask arrays: their smallest capacity)
  for (int i = 0; i < download->array_count; ++i)
    if (download->arrays[i].kind != FRZ_OBS_DENSE) limit = std::min(limit, download->arrays[i].capacity);

  // every host pointer must be page-locked memory mapped for this device: checked before anything is launched
  uint32_t* const overflow = mapped(download->status);  // (status[0] is the overflow flag)
  int32_t* const host_offsets = download->host_offsets != nullptr ? mapped(download->host_offsets) : nullptr;
  std::vector<FrzObsArray> arrays(download->arrays, download->arrays + download->array_count);
  bool all_mapped = overflow != nullptr && (download->host_offsets == nullptr || host_offsets != nullptr);
  for (FrzObsArray& a : arrays) {
    if (a.host != nullptr) a.host = mapped(a.host);
    all_mapped &= a.host != nullptr || download->arrays[&a - arrays.data()].host == nullptr;
  }
  if (!all_mapped) {
    set_error("%s: status / host_offsets / host must be page-locked host memory mapped for the current device", what);
    return FRZ_ERR_UNSUPPORTED;
  }

  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int2* const scan = reinterpret_cast<int2*>(download->scan);
  int2* const block_sums = reinterpret_cast<int2*>(download->scratch);
  const int blocks = (B + kScanBlock - 1) / kScanBlock;
  obs_block_sums<<<blocks, kScanThreads, 0, s>>>(download->counts, B, limit, mask_groups, block_sums);
  obs_top_scan<<<1, kScanThreads, 0, s>>>(block_sums, blocks);
  obs_offsets<<<blocks, kScanThreads, 0, s>>>(download->counts, B, limit, mask_groups, block_sums, blocks, scan,
                                              download->offsets, overflow);
  if (host_offsets != nullptr) {
    const long long bytes = 4LL * (B + 1);
    obs_flush<<<flush_grid(bytes), 256, 0, s>>>(reinterpret_cast<const uint4*>(download->offsets),
                                                 reinterpret_cast<uint4*>(host_offsets), scan + B, 0, 0, bytes);
  }
  for (const FrzObsArray& a : arrays) {
    if (a.kind == FRZ_OBS_DENSE) {
      const size_t words = (size_t(B) * a.capacity * a.columns * type_bytes(a.dst_type) + 3) / 4;
      obs_dense<<<persistent_grid(int(std::min<size_t>((words + 255) / 256, 1u << 30)), 8), 256, 0, s>>>(a, B, overflow);
    } else if (a.kind == FRZ_OBS_ROWS) {
      const long long segments = (long long)B * a.groups;
      obs_rows<<<persistent_grid(int(std::min<long long>((segments + 7) / 8, 1 << 30)), 8), 256, 0, s>>>(
          a, download->counts, scan, B, limit, overflow);
    } else {
      obs_mask<<<persistent_grid((B + 7) / 8, 8), 256, 0, s>>>(a, download->counts, scan, B, limit, overflow);
    }
    if (a.host == nullptr) continue;
    const long long item = type_bytes(a.dst_type);
    const long long padded = (long long)B * a.groups * a.capacity * a.columns * item;
    const uint4* const from = static_cast<const uint4*>(a.dst);
    uint4* const to = static_cast<uint4*>(a.host);
    if (a.kind == FRZ_OBS_DENSE) {
      obs_flush<<<flush_grid(padded), 256, 0, s>>>(from, to, scan + B, 0, 0, padded);
    } else if (a.kind == FRZ_OBS_ROWS) {
      obs_flush<<<flush_grid(padded), 256, 0, s>>>(from, to, scan + B, 1, (long long)a.groups * a.columns * item, 0);
    } else {
      obs_flush<<<flush_grid(padded / 8 + B), 256, 0, s>>>(from, to, scan + B, 2, 1, 0);
    }
  }
  return check_launch(what);
}

}  // extern "C"
