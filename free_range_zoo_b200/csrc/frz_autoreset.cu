// Same-step autoreset of finished environments (frz_autoreset, include/frz_autoreset.h).
//
// Runs after a step on the same stream, two launches with no host read in between, so it also runs inside the
// step's CUDA graph:
//   autoreset_scan     one pass over the batch: copies of the step's done flags, the finished episodes' returns and
//                      lengths, the agents_with_tasks bits (task counts of the environments that go on, snapshot counts
//                      of those that restart) and the compacted list of finished environments (block scan of
//                      frz_scan.cuh, one atomic per CTA for its place in the list).  Its last CTA publishes the list
//                      length and the batch-wide flags, as finish_launch does at the end of a refresh.
//   autoreset_restore  persistent grid over (row, group of listed environments) warp items: a row gets as many lanes per
//                      environment as it has words (up to 32), so one warp restores 32 one-word rows or one long row;
//                      16-byte words where the addresses and the row size allow.  No atomics, nothing to publish.
//                      A row with a `keep` array has each word's old value stored there before the word is restored.
// Work is proportional to the number of finished environments, plus the scan's read of the flags and, for the
// environments that go on, their per-agent task counts.
#include "frz_autoreset.h"
#include "frz_scan.cuh"

namespace frz {
namespace {

constexpr int kRestoreThreads = 256;

struct RowTable {
  FrzAutoresetRow row[FRZ_AUTORESET_MAX_ROWS];
  int32_t word[FRZ_AUTORESET_MAX_ROWS];   // bytes per copy: 16, 8, 4 or 1, as the row's alignment allows
  int32_t lanes[FRZ_AUTORESET_MAX_ROWS];  // lanes per environment: the row's words rounded up to a power of two, <= 32
  int32_t count;
  int32_t reserved;
};

__global__ void __launch_bounds__(kScanThreads) autoreset_scan_kernel(const FrzAutoreset a, const int B) {
  __shared__ int s_total, s_base;
  __shared__ unsigned s_agents;
  const int A = a.num_agents;
  if (threadIdx.x == 0) s_agents = 0u;
  unsigned finished_items = 0u, agent_bits = 0u;
  int finished = 0;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    const int env = blockIdx.x * kScanBlock + i * kScanThreads + threadIdx.x;
    if (env < B) {
      const uint8_t terminated = a.terminated[env], truncated = a.truncated[env];
      const bool done = (terminated | truncated) != 0;
      a.step_terminated[env] = terminated;
      a.step_truncated[env] = truncated;
      a.done[env] = done;
      if (done) {
        for (int g = 0; g < A; ++g) a.episode_return[size_t(env) * A + g] = a.cumulative_rewards[size_t(env) * A + g];
        a.episode_length[env] = a.num_moves[env];
        finished_items |= 1u << i;
        ++finished;
      }
      // the task counts the environment has after the restart: the snapshot's if it restarts
      const int32_t* counts = done ? a.reset_agent_task_count : a.agent_task_count;
      if (counts != nullptr)
        for (int g = 0; g < A; ++g) agent_bits |= (counts[size_t(env) * A + g] > 0 ? 1u : 0u) << g;
    }
  }
  const int prefix = cta_exclusive_scan(finished, &s_total);  // (synchronises: s_agents is initialised)
  agent_bits = __reduce_or_sync(kFullMask, agent_bits);
  if ((threadIdx.x & 31) == 0 && agent_bits) atomicOr(&s_agents, agent_bits);
  if (threadIdx.x == 0) s_base = s_total > 0 ? int(atomicAdd(&a.scratch[0], unsigned(s_total))) : 0;
  __syncthreads();
  int at = s_base + prefix;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i)
    if (finished_items >> i & 1u) a.finished[at++] = blockIdx.x * kScanBlock + i * kScanThreads + threadIdx.x;
  if (threadIdx.x == 0) {
    if (s_agents) atomicOr(&a.control->agents_with_tasks_acc, s_agents);
    // the last CTA publishes the list length and the batch-wide flags, and leaves the scratch zero for the next call;
    // the flags are read by the next step, which runs after the restore
    __threadfence();
    if (atomicAdd(&a.scratch[1], 1u) + 1u == gridDim.x) {
      __threadfence();
      *a.finished_count = int(atomicExch(&a.scratch[0], 0u));
      a.scratch[1] = 0u;
      a.control->agents_with_tasks = atomicExch(&a.control->agents_with_tasks_acc, 0u);
      a.control->alive = 3u;  // after the restart no environment is terminated or truncated
    }
  }
}

// the `rank`-th of `threads` threads copies its share of one row of `bytes` bytes in words of type Word; with kKeep it
// first stores each word's current value to `keep` (the same thread loads and overwrites the same address: no ordering)
template <class Word, bool kKeep>
__device__ __forceinline__ void copy_words(char* dst, const char* src, char* keep, size_t bytes, int rank, int threads) {
  const size_t words = bytes / sizeof(Word);
  for (size_t i = rank; i < words; i += threads) {
    if (kKeep) reinterpret_cast<Word*>(keep)[i] = reinterpret_cast<const Word*>(dst)[i];
    reinterpret_cast<Word*>(dst)[i] = src != nullptr ? reinterpret_cast<const Word*>(src)[i] : Word{};
  }
}

template <bool kKeep>
__device__ __forceinline__ void restore_words(char* dst, const char* src, char* keep, size_t bytes, int word, int rank,
                                              int threads) {
  switch (word) {
    case 16: copy_words<uint4, kKeep>(dst, src, keep, bytes, rank, threads); break;
    case 8: copy_words<uint2, kKeep>(dst, src, keep, bytes, rank, threads); break;
    case 4: copy_words<uint32_t, kKeep>(dst, src, keep, bytes, rank, threads); break;
    default: copy_words<uint8_t, kKeep>(dst, src, keep, bytes, rank, threads); break;
  }
}

__device__ __forceinline__ void restore_row(const FrzAutoresetRow& row, int word, int env, int rank, int threads) {
  const size_t bytes = size_t(row.bytes);
  char* dst = static_cast<char*>(row.dst) + size_t(env) * bytes;
  const char* src = row.src != nullptr ? static_cast<const char*>(row.src) + size_t(env) * bytes : nullptr;
  if (row.keep != nullptr)
    restore_words<true>(dst, src, static_cast<char*>(row.keep) + size_t(env) * bytes, bytes, word, rank, threads);
  else
    restore_words<false>(dst, src, nullptr, bytes, word, rank, threads);
}

__global__ void __launch_bounds__(kRestoreThreads) autoreset_restore_kernel(const FrzAutoreset a, const RowTable rows) {
  const int count = *a.finished_count;
  if (count == 0) return;
  const int lane = threadIdx.x & 31;
  const int warps = gridDim.x * (kRestoreThreads / 32);
  // warp items row after row: row r has ceil(count / envs per warp) of them; `first` = the first item of row r
  int r = 0, first = 0;
  for (int item = blockIdx.x * (kRestoreThreads / 32) + (threadIdx.x >> 5);; item += warps) {
    for (; r < rows.count; ++r) {
      const int per_warp = 32 / rows.lanes[r];
      const int items = (count + per_warp - 1) / per_warp;
      if (item < first + items) break;
      first += items;
    }
    if (r == rows.count) break;
    const int lanes = rows.lanes[r];
    const int slot = (item - first) * (32 / lanes) + lane / lanes;
    if (slot < count) restore_row(rows.row[r], rows.word[r], a.finished[slot], lane % lanes, lanes);
  }
}

}  // namespace
}  // namespace frz

extern "C" int frz_autoreset(const FrzAutoreset* autoreset, int32_t parallel_envs, void* stream) {
  using namespace frz;
  const char* what = "frz_autoreset";
  const FrzAutoreset* a = autoreset;
  if (a == nullptr || a->terminated == nullptr || a->truncated == nullptr || a->step_terminated == nullptr ||
      a->step_truncated == nullptr || a->done == nullptr || a->cumulative_rewards == nullptr ||
      a->episode_return == nullptr || a->num_moves == nullptr || a->episode_length == nullptr || a->control == nullptr ||
      a->finished == nullptr || a->finished_count == nullptr || a->scratch == nullptr ||
      (a->agent_task_count == nullptr) != (a->reset_agent_task_count == nullptr) ||
      (a->row_count > 0 && a->rows == nullptr)) {
    set_error("%s: a required pointer is NULL", what);
    return FRZ_ERR_NULL;
  }
  if (parallel_envs <= 0 || a->num_agents < 1 || a->num_agents > FRZ_MAX_AGENTS || a->row_count < 0 ||
      a->row_count > FRZ_AUTORESET_MAX_ROWS) {
    set_error("%s: unsupported shape B=%d agents=%d rows=%d (<= %d)", what, parallel_envs, a->num_agents, a->row_count,
              FRZ_AUTORESET_MAX_ROWS);
    return FRZ_ERR_SHAPE;
  }
  RowTable table = {};
  int64_t warp_items = 0;  // when every environment restarts
  for (int r = 0; r < a->row_count; ++r) {
    const FrzAutoresetRow& row = a->rows[r];
    if (row.dst == nullptr) {
      set_error("%s: row %d has a NULL destination", what, r);
      return FRZ_ERR_NULL;
    }
    if (row.bytes <= 0) {
      set_error("%s: row %d has %lld bytes per environment", what, r, static_cast<long long>(row.bytes));
      return FRZ_ERR_SHAPE;
    }
    const uintptr_t alignment = reinterpret_cast<uintptr_t>(row.dst) | reinterpret_cast<uintptr_t>(row.src) |
                                reinterpret_cast<uintptr_t>(row.keep) | uintptr_t(row.bytes);
    const int word = (alignment & 15u) == 0 ? 16 : (alignment & 7u) == 0 ? 8 : (alignment & 3u) == 0 ? 4 : 1;
    const int64_t words = row.bytes / word;
    int lanes = 1;
    while (lanes < 32 && lanes < words) lanes <<= 1;
    table.row[r] = row;
    table.word[r] = word;
    table.lanes[r] = lanes;
    warp_items += (int64_t(parallel_envs) + 32 / lanes - 1) / (32 / lanes);
  }
  table.count = a->row_count;
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  autoreset_scan_kernel<<<(parallel_envs + kScanBlock - 1) / kScanBlock, kScanThreads, 0, s>>>(*a, parallel_envs);
  const int status = check_launch("autoreset_scan_kernel");
  if (status != FRZ_OK) return status;
  // enough warps for every item when the whole batch restarts, up to a full SM's worth of CTAs per SM
  const int64_t work_ctas = (warp_items * 32 + kRestoreThreads - 1) / kRestoreThreads;
  const int grid = persistent_grid(int(work_ctas < (1 << 20) ? (work_ctas < 1 ? 1 : work_ctas) : (1 << 20)),
                                   2048 / kRestoreThreads);
  autoreset_restore_kernel<<<grid, kRestoreThreads, 0, s>>>(*a, table);
  return check_launch("autoreset_restore_kernel");
}
