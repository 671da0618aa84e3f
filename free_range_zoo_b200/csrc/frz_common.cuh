// Shared device helpers for the fused step kernels (sm_100a).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

#include "frz.h"

// State of one caller's pipelined host step (include/frz.h): its events and, once the pipeline has run, the whole
// multi-stream pipeline of one step as an instantiated CUDA graph -- later steps with the same buffers cost one
// cudaGraphLaunch (plus one node update per slice when the caller hands in a different page-locked action buffer)
// instead of ~40 stream API calls, which is what bounds a host-driven step once the copies overlap the kernels.
struct FrzHostPipeline {
  int device = -1;
  cudaEvent_t events[1 + 2 * FRZ_MAX_CHUNKS] = {};
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  std::vector<unsigned char> signature;  // everything the captured work depends on except the host action pointer
  struct ActionCopy {
    cudaGraphNode_t node;
    void* dst;
    size_t offset, bytes;  // source = host action buffer + offset
  };
  std::vector<ActionCopy> action_copies;
  const void* captured_actions = nullptr;
};

namespace frz {

constexpr unsigned kFullMask = 0xffffffffu;
constexpr int kMaxDevices = 64;  // launch-geometry caches are kept per device ordinal

// ---------------------------------------------------------------------------------------------- host side

void set_error(const char* fmt, ...);
int check_launch(const char* what);

inline int current_device() {
  int device = 0;
  cudaGetDevice(&device);
  return device;
}

// SMs of the current device (B200: 148 = 2 dies x 74), queried once per device
inline int sm_count() {
  static int cache[kMaxDevices] = {};
  const int device = current_device();
  int count = (device >= 0 && device < kMaxDevices) ? cache[device] : 0;
  if (count == 0) {
    cudaDeviceGetAttribute(&count, cudaDevAttrMultiProcessorCount, device);
    if (count < 1) count = 1;
    if (device >= 0 && device < kMaxDevices) cache[device] = count;
  }
  return count;
}

// resident CTAs per SM of `kernel` on the current device; cached per (instantiation, device), re-queried when the
// dynamic shared-memory footprint changes
template <class Kernel>
int resident_ctas(Kernel kernel, int threads, size_t smem) {
  static int ctas[kMaxDevices] = {};
  static size_t smem_of[kMaxDevices] = {};
  const int device = current_device();
  const bool cacheable = device >= 0 && device < kMaxDevices;
  if (cacheable && ctas[device] > 0 && smem_of[device] == smem) return ctas[device];
  int count = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&count, kernel, threads, smem);
  if (count < 1) count = 1;
  if (cacheable) {
    ctas[device] = count;
    smem_of[device] = smem;
  }
  return count;
}

inline int persistent_grid(int work_ctas, int ctas_per_sm) {
  const int cap = sm_count() * ctas_per_sm;
  return work_ctas < cap ? (work_ctas < 1 ? 1 : work_ctas) : cap;
}

// pipelined host-buffer step (frz_host.cuh): chunk control blocks <- main block before the slices run, main block <-
// OR of the chunks' published flags afterwards; events[0] = "broadcast done", then FRZ_MAX_CHUNKS "slice i uploaded"
// and FRZ_MAX_CHUNKS "slice i finished"
int control_broadcast(FrzControl* main_block, FrzControl* chunk_blocks, int count, cudaStream_t stream);
int control_merge(FrzControl* main_block, FrzControl* chunk_blocks, int count, cudaStream_t stream);
// the events of `pipeline`, or (NULL) of the calling thread on the current device; nullptr + error string on failure
cudaEvent_t* pipeline_events(FrzHostPipeline* pipeline);
// int16 / int8 [count] (element_bytes = 2 / 1) -> int32 [count] on the device (FRZ_HOST_ACTIONS_I16 / _I8)
int widen_actions(const void* packed, int element_bytes, int32_t* actions, size_t count, cudaStream_t stream);

// ---------------------------------------------------------------------------------------------- Philox4x32-10

struct Philox {
  uint32_t key0, key1;
  __device__ __forceinline__ Philox(uint64_t seed) : key0(uint32_t(seed)), key1(uint32_t(seed >> 32)) {}

  // Counter-based: (env, step, stream) -> 4 x 32 random bits.  Trajectories depend only on the global environment
  // index, the per-environment step counter and the event stream, never on the launch geometry or GPU count.
  __device__ __forceinline__ uint4 operator()(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3) const {
    uint32_t k0 = key0, k1 = key1;
#pragma unroll
    for (int round = 0; round < 10; ++round) {
      const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
      const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
      c0 = hi1 ^ c1 ^ k0;
      c1 = lo1;
      c2 = hi0 ^ c3 ^ k1;
      c3 = lo0;
      k0 += 0x9E3779B9u;
      k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
  }
};

// 24 random bits -> uniform in [0, 1) on the fp32 grid k * 2^-24 (same support as torch.rand's fp32 output)
__device__ __forceinline__ float u01(uint32_t bits) { return float(bits >> 8) * 5.9604644775390625e-08f; }

// position of the k-th (0-based) set bit of w; caller guarantees k < popc(w)
__device__ __forceinline__ int select_bit(uint32_t w, int k) {
  int pos = 0;
#pragma unroll
  for (int span = 16; span >= 1; span >>= 1) {
    const int below = __popc(w & ((1u << span) - 1u));
    if (k >= below) {
      k -= below;
      w >>= span;
      pos += span;
    }
  }
  return pos;
}

// ---------------------------------------------------------------------------------------------- shared memory

// Shared memory is addressed through explicit 32-bit shared-window addresses (one base register + immediates) instead
// of generic pointers: the compiler then emits plain LDS/STS [R + imm] and never re-derives the window base.
__device__ __forceinline__ uint32_t shared_address(const void* pointer) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(pointer));
}
// read-only tables (written once before a __syncthreads): loads may be combined / moved freely
__device__ __forceinline__ uint32_t lds_const(uint32_t address) {
  uint32_t value;
  asm("ld.shared.u32 %0, [%1];" : "=r"(value) : "r"(address));
  return value;
}
__device__ __forceinline__ uint4 lds_const_v4(uint32_t address) {
  uint4 value;
  asm("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(value.x), "=r"(value.y), "=r"(value.z), "=r"(value.w) : "r"(address));
  return value;
}
// scratch that changes between warp-level synchronisation points: ordered with respect to each other
__device__ __forceinline__ uint32_t lds(uint32_t address) {
  uint32_t value;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(value) : "r"(address) : "memory");
  return value;
}
__device__ __forceinline__ uint4 lds_v4(uint32_t address) {
  uint4 value;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(value.x), "=r"(value.y), "=r"(value.z), "=r"(value.w) : "r"(address) : "memory");
  return value;
}
__device__ __forceinline__ void sts(uint32_t address, uint32_t value) {
  asm volatile("st.shared.u32 [%0], %1;" : : "r"(address), "r"(value) : "memory");
}

// Ampere-style asynchronous copies (LDGSTS) for pieces that are not 16-byte multiples
__device__ __forceinline__ void cp_async_4(uint32_t shared_dst, const void* global_src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" : : "r"(shared_dst), "l"(global_src) : "memory");
}
__device__ __forceinline__ void cp_async_8(uint32_t shared_dst, const void* global_src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" : : "r"(shared_dst), "l"(global_src) : "memory");
}
__device__ __forceinline__ void cp_async_16(uint32_t shared_dst, const void* global_src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" : : "r"(shared_dst), "l"(global_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" : : : "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" : : : "memory"); }

// ---------------------------------------------------------------------------------------------- bulk async copies

// true in exactly one lane of a fully converged warp (the hardware's choice): the issuer of warp-uniform work such as
// bulk copies -- the compiler emits them once, without the serialisation loop a `lane == 0` test makes it build
__device__ __forceinline__ bool elect_one() {
  uint32_t elected;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "elect.sync _|p, 0xffffffff;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(elected));
  return elected != 0u;
}

// 1-D bulk copies of the async proxy (the TMA unit; SASS UBLKCP): one elected thread moves a whole tile between global
// and shared memory, completion of loads is signalled on an mbarrier, stores are tracked as bulk groups.  Addresses and
// sizes must be multiples of 16 bytes.
__device__ __forceinline__ void mbarrier_init(uint32_t barrier, uint32_t arrivals) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" : : "r"(barrier), "r"(arrivals) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" : : : "memory");
}
__device__ __forceinline__ void mbarrier_expect_bytes(uint32_t barrier, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" : : "r"(barrier), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbarrier_arrive(uint32_t barrier) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" : : "r"(barrier) : "memory");
}
// barrier among a subset of the CTA's warps (named barrier `id`, `threads` = participating threads, a multiple of 32)
__device__ __forceinline__ void named_barrier_sync(int id, int threads) {
  asm volatile("bar.sync %0, %1;" : : "r"(id), "r"(threads) : "memory");
}
__device__ __forceinline__ void mbarrier_wait(uint32_t barrier, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred done;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 done, [%0], %1;\n"
      "@!done bra WAIT_LOOP;\n"
      "}\n"
      : : "r"(barrier), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_load(uint32_t shared_dst, const void* global_src, uint32_t bytes, uint32_t barrier) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               : : "r"(shared_dst), "l"(global_src), "r"(bytes), "r"(barrier) : "memory");
}
__device__ __forceinline__ void bulk_store(void* global_dst, uint32_t shared_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
               : : "l"(global_dst), "r"(shared_src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" : : : "memory"); }
// wait until the committed bulk stores have finished READING shared memory (it may then be reused / the CTA may exit)
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" : : : "memory"); }
// ... until at most `pending` of the most recently committed bulk-store groups are still reading shared memory
template <int pending>
__device__ __forceinline__ void bulk_wait_read_all_but() {
  asm volatile("cp.async.bulk.wait_group.read %0;" : : "n"(pending) : "memory");
}
// make generic-proxy writes to shared memory visible to the async proxy before a bulk store reads them
__device__ __forceinline__ void fence_async_shared() { asm volatile("fence.proxy.async.shared::cta;" : : : "memory"); }

// ---------------------------------------------------------------------------------------------- launch epilogue

// Called by every CTA once, after its last environment.
//   alive_bits: bit0 = this CTA saw an env that is still not terminated, bit1 = one that is still not truncated
//   agent_bits: bit a = agent a has at least one task in some env of this CTA (after this launch)
// The last CTA to arrive publishes the accumulated flags for the next launch (a step and a refresh both do: a refresh
// follows every reset, checkpoint restore and hand edit of the state, whose done flags the next step must see) and, after
// a step, advances the step counter -- every CTA read control->step / alive / agents_with_tasks at its start, so no
// reader is left when they change.
enum Publish { kPublishNothing = 0, kPublishRefresh = 1, kPublishStep = 2 };

__device__ __forceinline__ void finish_launch(FrzControl* control, unsigned alive_bits, unsigned fault_bits,
                                              unsigned agent_bits, int publish) {
  __shared__ unsigned s_alive, s_fault, s_agents;
  if (threadIdx.x == 0) {
    s_alive = 0;
    s_fault = 0;
    s_agents = 0;
  }
  __syncthreads();
  if (alive_bits) atomicOr(&s_alive, alive_bits);
  if (fault_bits) atomicOr(&s_fault, fault_bits);
  if (agent_bits) atomicOr(&s_agents, agent_bits);
  __syncthreads();
  if (threadIdx.x == 0) {
    if (s_alive) atomicOr(&control->alive_acc, s_alive);
    if (s_fault) atomicOr(&control->error_word, s_fault);
    if (s_agents) atomicOr(&control->agents_with_tasks_acc, s_agents);
    __threadfence();
    const unsigned arrived = atomicAdd(&control->ctas_done, 1u) + 1u;
    if (arrived == gridDim.x) {
      __threadfence();
      const unsigned alive = atomicExch(&control->alive_acc, 0u);
      const unsigned agents = atomicExch(&control->agents_with_tasks_acc, 0u);
      if (publish == kPublishStep) {
        control->alive = alive;
        control->step += 1;
      }
      if (publish != kPublishNothing) control->agents_with_tasks = agents;
      if (publish == kPublishRefresh) control->alive = alive;
      control->ctas_done = 0u;
    }
  }
}

}  // namespace frz
