// Policy actions from logits over the fixed-width slot layout (frz_<domain>_policy_actions, include/frz_policy.h).
//
// One launch, a group of G lanes per (environment, agent) row, the row mapping of frz_slots.cuh: slot t of a row belongs
// to lane t % G of its group, in round t / G, so every round's loads of a group are consecutive elements (coalesced, no
// alignment needed, any row stride).  G is chosen from C: one thread per row for C <= 16 (cybersecurity, small wildfire
// grids), else the smallest group that leaves at most 4 slots per lane, up to a warp (9 slots per lane for the largest
// grids).
//   pass 1  legality of every slot from the domain's own buffers (the Rule below), in registers; SAMPLE loads the
//           legal slots' logits, checks them and reduces their max m over the group
//   pass 2  SAMPLE: running sums of exp(l - m) in slot order, round by round (group inclusive scan + the carry of the
//           earlier rounds); the last one is S, computed by the same additions
//   pass 3  the target slot, uniform over the group: SAMPLE the first legal slot whose running sum exceeds u * S (the
//           last legal slot if none does), DECODE the caller's slot; the noop on a fault
//   pass 4  the lane owning the target writes the action (k = the slot's rank among the legal slots, its id), the slot
//           and the log-probability; every lane writes its legality bytes when asked to (with
//           FRZ_POLICY_PACKED_LEGAL, lane 0 of the group writes the row's words, built from the rounds' ballots)
// Equal logits: every exp term is exactly 1 and S is the exact count n + 1, so u * S is the single multiply of the
// uniform sampler (u01(r.x) * float(n + 1)) and the first running sum above it is at choice int(u * S): the choice is
// exactly frz_<domain>_sample_actions'.
#include <cuda_bf16.h>

#include "frz_common.cuh"
#include "frz_policy.h"
#include "frz_slots.cuh"

namespace frz {
namespace {

constexpr int kPolicyThreads = 256;

// ---------------------------------------------------------------------------------------------- legality per domain

// wildfire: task t < H*W is legal iff its action_mask byte is set (with show_bad_actions: iff t is a live task);
// slot H*W is the noop
struct WildfireRule {
  const uint8_t* action_mask;
  const int32_t* env_task_count;
  int32_t A, C, cells, mask_stride;
  bool show_bad;
  struct Row {
    const uint8_t* mask;
    int live;
  };
  __device__ __forceinline__ Row row(int env, int agent) const {
    if (show_bad) return {nullptr, env_task_count[env]};
    return {action_mask + (size_t(env) * A + agent) * size_t(mask_stride), 0};
  }
  __device__ __forceinline__ bool legal(const Row& r, int t) const {
    if (t >= cells) return t == cells;
    return show_bad ? t < r.live : r.mask[t] != 0;
  }
  __device__ __forceinline__ int ident(int env, int t) const { return t == cells ? -1 : 0; }
  __device__ __forceinline__ int noop() const { return cells; }
};

// rideshare: table row t < K is legal iff its task_mask byte is set, its id is the passenger's state (riding 2,
// accepted 1, else 0, from task_obs columns 5 and 4); slot K is the noop
struct RideshareRule {
  const uint8_t* task_mask;
  const int32_t* task_obs;
  int32_t A, C, capacity, reserved;
  struct Row {
    const uint8_t* mask;
  };
  __device__ __forceinline__ Row row(int env, int agent) const {
    return {task_mask + (size_t(env) * A + agent) * size_t(capacity)};
  }
  __device__ __forceinline__ bool legal(const Row& r, int t) const {
    if (t >= capacity) return t == capacity;
    return r.mask[t] != 0;
  }
  __device__ __forceinline__ int ident(int env, int t) const {
    if (t == capacity) return -1;
    const int32_t* obs = task_obs + (size_t(env) * capacity + t) * FRZ_RS_TASK_COLUMNS;
    return obs[5] != FRZ_PAD ? 2 : (obs[4] != FRZ_PAD ? 1 : 0);
  }
  __device__ __forceinline__ int noop() const { return capacity; }
};

// cybersecurity: node t < n (n = N for an agent that may act, 0 otherwise), the noop N, and for a defender that may
// act: patch N+1 (unless it is at its home node without show_bad_actions) and monitor N+2
struct CyberRule {
  const int32_t* env_task_count;
  const int32_t* agent_task_count;
  const int32_t* location;
  int32_t A, C, nodes, attackers;
  bool show_bad;
  struct Row {
    int n;
    bool acts, can_patch;  // a defender with n > 0 / that may also patch
  };
  __device__ __forceinline__ Row row(int env, int agent) const {
    const int n = show_bad ? env_task_count[env] : agent_task_count[size_t(env) * A + agent];
    const bool acts = agent >= attackers && n > 0;
    const bool can_patch =
        acts && (show_bad || location[size_t(env) * (A - attackers) + (agent - attackers)] != -1);
    return {n, acts, can_patch};
  }
  __device__ __forceinline__ bool legal(const Row& r, int t) const {
    if (t < nodes) return t < r.n;
    return t == nodes || (t == nodes + 1 ? r.can_patch : r.acts);
  }
  __device__ __forceinline__ int ident(int env, int t) const { return t < nodes ? 0 : nodes - 1 - t; }
  __device__ __forceinline__ int noop() const { return nodes; }
};

// ---------------------------------------------------------------------------------------------- the kernel

struct Launch {
  FrzPolicyActions policy;
  int32_t* actions;  // [B, A, 2]
  FrzControl* control;
  int64_t env_offset;
  int32_t rows;      // B * A
  int32_t reserved;
};

__device__ __forceinline__ float logit(const float* p) { return *p; }
__device__ __forceinline__ float logit(const __nv_bfloat16* p) { return __bfloat162float(*p); }

// PACKED: `legal` receives the packed words of include/frz_policy.h instead of bytes.  (Its minimum of one CTA per SM
// lets ptxas use the registers it needs instead of spilling a few bytes; 0 leaves the byte instantiations as they were.)
template <class Rule, int G, int PER, class T, bool PACKED>
__global__ void __launch_bounds__(kPolicyThreads, PACKED ? 1 : 0) policy_kernel(const Rule rule, const Launch L) {
  const FrzPolicyActions& P = L.policy;
  const int lane = threadIdx.x & 31, glane = lane & (G - 1), base = lane - glane;
  const int C = rule.C, A = rule.A;
  const uint64_t step = L.control->step;
  const Philox philox(P.sampler_seed);
  const T* logits = static_cast<const T*>(P.logits);
  constexpr int kRowsPerWarp = 32 / G;
  const int warps = gridDim.x * (kPolicyThreads / 32);
  // whole warps iterate together (ballots and shuffles need every lane); rows past the end are inactive
  for (int first = (blockIdx.x * (kPolicyThreads / 32) + (threadIdx.x >> 5)) * kRowsPerWarp; first < L.rows;
       first += warps * kRowsPerWarp) {
    const int row = first + lane / G;
    const bool active = row < L.rows;
    const int env = active ? row / A : 0, agent = active ? row - env * A : 0;
    typename Rule::Row r{};
    if (active) r = rule.row(env, agent);

    // pass 1: legality (bit j = slot j * G + glane) and, for SAMPLE, the legal logits and their max
    uint32_t legal_bits = 0u;
    float l[PER];
    float m = -INFINITY;
    bool bad = false;
#pragma unroll
    for (int j = 0; j < PER; ++j) {
      const int t = j * G + glane;
      const bool ok = active && t < C && rule.legal(r, t);
      legal_bits |= uint32_t(ok) << j;
      l[j] = -INFINITY;
      if (P.mode == FRZ_POLICY_SAMPLE && ok) {
        l[j] = logit(logits + size_t(row) * size_t(P.row_stride) + t);
        bad |= l[j] != l[j] || l[j] == INFINITY;
        m = fmaxf(m, l[j]);
      }
      if (!PACKED && P.legal != nullptr && active && t < C) P.legal[size_t(row) * C + t] = ok;
    }
    if (PACKED && P.legal != nullptr) {
      // round j's group ballot holds slots j * G .. j * G + G - 1, at shift (j * G) % 32 of word (j * G) / 32; a word
      // is stored as soon as its last round is in
      uint32_t* words = reinterpret_cast<uint32_t*>(P.legal) + size_t(row) * size_t((C + 31) / 32);
      const bool store = active && glane == 0;
      if (G == 1) {
        if (store) words[0] = legal_bits;
      } else {
        uint32_t word = 0u;
#pragma unroll
        for (int j = 0; j < PER; ++j) {
          word |= group_ballot<G>(legal_bits >> j & 1u, base) << (j * G % 32);
          if ((j + 1) * G % 32 == 0 || j == PER - 1) {
            if (store && j * G / 32 * 32 < C) words[j * G / 32] = word;
            word = 0u;
          }
        }
      }
    }
    if (P.mode == FRZ_POLICY_LEGAL) continue;

    int target = -1;  // uniform over the group
    float S = 0.f;
    if (P.mode == FRZ_POLICY_SAMPLE) {
#pragma unroll
      for (int o = G / 2; o >= 1; o >>= 1) m = fmaxf(m, __shfl_xor_sync(kFullMask, m, o, G));
      bad = group_ballot<G>(bad, base) != 0u || m == -INFINITY;
      // pass 2: running sums in slot order
      float running[PER];
#pragma unroll
      for (int j = 0; j < PER; ++j) running[j] = running_sum<G>(slot_term(legal_bits >> j & 1u, l[j], m), glane, S);
      // pass 3: the first legal slot whose running sum exceeds u * S, else the last legal slot
      const uint64_t genv = uint64_t(L.env_offset + env);
      const uint4 bits = philox(uint32_t(genv), uint32_t(step), 0xC0000000u | uint32_t(agent),
                                uint32_t(step >> 32) ^ uint32_t(genv >> 32));
      const float threshold = u01(bits.x) * S;
      int last = -1;
#pragma unroll
      for (int j = 0; j < PER; ++j) {
        const bool ok = legal_bits >> j & 1u;
        const uint32_t hit = group_ballot<G>(ok && running[j] > threshold, base);
        const uint32_t any = group_ballot<G>(ok, base);
        if (target < 0 && hit != 0u) target = j * G + __ffs(hit) - 1;
        if (any != 0u) last = j * G + 31 - __clz(any);
      }
      if (target < 0) target = last;
      if (bad) target = rule.noop();
    } else {  // DECODE
      const int wanted = active ? P.slot[row] : -1;
      bool mine = false;
#pragma unroll
      for (int j = 0; j < PER; ++j) mine |= j * G + glane == wanted && (legal_bits >> j & 1u);
      bad = group_ballot<G>(mine, base) == 0u;  // out of range or illegal
      target = bad ? rule.noop() : wanted;
    }

    // pass 4: the owner of the target writes the row's outputs
    int rank = 0, k = -1;
    float chosen = 0.f;
#pragma unroll
    for (int j = 0; j < PER; ++j) {
      const uint32_t any = group_ballot<G>(legal_bits >> j & 1u, base);
      if (j * G + glane == target) {
        k = rank + __popc(any & ((1u << glane) - 1u));
        chosen = l[j];
      }
      rank += __popc(any);
    }
    if (active && k >= 0) {
      reinterpret_cast<int2*>(L.actions)[row] = make_int2(k, rule.ident(env, target));
      if (P.mode == FRZ_POLICY_SAMPLE) {
        P.slot[row] = target;
        if (P.log_prob != nullptr) P.log_prob[row] = bad ? __int_as_float(0x7fc00000) : (chosen - m) - logf(S);
      }
      if (bad) atomicOr(&L.control->error_word, P.mode == FRZ_POLICY_SAMPLE ? FRZ_FAULT_BAD_LOGITS : FRZ_FAULT_ILLEGAL_SLOT);
    }
  }
}

// ---------------------------------------------------------------------------------------------- launch

template <class Rule, int G, int PER, bool PACKED>
void launch_typed(const Rule& rule, const Launch& launch, cudaStream_t stream) {
  const int64_t threads = int64_t(launch.rows) * G;
  const int work_ctas = int((threads + kPolicyThreads - 1) / kPolicyThreads);
  const int grid = persistent_grid(work_ctas, 2048 / kPolicyThreads);
  if (launch.policy.mode == FRZ_POLICY_SAMPLE && launch.policy.logits_type == FRZ_LOGITS_BF16)
    policy_kernel<Rule, G, PER, __nv_bfloat16, PACKED><<<grid, kPolicyThreads, 0, stream>>>(rule, launch);
  else
    policy_kernel<Rule, G, PER, float, PACKED><<<grid, kPolicyThreads, 0, stream>>>(rule, launch);
}

// lanes per row and slots per lane from C (<= FRZ_MAX_CELLS + 1), legality bytes or packed words
template <class Rule>
int launch(const Rule& rule, const Launch& launch, bool packed, cudaStream_t stream) {
  with_row_mapping(rule.C, [&](auto map) {
    using M = decltype(map);
    if (packed)
      launch_typed<Rule, M::G, M::PER, true>(rule, launch, stream);
    else
      launch_typed<Rule, M::G, M::PER, false>(rule, launch, stream);
    return 0;
  });
  return check_launch("policy_kernel");
}

// argument checks shared by the three domains; fills `launch`
int check_policy(const FrzPolicyActions* policy, int32_t* actions, FrzControl* control, int B, int A, int C,
                 const char* what, Launch* launch) {
  if (policy == nullptr || control == nullptr) {
    set_error("%s: NULL params / buffers / policy block", what);
    return FRZ_ERR_NULL;
  }
  const int mode = policy->mode & ~int32_t(FRZ_POLICY_PACKED_LEGAL);
  if (mode != FRZ_POLICY_SAMPLE && mode != FRZ_POLICY_DECODE && mode != FRZ_POLICY_LEGAL) {
    set_error("%s: unknown mode %d", what, policy->mode);
    return FRZ_ERR_UNSUPPORTED;
  }
  if (mode == FRZ_POLICY_SAMPLE && policy->logits_type != FRZ_LOGITS_F32 && policy->logits_type != FRZ_LOGITS_BF16) {
    set_error("%s: unknown logits type %d", what, policy->logits_type);
    return FRZ_ERR_UNSUPPORTED;
  }
  if ((mode == FRZ_POLICY_SAMPLE && (policy->logits == nullptr || policy->slot == nullptr)) ||
      (mode == FRZ_POLICY_DECODE && policy->slot == nullptr) || (mode != FRZ_POLICY_LEGAL && actions == nullptr) ||
      (mode == FRZ_POLICY_LEGAL && policy->legal == nullptr)) {
    set_error("%s: a pointer the mode needs is NULL", what);
    return FRZ_ERR_NULL;
  }
  if (B <= 0 || A < 1 || A > FRZ_MAX_AGENTS || int64_t(B) * A > INT32_MAX) {
    set_error("%s: unsupported shape B=%d agents=%d", what, B, A);
    return FRZ_ERR_SHAPE;
  }
  if (policy->slots != C) {
    set_error("%s: slots=%d, but this configuration has %d", what, policy->slots, C);
    return FRZ_ERR_SHAPE;
  }
  if (mode == FRZ_POLICY_SAMPLE && policy->row_stride < C) {
    set_error("%s: row_stride=%d < slots=%d", what, policy->row_stride, C);
    return FRZ_ERR_SHAPE;
  }
  if ((policy->mode & FRZ_POLICY_PACKED_LEGAL) != 0 && reinterpret_cast<uintptr_t>(policy->legal) % 4 != 0) {
    set_error("%s: packed legal mask is not 4-byte aligned", what);
    return FRZ_ERR_SHAPE;
  }
  launch->policy = *policy;
  launch->policy.mode = mode;
  launch->actions = actions;
  launch->control = control;
  launch->rows = B * A;
  launch->reserved = 0;
  return FRZ_OK;
}

}  // namespace
}  // namespace frz

extern "C" {

int frz_wildfire_policy_actions(const FrzWildfireParams* params, const FrzWildfireBuffers* io, int32_t parallel_envs,
                                const FrzPolicyActions* policy, void* stream) {
  using namespace frz;
  const char* what = "frz_wildfire_policy_actions";
  if (params == nullptr || io == nullptr) {
    set_error("%s: NULL params / buffers", what);
    return FRZ_ERR_NULL;
  }
  const int cells = params->height * params->width;
  if (params->height < 1 || params->width < 1 || cells > FRZ_MAX_CELLS) {
    set_error("%s: unsupported grid %dx%d", what, params->height, params->width);
    return FRZ_ERR_SHAPE;
  }
  Launch launch;
  int status = check_policy(policy, const_cast<int32_t*>(io->actions), io->control, parallel_envs, params->num_agents,
                            cells + 1, what, &launch);
  if (status != FRZ_OK) return status;
  const bool show_bad = (params->flags & FRZ_WF_SHOW_BAD_ACTIONS) != 0;
  if ((show_bad ? static_cast<const void*>(io->env_task_count) : io->action_mask) == nullptr) {
    set_error("%s: NULL %s", what, show_bad ? "env_task_count" : "action_mask");
    return FRZ_ERR_NULL;
  }
  if (!show_bad && io->mask_stride < cells) {
    set_error("%s: mask_stride=%d < %d cells", what, io->mask_stride, cells);
    return FRZ_ERR_SHAPE;
  }
  launch.env_offset = params->env_offset;
  const WildfireRule rule{io->action_mask, io->env_task_count, params->num_agents, cells + 1, cells, io->mask_stride,
                          show_bad};
  return frz::launch(rule, launch, (policy->mode & FRZ_POLICY_PACKED_LEGAL) != 0, static_cast<cudaStream_t>(stream));
}

int frz_rideshare_policy_actions(const FrzRideshareParams* params, const FrzRideshareBuffers* io,
                                 int32_t parallel_envs, const FrzPolicyActions* policy, void* stream) {
  using namespace frz;
  const char* what = "frz_rideshare_policy_actions";
  if (params == nullptr || io == nullptr) {
    set_error("%s: NULL params / buffers", what);
    return FRZ_ERR_NULL;
  }
  if (params->capacity < 1 || params->capacity > FRZ_MAX_PASSENGERS) {
    set_error("%s: unsupported capacity %d", what, params->capacity);
    return FRZ_ERR_SHAPE;
  }
  Launch launch;
  int status = check_policy(policy, const_cast<int32_t*>(io->actions), io->control, parallel_envs, params->num_agents,
                            params->capacity + 1, what, &launch);
  if (status != FRZ_OK) return status;
  if (io->task_mask == nullptr || io->task_obs == nullptr) {
    set_error("%s: NULL task_mask / task_obs", what);
    return FRZ_ERR_NULL;
  }
  launch.env_offset = params->env_offset;
  const RideshareRule rule{io->task_mask, io->task_obs, params->num_agents, params->capacity + 1, params->capacity, 0};
  return frz::launch(rule, launch, (policy->mode & FRZ_POLICY_PACKED_LEGAL) != 0, static_cast<cudaStream_t>(stream));
}

int frz_cyber_policy_actions(const FrzCyberParams* params, const FrzCyberBuffers* io, int32_t parallel_envs,
                             const FrzPolicyActions* policy, void* stream) {
  using namespace frz;
  const char* what = "frz_cyber_policy_actions";
  if (params == nullptr || io == nullptr) {
    set_error("%s: NULL params / buffers", what);
    return FRZ_ERR_NULL;
  }
  if (params->num_nodes < 1 || params->num_nodes > FRZ_MAX_NODES || params->num_attackers < 0 ||
      params->num_defenders < 0) {
    set_error("%s: unsupported network N=%d attackers=%d defenders=%d", what, params->num_nodes, params->num_attackers,
              params->num_defenders);
    return FRZ_ERR_SHAPE;
  }
  const int A = params->num_attackers + params->num_defenders;
  Launch launch;
  int status = check_policy(policy, const_cast<int32_t*>(io->actions), io->control, parallel_envs, A,
                            params->num_nodes + 3, what, &launch);
  if (status != FRZ_OK) return status;
  const bool show_bad = (params->flags & FRZ_CY_SHOW_BAD_ACTIONS) != 0;
  if ((show_bad ? io->env_task_count : io->agent_task_count) == nullptr ||
      (params->num_defenders > 0 && io->location == nullptr)) {
    set_error("%s: NULL task counts / location", what);
    return FRZ_ERR_NULL;
  }
  launch.env_offset = params->env_offset;
  const CyberRule rule{io->env_task_count, io->agent_task_count, io->location, A, params->num_nodes + 3,
                       params->num_nodes, params->num_attackers, show_bad};
  return frz::launch(rule, launch, (policy->mode & FRZ_POLICY_PACKED_LEGAL) != 0, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
