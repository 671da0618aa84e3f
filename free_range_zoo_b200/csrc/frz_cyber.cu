// Fused cybersecurity environment step for sm_100a.
//
// One launch = for every environment: attacker / defender action decode -> movement -> presence -> subnetwork state
// transition -> rewards -> num_moves / truncation -> reward accumulation -> observations -> task counts.  Replaces,
// with identical results, the reference's envs/cybersecurity/env/cybersecurity.py:296-526,
// env/transitions/{movement,presence,subnetwork}.py and utils/env.py:215-237.
//
// Mapping: one thread per environment (state is 24 B .. a few hundred bytes).  Rows of the [B, *] arrays are
// contiguous per environment, so the 32 rows a warp touches form one contiguous span and every sector fetched is
// fully used (L1 merges the strided per-thread accesses of a warp).
//
// The only transcendental on the path is tanh((patches - attacks) / T) (subnetwork.py:54) whose result is compared
// with a uniform draw.  Because few agents act on a node, the score takes at most 2^(Att+D) distinct values: they are
// tabulated on the host with the reference's own torch.tanh and indexed here by the set of agents acting on the node,
// so the threshold compare is bit-exact.
#include <cstdlib>

#include "frz_common.cuh"
#include "frz_host.cuh"

namespace frz {
namespace {

constexpr int kCyThreads = 128;
enum CyMode { kCyStep = 0, kCyRefresh = 1 };

// The rows of one environment in every array the step touches.  They point into global memory (direct kernel) or into
// the CTA's staged tile in shared memory (tiled kernel); the step itself is the same code.
struct CyberRows {
  int32_t* state;           // [N]
  int32_t* location;        // [D]
  uint8_t* presence;        // [n]
  const int2* actions;      // [n]
  float* rewards;           // [n]
  float* cumulative;        // [n]
  int32_t* num_moves;       // [1]
  uint8_t* truncated;       // [1]
  int32_t* env_task_count;  // [1]
  int32_t* agent_task_count;// [n]
  float2* attacker_self;    // [Att]
  float* defender_self;     // [D * 3]
  int2* task_obs;           // [N]
  uint8_t* monitored;       // [D]
  const float* network_uniforms;  // [N] or nullptr
  const float* agent_uniforms;    // [n] or nullptr
};

// One environment, one thread.  Returns the launch-epilogue bits through alive_bits / faults.
//
// MAXN / MAXATT / MAXDEF are compile-time upper bounds of the node / attacker / defender counts (0 = no bound: runtime
// loops).  With bounds every loop is fully unrolled and the environment's actions, locations and presence live in
// registers for the whole step; the runtime counts only predicate the unrolled iterations.
template <int MODE, int MAXN, int MAXATT, int MAXDEF>
__device__ __forceinline__ void cyber_env_step(const FrzCyberParams& p, const CyberRows& r, const float* score_lut,
                                               const Philox& philox, const uint64_t step, const int64_t global_env,
                                               unsigned& alive_bits, unsigned& faults) {
  constexpr bool kBounded = MAXN > 0;
  const int N = p.num_nodes, n_att = p.num_attackers, n_def = p.num_defenders;
  // loop bounds: the compile-time bound when there is one (the body is then predicated by the runtime count)
  const int kNodes = kBounded ? MAXN : N, kAtt = kBounded ? MAXATT : n_att, kDef = kBounded ? MAXDEF : n_def;
  const bool show_bad = p.flags & FRZ_CY_SHOW_BAD_ACTIONS;
  const bool stochastic = p.flags & FRZ_CY_STOCHASTIC_STATE;

  // register copies of the rows (bounded variant); the unbounded variant re-reads the rows instead
  int2 att_act[kBounded ? MAXATT : 1] = {}, def_act[kBounded ? MAXDEF : 1] = {};
  int def_loc[kBounded ? MAXDEF : 1] = {};
  const auto attacker_action = [&](int i) { return kBounded ? att_act[kBounded ? i : 0] : r.actions[i]; };
  const auto defender_action = [&](int d) { return kBounded ? def_act[kBounded ? d : 0] : r.actions[n_att + d]; };
  const auto defender_location = [&](int d) { return kBounded ? def_loc[kBounded ? d : 0] : r.location[d]; };

  uint32_t present = 0;  // bit a = agent a is present (attackers first)
#pragma unroll
  for (int i = 0; i < kAtt; ++i) {
    if (i < n_att) {
      present |= uint32_t(r.presence[i] != 0) << i;
      if (kBounded && MODE == kCyStep) att_act[kBounded ? i : 0] = r.actions[i];
    }
  }
#pragma unroll
  for (int d = 0; d < kDef; ++d) {
    if (d < n_def) {
      present |= uint32_t(r.presence[n_att + d] != 0) << (n_att + d);
      if (kBounded) def_loc[kBounded ? d : 0] = r.location[d];
      if (kBounded && MODE == kCyStep) def_act[kBounded ? d : 0] = r.actions[n_att + d];
    }
  }

  if (MODE == kCyStep) {
    const uint32_t env_lo = uint32_t(global_env), env_hi = uint32_t(uint64_t(global_env) >> 32);
    const uint32_t step_lo = uint32_t(step), step_hi = uint32_t(step >> 32) ^ env_hi;

    // ---------------------------------------------------------------- decode (cybersecurity.py:317-384)
    // The subnetwork transition only depends on the attacks / patches decided here -- patches use the defender's
    // location BEFORE this step's move -- so it runs before movement / presence change the rows.
    uint32_t patching = 0, monitoring = 0;  // bit d = defender d
#pragma unroll
    for (int i = 0; i < kAtt; ++i) {
      if (i < n_att) {
        const int2 act = attacker_action(i);
        if (!show_bad && !((present >> i) & 1u) && act.y != -1) faults |= FRZ_FAULT_ABSENT_ACTED;  // :345
        if (act.y == 0 && (act.x < 0 || act.x >= N)) faults |= FRZ_FAULT_BAD_NODE;                 // :341
      }
    }
#pragma unroll
    for (int d = 0; d < kDef; ++d) {
      if (d < n_def) {
        const int2 act = defender_action(d);
        if (!show_bad && !((present >> (n_att + d)) & 1u) && act.y != -1) faults |= FRZ_FAULT_ABSENT_ACTED;  // :362
        if (act.y == 0 && (act.x < 0 || act.x >= N)) faults |= FRZ_FAULT_BAD_NODE;                           // :357
        if (act.y == -2 && defender_location(d) != -1) patching |= 1u << d;                                  // :354
        if (act.y == -3) monitoring |= 1u << d;
      }
    }

    // ---------------------------------------------------------------- subnetwork.py:40-72 + rewards :395-409
    float network_reward = 0.f;
    uint4 bits = make_uint4(0u, 0u, 0u, 0u);  // one Philox call serves four consecutive nodes / agents
#pragma unroll
    for (int node = 0; node < kNodes; ++node) {
      if (node < N) {
        uint32_t actors = 0;
        float attacks = 0.f, patches = 0.f;
#pragma unroll
        for (int i = 0; i < kAtt; ++i) {
          if (i < n_att) {
            const int2 act = attacker_action(i);
            if (act.y == 0 && act.x == node) {  // attack node act.x
              actors |= 1u << i;
              attacks = __fadd_rn(attacks, p.power[i]);
            }
          }
        }
#pragma unroll
        for (int d = 0; d < kDef; ++d) {
          if (d < n_def && ((patching >> d) & 1u) && defender_location(d) == node) {  // patch the node stood on
            actors |= 1u << (n_att + d);
            patches = __fadd_rn(patches, p.power[n_att + d]);
          }
        }
        float score;
        if (p.lut_bits > 0) score = score_lut[actors];
        else score = tanhf(__fdiv_rn(__fadd_rn(patches, -attacks), p.temperature));
        bool better = score > 0.f, worse = score < 0.f;
        if (stochastic) {
          float u;
          if (r.network_uniforms != nullptr) {
            u = r.network_uniforms[node];
          } else {
            if ((node & 3) == 0) bits = philox(env_lo, step_lo, uint32_t(node >> 2), step_hi);
            const uint32_t word = (node & 3) == 0 ? bits.x : (node & 3) == 1 ? bits.y : (node & 3) == 2 ? bits.z : bits.w;
            u = u01(word);
          }
          const bool within = fabsf(score) <= u;  // larger |score| => LESS likely, as in the reference
          better = better && within;
          worse = worse && within;
        }
        int s = r.state[node] - int(better) + int(worse);
        s = min(max(s, 0), p.num_states - 1);
        r.state[node] = s;
        network_reward = __fadd_rn(network_reward, __fmul_rn(p.state_rewards[s], p.criticality[node]));
        r.task_obs[node] = make_int2(s, int(p.criticality[node]));
      }
    }

    // ---------------------------------------------------------------- movement.py:17-32 + presence.py:35-60
    // one uniform per agent, agent a uses word a of the agent stream (attackers first)
    uint32_t now_present = 0;
    const auto presence_step = [&](int a) {
      float u;
      if (r.agent_uniforms != nullptr) {
        u = r.agent_uniforms[a];
      } else {
        if ((a & 3) == 0 || a == n_att) bits = philox(env_lo, step_lo, 0x80000000u | uint32_t(a >> 2), step_hi);
        const uint32_t word = (a & 3) == 0 ? bits.x : (a & 3) == 1 ? bits.y : (a & 3) == 2 ? bits.z : bits.w;
        u = u01(word);
      }
      const bool was = (present >> a) & 1u;
      const bool returning = !was && u < p.returns[a];
      const bool leaving = was && u >= p.persist[a];
      const bool is = (was || returning) && !leaving;
      now_present |= uint32_t(is) << a;
      r.presence[a] = is;
      return returning;
    };
#pragma unroll
    for (int i = 0; i < kAtt; ++i)
      if (i < n_att) presence_step(i);
#pragma unroll
    for (int d = 0; d < kDef; ++d) {
      if (d < n_def) {
        const bool returning = presence_step(n_att + d);
        const int2 act = defender_action(d);
        int loc = defender_location(d);
        if (act.y == 0) loc = act.x;  // move to node act.x (no adjacency check, movement.py:17-32)
        if (returning) loc = -1;      // returning defenders start at the home node
        r.location[d] = loc;
        if (kBounded) def_loc[kBounded ? d : 0] = loc;
      }
    }

    const int moves = r.num_moves[0] + 1;
    const bool truncated = moves >= p.max_steps;
    r.num_moves[0] = moves;
    r.truncated[0] = truncated;
    alive_bits |= 1u | (truncated ? 0u : 2u);  // cybersecurity never terminates (:299)
#pragma unroll
    for (int i = 0; i < kAtt; ++i) {
      if (i < n_att) {
        const float reward = __fadd_rn(0.f, -network_reward);
        r.rewards[i] = reward;
        r.cumulative[i] = __fadd_rn(r.cumulative[i], reward);
      }
    }
#pragma unroll
    for (int d = 0; d < kDef; ++d) {
      if (d < n_def) {
        const int a = n_att + d;
        // :376 (the bad-action branch :379-381 is dead)
        const float reward = __fadd_rn(((patching >> d) & 1u) ? p.patch_reward : 0.f, network_reward);
        r.rewards[a] = reward;
        r.cumulative[a] = __fadd_rn(r.cumulative[a], reward);
        r.monitored[d] = (monitoring >> d) & 1u;
      }
    }
    present = now_present;
  } else {
#pragma unroll
    for (int node = 0; node < kNodes; ++node)
      if (node < N) r.task_obs[node] = make_int2(r.state[node], int(p.criticality[node]));
  }

  // ------------------------------------------------------------------ update_actions / update_observations
  r.env_task_count[0] = N;
#pragma unroll
  for (int i = 0; i < kAtt; ++i) {
    if (i < n_att) {
      const bool is = (present >> i) & 1u;
      r.agent_task_count[i] = is ? N : 0;
      r.attacker_self[i] = make_float2(p.power[i], is ? 1.f : 0.f);
    }
  }
#pragma unroll
  for (int d = 0; d < kDef; ++d) {
    if (d < n_def) {
      const int a = n_att + d;
      const bool is = (present >> a) & 1u;
      r.agent_task_count[a] = is ? N : 0;
      float* out = r.defender_self + d * 3;
      out[0] = p.power[a];
      out[1] = is ? 1.f : 0.f;
      out[2] = float(defender_location(d));
    }
  }
}

// ---------------------------------------------------------------------------------------------- direct kernel
// One thread per environment straight on global memory: refresh / reset, and steps whose tile would not fit in shared
// memory.
template <int MODE>
__global__ void __launch_bounds__(kCyThreads)
cyber_step_kernel(const __grid_constant__ FrzCyberParams p, const __grid_constant__ FrzCyberBuffers io, const int B) {
  const int N = p.num_nodes, n_att = p.num_attackers, n_def = p.num_defenders, n_agents = n_att + n_def;
  FrzControl* control = io.control;
  const uint64_t step = control->step;
  const uint32_t alive_prev = control->alive;
  const Philox philox(control->seed);
  const bool skip = (MODE == kCyStep) && ((alive_prev & 3u) != 3u);  // utils/env.py:212
  unsigned alive_bits = 0, faults = 0;

  if (!skip) {
    for (int env = blockIdx.x * blockDim.x + threadIdx.x; env < B; env += gridDim.x * blockDim.x) {
      const size_t e = size_t(env);
      CyberRows r;
      r.state = io.network_state + e * N;
      r.location = io.location + e * n_def;
      r.presence = io.presence + e * n_agents;
      r.actions = reinterpret_cast<const int2*>(io.actions) + e * n_agents;
      r.rewards = io.rewards + e * n_agents;
      r.cumulative = io.cumulative_rewards + e * n_agents;
      r.num_moves = io.num_moves + e;
      r.truncated = io.truncated + e;
      r.env_task_count = io.env_task_count + e;
      r.agent_task_count = io.agent_task_count + e * n_agents;
      r.attacker_self = reinterpret_cast<float2*>(io.attacker_self) + e * n_att;
      r.defender_self = io.defender_self + e * n_def * 3;
      r.task_obs = reinterpret_cast<int2*>(io.task_obs) + e * N;
      r.monitored = io.monitored + e * n_def;
      r.network_uniforms = io.network_uniforms != nullptr ? io.network_uniforms + e * N : nullptr;
      r.agent_uniforms = io.agent_uniforms != nullptr ? io.agent_uniforms + e * n_agents : nullptr;
      cyber_env_step<MODE, 0, 0, 0>(p, r, io.score_lut, philox, step, p.env_offset + env, alive_bits, faults);
      // refresh: the done flags as a reset, a restore or a hand edit left them
      if (MODE == kCyRefresh) alive_bits |= (io.terminated[e] ? 0u : 1u) | (io.truncated[e] ? 0u : 2u);
    }
  }
  finish_launch(control, alive_bits, faults, 0u,
                skip ? kPublishNothing : (MODE == kCyStep ? kPublishStep : kPublishRefresh));
}

// ---------------------------------------------------------------------------------------------- tiled kernel
// The step path.  A CTA owns a tile of kCyThreads consecutive environments.  Every [B, *] array is environment-major,
// so the tile of each array is ONE contiguous byte range: a single elected thread streams all of them into shared
// memory with bulk async copies (the TMA unit, completion on an mbarrier), every thread then steps its environment
// entirely in shared memory, and the elected thread streams the results back with bulk stores.  HBM sees only full,
// aligned bursts; the per-thread row accesses (stride = row size) never leave the SM.
struct CyberTileLayout {  // byte offsets of the staged arrays inside the tile (each a multiple of 16)
  int state, location, presence, cumulative, num_moves;                     // read and written
  int actions, network_uniforms, agent_uniforms;                            // read only
  int rewards, truncated, env_task_count, agent_task_count, attacker_self,  // written only
      defender_self, task_obs, monitored;
  int total;
};

__host__ __device__ inline CyberTileLayout cyber_tile_layout(int N, int n_att, int n_def, bool injected, int T = kCyThreads) {
  const int n = n_att + n_def;
  CyberTileLayout L;
  int at = 0;
  auto take = [&at](int bytes) {
    const int offset = at;
    at += (bytes + 15) & ~15;
    return offset;
  };
  L.state = take(T * N * 4);
  L.location = take(T * n_def * 4);
  L.presence = take(T * n);
  L.cumulative = take(T * n * 4);
  L.num_moves = take(T * 4);
  L.actions = take(T * n * 8);
  L.network_uniforms = take(injected ? T * N * 4 : 0);
  L.agent_uniforms = take(injected ? T * n * 4 : 0);
  L.rewards = take(T * n * 4);
  L.truncated = take(T);
  L.env_task_count = take(T * 4);
  L.agent_task_count = take(T * n * 4);
  L.attacker_self = take(T * n_att * 8);
  L.defender_self = take(T * n_def * 12);
  L.task_obs = take(T * N * 8);
  L.monitored = take(T * n_def);
  L.total = at;
  return L;
}

// cooperative copy for the (at most one) partial tile at the end of the batch: sizes need not be multiples of 16
__device__ __forceinline__ void tile_copy(uint8_t* dst, const uint8_t* src, int bytes, int threads) {
  for (int i = threadIdx.x; i < bytes; i += threads) dst[i] = src[i];
}

// Persistent and warp-specialised: a CTA walks the tiles blockIdx.x, blockIdx.x + gridDim.x, ...; its first kCyThreads
// threads step one environment each, the extra warp's first thread does nothing but move tiles.  With two or three tile
// buffers (as many as fit, when the batch is large) the copy thread requests tile i, then stores tile i-1 as soon as the
// stepping threads are done with it, then waits until the stores that last read the next buffer have left shared memory
// and requests tile i+1 into it -- so the loads of one tile, the stepping of the next and the write-back of the
// previous ones overlap inside the CTA, and no stepping thread ever waits for a store to drain.  Hand-offs: full[b] (mbarrier armed with the
// tile's byte count, completed by the bulk loads) and done[b] (mbarrier the kCyThreads stepping threads arrive on).
constexpr int kCyBlock = kCyThreads + 32;
constexpr int kCyMaxBuffers = 3;

template <bool INJECTED, int MAXN, int MAXATT, int MAXDEF>
__global__ void __launch_bounds__(kCyBlock, 4)
cyber_step_tiled_kernel(const __grid_constant__ FrzCyberParams p, const __grid_constant__ FrzCyberBuffers io, const int B,
                        const int buffers, const int tile_envs) {
  const int T = tile_envs;  // environments per tile = stepping threads (64 or 128; the CTA has one more warp)
  extern __shared__ __align__(128) uint8_t tiles_storage[];
  __shared__ __align__(8) uint64_t barrier_storage[2 * kCyMaxBuffers];  // full[b], then done[b]
  const int N = p.num_nodes, n_att = p.num_attackers, n_def = p.num_defenders, n = n_att + n_def;
  FrzControl* control = io.control;
  const uint64_t step = control->step;
  const uint32_t alive_prev = control->alive;
  const Philox philox(control->seed);
  const bool skip = (alive_prev & 3u) != 3u;  // utils/env.py:212
  unsigned alive_bits = 0, faults = 0;

  if (!skip) {
    const CyberTileLayout L = cyber_tile_layout(N, n_att, n_def, INJECTED, T);
    const bool inject_network = INJECTED && io.network_uniforms != nullptr;
    const bool inject_agent = INJECTED && io.agent_uniforms != nullptr;
    const int tile_count = (B + T - 1) / T;
    const uint32_t storage_s = shared_address(tiles_storage);
    const auto full_barrier = [&](int b) { return shared_address(&barrier_storage[b]); };
    const auto done_barrier = [&](int b) { return shared_address(&barrier_storage[kCyMaxBuffers + b]); };
    if (threadIdx.x == 0) {
      for (int b = 0; b < kCyMaxBuffers; ++b) {
        mbarrier_init(full_barrier(b), 1);
        mbarrier_init(done_barrier(b), T);
      }
    }
    __syncthreads();
    const auto is_full = [&](int tile_index) { return (tile_index + 1) * T <= B; };

    if (threadIdx.x >= T) {
      // ================================================================== the copy thread
      if (threadIdx.x == T) {
        const uint32_t T = uint32_t(tile_envs);
        // the bulk loads of one full tile into buffer b
        const auto request = [&](int tile_index, int b) {
          const size_t e = size_t(tile_index) * T;
          const uint32_t tile_s = storage_s + uint32_t(b) * uint32_t(L.total), barrier = full_barrier(b);
          uint32_t bytes = T * (N * 4 + n_def * 4 + n + n * 4 + 4 + n * 8);
          if (inject_network) bytes += T * N * 4;
          if (inject_agent) bytes += T * n * 4;
          mbarrier_expect_bytes(barrier, bytes);
          bulk_load(tile_s + L.state, io.network_state + e * N, T * N * 4, barrier);
          bulk_load(tile_s + L.location, io.location + e * n_def, T * n_def * 4, barrier);
          bulk_load(tile_s + L.presence, io.presence + e * n, T * n, barrier);
          bulk_load(tile_s + L.cumulative, io.cumulative_rewards + e * n, T * n * 4, barrier);
          bulk_load(tile_s + L.num_moves, io.num_moves + e, T * 4, barrier);
          bulk_load(tile_s + L.actions, io.actions + e * n * 2, T * n * 8, barrier);
          if (inject_network) bulk_load(tile_s + L.network_uniforms, io.network_uniforms + e * N, T * N * 4, barrier);
          if (inject_agent) bulk_load(tile_s + L.agent_uniforms, io.agent_uniforms + e * n, T * n * 4, barrier);
        };
        // the bulk stores of one stepped full tile out of buffer b (one bulk group)
        const auto write_back = [&](int tile_index, int b) {
          const size_t e = size_t(tile_index) * T;
          const uint32_t tile_s = storage_s + uint32_t(b) * uint32_t(L.total);
          bulk_store(io.network_state + e * N, tile_s + L.state, T * N * 4);
          bulk_store(io.location + e * n_def, tile_s + L.location, T * n_def * 4);
          bulk_store(io.presence + e * n, tile_s + L.presence, T * n);
          bulk_store(io.cumulative_rewards + e * n, tile_s + L.cumulative, T * n * 4);
          bulk_store(io.num_moves + e, tile_s + L.num_moves, T * 4);
          bulk_store(io.rewards + e * n, tile_s + L.rewards, T * n * 4);
          bulk_store(io.truncated + e, tile_s + L.truncated, T);
          bulk_store(io.env_task_count + e, tile_s + L.env_task_count, T * 4);
          bulk_store(io.agent_task_count + e * n, tile_s + L.agent_task_count, T * n * 4);
          bulk_store(io.attacker_self + e * n_att * 2, tile_s + L.attacker_self, T * n_att * 8);
          bulk_store(io.defender_self + e * n_def * 3, tile_s + L.defender_self, T * n_def * 12);
          bulk_store(io.task_obs + e * N * 2, tile_s + L.task_obs, T * N * 8);
          bulk_store(io.monitored + e * n_def, tile_s + L.monitored, T * n_def);
          bulk_commit();
        };
        uint32_t done_parity = 0u;  // bit b = phase parity of done[b]
        const auto finish_tile = [&](int tile_index, int b) {  // once its environments are stepped, write the tile back
          if (!is_full(tile_index)) return;  // (the stepping threads store a partial tile themselves)
          mbarrier_wait(done_barrier(b), (done_parity >> b) & 1u);
          done_parity ^= 1u << b;
          write_back(tile_index, b);
        };
        int previous = -1, previous_buffer = 0, iteration = 0;
        for (int tile_index = blockIdx.x; tile_index < tile_count; tile_index += gridDim.x, ++iteration) {
          const int b = iteration % buffers;
          if (buffers == 1 && previous >= 0) finish_tile(previous, previous_buffer);
          // buffer b is free once the stores that read it last (tile `iteration - buffers`) have left shared memory:
          // all but the `buffers - 2` groups committed after them
          if (buffers == 3) bulk_wait_read_all_but<1>();
          else bulk_wait_read();
          if (is_full(tile_index)) request(tile_index, b);
          else mbarrier_arrive(full_barrier(b));  // partial tile: the stepping threads copy it themselves
          if (buffers >= 2 && previous >= 0) finish_tile(previous, previous_buffer);
          previous = tile_index;
          previous_buffer = b;
        }
        if (previous >= 0) finish_tile(previous, previous_buffer);
        bulk_wait_read();  // the last stores have left shared memory before the CTA exits
      }
    } else {
      // ================================================================== the stepping threads
      uint32_t full_parity = 0u;  // bit b = phase parity of full[b]
      int iteration = 0;
      for (int tile_index = blockIdx.x; tile_index < tile_count; tile_index += gridDim.x, ++iteration) {
        const int b = iteration % buffers;
        const int first = tile_index * T;
        const int count = min(T, B - first);
        const size_t e = size_t(first);
        const bool full = count == T;
        uint8_t* const tile = tiles_storage + size_t(b) * size_t(L.total);

        // ------------------------------------------------------------------ the tile has arrived (or the buffer is free)
        mbarrier_wait(full_barrier(b), (full_parity >> b) & 1u);
        full_parity ^= 1u << b;
        if (!full) {
          tile_copy(tile + L.state, reinterpret_cast<const uint8_t*>(io.network_state + e * N), count * N * 4, T);
          tile_copy(tile + L.location, reinterpret_cast<const uint8_t*>(io.location + e * n_def), count * n_def * 4, T);
          tile_copy(tile + L.presence, io.presence + e * n, count * n, T);
          tile_copy(tile + L.cumulative, reinterpret_cast<const uint8_t*>(io.cumulative_rewards + e * n), count * n * 4, T);
          tile_copy(tile + L.num_moves, reinterpret_cast<const uint8_t*>(io.num_moves + e), count * 4, T);
          tile_copy(tile + L.actions, reinterpret_cast<const uint8_t*>(io.actions + e * n * 2), count * n * 8, T);
          if (inject_network)
            tile_copy(tile + L.network_uniforms, reinterpret_cast<const uint8_t*>(io.network_uniforms + e * N), count * N * 4, T);
          if (inject_agent)
            tile_copy(tile + L.agent_uniforms, reinterpret_cast<const uint8_t*>(io.agent_uniforms + e * n), count * n * 4, T);
          named_barrier_sync(1, T);
        }

        // ------------------------------------------------------------------ step, entirely in shared memory
        const int t = threadIdx.x;
        if (t < count) {
          CyberRows r;
          r.state = reinterpret_cast<int32_t*>(tile + L.state) + t * N;
          r.location = reinterpret_cast<int32_t*>(tile + L.location) + t * n_def;
          r.presence = tile + L.presence + t * n;
          r.actions = reinterpret_cast<const int2*>(tile + L.actions) + t * n;
          r.rewards = reinterpret_cast<float*>(tile + L.rewards) + t * n;
          r.cumulative = reinterpret_cast<float*>(tile + L.cumulative) + t * n;
          r.num_moves = reinterpret_cast<int32_t*>(tile + L.num_moves) + t;
          r.truncated = tile + L.truncated + t;
          r.env_task_count = reinterpret_cast<int32_t*>(tile + L.env_task_count) + t;
          r.agent_task_count = reinterpret_cast<int32_t*>(tile + L.agent_task_count) + t * n;
          r.attacker_self = reinterpret_cast<float2*>(tile + L.attacker_self) + t * n_att;
          r.defender_self = reinterpret_cast<float*>(tile + L.defender_self) + t * n_def * 3;
          r.task_obs = reinterpret_cast<int2*>(tile + L.task_obs) + t * N;
          r.monitored = tile + L.monitored + t * n_def;
          r.network_uniforms = inject_network ? reinterpret_cast<const float*>(tile + L.network_uniforms) + t * N : nullptr;
          r.agent_uniforms = inject_agent ? reinterpret_cast<const float*>(tile + L.agent_uniforms) + t * n : nullptr;
          cyber_env_step<kCyStep, MAXN, MAXATT, MAXDEF>(p, r, io.score_lut, philox, step, p.env_offset + first + t, alive_bits, faults);
        }

        // ------------------------------------------------------------------ hand the tile to the copy thread
        if (full) {
          fence_async_shared();  // this thread's writes become visible to the bulk stores
          mbarrier_arrive(done_barrier(b));
        } else {
          named_barrier_sync(1, T);
          tile_copy(reinterpret_cast<uint8_t*>(io.network_state + e * N), tile + L.state, count * N * 4, T);
          tile_copy(reinterpret_cast<uint8_t*>(io.location + e * n_def), tile + L.location, count * n_def * 4, T);
          tile_copy(io.presence + e * n, tile + L.presence, count * n, T);
          tile_copy(reinterpret_cast<uint8_t*>(io.cumulative_rewards + e * n), tile + L.cumulative, count * n * 4, T);
          tile_copy(reinterpret_cast<uint8_t*>(io.num_moves + e), tile + L.num_moves, count * 4, T);
          tile_copy(reinterpret_cast<uint8_t*>(io.rewards + e * n), tile + L.rewards, count * n * 4, T);
          tile_copy(io.truncated + e, tile + L.truncated, count, T);
          tile_copy(reinterpret_cast<uint8_t*>(io.env_task_count + e), tile + L.env_task_count, count * 4, T);
          tile_copy(reinterpret_cast<uint8_t*>(io.agent_task_count + e * n), tile + L.agent_task_count, count * n * 4, T);
          tile_copy(reinterpret_cast<uint8_t*>(io.attacker_self + e * n_att * 2), tile + L.attacker_self, count * n_att * 8, T);
          tile_copy(reinterpret_cast<uint8_t*>(io.defender_self + e * n_def * 3), tile + L.defender_self, count * n_def * 12, T);
          tile_copy(reinterpret_cast<uint8_t*>(io.task_obs + e * N * 2), tile + L.task_obs, count * N * 8, T);
          tile_copy(io.monitored + e * n_def, tile + L.monitored, count * n_def, T);
        }
      }
    }
  }
  finish_launch(control, alive_bits, faults, 0u, skip ? kPublishNothing : kPublishStep);
}

__global__ void cyber_restore_kernel(const FrzCyberParams p, const FrzCyberBuffers io, const int B,
                                     const uint8_t* __restrict__ env_mask) {
  const int N = p.num_nodes, n_def = p.num_defenders, n_agents = p.num_attackers + p.num_defenders;
  for (int env = blockIdx.x * blockDim.x + threadIdx.x; env < B; env += gridDim.x * blockDim.x) {
    if (env_mask != nullptr && !env_mask[env]) continue;
    for (int i = 0; i < N; ++i) io.network_state[size_t(env) * N + i] = io.init_network_state[size_t(env) * N + i];
    for (int i = 0; i < n_def; ++i) {
      io.location[size_t(env) * n_def + i] = io.init_location[size_t(env) * n_def + i];
      io.monitored[size_t(env) * n_def + i] = 0;  // actions are re-initialised to -2 (cybersecurity.py:233-236)
    }
    for (int i = 0; i < n_agents; ++i) {
      io.presence[size_t(env) * n_agents + i] = io.init_presence[size_t(env) * n_agents + i];
      io.rewards[size_t(env) * n_agents + i] = 0.f;
      io.cumulative_rewards[size_t(env) * n_agents + i] = 0.f;
    }
    io.terminated[env] = 0;
    io.truncated[env] = 0;
    io.num_moves[env] = 0;
  }
}

// Uniform over the legal choices of spaces/actions.py:11-99:
//   attacker: [attack node 0..n-1, noop]           defender: [move 0..n-1, noop, (patch), monitor]
// with n = N if the agent is present (or show_bad_actions) else 0 (noop only); patch is offered unless
// show_bad_actions is off and the defender is at the home node.
__global__ void cyber_sample_kernel(const FrzCyberParams p, const FrzCyberBuffers io, const int B,
                                    const uint64_t sampler_seed) {
  const int n_att = p.num_attackers, n_agents = p.num_attackers + p.num_defenders;
  const Philox philox(sampler_seed);
  const uint64_t step = io.control->step;
  const bool show_bad = p.flags & FRZ_CY_SHOW_BAD_ACTIONS;
  const int total = B * n_agents;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int env = i / n_agents, a = i - env * n_agents;
    const int n = show_bad ? io.env_task_count[env] : io.agent_task_count[i];
    const uint64_t genv = uint64_t(p.env_offset + env);
    const uint4 r = philox(uint32_t(genv), uint32_t(step), 0xC0000000u | uint32_t(a), uint32_t(step >> 32) ^ uint32_t(genv >> 32));
    int choices = n + 1;
    bool can_patch = false;
    if (a >= n_att && n > 0) {
      can_patch = show_bad || io.location[size_t(env) * p.num_defenders + (a - n_att)] != -1;
      choices += can_patch ? 2 : 1;
    }
    const int k = min(int(u01(r.x) * float(choices)), choices - 1);
    int ident;
    if (k < n) ident = 0;
    else if (k == n) ident = -1;
    else if (k == n + 1 && can_patch) ident = -2;
    else ident = -3;
    reinterpret_cast<int2*>(const_cast<int32_t*>(io.actions))[i] = make_int2(k, ident);
  }
}

int cyber_validate(const FrzCyberParams* p, const FrzCyberBuffers* io, int B, const char* what) {
  if (p == nullptr || io == nullptr || io->control == nullptr || io->network_state == nullptr) {
    set_error("%s: NULL params / buffers", what);
    return FRZ_ERR_NULL;
  }
  const int n_agents = p->num_attackers + p->num_defenders;
  if (B <= 0 || p->num_nodes < 1 || p->num_nodes > FRZ_MAX_NODES || n_agents < 1 || n_agents > FRZ_MAX_AGENTS ||
      p->num_states < 1 || p->num_states > FRZ_MAX_NET_STATES ||
      (p->lut_bits != 0 && (p->lut_bits != n_agents || n_agents > FRZ_CY_MAX_LUT_BITS || io->score_lut == nullptr))) {
    set_error("%s: unsupported shape B=%d N=%d attackers=%d defenders=%d states=%d lut_bits=%d", what, B, p->num_nodes,
              p->num_attackers, p->num_defenders, p->num_states, p->lut_bits);
    return FRZ_ERR_SHAPE;
  }
  return FRZ_OK;
}

constexpr int kCyMaxTileBytes = 72 * 1024;  // keeps >= 3 tiles resident per SM

// tuning experiment knob (profiles/README.md): FRZ_CYBER_BUFFERS=1|2|3 fixes the tile buffers per CTA for large batches
inline int cyber_buffer_override() {
  static const int value = [] {
    const char* text = std::getenv("FRZ_CYBER_BUFFERS");
    const int n = text != nullptr ? std::atoi(text) : 0;
    return n >= 1 && n <= kCyMaxBuffers ? n : 0;
  }();
  return value;
}

int cyber_launch(const FrzCyberParams* p, const FrzCyberBuffers* io, int B, int mode, void* stream) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (mode == kCyStep) {
    const bool injected = io->network_uniforms != nullptr || io->agent_uniforms != nullptr;
    // tiles of 128 environments; 64 when that is what it takes to put a tile on every SM (the named 16 384 environments
    // are 128 tiles of 128 on a 148-SM B200)
    const int tile_envs = (B + kCyThreads - 1) / kCyThreads < sm_count() ? kCyThreads / 2 : kCyThreads;
    const int tile_count = (B + tile_envs - 1) / tile_envs;
    const CyberTileLayout layout = cyber_tile_layout(p->num_nodes, p->num_attackers, p->num_defenders, injected, tile_envs);
    if (layout.total <= kCyMaxTileBytes) {
      // size classes: loops over nodes / attackers / defenders are unrolled to the class bound (0 = runtime loops)
      void (*kernel)(FrzCyberParams, FrzCyberBuffers, int, int, int);
      const int N = p->num_nodes, att = p->num_attackers, def = p->num_defenders;
      if (N <= 4 && att <= 2 && def <= 2)
        kernel = injected ? cyber_step_tiled_kernel<true, 4, 2, 2> : cyber_step_tiled_kernel<false, 4, 2, 2>;
      else if (N <= 8 && att <= 4 && def <= 4)
        kernel = injected ? cyber_step_tiled_kernel<true, 8, 4, 4> : cyber_step_tiled_kernel<false, 8, 4, 4>;
      else if (N <= 16 && att <= 8 && def <= 8)
        kernel = injected ? cyber_step_tiled_kernel<true, 16, 8, 8> : cyber_step_tiled_kernel<false, 16, 8, 8>;
      else
        kernel = injected ? cyber_step_tiled_kernel<true, 0, 0, 0> : cyber_step_tiled_kernel<false, 0, 0, 0>;
      // two tile buffers per CTA (the next tile is fetched while this one is stepped) when that still leaves several
      // CTAs per SM, and when the batch has more tiles than one wave of CTAs anyway
      int buffers = 1;
      if (tile_count > sm_count() * 4) {
        if (cyber_buffer_override() > 0) buffers = cyber_buffer_override();
        else buffers = 2 * layout.total <= kCyMaxTileBytes ? 2 : 1;  // (three buffers = one CTA fewer per SM: 205 us against 181 at 4 M envs)
      }
      const int smem = buffers * layout.total;
      if (smem > 48 * 1024 && cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess)
        return check_launch("cyber tile shared memory");
      cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
      int ctas_per_sm = 0;  // (not cached: the same instantiation runs with one or two buffers)
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, kernel, tile_envs + 32, size_t(smem));
      const int grid = persistent_grid(tile_count, ctas_per_sm < 1 ? 1 : ctas_per_sm);
      kernel<<<grid, tile_envs + 32, smem, s>>>(*p, *io, B, buffers, tile_envs);
      return check_launch("cyber_step_tiled_kernel");
    }
  }
  const int work = (B + kCyThreads - 1) / kCyThreads;
  const int grid = persistent_grid(work, 8);
  if (mode == kCyStep) cyber_step_kernel<kCyStep><<<grid, kCyThreads, 0, s>>>(*p, *io, B);
  else cyber_step_kernel<kCyRefresh><<<grid, kCyThreads, 0, s>>>(*p, *io, B);
  return check_launch("cyber_step_kernel");
}

}  // namespace
}  // namespace frz

extern "C" {

int frz_cyber_step(const FrzCyberParams* params, const FrzCyberBuffers* io, int32_t parallel_envs, void* stream) {
  const int status = frz::cyber_validate(params, io, parallel_envs, "frz_cyber_step");
  if (status != FRZ_OK) return status;
  if (io->actions == nullptr) {
    frz::set_error("frz_cyber_step: actions is NULL");
    return FRZ_ERR_NULL;
  }
  return frz::cyber_launch(params, io, parallel_envs, frz::kCyStep, stream);
}

int frz_cyber_step_host(const FrzCyberParams* params, const FrzCyberBuffers* io, int32_t parallel_envs,
                        const FrzHostStep* host, void* stream) {
  const int status = frz::cyber_validate(params, io, parallel_envs, "frz_cyber_step_host");
  if (status != FRZ_OK) return status;
  if (io->actions == nullptr || io->rewards == nullptr) {
    frz::set_error("frz_cyber_step_host: actions / rewards is NULL");
    return FRZ_ERR_NULL;
  }
  if (io->network_uniforms != nullptr || io->agent_uniforms != nullptr) {
    frz::set_error("frz_cyber_step_host: injected uniforms are not supported on the pipelined host path");
    return FRZ_ERR_UNSUPPORTED;
  }
  const size_t N = size_t(params->num_nodes), att = size_t(params->num_attackers), dfd = size_t(params->num_defenders);
  const size_t n = att + dfd;
  const frz::HostArrays arrays{io->actions, io->rewards, io->terminated, io->truncated, io->control, int(n),
                                 params, sizeof(FrzCyberParams), io, sizeof(FrzCyberBuffers)};
  return frz::run_host_pipeline(
      "frz_cyber_step_host", host, arrays, parallel_envs, static_cast<cudaStream_t>(stream),
      [&](int first, int count, FrzControl* control, cudaStream_t slice_stream) {
        FrzCyberParams p = *params;
        p.env_offset += first;
        FrzCyberBuffers slice = *io;
        const size_t e = size_t(first);
        slice.network_state += e * N;
        slice.location += e * dfd;
        slice.presence += e * n;
        slice.actions += e * n * 2;
        slice.rewards += e * n;
        slice.cumulative_rewards += e * n;
        slice.terminated += e;
        slice.truncated += e;
        slice.num_moves += e;
        slice.env_task_count += e;
        slice.agent_task_count += e * n;
        slice.attacker_self += e * att * 2;
        slice.defender_self += e * dfd * 3;
        slice.task_obs += e * N * 2;
        slice.monitored += e * dfd;
        slice.control = control;
        return frz::cyber_launch(&p, &slice, count, frz::kCyStep, slice_stream);
      });
}

int frz_cyber_refresh(const FrzCyberParams* params, const FrzCyberBuffers* io, int32_t parallel_envs, void* stream) {
  const int status = frz::cyber_validate(params, io, parallel_envs, "frz_cyber_refresh");
  if (status != FRZ_OK) return status;
  return frz::cyber_launch(params, io, parallel_envs, frz::kCyRefresh, stream);
}

int frz_cyber_reset(const FrzCyberParams* params, const FrzCyberBuffers* io, int32_t parallel_envs,
                    const uint8_t* env_mask, void* stream) {
  int status = frz::cyber_validate(params, io, parallel_envs, "frz_cyber_reset");
  if (status != FRZ_OK) return status;
  if (io->init_network_state == nullptr) {
    frz::set_error("frz_cyber_reset: initial state is NULL");
    return FRZ_ERR_NULL;
  }
  const int grid = frz::persistent_grid((parallel_envs + 255) / 256, 8);
  frz::cyber_restore_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(*params, *io, parallel_envs, env_mask);
  status = frz::check_launch("cyber_restore_kernel");
  if (status != FRZ_OK) return status;
  return frz::cyber_launch(params, io, parallel_envs, frz::kCyRefresh, stream);
}

int frz_cyber_sample_actions(const FrzCyberParams* params, const FrzCyberBuffers* io, int32_t parallel_envs,
                             uint64_t sampler_seed, void* stream) {
  const int status = frz::cyber_validate(params, io, parallel_envs, "frz_cyber_sample_actions");
  if (status != FRZ_OK) return status;
  const int total = parallel_envs * (params->num_attackers + params->num_defenders);
  const int grid = frz::persistent_grid((total + 255) / 256, 8);
  frz::cyber_sample_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(*params, *io, parallel_envs, sampler_seed);
  return frz::check_launch("cyber_sample_kernel");
}

}  // extern "C"
