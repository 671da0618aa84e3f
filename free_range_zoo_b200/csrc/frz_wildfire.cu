// Fused wildfire environment step for sm_100a.
//
// One launch = for every environment: action decode -> suppressant decrease -> equipment -> refill -> capacity ->
// fire increase -> fire decrease -> fire spread -> rewards -> termination -> num_moves / truncation -> reward
// accumulation -> observations -> task counts -> action masks.  It replaces, with identical results, the reference's
//   envs/wildfire/env/wildfire.py:400-717 (step_environment, update_actions, update_observations),
//   envs/wildfire/env/transitions/*.py (seven nn.Module transitions) and utils/env.py:215-237 (AEC bookkeeping).
//
// Mapping: a group of G lanes (8, 16 or 32) owns one environment.  Lane l of the group owns grid cells
// l, l+G, l+2G, ... (CPL cells per lane) AND agent l.  Everything that couples cells or agents inside an environment
// is a warp primitive: lit / burning / available sets are ballots (bit c = cell c, i.e. row-major nonzero() order, so
// an env-local task index is a popcount), neighbour fire spread is a bit test on the burning ballot, the agents'
// attacks reach the cells through width-G shuffles in agent order (fp32 sums associate exactly as the reference's
// per-agent loop), per-environment reductions are shuffles / popcounts.  All global traffic is issued as contiguous
// per-environment rows ([B, H*W] / [B, A] layouts) so a warp's loads and stores coalesce.
#include <cmath>
#include <math_constants.h>

#include "frz_common.cuh"
#include "frz_host.cuh"

namespace frz {
namespace {

#ifndef FRZ_WF_THREADS
#define FRZ_WF_THREADS 256
#endif
constexpr int kThreads = FRZ_WF_THREADS;
enum Mode { kStep = 0, kRefresh = 1 };

template <int NW>
__device__ __forceinline__ uint32_t word_at(const uint32_t (&words)[NW], int index) {
  uint32_t w = words[0];
#pragma unroll
  for (int i = 1; i < NW; ++i) w = (index == i) ? words[i] : w;
  return w;
}

template <int NW>
__device__ __forceinline__ bool bit_at(const uint32_t (&words)[NW], int cell) {
  return (word_at<NW>(words, cell >> 5) >> (cell & 31)) & 1u;
}

template <int G>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int offset = G / 2; offset >= 1; offset >>= 1) v += __shfl_xor_sync(kFullMask, v, offset, G);
  return v;
}

template <int G>
__device__ __forceinline__ int group_sum(int v) {
#pragma unroll
  for (int offset = G / 2; offset >= 1; offset >>= 1) v += __shfl_xor_sync(kFullMask, v, offset, G);
  return v;
}

// ballot restricted to the G lanes of this lane's group; bit j = lane j of the group
template <int G>
__device__ __forceinline__ uint32_t group_ballot(bool pred, int group_base, uint32_t group_mask) {
  const uint32_t ballot = __ballot_sync(kFullMask, pred);
  return (G == 32) ? ballot : ((ballot >> group_base) & group_mask);
}

// Shared memory of one CTA (32-bit words):
//   static, filled once per CTA from the configuration tables
//     cell_y[kCells], cell_x[kCells]   grid coordinates of cell c
//     cell_ignition[kCells]    fire_config.ignition_temp
//     cell_reward[kCells]      reward_config.fire_rewards (fp32)
//   per group (= per environment in flight), groups_per_cta times
//     attack[kCells]           fp32 attack power per cell; all zero between environments
//     task_agents[kCells]      env-local task t -> bitmask of the agents that may fight it
//   static again (sizes depend on the configuration, so they come last: every offset above is a constant)
//     cell_agents[E][kCells]   bit a = agent a reaches cell c when its equipment is in state e
//     range_mask[A][E][NW]     bit c = cell c is within agent a's reach in equipment state e
//     (half-warp groups with more than 4 cells per lane only) 2 x { fires, intensity, fuel [kCells each] }: the cell
//     state stays here instead of in registers, padded so that the two groups of a warp hit different banks.  Two
//     buffers: when the rows are 16-byte multiples the state planes move with bulk async copies (cp.async.bulk,
//     completion on an mbarrier) -- the next environment's planes are fetched while the current one is stepped, and
//     the stepped planes are written back with three bulk stores instead of 3 * CPL per-lane stores
#ifndef FRZ_WF_CELLS_IN_SMEM
#define FRZ_WF_CELLS_IN_SMEM 1
#endif
__host__ __device__ constexpr bool split_geometry(int group, int cells_per_lane) { return group == 16 && cells_per_lane > 4; }
__host__ __device__ constexpr bool cells_in_smem(int group, int cells_per_lane) {
  return FRZ_WF_CELLS_IN_SMEM && split_geometry(group, cells_per_lane);
}
__host__ __device__ constexpr int group_smem_words(int group, int cells_per_lane) {
  const int cells = group * cells_per_lane;
  // (bulk path: + a one-deep staging area for the next environment's agent rows: suppressant, capacity, equipment, action pair)
  const int words = cells_in_smem(group, cells_per_lane) ? 8 * cells + 5 * group : 2 * cells;
  return (group == 16 && words % 32 == 0) ? words + 16 : words;
}
__host__ __device__ inline int static_smem_words(int cells, int agents, int states) {
  const int words = (cells + 31) / 32;
  return 4 * cells + states * cells + agents * states * words;
}

// Row ballots -> the group's bit words (bit c = cell c).  Row i of a group holds cells i*G .. i*G+G-1, so 32 / G rows
// share one word: for 32-lane groups a row IS a word; for 16-lane groups the group's halfword of two consecutive row
// ballots is packed with one byte permute; one-row groups just shift their lanes down.
template <int G, int CPL, int NW>
__device__ __forceinline__ void assemble_words(const uint32_t (&rows)[CPL], uint32_t (&words)[NW], int group_base,
                                               uint32_t group_mask, uint32_t half_selector) {
  if constexpr (G == 32) {
#pragma unroll
    for (int i = 0; i < CPL; ++i) words[i] = rows[i];
  } else if constexpr (CPL == 1) {
    words[0] = (rows[0] >> group_base) & group_mask;
  } else if constexpr (G == 16) {
#pragma unroll
    for (int w = 0; w < NW; ++w) words[w] = __byte_perm(rows[2 * w], (2 * w + 1 < CPL) ? rows[(2 * w + 1 < CPL) ? 2 * w + 1 : 0] : 0u, half_selector);
  } else {  // G == 8: up to four rows share the one word; byte i = the group's byte of row ballot i
    static_assert(G == 8 && CPL <= 4, "8-lane groups hold at most 4 cells per lane");
    const uint32_t lo = __byte_perm(rows[0], rows[1], half_selector);  // bytes 0, 1
    const uint32_t hi = CPL > 2 ? __byte_perm(rows[2], rows[CPL - 1], half_selector) : 0u;
    uint32_t word = __byte_perm(lo, hi, 0x5410);
    if (CPL == 2) word &= 0xffffu;
    if (CPL == 3) word &= 0xffffffu;
    words[0] = word;
  }
}

// the NW range-mask words of one (agent, equipment state) row; one 16-byte load when the row is four words
template <int NW>
__device__ __forceinline__ void load_range_words(uint32_t address, uint32_t (&words)[NW]) {
  if constexpr (NW == 4) {
    const uint4 v = lds_const_v4(address);
    words[0] = v.x;
    words[1] = v.y;
    words[2] = v.z;
    words[3] = v.w;
  } else {
#pragma unroll
    for (int w = 0; w < NW; ++w) words[w] = lds_const(address + 4u * w);
  }
}

#ifndef FRZ_WF_MIN_BLOCKS
#define FRZ_WF_MIN_BLOCKS 3
#endif

// MODE: kStep or kRefresh.  INJECTED: the caller supplies uniforms (parity mode) for the field and / or the agents;
// the production path (in-kernel Philox only) is compiled without those loads.
// Launch-time constants derived from the configuration on the host (fold_configuration below).
struct Derived {
  uint32_t west_ok[FRZ_MAX_CELLS / 32];  // bit c: cell c has a western neighbour (x > 0)
  uint32_t east_ok[FRZ_MAX_CELLS / 32];  // bit c: cell c has an eastern neighbour (x < W - 1)
  int32_t spare_lanes_feed_agents;       // Philox: the agents' four words come from lanes whose last cell is off-grid
  // Philox mode compares the 24 random bits k of a draw (u = k * 2^-24) with integer thresholds: u < p  <=>  k < ceil(p * 2^24),
  // u > c  <=>  k > floor(c * 2^24) -- the same outcome as the fp32 compare for every k, without the int -> float conversion
  uint32_t t_increase, t_burnout, t_suppressant_decrease, t_repair, t_critical, t_degrade, t_refill, t_tank_switch;
  int32_t t_capacity_cum[FRZ_MAX_CAPACITIES];
  int32_t almost_state, burned_state;    // num_fire_states - 2 / - 1
  int32_t cells;                         // height * width
};

template <int G, int CPL, int MODE, bool INJECTED, bool BULK>
__global__ void __launch_bounds__(kThreads, (G * CPL > 128) ? 1 : FRZ_WF_MIN_BLOCKS)
wildfire_step_kernel(const __grid_constant__ FrzWildfireParams p, const __grid_constant__ FrzWildfireBuffers io,
                     const __grid_constant__ Derived derived, const int B) {
  constexpr int mode = MODE;
  constexpr int kGroupsPerWarp = 32 / G;
  constexpr int kCells = G * CPL;
  constexpr int NW = (kCells + 31) / 32;
  // Philox words per lane: two per cell (a cell consumes either its fire-increase or its fire-decrease draw, never
  // both, so the two events share a word; the other word is the spread draw) and four per agent
  constexpr int kCalls = (2 * CPL + 3) / 4;
  static_assert(G == 32 || G == 16 || CPL <= 4, "8-lane groups hold at most four cells per lane (one mask word)");
  constexpr int RPW = (CPL == 1) ? 1 : 32 / G;  // grid rows (of G cells) per 32-bit word
  // rows that the geometry choice guarantees to lie entirely inside the grid (pick_geometry())
  constexpr int kFullRows = (G == 32) ? CPL / 2 : (CPL - 1);
  extern __shared__ __align__(16) uint32_t smem[];

  const int lane = threadIdx.x & 31;
  // broadcast from lane 0: tells the compiler the warp index (and everything derived from it: the environment loop,
  // its trip count, every ballot word) is warp-uniform, so control flow stays convergent and votes need no re-sync
  const int warp_in_cta = __shfl_sync(kFullMask, int(threadIdx.x >> 5), 0);
  const int sub = lane % G;
  const int group_base = lane - sub;
  const uint32_t group_mask = (G == 32) ? 0xffffffffu : ((1u << G) - 1u);
  // (per-lane constants used all over the loop are made opaque to the compiler, which otherwise re-derives them from
  // %tid at every use instead of keeping them in a register: -4 % kernel time)
  uint32_t lane_bit = 1u << sub;
  asm volatile("" : "+r"(lane_bit));
  // this lane's cell of row i is bit (i % RPW) * G + sub of word i / RPW
  const auto row_bit = [&](int i) { return lane_bit << ((i % RPW) * G); };
  // byte-permute selector that pulls this group's slice out of two row ballots (assemble_words): halfword g for
  // 16-lane groups, byte g for 8-lane groups
  const uint32_t half_selector = (G == 16) ? ((group_base & 16) ? 0x7632u : 0x5410u)
                                           : (uint32_t(group_base >> 3) | ((4u + uint32_t(group_base >> 3)) << 4));
  const int W = p.width, HW = derived.cells;
  const int A = p.num_agents;
  const int E = p.num_equipment_states;
  const uint32_t flags = p.flags;
  const bool show_bad = flags & FRZ_WF_SHOW_BAD_ACTIONS;
  const bool use_fuel = flags & FRZ_WF_FIRE_FUEL;
  const int mask_words_row = io.mask_stride >> 2;
  const int table_words = io.mask_words;

  // word offsets into smem[] (see the layout above): everything but the range-mask base is a compile-time constant
  // plus, for the per-group region, one per-thread register -- shared memory is only ever addressed as smem[offset]
  constexpr int kYOff = 0, kXOff = kCells, kIgnitionOff = 2 * kCells, kRewardOff = 3 * kCells, kRegionOff = 4 * kCells;
  constexpr int kCellAgentsOff = kRegionOff + (kThreads / 32) * kGroupsPerWarp * group_smem_words(G, CPL);
  constexpr bool kCellsInSmem = cells_in_smem(G, CPL);
  const int range_off = kCellAgentsOff + E * kCells;
  const int attack_off = kRegionOff + (warp_in_cta * kGroupsPerWarp + lane / G) * group_smem_words(G, CPL);
  const int tasks_off = attack_off + kCells;
  // 32-bit shared-window byte addresses: static tables at this lane's cell column, this group's scratch region
  const uint32_t s_base = shared_address(smem);
  uint32_t s_cell = s_base + 4u * uint32_t(sub);
  asm volatile("" : "+r"(s_cell));
  uint32_t s_attack = s_base + 4u * uint32_t(attack_off);
  asm volatile("" : "+r"(s_attack));
  const uint32_t s_tasks = s_base + 4u * uint32_t(tasks_off);
  const uint32_t s_range = s_base + 4u * uint32_t(range_off);
  uint32_t* my_state = smem + tasks_off + kCells + sub;  // this lane's column of the group's current state planes
  // bulk-copy path of the state planes (kCellsInSmem geometries whose rows are 16-byte multiples): one mbarrier per
  // (warp, buffer); lane 0 of the warp issues the copies of both groups -- every operand of a bulk copy is then
  // warp-uniform (a per-group issuer makes the compiler serialise the copies lane by lane) -- and all lanes wait
  // (the barriers sit behind the range masks in the dynamic region, so that their addresses derive from the same
  // warp-uniform base as everything else)
  constexpr bool bulk = BULK;
  static_assert(!BULK || kCellsInSmem, "the bulk path moves the shared-memory state planes");
  const uint32_t s_barriers = s_base + 4u * uint32_t((range_off + A * E * NW + 3) & ~3) + 16u * uint32_t(warp_in_cta);
  const uint32_t s_planes = s_base + 4u * uint32_t(tasks_off + kCells);  // buffer 0 of this group's state planes
  // the same for group g of this warp, from warp-uniform values only
  const auto planes_of_group = [&](int g) {
    return s_base + 4u * uint32_t(kRegionOff + (warp_in_cta * kGroupsPerWarp + g) * group_smem_words(G, CPL) + 2 * kCells);
  };
  constexpr uint32_t kBufferBytes = 4u * 3u * kCells;
  // staging area of the next environment's agent rows (this lane's slots): [G] suppressant, [G] capacity, [G] equipment,
  // [G] x 8 bytes action pair -- filled by cp.async one iteration ahead, so the decode does not wait for global memory
  const uint32_t s_stage = s_planes + 2u * kBufferBytes + 4u * uint32_t(sub);

  for (int i = threadIdx.x; i < E * kCells; i += kThreads) {
    const int e = i / kCells, c = i - e * kCells;
    smem[kCellAgentsOff + i] = c < HW ? io.cell_agents[e * HW + c] : 0u;
  }
  for (int i = threadIdx.x; i < A * E * NW; i += kThreads) {
    const int row = i / NW, w = i - row * NW;
    smem[range_off + i] = w < table_words ? io.range_mask[row * table_words + w] : 0u;
  }
  for (int c = threadIdx.x; c < kCells; c += kThreads) {
    const int y = c / W, x = c - y * W;
    const bool in_grid = c < HW;
    smem[kYOff + c] = uint32_t(y);
    smem[kXOff + c] = uint32_t(x);
    smem[kIgnitionOff + c] = in_grid ? uint32_t(io.cell_ignition[c]) : 0u;
    smem[kRewardOff + c] = in_grid ? __float_as_uint(io.cell_reward[c]) : 0u;
  }
#pragma unroll
  for (int i = 0; i < CPL; ++i) smem[attack_off + i * G + sub] = 0u;
  if constexpr (kCellsInSmem) {
    // (the cells past the end of the grid are never touched by the bulk copies: they stay zero = "no fire")
#pragma unroll
    for (int i = 0; i < 6 * CPL; ++i) my_state[i * G] = 0u;
    if (bulk && lane == 0) {
      mbarrier_init(s_barriers, 1);
      mbarrier_init(s_barriers + 8u, 1);
    }
  }
  __syncthreads();

  FrzControl* const control = io.control;
  const uint64_t step = control->step;
  const uint32_t alive_prev = control->alive;
  const uint32_t agents_with_tasks = control->agents_with_tasks;
  const Philox philox(control->seed);
  // BatchedAECEnv.step returns before doing anything once every env is terminated, or every env is truncated
  // (utils/env.py:212); the flags were published by the previous launch.
  const bool skip = (mode == kStep) && ((alive_prev & 3u) != 3u);

  const bool is_agent = sub < A;
  const float base_power = is_agent ? p.agent_power[sub] : 0.f;
  const float agent_yf = is_agent ? float(p.agent_y[sub]) : 0.f;
  const float agent_xf = is_agent ? float(p.agent_x[sub]) : 0.f;

  unsigned alive_bits = 0, faults = 0, agent_bits = 0;

  if (!skip) {
    const int groups_per_cta = (kThreads / 32) * kGroupsPerWarp;
    const int first_env0 = (blockIdx.x * (kThreads / 32) + warp_in_cta) * kGroupsPerWarp;
    // bulk path: fetch the three state rows of environment `which` into buffer `buffer` of this group (lane 0 of the
    // group only; the expected byte count arms the buffer's barrier)
    const uint32_t row_bytes = 4u * uint32_t(HW);
    const auto fetch_state = [&](int pair, uint32_t into) {  // pair = the warp's first environment of that iteration
      // (broadcast from lane 0: the buffer index is the same in every lane, which the compiler cannot see)
      const uint32_t buffer = __shfl_sync(kFullMask, into, 0);
      if (elect_one()) {
        const uint32_t barrier = s_barriers + 8u * buffer;
        mbarrier_expect_bytes(barrier, uint32_t(kGroupsPerWarp) * 3u * row_bytes);
#pragma unroll
        for (int g = 0; g < kGroupsPerWarp; ++g) {
          const size_t at = size_t(min(pair + g, B - 1)) * size_t(HW);
          const uint32_t planes = planes_of_group(g) + kBufferBytes * buffer;
          bulk_load(planes, io.fires + at, row_bytes, barrier);
          bulk_load(planes + 4u * kCells, io.intensity + at, row_bytes, barrier);
          bulk_load(planes + 8u * kCells, io.fuel + at, row_bytes, barrier);
        }
      }
      if (is_agent) {  // (the staged values were consumed at the top of the current iteration)
        const uint32_t at = uint32_t(min(pair + lane / G, B - 1)) * uint32_t(A) + uint32_t(sub);
        cp_async_4(s_stage, io.suppressants + at);
        cp_async_4(s_stage + 4u * G, io.capacity + at);
        cp_async_4(s_stage + 8u * G, io.equipment + at);
        if (mode == kStep) cp_async_8(s_stage + 12u * G + 4u * uint32_t(sub), io.actions + 2u * at);
      }
      cp_async_commit();
    };
    uint32_t buffer = 0u, parities = 0u;  // current state buffer; bit b = phase parity of buffer b's barrier
    if constexpr (kCellsInSmem) {
      if (bulk && first_env0 < B) fetch_state(first_env0, 0u);
    }
    for (int env0 = first_env0; env0 < B; env0 += gridDim.x * groups_per_cta) {
      const int env = env0 + lane / G;
      const bool valid = (G == 32) || env < B;  // sub-warp groups past the end stay for the warp-wide votes
      const int e = valid ? env : B - 1;
      // 32-bit element indices (the host rejects batches whose arrays exceed 2^32 elements): one IMAD.WIDE per access
      const uint32_t cell_row = uint32_t(e) * uint32_t(HW);
      const uint32_t agent_at = uint32_t(e) * uint32_t(A) + uint32_t(sub);
      int* const fires_row = io.fires + cell_row;
      int* const inten_row = io.intensity + cell_row;
      int* const fuel_row = io.fuel + cell_row;

      // ------------------------------------------------------------------ load
      // cell state of this lane's cells: plane 0 fires, 1 intensity, 2 fuel -- in registers, or (large half-warp
      // geometries, where 3 * CPL registers per lane would spill) in the group's shared-memory planes
      int cell_regs[3][kCellsInSmem ? 1 : CPL] = {};
      // (the planes are private to the lane -- it only ever touches its own column -- so these are plain accesses the
      // compiler may batch and interleave across the unrolled cell loops; the cross-lane tables go through lds / sts)
      const auto cell = [&](int plane, int i) -> int {
        if constexpr (kCellsInSmem) return int(my_state[plane * kCells + i * G]);
        else return cell_regs[plane][i];
      };
      const auto set_cell = [&](int plane, int i, int value) {
        if constexpr (kCellsInSmem) my_state[plane * kCells + i * G] = uint32_t(value);
        else cell_regs[plane][i] = value;
      };
      uint32_t litw[NW], rows[CPL];
      if constexpr (bulk) {
        // the planes of this environment were requested one iteration ago (or in the prologue)
        mbarrier_wait(s_barriers + 8u * buffer, (parities >> buffer) & 1u);
        parities ^= 1u << buffer;
#pragma unroll
        for (int i = 0; i < CPL; ++i) rows[i] = __ballot_sync(kFullMask, cell(0, i) > 0);
      } else {
#pragma unroll
        for (int i = 0; i < CPL; ++i) {
          const int c = i * G + sub;
          // pick_geometry() only chooses CPL cells per lane when the rows before the last one are full
          const bool in_grid = i < kFullRows || c < HW;
          const int f = in_grid ? fires_row[c] : 0;
          set_cell(0, i, f);
          set_cell(1, i, in_grid ? inten_row[c] : 0);
          set_cell(2, i, in_grid ? fuel_row[c] : 0);
          rows[i] = __ballot_sync(kFullMask, f > 0);
        }
      }
      float supp = 0.f, cap = 0.f;
      int equip = 0;
      int2 staged_action = make_int2(0, -1);
      if constexpr (bulk) {
        cp_async_wait_all();  // this lane's own copies: no other lane reads its staging slots
        if (is_agent) {
          supp = __uint_as_float(lds(s_stage));
          cap = __uint_as_float(lds(s_stage + 4u * G));
          equip = min(max(int(lds(s_stage + 8u * G)), 0), E - 1);
          if (mode == kStep) {
            staged_action.x = int(lds(s_stage + 12u * G + 4u * uint32_t(sub)));
            staged_action.y = int(lds(s_stage + 12u * G + 4u * uint32_t(sub) + 4u));
          }
        }
      } else if (is_agent) {
        supp = io.suppressants[agent_at];
        cap = io.capacity[agent_at];
        equip = min(max(io.equipment[agent_at], 0), E - 1);
      }

      int n_before = 0;  // tasks published by the previous launch: rows / mask bytes beyond are already padding
      assemble_words<G, CPL, NW>(rows, litw, group_base, group_mask, half_selector);
#pragma unroll
      for (int w = 0; w < NW; ++w) n_before += __popc(litw[w]);
      if (mode != kStep) n_before = HW;  // refresh / reset: (re)write every row

      float reward = 0.f, cumulative = 0.f;
      int moves = 0, total_burnouts = 0, n_burned = 0, n_putout = 0;
      bool terminated = false, truncated = false;

      // bulk path: request the next environment's planes into the other buffer.  Every lane finished with that buffer
      // at the end of the previous iteration; its write-back (the previous iteration's bulk stores, issued by the same
      // lane) must have finished reading it.  Called a third of the way into the step so that wait is over already.
      const auto prefetch_next = [&]() {
        if constexpr (kCellsInSmem) {
          const int next_env0 = env0 + gridDim.x * groups_per_cta;
          if (bulk && next_env0 < B) {
            if (lane == 0) bulk_wait_read();
            fetch_state(next_env0, buffer ^ 1u);
          }
        }
      };
      if (mode != kStep) prefetch_next();

      if (mode == kStep) {
        // ---------------------------------------------------------------- action decode (wildfire.py:412-486)
        int act_k = 0, act_id = -1;
        if (is_agent) {
          const int2 act = bulk ? staged_action : reinterpret_cast<const int2*>(io.actions)[agent_at];
          act_k = act.x;
          act_id = act.y;
          cumulative = io.cumulative_rewards[agent_at];
        }
        moves = io.num_moves[e];
        total_burnouts = io.num_burnouts[e];
        const bool was_terminated = io.terminated[e] != 0;

        // tasks this agent could fight at the start of the step == what update_actions published after the previous
        // step (wildfire.py:587-666): lit & in Chebyshev range (equipment bonus folded in) & has suppressant
        const bool refill = is_agent && act_id == -1;  // wildfire.py:431
        int target = -1;
        bool bad = false;
        // an agent without a single task in ANY environment is skipped by the reference's decode loop
        // (wildfire.py:434): no attack, no bad-action penalty -- only its refill flag is recorded
        if (is_agent && !refill && ((agents_with_tasks >> sub) & 1u)) {
          uint32_t availw[NW];
          load_range_words<NW>(s_range + 4u * uint32_t((sub * E + equip) * NW), availw);
#pragma unroll
          for (int w = 0; w < NW; ++w) availw[w] = supp > 0.f ? (litw[w] & availw[w]) : 0u;
          // the k-th set bit of the agent's choice words: pick the word by running popcounts, then one select
          int k = act_k, found = -1, base_bit = 0;
          uint32_t chosen = 0u;
          bool hit = false;
          if (k >= 0) {
#pragma unroll
            for (int w = 0; w < NW; ++w) {
              const uint32_t choices = show_bad ? litw[w] : availw[w];
              const int count = __popc(choices);
              if (!hit) {
                if (k < count) {
                  hit = true;
                  chosen = choices;
                  base_bit = 32 * w;
                } else {
                  k -= count;
                }
              }
            }
          }
          if (hit) found = base_bit + select_bit(chosen, k);
          if (found < 0) faults |= FRZ_FAULT_BAD_TASK_INDEX;
          else if (show_bad && !bit_at<NW>(availw, found)) bad = true;  // wildfire.py:464-477
          else target = found;
        }
        const bool user = target >= 0;
        const float power = base_power + p.equipment_power_bonus[equip];  // wildfire.py:455-457

        // attack power per cell (wildfire.py:470): agents aiming at the same cell find each other with match_any and
        // sum their powers in agent order (the association of the reference's per-agent `+=`), then scatter the sum
        {
          const uint32_t key = user ? (uint32_t(group_base) << 16 | uint32_t(target)) : (0x80000000u | uint32_t(lane));
          uint32_t peers = __match_any_sync(kFullMask, key);
          if (!user) peers = 0u;
          float total = 0.f;
          while (__any_sync(kFullMask, peers != 0u)) {
            const int source = (__ffs(peers) - 1) & 31;
            const float theirs = __shfl_sync(kFullMask, power, source);
            if (peers != 0u) total = __fadd_rn(total, theirs);
            peers &= peers - 1u;
          }
          if (user) sts(s_attack + 4u * uint32_t(target), __float_as_uint(total));
          __syncwarp();
        }

        // ---------------------------------------------------------------- randomness
        // Agent events: 0 suppressant decrease, 1 equipment, 2 refill, 3 capacity pick, 4 tank switch (wildfire.py:492-513).
        // "decrease" needs a fight action and "refill" a refill action, so in Philox mode events 0 and 2 share one draw.
        // Field events per cell: fire increase / decrease (a cell consumes one or the other: one word) and spread.
        // Philox words of a lane, bits[4 * call + j].  Split layout (production path, when it needs no extra call):
        // the first half of the calls feeds increase / decrease (word i = cell i), the second half -- generated only
        // after that loop, so its words are not alive across it -- feeds the spread; used by the geometries that keep
        // the cell state in shared memory (register-bound; measured 6 % slower on the others).  Otherwise the words of
        // cell i are 2i and 2i + 1 and every call is made up front.
        constexpr bool kSplit = !INJECTED && split_geometry(G, CPL) && 2 * ((CPL + 3) / 4) == kCalls;
        constexpr int kCallsA = kSplit ? kCalls / 2 : kCalls;
        const auto grow_word = [](int i) { return kSplit ? i : 2 * i; };
        const auto spread_word = [](int i) { return kSplit ? 4 * kCallsA + i : 2 * i + 1; };
        float ua[5], uf[INJECTED ? 3 * CPL : 1];  // uf[3*i + event]: injected / pre-converted uniforms (parity mode)
        uint32_t ka[5];                           // Philox mode: the agents' draws as 24-bit integers
        uint32_t bits[4 * kCalls];
        const bool inject_agent = INJECTED && io.agent_uniforms != nullptr;
        const bool inject_field = INJECTED && io.field_uniforms != nullptr;
        const uint32_t env_lo = uint32_t(p.env_offset + e), env_hi = uint32_t(uint64_t(p.env_offset + e) >> 32);
        const uint32_t step_lo = uint32_t(step), step_hi = uint32_t(step >> 32) ^ env_hi;
        const auto draw = [&](int first_call, int last_call) {
#pragma unroll
          for (int k = first_call; k < last_call; ++k) {
            const uint4 r = philox(env_lo, step_lo, uint32_t(k * G + sub), step_hi);
            bits[4 * k] = r.x;
            bits[4 * k + 1] = r.y;
            bits[4 * k + 2] = r.z;
            bits[4 * k + 3] = r.w;
          }
        };
        if (!inject_field || !inject_agent) draw(0, kCallsA);
        if constexpr (INJECTED) {
          const size_t plane = size_t(B) * HW;
#pragma unroll
          for (int i = 0; i < CPL; ++i) {
            const int c = i * G + sub;
            if (inject_field) {
#pragma unroll
              for (int ev = 0; ev < 3; ++ev) uf[3 * i + ev] = c < HW ? io.field_uniforms[ev * plane + cell_row + c] : 1.f;
            } else {
              uf[3 * i] = uf[3 * i + 1] = u01(bits[grow_word(i)]);
              uf[3 * i + 2] = u01(bits[spread_word(i)]);
            }
          }
        }
        const auto field_uniform = [&](int i, int event) -> float {  // event: 0 increase, 1 decrease, 2 spread
          if constexpr (INJECTED) return uf[3 * i + event];
          else return u01(bits[event == 2 ? spread_word(i) : grow_word(i)]);
        };

        // ---------------------------------------------------------------- agent randomness + transitions
        // Independent of the fire transitions (they only meet again in update_actions), so the phase runs before them
        // or -- in the split Philox layout, where the agents' words exist only after the second half of the calls --
        // after the spread.
        const auto agent_phase = [&]() {
          if (inject_agent) {
#pragma unroll
            for (int ev = 0; ev < 5; ++ev)
              ua[ev] = is_agent ? io.agent_uniforms[(size_t(ev) * B + e) * A + sub] : 1.f;
          } else {
            uint32_t words[4];
            bool have_words = false;
            // Words this lane never consumes: 4 * kCalls - 2 * CPL of its own (kSpareOwn: 0 or 2), and the two words of
            // its last cell when that cell lies outside the grid ("spare lanes": the top lanes of the group).  When the
            // host found enough spare lanes for this grid, the agents' four words come from there instead of from a
            // Philox call of their own.
            constexpr int kSpareOwn = 4 * kCalls - 2 * CPL;
            constexpr int kOwnA = kSplit ? CPL : 2 * CPL, kOwnB = kSplit ? 4 * kCallsA + CPL : 2 * CPL + 1;
            if constexpr (CPL > 1) {
              if (derived.spare_lanes_feed_agents) {
                const int first = group_base + ((G - 1 - sub) & (G - 1)), second = group_base + ((G - 1 - A - sub) & (G - 1));
                const uint32_t a = __shfl_sync(kFullMask, bits[grow_word(CPL - 1)], first);
                const uint32_t b = __shfl_sync(kFullMask, bits[spread_word(CPL - 1)], first);
                if constexpr (kSpareOwn == 2) {
                  words[0] = bits[kOwnA < 4 * kCalls ? kOwnA : 0];
                  words[1] = bits[kOwnB < 4 * kCalls ? kOwnB : 0];
                  words[2] = a;
                  words[3] = b;
                } else {
                  words[0] = a;
                  words[1] = b;
                  words[2] = __shfl_sync(kFullMask, bits[grow_word(CPL - 1)], second);
                  words[3] = __shfl_sync(kFullMask, bits[spread_word(CPL - 1)], second);
                }
                have_words = true;
              }
            }
            if (!have_words) {
              const uint4 r = philox(env_lo, step_lo, 0x80000000u | uint32_t(sub), step_hi);
              words[0] = r.x;
              words[1] = r.y;
              words[2] = r.z;
              words[3] = r.w;
            }
            if constexpr (INJECTED) {
              ua[0] = ua[2] = u01(words[0]);
              ua[1] = u01(words[1]);
              ua[3] = u01(words[2]);
              ua[4] = u01(words[3]);
            } else {
              ka[0] = ka[2] = words[0] >> 8;
              ka[1] = words[1] >> 8;
              ka[3] = words[2] >> 8;
              ka[4] = words[3] >> 8;
            }
          }
          // event `ev` happens with probability p: fp32 compare on injected uniforms, integer compare on Philox bits
          const auto happens = [&](int ev, float p_event, uint32_t t_event) -> bool {
            if constexpr (INJECTED) return ua[ev] < p_event;
            else return ka[ev] < t_event;
          };

          // agent transitions (the host folded the StochasticConfiguration switches into the thresholds: 2 = always, -1 = never)
          // suppressant_decrease.py:34-63
          const bool decrease = user && happens(0, p.p_suppressant_decrease, derived.t_suppressant_decrease);
          supp = fmaxf(decrease ? __fadd_rn(supp, -1.f) : supp, 0.f);
          // equipment.py:42-77 -- masks from the pre-update state, one uniform for all three tests
          {
            const bool pristine = equip == E - 1, damaged = equip == 0;
            const bool wearable = pristine || !damaged;  // pristine | intermediate
            const bool repairs = damaged && happens(1, p.p_repair, derived.t_repair);
            const bool critical = pristine && happens(1, p.p_critical, derived.t_critical);
            const bool degrades = wearable && happens(1, p.p_degrade, derived.t_degrade) && !critical;
            if (repairs) equip = E - 1;
            if (critical) equip = 0;
            if (degrades) equip -= 1;
          }
          // suppressant_refill.py:43-74 -- bonus of the equipment state AFTER its transition
          const bool increased = refill && happens(2, p.p_refill, derived.t_refill);
          if (increased) supp = __fadd_rn(cap, p.equipment_capacity_bonus[max(equip, 0)]);
          // capacity.py:39-66 -- bucketize(right=False): first i with r <= cum[i]
          if (__any_sync(kFullMask, increased)) {
            // first i with r <= cum[i] == the number of entries below r (cum is non-decreasing; the host pads the unused
            // entries with +inf), capped at the last capacity like the reference's default
            int pick = 0;
#pragma unroll
            for (int i = 0; i < FRZ_MAX_CAPACITIES; ++i) {
              if constexpr (INJECTED) pick += ua[3] > p.capacity_cum[i] ? 1 : 0;
              else pick += int(ka[3]) > derived.t_capacity_cum[i] ? 1 : 0;
            }
            pick = min(pick, p.num_capacities - 1);
            const bool switches = increased && happens(4, p.p_tank_switch, derived.t_tank_switch);
            const float extra = __fadd_rn(supp, -cap);
            if (switches) {
              cap = p.capacity_value[pick];
              supp = __fadd_rn(cap, extra);
            }
          }
        };
        if constexpr (!kSplit) agent_phase();

        // ---------------------------------------------------------------- fire increase + decrease per cell
        // p.p_increase / p.p_burnout arrive clamped (and 1 when the increase is deterministic); a deterministic
        // decrease arrives as p_decrease = 2, bonus = 0, which the clamp turns into probability 1
        uint32_t burned_bits = 0, putout_bits = 0;  // bit i = this lane's cell i
        uint32_t burnw[NW];
#pragma unroll
        for (int i = 0; i < CPL; ++i) {
          const float attack = __uint_as_float(lds(s_attack + 4u * uint32_t(i * G + sub)));
          int f = cell(0, i), it = cell(1, i);
          // fire_increase.py:43-95
          const bool burning = f > 0 && it > 0;
          const float diff = __fadd_rn(f > 0 ? float(f) : 0.f, -attack);
          const bool unmet = burning && diff > 0.f;
          // (one Philox word serves both events of a cell)
          bool grow;
          float u_down;
          if constexpr (INJECTED) {
            u_down = field_uniform(i, 1);
            grow = unmet && field_uniform(i, 0) < (it == derived.almost_state ? p.p_burnout : p.p_increase);
          } else {
            const uint32_t k24 = bits[grow_word(i)] >> 8;
            u_down = float(k24) * 5.9604644775390625e-08f;
            grow = unmet && (it == derived.almost_state ? k24 < derived.t_burnout : k24 < derived.t_increase);
          }
          it += grow ? 1 : 0;
          const bool burned = grow && it >= derived.burned_state;
          // fire_decrease.py:36-80 sees the post-increase state: a cell that just burned out is no longer lit, any other
          // burning cell kept its sign and a positive intensity, so `diff` is unchanged; the product and the sum are
          // rounded separately like the reference's two aten ops
          const bool met = burning && !burned && diff <= 0.f;
          const float prob_down = fminf(fmaxf(__fadd_rn(p.p_decrease, __fmul_rn(-diff, p.decrease_bonus)), 0.f), 1.f);
          const bool shrink = met && u_down < prob_down;
          it -= shrink ? 1 : 0;
          const bool put = shrink && it <= 0;
          if (burned || put) {
            // burn-out clamps the fuel (fire_increase.py:90), putting out does not (fire_decrease.py:75)
            const int fuel = cell(2, i) - 1;
            set_cell(2, i, burned ? max(fuel, 0) : fuel);
            f = -f;
          }
          burned_bits |= uint32_t(burned) << i;
          putout_bits |= uint32_t(put) << i;
          if (!kCellsInSmem || burned || put) set_cell(0, i, f);
          if (!kCellsInSmem || grow || shrink) set_cell(1, i, it);
          rows[i] = __ballot_sync(kFullMask, burning && !burned && !put);
        }
        assemble_words<G, CPL, NW>(rows, burnw, group_base, group_mask, half_selector);
        // the agents that scattered an attack clear it again: the table is all zero between environments
        __syncwarp();
        if (user) sts(s_attack + 4u * uint32_t(target), 0u);

        // ---------------------------------------------------------------- fire spread (fire_spreads.py:33-59)
        if constexpr (kSplit) draw(kCallsA, kCalls);
        prefetch_next();
#pragma unroll
        for (int w = 0; w < NW; ++w) {  // word by word: the neighbour words are shared by the RPW rows of a word
          int f[RPW], it[RPW];
          bool unlit[RPW], any_unlit = false;
#pragma unroll
          for (int r = 0; r < RPW; ++r) {
            const int i = w * RPW + r;
            unlit[r] = false;
            if (i < CPL) {
              f[r] = cell(0, i);
              it[r] = cell(1, i);
              unlit[r] = f[r] < 0 && it[r] == 0 && (!use_fuel || cell(2, i) > 0);
              any_unlit = any_unlit || unlit[r];
            }
          }
          if (__any_sync(kFullMask, any_unlit)) {
            // burning neighbours of cell c as bit c of four words: N = cell c-W, W = c-1, E = c+1, S = c+W
            const uint32_t cur = burnw[w];
            const uint32_t prev = w > 0 ? burnw[w > 0 ? w - 1 : 0] : 0u;
            const uint32_t next = w + 1 < NW ? burnw[w + 1 < NW ? w + 1 : 0] : 0u;
            uint32_t north, south;
            if (W < 32) {
              north = __funnelshift_l(prev, cur, W);
              south = __funnelshift_r(cur, next, W);
            } else {  // a row is at least one word: the neighbour word is W / 32 (+ 1) words away
              const int q = W >> 5, r = W & 31;
              const auto word_or_zero = [&](int v) { return (v >= 0 && v < NW) ? word_at<NW>(burnw, v) : 0u; };
              north = __funnelshift_l(word_or_zero(w - q - 1), word_or_zero(w - q), r);
              south = __funnelshift_r(word_or_zero(w + q), word_or_zero(w + q + 1), r);
            }
            const uint32_t west = __funnelshift_l(prev, cur, 1) & derived.west_ok[w];
            const uint32_t east = __funnelshift_r(cur, next, 1) & derived.east_ok[w];
#pragma unroll
            for (int r = 0; r < RPW; ++r) {
              const int i = w * RPW + r;
              if (i < CPL) {
                const uint32_t my_bit = row_bit(i);
                // the conv sum in the reference's accumulation order N, W, E, S, starting from zero (spread_lut[1 << k]
                // is the weight of direction k; see spread_lut() on the host for the order)
                float prob = 0.f;
                if (north & my_bit) prob = p.spread_lut[1];
                if (west & my_bit) prob = __fadd_rn(prob, p.spread_lut[2]);
                if (east & my_bit) prob = __fadd_rn(prob, p.spread_lut[4]);
                if (south & my_bit) prob = __fadd_rn(prob, p.spread_lut[8]);
                prob = __fadd_rn(prob, p.p_random_ignition);
                if (unlit[r] && field_uniform(i, 2) < prob) {
                  f[r] = -f[r];
                  it[r] = int(lds_const(s_cell + 4u * (kIgnitionOff + i * G)));
                  if (kCellsInSmem) {
                    set_cell(0, i, f[r]);
                    set_cell(1, i, it[r]);
                  }
                }
              }
            }
          }
#pragma unroll
          for (int r = 0; r < RPW; ++r) {
            const int i = w * RPW + r;
            if (i < CPL) {
              if (!kCellsInSmem) {
                set_cell(0, i, f[r]);
                set_cell(1, i, it[r]);
              }
              rows[i] = __ballot_sync(kFullMask, f[r] > 0);
            }
          }
        }
        assemble_words<G, CPL, NW>(rows, litw, group_base, group_mask, half_selector);

        if constexpr (kSplit) agent_phase();

        // ---------------------------------------------------------------- rewards + termination (wildfire.py:534-582)
        // burn-outs and put-outs are rare: count them with one reduction each and only then look at which cells
        if constexpr (G == 32) {
          n_burned = __reduce_add_sync(kFullMask, __popc(burned_bits));
          n_putout = __reduce_add_sync(kFullMask, __popc(putout_bits));
        } else {
          n_burned = group_sum<G>(__popc(burned_bits));
          n_putout = group_sum<G>(__popc(putout_bits));
        }
        float put_total = 0.f, burn_total = 0.f;
        uint32_t putw[NW];
#pragma unroll
        for (int w = 0; w < NW; ++w) putw[w] = 0u;
        const bool localize = flags & FRZ_WF_LOCALIZE_PUTOUTS, scaled = flags & FRZ_WF_BURNOUT_SCALED;
        if (__any_sync(kFullMask, n_putout != 0) && !localize) {  // warp-uniform tests
          float my_put_reward = 0.f;
#pragma unroll
          for (int i = 0; i < CPL; ++i)
            if ((putout_bits >> i) & 1u) my_put_reward += __uint_as_float(lds_const(s_cell + 4u * (kRewardOff + i * G)));
          put_total = group_sum<G>(my_put_reward);
        }
        if (__any_sync(kFullMask, n_putout != 0) && localize) {
#pragma unroll
          for (int i = 0; i < CPL; ++i) rows[i] = __ballot_sync(kFullMask, (putout_bits >> i) & 1u);
          assemble_words<G, CPL, NW>(rows, putw, group_base, group_mask, half_selector);
        }
        if (__any_sync(kFullMask, n_burned != 0) && scaled) {
          float my_burn_reward = 0.f;
#pragma unroll
          for (int i = 0; i < CPL; ++i)
            if ((burned_bits >> i) & 1u) my_burn_reward += __uint_as_float(lds_const(s_cell + 4u * (kRewardOff + i * G)));
          burn_total = group_sum<G>(my_burn_reward);
        }
        const float penalty_total =
            (flags & FRZ_WF_BURNOUT_SCALED) ? -burn_total : __fmul_rn(p.burnout_penalty, float(n_burned));
        uint32_t any_lit = 0;
#pragma unroll
        for (int w = 0; w < NW; ++w) any_lit |= litw[w];
        bool dead = any_lit == 0;
        if (use_fuel && __any_sync(kFullMask, dead)) {
          int my_fuel = 0;
#pragma unroll
          for (int i = 0; i < CPL; ++i) my_fuel += cell(2, i);
          const int fuel_left = group_sum<G>(my_fuel);  // every lane takes part: no short-circuit around the shuffles
          dead = dead && fuel_left <= 0;
        }
        if (dead) {  // wildfire.py:570
#pragma unroll
          for (int i = 0; i < CPL; ++i) set_cell(0, i, 0);
#pragma unroll
          for (int w = 0; w < NW; ++w) litw[w] = 0;
        }
        const bool newly = !was_terminated && dead;
        terminated = was_terminated || dead;
        reward = bad ? p.bad_attack_penalty : 0.f;
        float gain = put_total;
        if (flags & FRZ_WF_LOCALIZE_PUTOUTS)
          gain = (target >= 0 && bit_at<NW>(putw, target)) ? __uint_as_float(lds_const(s_base + 4u * uint32_t(kRewardOff + target))) : 0.f;
        reward = __fadd_rn(reward, __fadd_rn(gain, penalty_total));
        if (newly) {
          const float penalty = __fmul_rn(p.termination_kappa, logf(__fadd_rn(float(total_burnouts), 1.f)));
          reward = __fadd_rn(reward, fmaxf(__fadd_rn(p.termination_reward, -penalty), 0.f));
        }
        total_burnouts += n_burned;
        // utils/env.py:228-235
        moves += 1;
        truncated = moves >= p.max_steps;
        cumulative = __fadd_rn(cumulative, reward);
        if (valid) alive_bits |= (terminated ? 0u : 1u) | (truncated ? 0u : 2u);
      } else if (valid) {  // refresh: the done flags as a reset, a restore or a hand edit left them
        alive_bits |= (io.terminated[e] ? 0u : 1u) | (io.truncated[e] ? 0u : 2u);
      }

      // ------------------------------------------------------------------ update_actions / update_observations
      if constexpr (G != 32) {
        if (!valid) {  // a group past the end of the batch has no tasks to publish: no rows, no mask words below
          n_before = 0;
#pragma unroll
          for (int w = 0; w < NW; ++w) litw[w] = 0u;
        }
      }
      int n_lit = 0;
#pragma unroll
      for (int w = 0; w < NW; ++w) n_lit += __popc(litw[w]);
      const int n_rows = max(n_lit, n_before);  // rows / mask bytes that may differ from their padding value

      int n_avail = 0;
      if (is_agent && supp > 0.f) {
        uint32_t reach[NW];
        load_range_words<NW>(s_range + 4u * uint32_t((sub * E + max(equip, 0)) * NW), reach);
#pragma unroll
        for (int w = 0; w < NW; ++w) n_avail += __popc(litw[w] & reach[w]);
      }
      // agents able to act right now, grouped by equipment state: a cell's fighters are the union over equipment
      // states of (agents that reach the cell in that state) & (agents in that state with suppressant left)
      uint32_t fighters[CPL];
#pragma unroll
      for (int i = 0; i < CPL; ++i) fighters[i] = 0u;
      for (int q = 0; q < E; ++q) {
        const uint32_t ready = group_ballot<G>(is_agent && supp > 0.f && equip == q, group_base, group_mask);
#pragma unroll
        for (int i = 0; i < CPL; ++i) fighters[i] |= lds_const(s_cell + 4u * uint32_t(kCellAgentsOff + q * kCells + i * G)) & ready;
      }
      int4* const task_rows = reinterpret_cast<int4*>(io.task_obs);
      {
        int rank = 0;  // lit cells in the words before the current one
#pragma unroll
        for (int i = 0; i < CPL; ++i) {
          const uint32_t word = litw[i / RPW], my_bit = row_bit(i);
          if (i > 0 && i % RPW == 0) rank += __popc(litw[i > 0 ? i / RPW - 1 : 0]);
          if (word & my_bit) {
            const int t = rank + __popc(word & (my_bit - 1u));  // env-local task index = rank in row-major lit order
            sts(s_tasks + 4u * uint32_t(t), fighters[i]);
            task_rows[cell_row + uint32_t(t)] = make_int4(int(lds_const(s_cell + 4u * (kYOff + i * G))), int(lds_const(s_cell + 4u * (kXOff + i * G))),
                                      cell(0, i), cell(1, i));
          }
        }
      }
      // tasks of the previous launch that no longer exist: their rows go back to padding, their mask bytes to zero
      const int quads = (n_rows + 3) >> 2;
      const int quads_warp = __reduce_max_sync(kFullMask, quads);  // (every lane of the warp: not under `valid`)
      for (int first = n_lit; first < 4 * quads; first += G) {
        const int t = first + sub;
        if (t < 4 * quads) {
          sts(s_tasks + 4u * uint32_t(t), 0u);
          if (t < n_before) task_rows[cell_row + uint32_t(t)] = make_int4(FRZ_PAD, FRZ_PAD, FRZ_PAD, FRZ_PAD);
        }
      }
      __syncwarp();

      if (valid) {
        // action mask [A, mask_stride] bytes indexed by env-local task, four tasks per 4-byte store.  The group's
        // lanes are cut into (agent slot, task quad): `span` = the smallest power of two that holds the quads of
        // every environment of the warp (at most G), G / span agent slots.  A lane packs the fighter sets of its
        // four tasks into byte planes (byte j of plane k = agents 8k .. 8k+7 of task 4q+j) and emits
        // (plane >> (a & 7)) & 0x01010101 for the agents a = slot, slot + slots, ... -- lanes of one slot write
        // consecutive words of one agent's row, and few tasks mean many slots, i.e. few passes over the agents.
        uint32_t* const mask_words = reinterpret_cast<uint32_t*>(io.action_mask);
        const uint32_t mask_env = uint32_t(env) * uint32_t(A) * uint32_t(mask_words_row);
        const int span_shift = min(32 - __clz(max(quads_warp, 1) - 1), (G == 32) ? 5 : (G == 16) ? 4 : 3);
        const int span = 1 << span_shift, slots = G >> span_shift;
        const int slot = sub >> span_shift, quad_in_span = sub & (span - 1);
        for (int first = 0; first < quads; first += span) {
          const int q = first + quad_in_span;
          if (q < quads) {
            const uint4 m = lds_v4(s_tasks + 16u * uint32_t(q));
            // a group of G lanes holds at most G agents: one byte plane per eight of them; the agents are visited
            // plane by plane (the plane index is a compile-time constant inside each inner loop)
            constexpr int kPlanes = G / 8;
            uint32_t at = mask_env + uint32_t(slot * mask_words_row + q);
            const uint32_t stride = uint32_t(slots * mask_words_row);
            int a = slot;
#pragma unroll
            for (int k = 0; k < kPlanes; ++k) {
              if (k > 0 && 8 * k >= A) break;
              const uint32_t selector = uint32_t(k | ((4 + k) << 4));
              const uint32_t plane = __byte_perm(__byte_perm(m.x, m.y, selector), __byte_perm(m.z, m.w, selector), 0x5410);
              const int end = min(A, 8 * k + 8);
              for (; a < end; a += slots, at += stride) mask_words[at] = (plane >> (a & 7)) & 0x01010101u;
            }
          }
        }

        if (is_agent) {
          io.agent_task_count[agent_at] = n_avail;
          if (n_avail > 0) agent_bits |= lane_bit;
          reinterpret_cast<float4*>(io.self_obs)[agent_at] =
              make_float4(agent_yf, agent_xf, base_power, supp);
        }
        if (sub == 0) io.env_task_count[env] = n_lit;

        if (mode == kStep) {
          if (!bulk) {
#pragma unroll
            for (int i = 0; i < CPL; ++i) {
              const int c = i * G + sub;
              if (i < kFullRows || c < HW) {
                fires_row[c] = cell(0, i);
                inten_row[c] = cell(1, i);
                fuel_row[c] = cell(2, i);
              }
            }
          }
          if (is_agent) {
            io.suppressants[agent_at] = supp;
            io.capacity[agent_at] = cap;
            io.equipment[agent_at] = equip;
            io.rewards[agent_at] = reward;
            io.cumulative_rewards[agent_at] = cumulative;
          }
          if (sub == 0) {
            io.terminated[env] = terminated;
            io.truncated[env] = truncated;
            io.num_moves[env] = moves;
            io.num_burnouts[env] = total_burnouts;
            io.burnouts[env] = n_burned;
            io.putouts[env] = n_putout;
          }
        }
      }
      if constexpr (kCellsInSmem) {
        if (bulk) {
          if (mode == kStep) {
            // write the stepped planes back: the lanes' shared-memory writes become visible to the async proxy, then
            // lane 0 stores the three rows of both groups
            fence_async_shared();
            __syncwarp();
            const uint32_t from = __shfl_sync(kFullMask, buffer, 0);
            if (lane == 0) {
#pragma unroll
              for (int g = 0; g < kGroupsPerWarp; ++g) {
                if (env0 + g < B) {
                  const size_t at = size_t(env0 + g) * size_t(HW);
                  const uint32_t planes = planes_of_group(g) + kBufferBytes * from;
                  bulk_store(io.fires + at, planes, row_bytes);
                  bulk_store(io.intensity + at, planes + 4u * kCells, row_bytes);
                  bulk_store(io.fuel + at, planes + 8u * kCells, row_bytes);
                }
              }
              bulk_commit();
            }
          }
          buffer ^= 1u;
          my_state = smem + tasks_off + kCells + sub + buffer * (3 * kCells);
        }
      }
      __syncwarp();
    }
    if constexpr (kCellsInSmem) {
      if (bulk && lane == 0) bulk_wait_read();  // shared memory must outlive the last write-back
    }
  }
  finish_launch(control, alive_bits, faults, agent_bits,
                skip ? kPublishNothing : (mode == kStep ? kPublishStep : kPublishRefresh));
}

// ------------------------------------------------------------------------------------------------ reset / sampling

__global__ void wildfire_restore_kernel(const FrzWildfireParams p, const FrzWildfireBuffers io, const int B,
                                        const uint8_t* __restrict__ env_mask) {
  const int HW = p.height * p.width, A = p.num_agents;
  const int per_env = HW > A ? HW : A;
  const size_t total = size_t(B) * per_env;
  for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += size_t(gridDim.x) * blockDim.x) {
    const int env = int(i / per_env), j = int(i % per_env);
    if (env_mask != nullptr && !env_mask[env]) continue;
    if (j < HW) {
      const size_t at = size_t(env) * HW + j;
      io.fires[at] = io.init_fires[at];
      io.intensity[at] = io.init_intensity[at];
      io.fuel[at] = io.init_fuel[at];
    }
    if (j < A) {
      const size_t at = size_t(env) * A + j;
      io.suppressants[at] = io.init_suppressants[at];
      io.capacity[at] = io.init_capacity[at];
      io.equipment[at] = io.init_equipment[at];
      io.rewards[at] = 0.f;
      io.cumulative_rewards[at] = 0.f;
    }
    if (j == 0) {
      io.terminated[env] = 0;
      io.truncated[env] = 0;
      io.num_moves[env] = 0;
      io.num_burnouts[env] = 0;
      io.burnouts[env] = 0;
      io.putouts[env] = 0;
    }
  }
}

__global__ void wildfire_sample_kernel(const FrzWildfireParams p, const FrzWildfireBuffers io, const int B,
                                       const uint64_t sampler_seed) {
  const int A = p.num_agents;
  const Philox philox(sampler_seed);
  const uint64_t step = io.control->step;
  const bool show_bad = p.flags & FRZ_WF_SHOW_BAD_ACTIONS;
  const int total = B * A;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int env = i / A, agent = i - env * A;
    const int n = show_bad ? io.env_task_count[env] : io.agent_task_count[i];
    const uint64_t genv = uint64_t(p.env_offset + env);
    const uint4 r = philox(uint32_t(genv), uint32_t(step), 0xC0000000u | uint32_t(agent), uint32_t(step >> 32) ^ uint32_t(genv >> 32));
    const int k = min(int(u01(r.x) * float(n + 1)), n);
    reinterpret_cast<int2*>(const_cast<int32_t*>(io.actions))[i] = make_int2(k, k == n ? -1 : 0);
  }
}

// Largest grid (in cells) that is stepped by half-warp groups (when the agents fit 16 lanes).  Measured on B200:
//   3x3 / 3 agents (524 288 envs)    16-lane groups 258 us   8-lane groups, 2 cells per lane 157 us
//   5x6 / 6 agents (262 144 envs)    32-lane groups 269 us   half-warp groups 178 us   8-lane groups 159 us
//   7x8 / 5 agents (262 144 envs)                   310 us                    245 us
//   10x10 / 10 agents (65 536 envs)                 116 us                    110 us with the cell state in shared
//                                                   memory (124 us with 7 cells per lane in registers: spills)
#ifndef FRZ_WF_HALF_WARP_CELLS
#define FRZ_WF_HALF_WARP_CELLS 128
#endif

struct Geometry {
  int group, cells_per_lane;
};

bool pick_geometry(const FrzWildfireParams& p, Geometry* g) {
  const int HW = p.height * p.width, A = p.num_agents;
  if (A < 1 || A > FRZ_MAX_AGENTS || HW < 1 || HW > FRZ_MAX_CELLS) return false;
  // Half-warp groups for small and mid-size grids whose agents fit 16 lanes: two environments share every instruction
  // of the agent phase, and ceil(H*W / 16) cells per lane waste fewer lanes than a power-of-two count over 32 lanes.
  if (HW <= 8 && A <= 8) *g = {8, 1};
  else if (HW <= 32 && A <= 8) *g = {8, (HW + 7) / 8};  // four environments per warp
  else if (HW <= 16 && A <= 16) *g = {16, 1};
  else if (HW <= FRZ_WF_HALF_WARP_CELLS && A <= 16) *g = {16, (HW + 15) / 16};
  else if (HW <= 32) *g = {32, 1};
  else if (HW <= 64) *g = {32, 2};
  else if (HW <= 128) *g = {32, 4};
  else *g = {32, 8};
  return true;
}

// What the kernel receives instead of the caller's FrzWildfireParams: the StochasticConfiguration switches
// (structures/configuration.py:271-322) are folded into the thresholds the uniforms are compared with -- every draw is
// in [0, 1), so a threshold of 2 makes the event certain and -1 impossible, exactly what the reference's
// "if not stochastic: skip the randomness test" branches do -- and the per-word neighbour masks are tabulated.
void fold_configuration(const FrzWildfireParams& in, int group, int cells_per_lane, FrzWildfireParams* out, Derived* derived) {
  *out = in;
  const uint32_t flags = in.flags;
  const auto clamp01 = [](float v) { return v < 0.f ? 0.f : (v > 1.f ? 1.f : v); };
  if (!(flags & FRZ_WF_STOCH_SUPPRESSANT_DECREASE)) out->p_suppressant_decrease = 2.f;  // suppressant_decrease.py:49-53
  if (!(flags & FRZ_WF_STOCH_REFILL)) out->p_refill = 2.f;                                // suppressant_refill.py:58-62
  if (!(flags & FRZ_WF_STOCH_TANK_SWITCH)) out->p_tank_switch = 2.f;                      // capacity.py:54-58
  if (!(flags & FRZ_WF_CRITICAL_ERROR)) out->p_critical = -1.f;                           // equipment.py:60-63
  if (!(flags & FRZ_WF_STOCH_DEGRADE)) out->p_degrade = 2.f;                              // equipment.py:65-69
  if (!(flags & FRZ_WF_STOCH_REPAIR)) out->p_repair = 2.f;                                // equipment.py:54-58
  // fire_increase.py:62-78: probability 1 when deterministic; "almost burned out" cells use the burnout probability
  out->p_increase = (flags & FRZ_WF_STOCH_FIRE_INCREASE) ? clamp01(in.p_increase) : 1.f;
  out->p_burnout = clamp01((flags & FRZ_WF_SPECIAL_BURNOUT) ? in.p_burnout : in.p_increase);
  if (!(flags & FRZ_WF_STOCH_FIRE_DECREASE)) {  // fire_decrease.py:60-66: clamp(2 + x * 0) = 1
    out->p_decrease = 2.f;
    out->decrease_bonus = 0.f;
  }
  for (int i = in.num_capacities; i < FRZ_MAX_CAPACITIES; ++i) out->capacity_cum[i] = INFINITY;  // capacity.py:52
  const int H = in.height, W = in.width, HW = H * W;
  for (int w = 0; w < FRZ_MAX_CELLS / 32; ++w) derived->west_ok[w] = derived->east_ok[w] = 0u;
  for (int c = 0; c < HW; ++c) {
    const int x = c % W;
    if (x > 0) derived->west_ok[c >> 5] |= 1u << (c & 31);
    if (x < W - 1) derived->east_ok[c >> 5] |= 1u << (c & 31);
  }
  {
    const auto below = [](float probability) {  // u < p  <=>  k < ceil(p * 2^24)
      const double scaled = std::ceil(double(probability) * 16777216.0);
      return uint32_t(scaled < 0.0 ? 0.0 : (scaled > 16777216.0 ? 16777216.0 : scaled));
    };
    derived->t_increase = below(out->p_increase);
    derived->t_burnout = below(out->p_burnout);
    derived->t_suppressant_decrease = below(out->p_suppressant_decrease);
    derived->t_repair = below(out->p_repair);
    derived->t_critical = below(out->p_critical);
    derived->t_degrade = below(out->p_degrade);
    derived->t_refill = below(out->p_refill);
    derived->t_tank_switch = below(out->p_tank_switch);
    for (int i = 0; i < FRZ_MAX_CAPACITIES; ++i) {  // u > c  <=>  k > floor(c * 2^24)
      const double scaled = std::floor(double(out->capacity_cum[i]) * 16777216.0);
      derived->t_capacity_cum[i] = std::isnan(scaled) ? (1 << 24) : int32_t(scaled < -1.0 ? -1.0 : (scaled > 16777216.0 ? 16777216.0 : scaled));
    }
    derived->almost_state = in.num_fire_states - 2;
    derived->burned_state = in.num_fire_states - 1;
    derived->cells = in.height * in.width;
  }
  // Philox layout (see the kernel): lanes whose last cell is off-grid have two unused words; with an odd number of
  // cells per lane every lane has two more.  The agents' four words are taken from those when enough lanes qualify.
  derived->spare_lanes_feed_agents = 0;
  if (cells_per_lane > 1) {
    const int last_row_cells = HW - group * (cells_per_lane - 1);  // cells of the last row that are inside the grid
    const int spare_lanes = group - (last_row_cells > 0 ? last_row_cells : 0);
    const int calls = (2 * cells_per_lane + 3) / 4, spare_own = 4 * calls - 2 * cells_per_lane;
    const int lanes_needed = spare_own == 2 ? in.num_agents : 2 * in.num_agents;
    derived->spare_lanes_feed_agents = lanes_needed <= spare_lanes ? 1 : 0;
  }
}

#include "frz_wildfire_tile.cuh"

// The tiled kernel for small grids: a one-warp CTA per tile of 32 environments, persistent grid in whole rounds.
template <int MAXA, int MODE, bool INJECTED>
int launch_tiles(const FrzWildfireParams& caller_params, const FrzWildfireBuffers& io, int B, const Geometry& g,
                 cudaStream_t stream) {
  FrzWildfireParams p;
  Derived derived;
  fold_configuration(caller_params, g.group, g.cells_per_lane, &p, &derived);
  const SmallRandomLayout layout = small_random_layout(p.height * p.width, p.num_agents, g.group, g.cells_per_lane,
                                                       derived.spare_lanes_feed_agents != 0);
  const size_t smem = size_t(small_tile(p.height * p.width, p.num_agents).total) * sizeof(uint32_t);
  auto kernel = wildfire_tile_kernel<MAXA, MODE, INJECTED>;
  if (smem > 48 * 1024 && cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)) != cudaSuccess)
    return check_launch("wildfire tile shared memory");
  cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  const int tiles = (B + 31) / 32;
  const int resident = sm_count() * resident_ctas(kernel, 32, smem);
  const int rounds = (tiles + resident - 1) / resident;
  const int grid = (tiles + rounds - 1) / rounds;
  kernel<<<grid, 32, smem, stream>>>(p, io, derived, layout, B);
  return check_launch("wildfire_tile_kernel");
}

template <int MAXA>
int launch_tiles_mode(const FrzWildfireParams& p, const FrzWildfireBuffers& io, int B, int mode, const Geometry& g,
                      cudaStream_t stream) {
  if (mode != kStep) return launch_tiles<MAXA, kRefresh, false>(p, io, B, g, stream);
  if (io.field_uniforms != nullptr || io.agent_uniforms != nullptr) return launch_tiles<MAXA, kStep, true>(p, io, B, g, stream);
  return launch_tiles<MAXA, kStep, false>(p, io, B, g, stream);
}

template <int G, int CPL, int MODE, bool INJECTED, bool BULK>
int launch_variant(const FrzWildfireParams& caller_params, const FrzWildfireBuffers& io, int B, cudaStream_t stream) {
  FrzWildfireParams p;
  Derived derived;
  fold_configuration(caller_params, G, CPL, &p, &derived);
  const int groups_per_cta = (kThreads / 32) * (32 / G);
  const size_t smem = (size_t(static_smem_words(G * CPL, p.num_agents, p.num_equipment_states)) +
                       size_t(groups_per_cta) * group_smem_words(G, CPL)) * sizeof(uint32_t) +
                      (BULK ? 16 + 16 * (kThreads / 32) : 0);  // bulk path: two mbarriers per warp
  auto kernel = wildfire_step_kernel<G, CPL, MODE, INJECTED, BULK>;
  if (smem > 48 * 1024) {
    if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)) != cudaSuccess)
      return check_launch("wildfire smem attribute");
  }
  const int grid = persistent_grid((B + groups_per_cta - 1) / groups_per_cta, resident_ctas(kernel, kThreads, smem));
  kernel<<<grid, kThreads, smem, stream>>>(p, io, derived, B);
  return check_launch("wildfire_step_kernel");
}

template <int G, int CPL, bool BULK>
int launch_mode(const FrzWildfireParams& p, const FrzWildfireBuffers& io, int B, int mode, cudaStream_t stream) {
  if (mode != kStep) return launch_variant<G, CPL, kRefresh, false, BULK>(p, io, B, stream);
  if (io.field_uniforms != nullptr || io.agent_uniforms != nullptr) return launch_variant<G, CPL, kStep, true, BULK>(p, io, B, stream);
  return launch_variant<G, CPL, kStep, false, BULK>(p, io, B, stream);
}

template <int G, int CPL>
int launch_step(const FrzWildfireParams& p, const FrzWildfireBuffers& io, int B, int mode, cudaStream_t stream) {
  if constexpr (cells_in_smem(G, CPL)) {
    // the state planes move with bulk async copies when every row is a 16-byte multiple at a 16-byte aligned address
    // (same results either way: the Philox layout only depends on the geometry)
    const uintptr_t bases = reinterpret_cast<uintptr_t>(io.fires) | reinterpret_cast<uintptr_t>(io.intensity) |
                            reinterpret_cast<uintptr_t>(io.fuel);
    if ((p.height * p.width) % 4 == 0 && bases % 16 == 0) return launch_mode<G, CPL, true>(p, io, B, mode, stream);
  }
  return launch_mode<G, CPL, false>(p, io, B, mode, stream);
}

int dispatch(const FrzWildfireParams* p, const FrzWildfireBuffers* io, int B, int mode, void* stream) {
  if (p == nullptr || io == nullptr || io->control == nullptr || io->fires == nullptr || io->cell_agents == nullptr ||
      io->range_mask == nullptr) {
    set_error("frz_wildfire: NULL params / buffers");
    return FRZ_ERR_NULL;
  }
  Geometry g;
  if (B <= 0 || !pick_geometry(*p, &g) || p->num_equipment_states < 1 || p->num_equipment_states > FRZ_MAX_EQUIPMENT ||
      p->num_capacities < 1 || p->num_capacities > FRZ_MAX_CAPACITIES || io->mask_stride % 4 != 0 ||
      io->mask_stride < p->height * p->width) {
    set_error("frz_wildfire: unsupported shape B=%d H=%d W=%d A=%d E=%d", B, p->height, p->width, p->num_agents,
              p->num_equipment_states);
    return FRZ_ERR_SHAPE;
  }
  {  // the kernels index every array with 32-bit element indices
    const uint64_t cells = uint64_t(B) * uint64_t(p->height * p->width);
    const uint64_t mask_words = uint64_t(B) * uint64_t(p->num_agents) * uint64_t(io->mask_stride / 4);
    if (cells >= (1ull << 32) || mask_words >= (1ull << 32)) {
      set_error("frz_wildfire: B=%d is too large for one launch (arrays exceed 2^32 elements); shard the batch", B);
      return FRZ_ERR_SHAPE;
    }
  }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  // small grids: one thread per environment once the batch fills the GPU with tiles (same random streams either way)
  if (small_grid(*p) && g.group == 8 &&
      ((p->flags & FRZ_WF_KERNEL_TILES) ||
       (!(p->flags & FRZ_WF_KERNEL_GROUPS) && tiny_grid(*p) && B >= kSmallTileMinimumBatch))) {
    return p->num_agents <= 4 ? launch_tiles_mode<4>(*p, *io, B, mode, g, s) : launch_tiles_mode<8>(*p, *io, B, mode, g, s);
  }
  if (g.group == 8) {
    switch (g.cells_per_lane) {
      case 1: return launch_step<8, 1>(*p, *io, B, mode, s);
      case 2: return launch_step<8, 2>(*p, *io, B, mode, s);
      case 3: return launch_step<8, 3>(*p, *io, B, mode, s);
      default: return launch_step<8, 4>(*p, *io, B, mode, s);
    }
  }
  if (g.group == 16) {
    switch (g.cells_per_lane) {
      case 1: return launch_step<16, 1>(*p, *io, B, mode, s);
      case 2: return launch_step<16, 2>(*p, *io, B, mode, s);
      case 3: return launch_step<16, 3>(*p, *io, B, mode, s);
      case 4: return launch_step<16, 4>(*p, *io, B, mode, s);
      case 5: return launch_step<16, 5>(*p, *io, B, mode, s);
      case 6: return launch_step<16, 6>(*p, *io, B, mode, s);
      case 7: return launch_step<16, 7>(*p, *io, B, mode, s);
      default: return launch_step<16, 8>(*p, *io, B, mode, s);
    }
  }
  switch (g.cells_per_lane) {
    case 1: return launch_step<32, 1>(*p, *io, B, mode, s);
    case 2: return launch_step<32, 2>(*p, *io, B, mode, s);
    case 4: return launch_step<32, 4>(*p, *io, B, mode, s);
    default: return launch_step<32, 8>(*p, *io, B, mode, s);
  }
}

}  // namespace
}  // namespace frz

extern "C" {

int frz_wildfire_step(const FrzWildfireParams* params, const FrzWildfireBuffers* io, int32_t parallel_envs, void* stream) {
  if (io != nullptr && io->actions == nullptr) {
    frz::set_error("frz_wildfire_step: actions is NULL");
    return FRZ_ERR_NULL;
  }
  return frz::dispatch(params, io, parallel_envs, frz::kStep, stream);
}

int frz_wildfire_step_host(const FrzWildfireParams* params, const FrzWildfireBuffers* io, int32_t parallel_envs,
                           const FrzHostStep* host, void* stream) {
  if (params == nullptr || io == nullptr || io->actions == nullptr || io->control == nullptr || io->rewards == nullptr) {
    frz::set_error("frz_wildfire_step_host: NULL params / buffers");
    return FRZ_ERR_NULL;
  }
  if (io->field_uniforms != nullptr || io->agent_uniforms != nullptr) {
    frz::set_error("frz_wildfire_step_host: injected uniforms are not supported on the pipelined host path");
    return FRZ_ERR_UNSUPPORTED;
  }
  const size_t HW = size_t(params->height) * params->width, A = size_t(params->num_agents);
  const frz::HostArrays arrays{io->actions, io->rewards, io->terminated, io->truncated, io->control, params->num_agents,
                                 params, sizeof(FrzWildfireParams), io, sizeof(FrzWildfireBuffers)};
  return frz::run_host_pipeline(
      "frz_wildfire_step_host", host, arrays, parallel_envs, static_cast<cudaStream_t>(stream),
      [&](int first, int count, FrzControl* control, cudaStream_t slice_stream) {
        FrzWildfireParams p = *params;
        p.env_offset += first;  // the Philox counters are keyed by the global environment index
        FrzWildfireBuffers slice = *io;
        const size_t e = size_t(first);
        slice.fires += e * HW;
        slice.intensity += e * HW;
        slice.fuel += e * HW;
        slice.suppressants += e * A;
        slice.capacity += e * A;
        slice.equipment += e * A;
        slice.actions += e * A * 2;
        slice.rewards += e * A;
        slice.cumulative_rewards += e * A;
        slice.terminated += e;
        slice.truncated += e;
        slice.num_moves += e;
        slice.num_burnouts += e;
        slice.burnouts += e;
        slice.putouts += e;
        slice.env_task_count += e;
        slice.agent_task_count += e * A;
        slice.action_mask += e * A * size_t(io->mask_stride);
        slice.self_obs += e * A * 4;
        slice.task_obs += e * HW * 4;
        slice.control = control;
        return frz::dispatch(&p, &slice, count, frz::kStep, slice_stream);
      });
}

int frz_wildfire_tile_random_layout(const FrzWildfireParams* params, uint32_t* streams, int8_t* destinations) {
  frz::Geometry g;
  if (params == nullptr || streams == nullptr || destinations == nullptr) {
    frz::set_error("frz_wildfire_tile_random_layout: NULL argument");
    return -FRZ_ERR_NULL;
  }
  if (!frz::pick_geometry(*params, &g) || !frz::small_grid(*params) || g.group != 8) {
    frz::set_error("frz_wildfire_tile_random_layout: H=%d W=%d A=%d is not a small grid", params->height, params->width,
                   params->num_agents);
    return -FRZ_ERR_SHAPE;
  }
  FrzWildfireParams folded;
  frz::Derived derived;
  frz::fold_configuration(*params, g.group, g.cells_per_lane, &folded, &derived);
  const frz::SmallRandomLayout layout = frz::small_random_layout(
      params->height * params->width, params->num_agents, g.group, g.cells_per_lane, derived.spare_lanes_feed_agents != 0);
  for (int i = 0; i < layout.calls; ++i) {
    streams[i] = layout.stream[i];
    for (int j = 0; j < 4; ++j) destinations[4 * i + j] = layout.dest[i][j];
  }
  return layout.calls;
}

int frz_wildfire_refresh(const FrzWildfireParams* params, const FrzWildfireBuffers* io, int32_t parallel_envs,
                         void* stream) {
  return frz::dispatch(params, io, parallel_envs, frz::kRefresh, stream);
}

int frz_wildfire_reset(const FrzWildfireParams* params, const FrzWildfireBuffers* io, int32_t parallel_envs,
                       const uint8_t* env_mask, void* stream) {
  if (params == nullptr || io == nullptr || io->init_fires == nullptr || io->control == nullptr) {
    frz::set_error("frz_wildfire_reset: NULL params / buffers");
    return FRZ_ERR_NULL;
  }
  if (parallel_envs <= 0) {
    frz::set_error("frz_wildfire_reset: parallel_envs=%d", parallel_envs);
    return FRZ_ERR_SHAPE;
  }
  const int HW = params->height * params->width;
  const size_t total = size_t(parallel_envs) * (HW > params->num_agents ? HW : params->num_agents);
  const int grid = frz::persistent_grid(int((total + 255) / 256 < (1u << 20) ? (total + 255) / 256 : (1u << 20)), 16);
  frz::wildfire_restore_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(*params, *io, parallel_envs, env_mask);
  const int status = frz::check_launch("wildfire_restore_kernel");
  if (status != FRZ_OK) return status;
  return frz::dispatch(params, io, parallel_envs, frz::kRefresh, stream);
}

int frz_wildfire_sample_actions(const FrzWildfireParams* params, const FrzWildfireBuffers* io, int32_t parallel_envs,
                                uint64_t sampler_seed, void* stream) {
  if (params == nullptr || io == nullptr || io->actions == nullptr || io->control == nullptr) {
    frz::set_error("frz_wildfire_sample_actions: NULL params / buffers");
    return FRZ_ERR_NULL;
  }
  const int total = parallel_envs * params->num_agents;
  const int grid = frz::persistent_grid((total + 255) / 256, 8);
  frz::wildfire_sample_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(*params, *io, parallel_envs, sampler_seed);
  return frz::check_launch("wildfire_sample_kernel");
}

}  // extern "C"
