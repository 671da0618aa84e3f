// Wildfire step for SMALL grids (at most 32 cells, at most 8 agents) and large batches: one THREAD per environment, a
// one-warp CTA per tile of 32 consecutive environments.  Included by frz_wildfire.cu (inside frz::<anonymous>).
//
// On a 3x3 grid the group kernel (8 lanes per environment) spends most of its instructions on ballots, shuffles and
// lanes without a cell: an environment is ~600 scalar operations.  Here a thread walks its environment's cells and
// agents serially -- cell sets are bit masks in a register -- so a warp instruction serves 32 environments instead
// of 4.  Every [B, *] array is environment-major, so a tile of each array is ONE contiguous byte range: the tile's
// state moves global -> shared -> global with one bulk async copy per array (cp.async.bulk, the TMA unit; completion on
// the warp's mbarrier), a thread then reads and writes its environment's rows in shared memory (row stride = row
// size: odd strides such as 9 cells are conflict-free).  The variable-length outputs (live task-observation rows, the
// action-mask words that can differ from their padding) are stored directly, in whole 16-byte / 4-byte pieces.
// (Measured alternative, not kept: staging only the three cell planes and letting every thread read / write its
// per-agent rows directly -- 6 KB of shared memory per tile instead of 12 -- was 27 % slower on the 3x3 grid.)
//
// Randomness: the SAME Philox calls and word assignment as the group kernel uses for this grid (a host-built table
// says which word of which call feeds which cell / agent event), so a trajectory does not depend on which of the two
// kernels the batch size selects -- in particular not on how a batch is sharded over GPUs.
#pragma once

constexpr int kSmallMaxCells = 32;
constexpr int kSmallMaxCalls = 24;  // 8 lanes x 2 calls of the group layout + one call per agent

// Which Philox call feeds what: call i uses stream[i] as its third counter word; its word j goes to slot dest[i][j] of
// the environment's random scratch (-1 = unused): [0, HW) increase / decrease of cell c, [HW, 2 HW) spread of cell c,
// 2 HW + 4 a + j = word j of agent a.
struct SmallRandomLayout {
  int32_t calls;
  uint32_t stream[kSmallMaxCalls];
  int8_t dest[kSmallMaxCalls][4];
};

// the same table the group kernel implements implicitly (see its "randomness" section and fold_configuration)
inline SmallRandomLayout small_random_layout(int HW, int A, int group, int cells_per_lane, bool spare_lanes_feed_agents) {
  SmallRandomLayout layout = {};
  const int calls = (2 * cells_per_lane + 3) / 4;  // per lane of the group layout (never split for 8-lane groups)
  const auto slot_of = [&](int sub, int word) -> int8_t* {  // word `word` of lane `sub`
    const int call = (word / 4) * group + sub;
    return &layout.dest[call][word % 4];
  };
  layout.calls = calls * group;
  for (int i = 0; i < layout.calls; ++i) {
    layout.stream[i] = uint32_t(i);
    for (int j = 0; j < 4; ++j) layout.dest[i][j] = -1;
  }
  for (int c = 0; c < HW; ++c) {
    const int i = c / group, sub = c % group;
    *slot_of(sub, 2 * i) = int8_t(c);
    *slot_of(sub, 2 * i + 1) = int8_t(HW + c);
  }
  const int spare_own = 4 * calls - 2 * cells_per_lane;
  for (int a = 0; a < A; ++a) {
    if (cells_per_lane > 1 && spare_lanes_feed_agents) {
      const int first = (group - 1 - a) & (group - 1), second = (group - 1 - A - a) & (group - 1);
      const int last = cells_per_lane - 1;
      if (spare_own == 2) {
        *slot_of(a, 2 * cells_per_lane) = int8_t(2 * HW + 4 * a);
        *slot_of(a, 2 * cells_per_lane + 1) = int8_t(2 * HW + 4 * a + 1);
        *slot_of(first, 2 * last) = int8_t(2 * HW + 4 * a + 2);
        *slot_of(first, 2 * last + 1) = int8_t(2 * HW + 4 * a + 3);
      } else {
        *slot_of(first, 2 * last) = int8_t(2 * HW + 4 * a);
        *slot_of(first, 2 * last + 1) = int8_t(2 * HW + 4 * a + 1);
        *slot_of(second, 2 * last) = int8_t(2 * HW + 4 * a + 2);
        *slot_of(second, 2 * last + 1) = int8_t(2 * HW + 4 * a + 3);
      }
    } else {
      const int call = layout.calls++;
      layout.stream[call] = 0x80000000u | uint32_t(a);
      for (int j = 0; j < 4; ++j) layout.dest[call][j] = int8_t(2 * HW + 4 * a + j);
    }
  }
  return layout;
}

// shared memory of a tile, in 32-bit words: the staged arrays (each a multiple of four words), then per-thread scratch
struct SmallTile {
  int fires, intensity, fuel, suppressants, capacity, equipment, cumulative, num_moves, num_burnouts, terminated;  // in + out
  int actions;                                                                                                   // in
  int rewards, truncated, burnouts, putouts, env_task_count, agent_task_count;                                    // out
  int attack, random;  // scratch: attack power per cell, random words
  int total;
};

__host__ __device__ inline SmallTile small_tile(int HW, int A) {
  SmallTile t;
  int at = 0;
  const auto take = [&at](int words) {
    const int offset = at;
    at += (words + 3) & ~3;
    return offset;
  };
  t.fires = take(32 * HW), t.intensity = take(32 * HW), t.fuel = take(32 * HW);
  t.suppressants = take(32 * A), t.capacity = take(32 * A), t.equipment = take(32 * A), t.cumulative = take(32 * A);
  t.num_moves = take(32), t.num_burnouts = take(32), t.terminated = take(8);
  t.actions = take(64 * A);
  t.rewards = take(32 * A), t.truncated = take(8), t.burnouts = take(32), t.putouts = take(32), t.env_task_count = take(32);
  t.agent_task_count = take(32 * A);
  t.attack = take(32 * HW), t.random = take(32 * (2 * HW + 4 * A));
  t.total = at;
  return t;
}

template <int MAXA, int MODE, bool INJECTED>
__global__ void __launch_bounds__(32)
wildfire_tile_kernel(const __grid_constant__ FrzWildfireParams p, const __grid_constant__ FrzWildfireBuffers io,
                     const __grid_constant__ Derived derived, const __grid_constant__ SmallRandomLayout random_layout,
                     const int B) {
  extern __shared__ __align__(16) uint32_t smem[];
  __shared__ __align__(8) uint64_t barrier_storage;
  const int lane = threadIdx.x;
  const int W = p.width, HW = derived.cells, A = p.num_agents, E = p.num_equipment_states;
  const uint32_t flags = p.flags;
  const bool show_bad = flags & FRZ_WF_SHOW_BAD_ACTIONS, use_fuel = flags & FRZ_WF_FIRE_FUEL;
  const bool localize = flags & FRZ_WF_LOCALIZE_PUTOUTS, scaled = flags & FRZ_WF_BURNOUT_SCALED;
  const SmallTile T = small_tile(HW, A);
  const uint32_t smem_s = shared_address(smem), barrier = shared_address(&barrier_storage);
  const int table_words = io.mask_words, mask_words_row = io.mask_stride >> 2;
  if (lane == 0) mbarrier_init(barrier, 1);
  __syncwarp();
  uint32_t parity = 0u;

  FrzControl* const control = io.control;
  const uint64_t step = control->step;
  const uint32_t alive_prev = control->alive;
  const uint32_t agents_with_tasks = control->agents_with_tasks;
  const Philox philox(control->seed);
  const bool skip = (MODE == kStep) && ((alive_prev & 3u) != 3u);  // utils/env.py:212
  unsigned alive_bits = 0, faults = 0, agent_bits = 0;

  // this thread's rows of the staged arrays
  int* const fires = reinterpret_cast<int*>(smem) + T.fires + lane * HW;
  int* const intensity = reinterpret_cast<int*>(smem) + T.intensity + lane * HW;
  int* const fuel = reinterpret_cast<int*>(smem) + T.fuel + lane * HW;
  float* const suppressants = reinterpret_cast<float*>(smem) + T.suppressants + lane * A;
  float* const capacity = reinterpret_cast<float*>(smem) + T.capacity + lane * A;
  int* const equipment = reinterpret_cast<int*>(smem) + T.equipment + lane * A;
  float* const cumulative = reinterpret_cast<float*>(smem) + T.cumulative + lane * A;
  const int2* const actions = reinterpret_cast<const int2*>(smem + T.actions) + lane * A;
  float* const rewards = reinterpret_cast<float*>(smem) + T.rewards + lane * A;
  int* const agent_task_count = reinterpret_cast<int*>(smem) + T.agent_task_count + lane * A;
  float* const attack = reinterpret_cast<float*>(smem) + T.attack + lane * HW;
  uint32_t* const random = smem + T.random + lane * (2 * HW + 4 * A);
  uint8_t* const terminated_tile = reinterpret_cast<uint8_t*>(smem + T.terminated);
  uint8_t* const truncated_tile = reinterpret_cast<uint8_t*>(smem + T.truncated);

  if (!skip) {
    for (int tile0 = blockIdx.x * 32; tile0 < B; tile0 += gridDim.x * 32) {
      const int env = tile0 + lane;
      const bool valid = env < B;
      const bool full = tile0 + 32 <= B;
      const size_t cells_at = size_t(tile0) * size_t(HW), agents_at = size_t(tile0) * size_t(A);

      // ------------------------------------------------------------------ stage in
      if (full) {
        if (elect_one()) {
          const uint32_t cell_bytes = 128u * uint32_t(HW), agent_bytes = 128u * uint32_t(A);
          mbarrier_expect_bytes(barrier, 3u * cell_bytes + 3u * agent_bytes +
                                             (MODE == kStep ? agent_bytes + 2u * agent_bytes + 128u + 128u + 32u : 0u));
          bulk_load(smem_s + 4u * T.fires, io.fires + cells_at, cell_bytes, barrier);
          bulk_load(smem_s + 4u * T.intensity, io.intensity + cells_at, cell_bytes, barrier);
          bulk_load(smem_s + 4u * T.fuel, io.fuel + cells_at, cell_bytes, barrier);
          bulk_load(smem_s + 4u * T.suppressants, io.suppressants + agents_at, agent_bytes, barrier);
          bulk_load(smem_s + 4u * T.capacity, io.capacity + agents_at, agent_bytes, barrier);
          bulk_load(smem_s + 4u * T.equipment, io.equipment + agents_at, agent_bytes, barrier);
          if (MODE == kStep) {
            bulk_load(smem_s + 4u * T.cumulative, io.cumulative_rewards + agents_at, agent_bytes, barrier);
            bulk_load(smem_s + 4u * T.actions, io.actions + 2 * agents_at, 2u * agent_bytes, barrier);
            bulk_load(smem_s + 4u * T.num_moves, io.num_moves + tile0, 128u, barrier);
            bulk_load(smem_s + 4u * T.num_burnouts, io.num_burnouts + tile0, 128u, barrier);
            bulk_load(smem_s + 4u * T.terminated, io.terminated + tile0, 32u, barrier);
          }
        }
        mbarrier_wait(barrier, parity);
        parity ^= 1u;
      } else if (valid) {  // the partial tile at the end of the batch: every thread fetches its own rows
        for (int c = 0; c < HW; ++c) {
          fires[c] = io.fires[cells_at + size_t(lane) * HW + c];
          intensity[c] = io.intensity[cells_at + size_t(lane) * HW + c];
          fuel[c] = io.fuel[cells_at + size_t(lane) * HW + c];
        }
        for (int a = 0; a < A; ++a) {
          suppressants[a] = io.suppressants[agents_at + size_t(lane) * A + a];
          capacity[a] = io.capacity[agents_at + size_t(lane) * A + a];
          equipment[a] = io.equipment[agents_at + size_t(lane) * A + a];
          if (MODE == kStep) {
            cumulative[a] = io.cumulative_rewards[agents_at + size_t(lane) * A + a];
            reinterpret_cast<int2*>(smem + T.actions)[lane * A + a] =
                reinterpret_cast<const int2*>(io.actions)[agents_at + size_t(lane) * A + a];
          }
        }
        if (MODE == kStep) {
          smem[T.num_moves + lane] = uint32_t(io.num_moves[env]);
          smem[T.num_burnouts + lane] = uint32_t(io.num_burnouts[env]);
          terminated_tile[lane] = io.terminated[env];
        }
      }

      uint32_t lit = 0u;
      int n_before = 0, n_lit = 0;
      if (valid) {
        for (int c = 0; c < HW; ++c) lit |= uint32_t(fires[c] > 0) << c;
        n_before = MODE == kStep ? __popc(lit) : HW;  // refresh / reset: (re)write every row

        if (MODE == kStep) {
          const int e = env;
          // ---------------------------------------------------------------- randomness
          // the group layout's Philox calls (see the header of this file); parity mode reads the injected uniforms
          // at their point of use instead
          const bool inject_agent = INJECTED && io.agent_uniforms != nullptr;
          const bool inject_field = INJECTED && io.field_uniforms != nullptr;
          if (!inject_agent || !inject_field) {
            const uint32_t env_lo = uint32_t(p.env_offset + e), env_hi = uint32_t(uint64_t(p.env_offset + e) >> 32);
            const uint32_t step_lo = uint32_t(step), step_hi = uint32_t(step >> 32) ^ env_hi;
            for (int i = 0; i < random_layout.calls; ++i) {
              const uint4 r = philox(env_lo, step_lo, random_layout.stream[i], step_hi);
              const int d0 = random_layout.dest[i][0], d1 = random_layout.dest[i][1], d2 = random_layout.dest[i][2],
                        d3 = random_layout.dest[i][3];
              if (d0 >= 0) random[d0] = r.x;
              if (d1 >= 0) random[d1] = r.y;
              if (d2 >= 0) random[d2] = r.z;
              if (d3 >= 0) random[d3] = r.w;
            }
          }
          const size_t plane = size_t(B) * HW;
          // field event 0 increase, 1 decrease (one shared word), 2 spread; as the 24 random bits and as a uniform
          const auto field_bits = [&](int c, int event) { return random[event == 2 ? HW + c : c] >> 8; };
          const auto field_uniform = [&](int c, int event) -> float {
            if (inject_field) return io.field_uniforms[event * plane + size_t(e) * HW + c];
            return float(field_bits(c, event)) * 5.9604644775390625e-08f;
          };
          // agent event 0 suppressant decrease and 2 refill (one shared word), 1 equipment, 3 capacity pick, 4 tank switch
          const auto agent_word = [](int event) { return event == 0 || event == 2 ? 0 : (event == 1 ? 1 : event - 1); };
          const auto happens = [&](int a, int event, float p_event, uint32_t t_event) -> bool {
            if (inject_agent) return io.agent_uniforms[(size_t(event) * B + e) * A + a] < p_event;
            return (random[2 * HW + 4 * a + agent_word(event)] >> 8) < t_event;
          };

          // ---------------------------------------------------------------- action decode (wildfire.py:412-486)
          for (int c = 0; c < HW; ++c) attack[c] = 0.f;
          uint32_t users = 0u, refills = 0u, bads = 0u;
          int target[MAXA];
#pragma unroll
          for (int a = 0; a < MAXA; ++a) {
            target[a] = -1;
            if (a < A) {
              const int2 act = actions[a];
              const int equip = min(max(equipment[a], 0), E - 1);
              const bool refill = act.y == -1;  // wildfire.py:431
              refills |= uint32_t(refill) << a;
              // an agent without a single task in ANY environment is skipped by the reference's decode loop
              // (wildfire.py:434): no attack, no bad-action penalty -- only its refill flag is recorded
              if (!refill && ((agents_with_tasks >> a) & 1u)) {
                const uint32_t reach = io.range_mask[(a * E + equip) * table_words];
                const uint32_t available = suppressants[a] > 0.f ? (lit & reach) : 0u;
                const uint32_t choices = show_bad ? lit : available;
                if (act.x >= 0 && act.x < __popc(choices)) {
                  const int found = select_bit(choices, act.x);
                  if (show_bad && !((available >> found) & 1u)) bads |= 1u << a;  // wildfire.py:464-477
                  else target[a] = found;
                } else {
                  faults |= FRZ_FAULT_BAD_TASK_INDEX;
                }
              }
              if (target[a] >= 0) {  // wildfire.py:455-470: powers add up in agent order
                users |= 1u << a;
                attack[target[a]] = __fadd_rn(attack[target[a]], __fadd_rn(p.agent_power[a], p.equipment_power_bonus[equip]));
              }
            }
          }
          const int moves = int(smem[T.num_moves + lane]) + 1;
          int total_burnouts = int(smem[T.num_burnouts + lane]);
          const bool was_terminated = terminated_tile[lane] != 0;

          // ---------------------------------------------------------------- agent transitions (wildfire.py:488-514)
          // (the host folded the StochasticConfiguration switches into the thresholds: 2 = always, -1 = never)
#pragma unroll
          for (int a = 0; a < MAXA; ++a) {
            if (a < A) {
              float supp = suppressants[a], cap = capacity[a];
              int equip = min(max(equipment[a], 0), E - 1);
              // suppressant_decrease.py:34-63
              const bool decrease = ((users >> a) & 1u) && happens(a, 0, p.p_suppressant_decrease, derived.t_suppressant_decrease);
              supp = fmaxf(decrease ? __fadd_rn(supp, -1.f) : supp, 0.f);
              // equipment.py:42-77 -- masks from the pre-update state, one uniform for all three tests
              {
                const bool pristine = equip == E - 1, damaged = equip == 0;
                const bool wearable = pristine || !damaged;
                const bool repairs = damaged && happens(a, 1, p.p_repair, derived.t_repair);
                const bool critical = pristine && happens(a, 1, p.p_critical, derived.t_critical);
                const bool degrades = wearable && happens(a, 1, p.p_degrade, derived.t_degrade) && !critical;
                if (repairs) equip = E - 1;
                if (critical) equip = 0;
                if (degrades) equip -= 1;
              }
              // suppressant_refill.py:43-74 -- bonus of the equipment state AFTER its transition
              const bool increased = ((refills >> a) & 1u) && happens(a, 2, p.p_refill, derived.t_refill);
              if (increased) {
                supp = __fadd_rn(cap, p.equipment_capacity_bonus[max(equip, 0)]);
                // capacity.py:39-66 -- bucketize(right=False): first i with r <= cum[i] == entries below r
                int pick = 0;
#pragma unroll
                for (int i = 0; i < FRZ_MAX_CAPACITIES; ++i) {
                  if (inject_agent) pick += io.agent_uniforms[(size_t(3) * B + e) * A + a] > p.capacity_cum[i] ? 1 : 0;
                  else pick += int(random[2 * HW + 4 * a + 2] >> 8) > derived.t_capacity_cum[i] ? 1 : 0;
                }
                pick = min(pick, p.num_capacities - 1);
                const float extra = __fadd_rn(supp, -cap);
                if (happens(a, 4, p.p_tank_switch, derived.t_tank_switch)) {
                  cap = p.capacity_value[pick];
                  supp = __fadd_rn(cap, extra);
                }
              }
              suppressants[a] = supp, capacity[a] = cap, equipment[a] = equip;
            }
          }

          // ---------------------------------------------------------------- fire increase + decrease per cell
          uint32_t burned = 0u, put_out = 0u, burning_after = 0u;
          for (int c = 0; c < HW; ++c) {
            int f = fires[c], it = intensity[c];
            // fire_increase.py:43-95
            const bool burning = f > 0 && it > 0;
            const float diff = __fadd_rn(f > 0 ? float(f) : 0.f, -attack[c]);
            const bool unmet = burning && diff > 0.f;
            bool grow;
            if (inject_field) grow = unmet && field_uniform(c, 0) < (it == derived.almost_state ? p.p_burnout : p.p_increase);
            else grow = unmet && field_bits(c, 0) < (it == derived.almost_state ? derived.t_burnout : derived.t_increase);
            it += grow ? 1 : 0;
            const bool burns_out = grow && it >= derived.burned_state;
            // fire_decrease.py:36-80 on the post-increase state; product and sum rounded separately
            const bool met = burning && !burns_out && diff <= 0.f;
            const float prob_down = fminf(fmaxf(__fadd_rn(p.p_decrease, __fmul_rn(-diff, p.decrease_bonus)), 0.f), 1.f);
            const bool shrink = met && field_uniform(c, 1) < prob_down;
            it -= shrink ? 1 : 0;
            const bool put = shrink && it <= 0;
            if (burns_out || put) {
              // burn-out clamps the fuel (fire_increase.py:90), putting out does not (fire_decrease.py:75)
              const int left = fuel[c] - 1;
              fuel[c] = burns_out ? max(left, 0) : left;
              f = -f;
            }
            fires[c] = f, intensity[c] = it;
            burned |= uint32_t(burns_out) << c;
            put_out |= uint32_t(put) << c;
            burning_after |= uint32_t(burning && !burns_out && !put) << c;
          }

          // ---------------------------------------------------------------- fire spread (fire_spreads.py:33-59)
          {
            // burning neighbours of cell c as bit c: N = cell c - W, W = c - 1, E = c + 1, S = c + W
            const uint32_t north = W < 32 ? burning_after << W : 0u, south = W < 32 ? burning_after >> W : 0u;
            const uint32_t west = (burning_after << 1) & derived.west_ok[0], east = (burning_after >> 1) & derived.east_ok[0];
            lit = 0u;
            for (int c = 0; c < HW; ++c) {
              int f = fires[c];
              const uint32_t bit = 1u << c;
              if (f < 0 && intensity[c] == 0 && (!use_fuel || fuel[c] > 0)) {
                // the conv sum in the reference's accumulation order N, W, E, S, starting from zero
                float prob = 0.f;
                if (north & bit) prob = p.spread_lut[1];
                if (west & bit) prob = __fadd_rn(prob, p.spread_lut[2]);
                if (east & bit) prob = __fadd_rn(prob, p.spread_lut[4]);
                if (south & bit) prob = __fadd_rn(prob, p.spread_lut[8]);
                prob = __fadd_rn(prob, p.p_random_ignition);
                if (field_uniform(c, 2) < prob) {
                  f = -f;
                  fires[c] = f;
                  intensity[c] = io.cell_ignition[c];
                }
              }
              lit |= uint32_t(f > 0) << c;
            }
          }

          // ---------------------------------------------------------------- rewards + termination (wildfire.py:534-582)
          const int n_burned = __popc(burned), n_putout = __popc(put_out);
          float put_total = 0.f, burn_total = 0.f;
          if (!localize)
            for (uint32_t m = put_out; m != 0u; m &= m - 1u) put_total += io.cell_reward[__ffs(int(m)) - 1];
          if (scaled)
            for (uint32_t m = burned; m != 0u; m &= m - 1u) burn_total += io.cell_reward[__ffs(int(m)) - 1];
          const float penalty_total = scaled ? -burn_total : __fmul_rn(p.burnout_penalty, float(n_burned));
          bool dead = lit == 0u;
          if (use_fuel && dead) {
            int fuel_left = 0;
            for (int c = 0; c < HW; ++c) fuel_left += fuel[c];
            dead = fuel_left <= 0;
          }
          if (dead) {  // wildfire.py:570
            for (int c = 0; c < HW; ++c) fires[c] = 0;
            lit = 0u;
          }
          const bool newly = !was_terminated && dead;
          const bool terminated = was_terminated || dead;
          float bonus = 0.f;
          if (newly) {
            const float penalty = __fmul_rn(p.termination_kappa, logf(__fadd_rn(float(total_burnouts), 1.f)));
            bonus = fmaxf(__fadd_rn(p.termination_reward, -penalty), 0.f);
          }
#pragma unroll
          for (int a = 0; a < MAXA; ++a) {
            if (a < A) {
              float reward = ((bads >> a) & 1u) ? p.bad_attack_penalty : 0.f;
              float gain = put_total;
              if (localize) gain = (target[a] >= 0 && ((put_out >> target[a]) & 1u)) ? io.cell_reward[target[a]] : 0.f;
              reward = __fadd_rn(reward, __fadd_rn(gain, penalty_total));
              if (newly) reward = __fadd_rn(reward, bonus);
              rewards[a] = reward;
              cumulative[a] = __fadd_rn(cumulative[a], reward);
            }
          }
          total_burnouts += n_burned;
          const bool truncated = moves >= p.max_steps;  // utils/env.py:228-235
          alive_bits |= (terminated ? 0u : 1u) | (truncated ? 0u : 2u);
          smem[T.num_moves + lane] = uint32_t(moves);
          smem[T.num_burnouts + lane] = uint32_t(total_burnouts);
          smem[T.burnouts + lane] = uint32_t(n_burned);
          smem[T.putouts + lane] = uint32_t(n_putout);
          terminated_tile[lane] = terminated;
          truncated_tile[lane] = truncated;
        } else {  // refresh: the done flags as a reset, a restore or a hand edit left them
          alive_bits |= (io.terminated[env] ? 0u : 1u) | (io.truncated[env] ? 0u : 2u);
        }

        // ------------------------------------------------------------------ update_actions / update_observations
        n_lit = __popc(lit);
        const int n_rows = max(n_lit, n_before);  // rows / mask bytes that may differ from their padding value
        smem[T.env_task_count + lane] = uint32_t(n_lit);
        // bit t of tasks[a] = agent a may fight env-local task t (the t-th lit cell in row-major order)
        uint32_t available[MAXA], tasks[MAXA];
#pragma unroll
        for (int a = 0; a < MAXA; ++a) {
          available[a] = tasks[a] = 0u;
          if (a < A) {
            const float supp = suppressants[a];
            const int equip = min(max(equipment[a], 0), E - 1);
            if (supp > 0.f) available[a] = lit & io.range_mask[(a * E + equip) * table_words];
            const int n_available = __popc(available[a]);
            agent_task_count[a] = n_available;
            if (n_available > 0) agent_bits |= 1u << a;
            reinterpret_cast<float4*>(io.self_obs)[size_t(env) * A + a] =
                make_float4(float(p.agent_y[a]), float(p.agent_x[a]), p.agent_power[a], supp);
          }
        }
        int4* const task_rows = reinterpret_cast<int4*>(io.task_obs) + size_t(env) * HW;
        {
          int t = 0;
          for (uint32_t m = lit; m != 0u; m &= m - 1u, ++t) {
            const int c = __ffs(int(m)) - 1;
            const int y = c / W;
            task_rows[t] = make_int4(y, c - y * W, fires[c], intensity[c]);
#pragma unroll
            for (int a = 0; a < MAXA; ++a) tasks[a] |= ((available[a] >> c) & 1u) << t;
          }
        }
        // tasks of the previous launch that no longer exist: their rows go back to padding
        for (int t = n_lit; t < n_before; ++t) task_rows[t] = make_int4(FRZ_PAD, FRZ_PAD, FRZ_PAD, FRZ_PAD);
        // action mask [A, mask_stride] bytes indexed by env-local task, four tasks per word (nibble x 0x204081 spreads
        // four bits over four bytes); words past the tasks of this and the previous launch are zero already
        const int quads = (n_rows + 3) >> 2;
        uint32_t* const mask_words = reinterpret_cast<uint32_t*>(io.action_mask) + size_t(env) * A * mask_words_row;
#pragma unroll
        for (int a = 0; a < MAXA; ++a) {
          if (a < A)
            for (int q = 0; q < quads; ++q)
              mask_words[a * mask_words_row + q] = (((tasks[a] >> (4 * q)) & 0xfu) * 0x00204081u) & 0x01010101u;
        }
      }

      // ------------------------------------------------------------------ stage out
      if (full) {
        fence_async_shared();
        __syncwarp();
        if (elect_one()) {
          const uint32_t cell_bytes = 128u * uint32_t(HW), agent_bytes = 128u * uint32_t(A);
          bulk_store(io.env_task_count + tile0, smem_s + 4u * T.env_task_count, 128u);
          bulk_store(io.agent_task_count + agents_at, smem_s + 4u * T.agent_task_count, agent_bytes);
          if (MODE == kStep) {
            bulk_store(io.fires + cells_at, smem_s + 4u * T.fires, cell_bytes);
            bulk_store(io.intensity + cells_at, smem_s + 4u * T.intensity, cell_bytes);
            bulk_store(io.fuel + cells_at, smem_s + 4u * T.fuel, cell_bytes);
            bulk_store(io.suppressants + agents_at, smem_s + 4u * T.suppressants, agent_bytes);
            bulk_store(io.capacity + agents_at, smem_s + 4u * T.capacity, agent_bytes);
            bulk_store(io.equipment + agents_at, smem_s + 4u * T.equipment, agent_bytes);
            bulk_store(io.cumulative_rewards + agents_at, smem_s + 4u * T.cumulative, agent_bytes);
            bulk_store(io.rewards + agents_at, smem_s + 4u * T.rewards, agent_bytes);
            bulk_store(io.num_moves + tile0, smem_s + 4u * T.num_moves, 128u);
            bulk_store(io.num_burnouts + tile0, smem_s + 4u * T.num_burnouts, 128u);
            bulk_store(io.burnouts + tile0, smem_s + 4u * T.burnouts, 128u);
            bulk_store(io.putouts + tile0, smem_s + 4u * T.putouts, 128u);
            bulk_store(io.terminated + tile0, smem_s + 4u * T.terminated, 32u);
            bulk_store(io.truncated + tile0, smem_s + 4u * T.truncated, 32u);
          }
        }
        bulk_commit();
        bulk_wait_read();  // the tile is loaded again right away
        __syncwarp();
      } else if (valid) {
        io.env_task_count[env] = n_lit;
        for (int a = 0; a < A; ++a) io.agent_task_count[agents_at + size_t(lane) * A + a] = agent_task_count[a];
        if (MODE == kStep) {
          for (int c = 0; c < HW; ++c) {
            io.fires[cells_at + size_t(lane) * HW + c] = fires[c];
            io.intensity[cells_at + size_t(lane) * HW + c] = intensity[c];
            io.fuel[cells_at + size_t(lane) * HW + c] = fuel[c];
          }
          for (int a = 0; a < A; ++a) {
            io.suppressants[agents_at + size_t(lane) * A + a] = suppressants[a];
            io.capacity[agents_at + size_t(lane) * A + a] = capacity[a];
            io.equipment[agents_at + size_t(lane) * A + a] = equipment[a];
            io.cumulative_rewards[agents_at + size_t(lane) * A + a] = cumulative[a];
            io.rewards[agents_at + size_t(lane) * A + a] = rewards[a];
          }
          io.num_moves[env] = int(smem[T.num_moves + lane]);
          io.num_burnouts[env] = int(smem[T.num_burnouts + lane]);
          io.burnouts[env] = int(smem[T.burnouts + lane]);
          io.putouts[env] = int(smem[T.putouts + lane]);
          io.terminated[env] = terminated_tile[lane];
          io.truncated[env] = truncated_tile[lane];
        }
      }
    }
  }
  finish_launch(control, alive_bits, faults, agent_bits,
                skip ? kPublishNothing : (MODE == kStep ? kPublishStep : kPublishRefresh));
}

// When the dispatcher picks the tiled kernel by itself: tiny grids (measured on B200: 3x3 / 3 agents at 524 288 envs
// 105 us against 188 us with groups of eight lanes; 5x6 / 6 agents at 262 144 envs 278 us against 159 us -- the serial
// walk over cells and agents grows with the grid while the group kernel's lanes fill up) from 49 152 environments up
// (below, a tile per warp leaves most of the GPU idle).  FRZ_WF_KERNEL_TILES forces it for any grid it can step.
constexpr int kSmallTileMinimumBatch = 49152;

inline bool small_grid(const FrzWildfireParams& p) { return p.height * p.width <= kSmallMaxCells && p.num_agents <= 8; }
inline bool tiny_grid(const FrzWildfireParams& p) { return p.height * p.width <= 16 && p.num_agents <= 4; }
