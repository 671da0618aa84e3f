// Fused rideshare environment step for sm_100a.
//
// One launch = for every environment: action decode -> movement -> passenger state (accept conflicts, picks) ->
// passenger exit -> passenger entry -> rewards -> num_moves / truncation -> reward accumulation -> observations ->
// task lists.  Replaces, with identical results, the reference's envs/rideshare/env/rideshare.py:249-467,
// env/transitions/{movement,passenger_state,passenger_exit,passenger_entry}.py and utils/env.py:215-237.
//
// The reference keeps all passengers of all environments in one flat table [N_total, 11] sorted by environment and
// re-sorts / compacts it with `unique`, boolean-mask indexing and a stable `argsort` every step.  Here environment b
// owns rows passengers[b, 0:count[b]] (same relative order).
//
// Two kernels with identical results; the batch size picks one (FRZ_RS_KERNEL_* force it):
//   * rideshare_tile_kernel (batches of 24 576 environments and more, tables with a multiple of four rows, at most
//     eight drivers): one THREAD per environment -- see the comment above that kernel;
//   * rideshare_step_kernel (everything else), described here.
//
// Mapping: a group of G lanes (8, 16 or 32, chosen from the table capacity and the number of drivers) owns one
// environment, so a warp steps 4, 2 or 1 environments at once.  The environment's rows are staged in shared memory
// (cp.async) for the whole step and edited in place; lane s of the group looks after rows s, s+G, ... (PPL of them)
// and driver s.  One table buffer per group: double buffering (prefetching the group's next environment) halved the
// resident warps and measured 8 % slower than letting twice as many warps cover the staging latency.  Task lists, conflict
// detection, compaction and the per-class "last row" reward quirk are ballots (cut to the group's lanes), match_any
// and popcounts on 64-bit row masks.
#include <algorithm>
#include <climits>
#include <math_constants.h>

#include <type_traits>

#include "frz_common.cuh"
#include "frz_host.cuh"

namespace frz {
namespace {

constexpr int kRsThreads = 128;
constexpr int kCols = FRZ_RS_PASSENGER_COLUMNS;
enum RsMode { kRsStep = 0, kRsRefresh = 1, kRsEntryRefresh = 2 };
enum Col { cBatch = 0, cY, cX, cDestY, cDestX, cFare, cState, cAssoc, cEntered, cAccepted, cPicked };
constexpr int kRemoved = -7;  // scratch value of the state column: the row left the table in this step

// stay, N, E, S, W, NW, NE, SE, SW (transitions/movement.py:27-45)
__constant__ int kDirY[9] = {0, -1, 0, 1, 0, -1, -1, 1, 1};
__constant__ int kDirX[9] = {0, 0, 1, 0, -1, -1, 1, 1, -1};

__device__ __forceinline__ int select_bit64(uint64_t mask, int k) {
  const uint32_t lo = uint32_t(mask);
  const int in_lo = __popc(lo);
  return k < in_lo ? select_bit(lo, k) : 32 + select_bit(uint32_t(mask >> 32), k - in_lo);
}

// Squared Euclidean length.  The reference compares fp32 L2 norms of small integer vectors (movement.py:57-116,
// passenger_state.py:48-74); sqrt is strictly increasing on these exactly representable integers (neighbouring values are
// > 1e-3 apart, far above an fp32 ulp), so argmin, ties, "== 0" and "< 1e-6" give the same answers on the squares.
__device__ __forceinline__ int squared(int dy, int dx) { return dy * dy + dx * dx; }

// Row mask of one environment from per-lane predicates: bit (s + G * i) = predicate i of the group's lane s.  Every
// lane of the warp must call it (the ballots are warp-wide); each lane receives its own group's mask.  The group's
// byte / halfword of up to four ballots is packed with byte permutes (`pack` = the group's selector, see the kernel).
template <int G, int PPL>
__device__ __forceinline__ uint64_t group_rows(const bool (&pred)[PPL], int group_base, uint32_t pack) {
  uint32_t ballot[PPL];
#pragma unroll
  for (int i = 0; i < PPL; ++i) ballot[i] = __ballot_sync(kFullMask, pred[i]);
  if constexpr (G == 32) {
    return uint64_t(ballot[0]) | (PPL > 1 ? uint64_t(ballot[PPL - 1]) << 32 : 0);
  } else if constexpr (PPL == 1) {
    return uint64_t((ballot[0] >> group_base) & ((1u << G) - 1u));
  } else if constexpr (G == 16) {  // halfwords: rows (0, 1) -> low word, rows (2, 3) -> high word
    const uint32_t lo = __byte_perm(ballot[0], ballot[1], pack);
    const uint32_t hi = PPL > 2 ? __byte_perm(ballot[2], ballot[PPL - 1], pack) : 0u;
    return uint64_t(lo) | (uint64_t(hi) << 32);
  } else {  // G == 8, bytes: byte i of the result is the group's byte of ballot i
    static_assert(G == 8 && (PPL == 2 || PPL == 4), "8-lane groups hold 1, 2 or 4 rows per lane");
    const uint32_t lo = __byte_perm(ballot[0], ballot[1], pack);  // bytes 0, 1 valid
    if constexpr (PPL == 2) return uint64_t(lo & 0xffffu);
    const uint32_t hi = __byte_perm(ballot[2], ballot[PPL - 1], pack);
    return uint64_t(__byte_perm(lo, hi, 0x5410));
  }
}

template <int G>
__device__ __forceinline__ int group_min(int v) {
#pragma unroll
  for (int offset = G / 2; offset >= 1; offset >>= 1) v = min(v, __shfl_xor_sync(kFullMask, v, offset, G));
  return v;
}

// MODE is a template parameter so that the refresh / reset variants carry none of the step's code.
template <int G, int PPL, int MODE>
__global__ void __launch_bounds__(kRsThreads)
rideshare_step_kernel(const __grid_constant__ FrzRideshareParams p, const __grid_constant__ FrzRideshareBuffers io,
                      const int B, const uint8_t* __restrict__ entry_mask, const int batch_base) {
  static_assert(G * PPL <= 64, "row masks are 64 bits wide");
  extern __shared__ int smem[];
  constexpr int kGroupsPerWarp = 32 / G;
  constexpr int kGroupsPerCta = (kRsThreads / 32) * kGroupsPerWarp;
  const int lane = threadIdx.x & 31;
  // broadcast from lane 0: makes the warp index, hence the environment loop and every ballot, provably warp-uniform
  const int warp = __shfl_sync(kFullMask, int(threadIdx.x >> 5), 0);
  const int sub = lane % G, group_base = lane - sub;
  const int K = p.capacity, A = p.num_agents, S = p.schedule_rows;
  // this group's passenger-table buffer as a 32-bit shared-window address: rows are read / written as [table + 4 * index]
  const uint32_t table_bytes = uint32_t(K * kCols) * 4u;
  const uint32_t table = shared_address(smem) + uint32_t(warp * kGroupsPerWarp + lane / G) * table_bytes;
  const uint64_t rows_below = (uint64_t(1) << sub) - 1u;  // rows before this lane's first row
  // byte-permute selector that pulls this group's slice out of two ballots (group_rows): 16-lane groups take halfword
  // g of each, 8-lane groups byte g of each
  const uint32_t pack = (G == 16) ? ((group_base & 16) ? 0x7632u : 0x5410u)
                                  : (uint32_t(group_base >> 3) | ((4u + uint32_t(group_base >> 3)) << 4));

  FrzControl* control = io.control;
  const uint32_t alive_prev = control->alive;
  const uint32_t agents_with_tasks = control->agents_with_tasks;
  const bool skip = (MODE == kRsStep) && ((alive_prev & 3u) != 3u);  // utils/env.py:212
  const bool is_agent = sub < A;
  const bool fast = p.flags & FRZ_RS_FAST_TRAVEL, diagonal = p.flags & FRZ_RS_DIAGONAL_TRAVEL;
  const int directions = diagonal ? 9 : 5;
  // task-mask stores: work item -> (agent, four consecutive table rows)
  const bool wide_rows = (K & 3) == 0;  // every environment's table starts on a 16-byte boundary
  const int quads = (K + 3) >> 2;
  const uint32_t inverse_quads = (65536u + uint32_t(quads) - 1u) / uint32_t(quads);  // item / quads for item < 512
  unsigned alive_bits = 0, faults = 0, agent_bits = 0;

  if (!skip) {
    const int stride = gridDim.x * kGroupsPerCta;
    for (int env0 = (blockIdx.x * (kRsThreads / 32) + warp) * kGroupsPerWarp; env0 < B; env0 += stride) {
      const int env = min(env0 + lane / G, B - 1);
      const bool valid = env0 + lane / G < B;  // groups past the end of the batch replay the last environment, storing nothing
      const uint32_t agent_at = uint32_t(env) * uint32_t(A) + uint32_t(sub);
      int* const global_rows = io.passengers + uint32_t(env) * uint32_t(K * kCols);
      // stage the environment's live rows (cp.async); the other warps of the SM cover the latency
      const int n_before = min(io.env_task_count[env], K);
      {
        // 16-byte pieces while they lie inside the live rows (table bases are 16-byte aligned when K is a multiple of
        // four), single words for the remaining one to three
        const int words = n_before * kCols, quads_of_words = wide_rows ? words >> 2 : 0;
        for (int i = sub; i < quads_of_words; i += G) cp_async_16(table + 16u * i, global_rows + 4 * i);
        for (int i = 4 * quads_of_words + sub; i < words; i += G) cp_async_4(table + 4u * i, global_rows + i);
      }
      cp_async_commit();

      int agent_y = 0, agent_x = 0;
      int2 act = make_int2(0, -100);
      if (is_agent) {
        const int2 at = reinterpret_cast<const int2*>(io.agents)[agent_at];
        agent_y = at.x;
        agent_x = at.y;
        if (MODE == kRsStep) act = reinterpret_cast<const int2*>(io.actions)[agent_at];
      }
      const int t_now = io.num_moves[env];
      int n_kept = n_before, fare_won = 0;
      float move_cost = 0.f;
      const bool noop = act.y == -1, accept = act.y == 0, pick = act.y == 1, drop = act.y == 2;
      cp_async_wait_all();
      __syncwarp();

      // state / association columns of this lane's rows (kept in registers, refreshed after every edit phase)
      int state[PPL], assoc[PPL];
      bool present[PPL];
      const auto load_rows = [&](int count) {
#pragma unroll
        for (int i = 0; i < PPL; ++i) {
          const int r = sub + G * i;
          present[i] = r < count;
          state[i] = present[i] ? int(lds(table + 4u * uint32_t(r * kCols + cState))) : -1;
          assoc[i] = present[i] ? int(lds(table + 4u * uint32_t(r * kCols + cAssoc))) : -1;
        }
      };
      bool pred[PPL];

      if (MODE == kRsStep) {
        load_rows(n_before);
        // ---------------------------------------------------------------- task lists (rideshare.py:374-386)
#pragma unroll
        for (int i = 0; i < PPL; ++i) pred[i] = present[i] && state[i] == 0;
        const uint64_t unaccepted = group_rows<G, PPL>(pred, group_base, pack);
        uint64_t mine = 0;
        for (int a = 0; a < A; ++a) {
#pragma unroll
          for (int i = 0; i < PPL; ++i) pred[i] = present[i] && assoc[i] == a;
          const uint64_t own = group_rows<G, PPL>(pred, group_base, pack);
          if (sub == a) mine = unaccepted | own;
        }

        // ---------------------------------------------------------------- decode (rideshare.py:255-300)
        int target = -1;
        // the reference only resolves targets of agents that have a task in SOME environment (rideshare.py:276)
        if (is_agent && !noop && ((agents_with_tasks >> sub) & 1u)) {
          if (act.x >= 0 && act.x < __popcll(mine)) target = select_bit64(mine, act.x);
          else if (valid && (accept || pick || drop)) faults |= FRZ_FAULT_BAD_TASK_INDEX;
        }
        const bool has_vector = target >= 0 && (accept || pick || drop);
        int goal_y = 0, goal_x = 0, fare_target = 0;
        if (has_vector) {
          const uint32_t t = table + 4u * uint32_t(target * kCols);
          goal_y = int(lds(t + 4u * (drop ? cDestY : cY)));
          goal_x = int(lds(t + 4u * (drop ? cDestX : cX)));
          fare_target = int(lds(t + 4u * cFare));
        }

        // ---------------------------------------------------------------- movement (transitions/movement.py:57-116)
        int move_y = 0, move_x = 0;
        int distance2 = INT_MAX;  // squared distance agent -> goal before moving (passenger_state.py:48-49)
        if (has_vector) {
          distance2 = squared(agent_y - goal_y, agent_x - goal_x);
          if (fast) {
            move_y = goal_y - agent_y;
            move_x = goal_x - agent_x;
          } else {
            int best = INT_MAX;
            for (int d = 0; d < directions; ++d) {  // first argmin: strict <
              const int candidate = squared(agent_y + kDirY[d] - goal_y, agent_x + kDirX[d] - goal_x);
              if (candidate < best) {
                best = candidate;
                move_y = kDirY[d];
                move_x = kDirX[d];
              }
            }
          }
          move_cost = diagonal ? __fsqrt_rn(float(squared(move_y, move_x))) : float(abs(move_y) + abs(move_x));
        }
        agent_y += move_y;
        agent_x += move_x;
        __syncwarp();  // every lane has read its goal from the table
        // riding passengers travel with their driver; association -1 wraps to the last agent like the tensor index
#pragma unroll
        for (int i = 0; i < PPL; ++i) {
          int driver = assoc[i] < 0 ? assoc[i] + A : assoc[i];
          driver = group_base + min(max(driver, 0), G - 1);
          const int dy = __shfl_sync(kFullMask, move_y, driver), dx = __shfl_sync(kFullMask, move_x, driver);
          if (present[i] && state[i] == 2 && (dy | dx) != 0) {
            const uint32_t t = table + 4u * uint32_t((sub + G * i) * kCols);
            sts(t + 4u * cY, uint32_t(int(lds(t + 4u * cY)) + dy));
            sts(t + 4u * cX, uint32_t(int(lds(t + 4u * cX)) + dx));
          }
        }

        // ---------------------------------------------------------------- accept conflicts (passenger_state.py:50-74)
        int claim = (accept && target >= 0) ? target : -1;
        {
          const unsigned key = claim >= 0 ? (unsigned(group_base) << 8 | unsigned(claim)) : (0x80000000u | unsigned(lane));
          const bool duplicated = __popc(__match_any_sync(kFullMask, key)) > 1;
          if (__any_sync(kFullMask, duplicated)) {
            // among ALL duplicated claims of the environment only the closest claimant (first on ties) survives
            const int contest = duplicated ? distance2 : INT_MAX;
            const int closest = group_min<G>(contest);
            const uint32_t tied = (__ballot_sync(kFullMask, duplicated && contest == closest) >> group_base);
            const int keeper = __ffs(G == 32 ? tied : (tied & ((1u << G) - 1u))) - 1;
            if (duplicated && sub != keeper) claim = -1;
          }
        }
        const int picked = (pick && target >= 0 && distance2 == 0) ? target : -1;   // passenger_state.py:89-92 (< 1e-6)
        const int dropped = (drop && target >= 0 && distance2 == 0) ? target : -1;  // passenger_exit.py:40-45 (== 0)
        fare_won = dropped >= 0 ? fare_target : 0;

        // ---------------------------------------------------------------- apply: the drivers edit the rows in place
        if (claim >= 0) {  // accept: all accepts land before any pick, like the reference's transition
          const uint32_t t = table + 4u * uint32_t(claim * kCols);
          sts(t + 4u * cState, 1u);
          sts(t + 4u * cAccepted, uint32_t(t_now));
          sts(t + 4u * cAssoc, uint32_t(sub));
        }
        __syncwarp();
        if (picked >= 0) {
          const uint32_t t = table + 4u * uint32_t(picked * kCols);
          sts(t + 4u * cState, 2u);
          sts(t + 4u * cPicked, uint32_t(t_now));
        }
        __syncwarp();
        if (dropped >= 0) sts(table + 4u * uint32_t(dropped * kCols + cState), uint32_t(kRemoved));  // after the picks
        __syncwarp();

        // ---------------------------------------------------------------- exit: order-preserving compaction
        if (__any_sync(kFullMask, dropped >= 0)) {
#pragma unroll
          for (int i = 0; i < PPL; ++i) {
            const int r = sub + G * i;
            pred[i] = r < n_before && int(lds(table + 4u * uint32_t(r * kCols + cState))) != kRemoved;
          }
          const uint64_t kept = group_rows<G, PPL>(pred, group_base, pack);
          n_kept = __popcll(kept);
          // rows move down to their rank among the kept rows; slab by slab (rows s + G * i for all lanes s), read then
          // write: a row lands either in an earlier slab (done) or on a row of this slab that was just read
#pragma unroll
          for (int i = 0; i < PPL; ++i) {
            const int r = sub + G * i;
            const int to = __popcll(kept & ((rows_below << (G * i)) | ((uint64_t(1) << (G * i)) - 1u)));
            const bool moves = pred[i] && to != r;
            int row[kCols];
            if (moves) {
#pragma unroll
              for (int c = 0; c < kCols; ++c) row[c] = int(lds(table + 4u * uint32_t(r * kCols + c)));
            }
            __syncwarp();
            if (moves) {
#pragma unroll
              for (int c = 0; c < kCols; ++c) sts(table + 4u * uint32_t(to * kCols + c), uint32_t(row[c]));
            }
            __syncwarp();
          }
        }
      }

      // ------------------------------------------------------------------ entry (passenger_entry.py:25-72)
      int n_rows = n_kept;
      const bool admits = MODE == kRsStep || (MODE == kRsEntryRefresh && (entry_mask == nullptr || entry_mask[env]));
      {
        const int t_entry = (MODE == kRsStep) ? t_now + 1 : t_now;  // rideshare.py:307 vs :212
        // rows of the time-sorted schedule that enter at t_entry: [schedule_index[t], schedule_index[t + 1])
        int lo = S, hi = S;
        if (admits && t_entry >= 0 && t_entry <= p.schedule_horizon) {
          lo = io.schedule_index[t_entry];
          hi = io.schedule_index[t_entry + 1];
        }
        if (__any_sync(kFullMask, lo < hi)) {  // (environments of one warp may be at different steps after a partial reset)
          const int64_t global_env = p.env_offset + env;
          constexpr uint32_t lanes = (G == 32) ? 0xffffffffu : ((1u << G) - 1u);
          for (int base = 0; __any_sync(kFullMask, lo + base < hi); base += G) {
            const int r = lo + base + sub;
            const bool now = r < hi;
            const int* s = io.schedule + r * 7;
            const int batch = now ? s[1] : 0;
            const bool enters = now && (batch == -1 || batch == global_env);
            const uint32_t entering = (__ballot_sync(kFullMask, enters) >> group_base) & lanes;
            const int slot = n_rows + __popc(entering & ((1u << sub) - 1u));
            if (enters) {
              if (slot < K) {
                const uint32_t out = table + 4u * uint32_t(slot * kCols);
                sts(out + 4u * cBatch, uint32_t(batch_base + env));  // index in the caller's batch (a slice starts at batch_base)
                sts(out + 4u * cY, uint32_t(s[2]));
                sts(out + 4u * cX, uint32_t(s[3]));
                sts(out + 4u * cDestY, uint32_t(s[4]));
                sts(out + 4u * cDestX, uint32_t(s[5]));
                sts(out + 4u * cFare, uint32_t(s[6]));
                sts(out + 4u * cState, 0u);
                sts(out + 4u * cAssoc, uint32_t(-1));
                sts(out + 4u * cEntered, uint32_t(t_entry));
                sts(out + 4u * cAccepted, uint32_t(-1));
                sts(out + 4u * cPicked, uint32_t(-1));
              } else if (valid) {
                faults |= FRZ_FAULT_TABLE_FULL;
              }
            }
            n_rows = min(n_rows + __popc(entering), K);
          }
        }
      }
      __syncwarp();

      // ------------------------------------------------------------------ the new table
      load_rows(n_rows);
#pragma unroll
      for (int i = 0; i < PPL; ++i) {
        const int r = sub + G * i;
        // task observation row (rideshare.py:398-416) + padding of rows that just became free
        if (valid && r < K && (present[i] || r < n_before || MODE != kRsStep)) {
          int4 head = make_int4(FRZ_PAD, FRZ_PAD, FRZ_PAD, FRZ_PAD), tail = head;
          if (present[i]) {
            const uint32_t t = table + 4u * uint32_t(r * kCols);
            head = make_int4(int(lds(t + 4u * cY)), int(lds(t + 4u * cX)), int(lds(t + 4u * cDestY)), int(lds(t + 4u * cDestX)));
            tail = make_int4(state[i] == 1 ? assoc[i] : FRZ_PAD, state[i] == 2 ? assoc[i] : FRZ_PAD, int(lds(t + 4u * cFare)),
                             int(lds(t + 4u * cEntered)));
          }
          int4* out = reinterpret_cast<int4*>(io.task_obs) + (uint32_t(env) * uint32_t(K) + uint32_t(r)) * 2u;
          out[0] = head;
          out[1] = tail;
        }
      }

      // row masks by passenger state, per-agent counts; lane a of the group keeps agent a's
      uint64_t in_state[3];
#pragma unroll
      for (int cls = 0; cls < 3; ++cls) {
#pragma unroll
        for (int i = 0; i < PPL; ++i) pred[i] = present[i] && state[i] == cls;
        in_state[cls] = group_rows<G, PPL>(pred, group_base, pack);
      }
      int associated = 0, n_accepted = 0, n_riding = 0, n_tasks = 0;
      uint64_t members_mine = 0;
      for (int a = 0; a < A; ++a) {
#pragma unroll
        for (int i = 0; i < PPL; ++i) pred[i] = present[i] && assoc[i] == a;
        const uint64_t own = group_rows<G, PPL>(pred, group_base, pack);
        if (sub == a) {
          associated = __popcll(own);
          n_accepted = __popcll(own & in_state[1]);
          n_riding = __popcll(own & in_state[2]);
          members_mine = in_state[0] | own;
          n_tasks = __popcll(members_mine);
        }
      }
      // task mask [A, K] bytes: work item (agent, four consecutive rows) -> one 4-byte store when K is a multiple of 4
      {
        const bool aligned = (K & 3) == 0;
        const int items = aligned ? A * quads : 0;
        uint32_t* const mask_words = reinterpret_cast<uint32_t*>(io.task_mask);
        const uint32_t mask_at = uint32_t(env) * uint32_t(A * quads);
        for (int first = 0; first < items; first += G) {
          const int item = first + sub;
          const int a = int((uint32_t(item) * inverse_quads) >> 16), q = item - a * quads;
          const int source = group_base + min(a, G - 1);
          const uint32_t lo = __shfl_sync(kFullMask, uint32_t(members_mine), source);
          const uint32_t hi = __shfl_sync(kFullMask, uint32_t(members_mine >> 32), source);
          const uint32_t nibble = ((q < 8 ? lo : hi) >> (4 * (q & 7))) & 0xfu;
          if (valid && item < items) mask_words[mask_at + item] = (nibble * 0x00204081u) & 0x01010101u;
        }
        if (!aligned) {
          for (int a = 0; a < A; ++a) {
            const uint64_t members = (uint64_t(__shfl_sync(kFullMask, uint32_t(members_mine >> 32), group_base + a)) << 32) |
                                     __shfl_sync(kFullMask, uint32_t(members_mine), group_base + a);
            uint8_t* mask_row = io.task_mask + (uint32_t(env) * uint32_t(A) + uint32_t(a)) * uint32_t(K);
#pragma unroll
            for (int i = 0; i < PPL; ++i) {
              const int r = sub + G * i;
              if (valid && r < K) mask_row[r] = (members >> r) & 1u;
            }
          }
        }
      }

      if (MODE == kRsStep) {
        // ---------------------------------------------------------------- rewards (rideshare.py:309-363)
        float shared = 0.f;
        if (p.flags & FRZ_RS_WAITING_COSTS) {
          // `global[idx] += v` with duplicate indices keeps ONE write per statement: the last row of the class
          int elapsed_unaccepted = 0;
#pragma unroll
          for (int cls = 0; cls < 3; ++cls) {
            if (in_state[cls]) {
              const int last = 63 - __clzll(in_state[cls]);
              const int when = int(lds(table + 4u * uint32_t(last * kCols + (cls == 0 ? cEntered : (cls == 1 ? cAccepted : cPicked)))));
              const int elapsed = t_now - when;
              shared = __fadd_rn(shared, __fmul_rn(elapsed >= p.wait_limit[cls] ? 1.f : 0.f, p.general_wait_cost));
              if (cls == 0) elapsed_unaccepted = elapsed;
            }
          }
          if (in_state[0])
            shared = __fadd_rn(shared, __fmul_rn(elapsed_unaccepted >= p.long_wait_time ? 1.f : 0.f, p.long_wait_cost));
          const int free_slots = A * p.pool_limit - n_rows;
          const float unserved = __fmul_rn(__popcll(in_state[0]) >= free_slots ? 1.f : 0.f, -0.5f);
          shared = __fadd_rn(shared, __fmul_rn(unserved, float(free_slots)));
        }
        const int moves = t_now + 1;
        const bool truncated = moves >= p.max_steps;
        if (is_agent && valid) {
          float reward = associated > p.pool_limit ? p.pool_limit_cost : 0.f;
          reward = __fadd_rn(reward, __fmul_rn(noop ? 1.f : 0.f, p.noop_cost));
          reward = __fadd_rn(reward, __fmul_rn(accept ? 1.f : 0.f, p.accept_cost));
          reward = __fadd_rn(reward, fare_won > 0 ? __fadd_rn(float(fare_won), -p.drop_cost) : 0.f);
          float move_reward = __fmul_rn(move_cost, p.move_cost);
          if (p.flags & FRZ_RS_VARIABLE_MOVE_COST) move_reward = __fdiv_rn(move_reward, float(associated + 1));
          reward = __fadd_rn(reward, move_reward);
          reward = __fadd_rn(reward, shared);
          io.rewards[agent_at] = reward;
          io.cumulative_rewards[agent_at] = __fadd_rn(io.cumulative_rewards[agent_at], reward);
          reinterpret_cast<int2*>(io.agents)[agent_at] = make_int2(agent_y, agent_x);
        }
        if (sub == 0 && valid) {
          io.num_moves[env] = moves;
          io.truncated[env] = truncated;
        }
        if (valid) alive_bits |= 1u | (truncated ? 0u : 2u);  // rideshare never terminates (rideshare.py:252)
      } else if (valid) {  // refresh: the done flags as a reset, a restore or a hand edit left them
        alive_bits |= (io.terminated[env] ? 0u : 1u) | (io.truncated[env] ? 0u : 2u);
      }

      // ------------------------------------------------------------------ publish
      if (valid) {
        if (is_agent) {
          io.agent_task_count[agent_at] = n_tasks;
          if (n_tasks > 0) agent_bits |= 1u << sub;
          reinterpret_cast<int4*>(io.self_obs)[agent_at] = make_int4(agent_y, agent_x, n_accepted, n_riding);
        }
        if (sub == 0) io.env_task_count[env] = n_rows;
        if (admits) {
          const int words = n_rows * kCols, quads_of_words = wide_rows ? words >> 2 : 0;
          for (int i = sub; i < quads_of_words; i += G) {
            const uint4 piece = lds_v4(table + 16u * i);
            reinterpret_cast<int4*>(global_rows)[i] = make_int4(int(piece.x), int(piece.y), int(piece.z), int(piece.w));
          }
          for (int i = 4 * quads_of_words + sub; i < words; i += G) global_rows[i] = int(lds(table + 4u * i));
        }
      }
      __syncwarp();
    }
  }
  finish_launch(control, alive_bits, faults, agent_bits,
                skip ? kPublishNothing : (MODE == kRsStep ? kPublishStep : kPublishRefresh));
}

// ------------------------------------------------------------------------------------------------ tiled kernel
//
// One THREAD per environment, a warp per tile of 32 consecutive environments (tables with a multiple of four rows and at
// most eight drivers -- the named configurations; everything else takes the group kernel above).  The arithmetic of a
// rideshare step is a few dozen decisions per environment, so a lane-per-row mapping spends its instructions on ballots
// and on lanes without a row; here a thread walks its environment's rows serially (row sets are bit masks in registers)
// and a warp instruction serves 32 environments instead of 4.
//
// What makes that possible is the staging: the live rows of an environment are one contiguous byte range of the table
// (rows 0 .. count-1 of its slot), so they move global -> shared as ONE 1-D bulk async copy per environment
// (cp.async.bulk, the TMA unit; completion on the warp's mbarrier), never through registers or the LSU.  The warp's
// buffer is carved up by a prefix sum over what its environments need this step (live rows + rows that may enter), so
// shared memory is sized for the typical table fill, not for the capacity; a tile whose environments do not fit in one
// go is stepped in several passes of similar size.
//
// The way back is selective: a step touches few rows (riding passengers that moved, an accept, a pick, the rows behind an
// exit, an entry), and task_obs / task_mask are functions of the table alone, so only the changed rows, their
// observation rows and the 16-row mask pieces whose membership changed are stored (directly, as 8- / 16-byte pieces).
// Measured: rewriting everything with coalescing sweeps cost 60 us of DRAM write traffic at 524 288 environments.
// Row sets (unaccepted / accepted / riding / per driver) live in registers as bit masks, built once from the table and
// kept up to date through every edit (an exit removes a bit position: bit-compress).
// One warp per CTA: the tile index is then a function of blockIdx alone, which the compiler can prove warp-uniform -- the
// addresses of the bulk copies stay in uniform registers -- and up to 20 such CTAs share an SM.
constexpr int kTileThreads = 32;
constexpr int kTileWarps = kTileThreads / 32;
// profiling experiments only (profiles/README.md; never defined in the shipped build): 1 = copies but no stepping,
// 2 = stepping but no copies, 3 = no observation / mask stores -- results are wrong on purpose, time only
#ifndef FRZ_RS_ABLATE
#define FRZ_RS_ABLATE 0
#endif
constexpr int kTileRowBudget = 8;   // rows per environment the warp buffers are sized for (32 * 8 rows per warp)

constexpr int kTileIndexWords = 2048;      // longest schedule_index copied to shared memory
constexpr int kTileMinimumBatch = 24576;   // environments from which the tiled kernel is used (measured cross-over:
                                           // 16 384 envs 10.9 us with groups / 12.3 with tiles, 32 768: 18.9 / 13.4)

// row sets of an environment: bit r = table row r (32 or 64 rows)
__device__ __forceinline__ int mask_count(uint32_t m) { return __popc(m); }
__device__ __forceinline__ int mask_count(uint64_t m) { return __popcll(m); }
__device__ __forceinline__ int mask_first(uint32_t m) { return __ffs(int(m)) - 1; }
__device__ __forceinline__ int mask_first(uint64_t m) { return __ffsll((long long)(m)) - 1; }
__device__ __forceinline__ int mask_last(uint32_t m) { return 31 - __clz(int(m)); }
__device__ __forceinline__ int mask_last(uint64_t m) { return 63 - __clzll((long long)(m)); }
__device__ __forceinline__ int mask_select(uint32_t m, int k) { return select_bit(m, k); }
__device__ __forceinline__ int mask_select(uint64_t m, int k) { return select_bit64(m, k); }
// bits 0 .. n-1 (n may equal the width of the set)
__device__ __forceinline__ uint32_t mask_below(uint32_t, int n) { return n >= 32 ? 0xffffffffu : (1u << n) - 1u; }
__device__ __forceinline__ uint64_t mask_below(uint64_t, int n) { return n >= 64 ? ~uint64_t(0) : (uint64_t(1) << n) - 1u; }

template <int MAXA, bool WIDE, int MODE>
__global__ void __launch_bounds__(kTileThreads, MAXA <= 4 ? 20 : 12)
rideshare_tile_kernel(const __grid_constant__ FrzRideshareParams p, const __grid_constant__ FrzRideshareBuffers io,
                      const int B, const uint8_t* __restrict__ entry_mask, const int batch_base,
                      const uint32_t warp_bytes, const int index_words) {
  using Mask = typename std::conditional<WIDE, uint64_t, uint32_t>::type;
  extern __shared__ __align__(16) int smem[];
  static_assert(kTileWarps == 1, "the tile loop below assumes one warp per CTA");
  const int lane = threadIdx.x;
  constexpr int warp = 0, warps = 1;
  const int K = p.capacity, A = p.num_agents, S = p.schedule_rows;
  const uint32_t table_words = uint32_t(K * kCols);
  const uint32_t buffer = shared_address(smem);
  int* const buffer_words = smem;
  // after the table buffers: the mbarriers, then schedule_index
  int* const after_masks = smem + warps * int(warp_bytes >> 2);
  const uint32_t barrier = shared_address(after_masks) + 8u * uint32_t(warp);
  // schedule_index[0 .. index_words) copied next to the barriers (index_words = 0: the schedule is too long, read it
  // from global memory): turns the dependent load "count -> step -> schedule rows entering now" into a shared-memory read
  int* const index_copy = after_masks + 2 * warps;
  for (int i = threadIdx.x; i < index_words; i += blockDim.x) index_copy[i] = io.schedule_index[i];
  if (lane == 0) mbarrier_init(barrier, 1);
  __syncthreads();
  uint32_t phase = 0;

  FrzControl* control = io.control;
  const uint32_t alive_prev = control->alive;
  const uint32_t agents_with_tasks = control->agents_with_tasks;
  const bool skip = (MODE == kRsStep) && ((alive_prev & 3u) != 3u);  // utils/env.py:212
  const bool fast = p.flags & FRZ_RS_FAST_TRAVEL, diagonal = p.flags & FRZ_RS_DIAGONAL_TRAVEL;
  const bool even_agents = (A & 1) == 0, quad_agents = (A & 3) == 0;
  const uint32_t one_table = (table_words * 4u + 15u) & ~15u;
  unsigned alive_bits = 0, faults = 0, agent_bits = 0;

  if (!skip) {
    const int tile_stride = gridDim.x * 32;
    int tile0 = blockIdx.x * 32;
    // table fill and step of the tile's environments: loaded one tile ahead
    int next_count = 0, next_moves = 0;
    if (tile0 + lane < B) {
      next_count = io.env_task_count[tile0 + lane];
      next_moves = io.num_moves[tile0 + lane];
    }
    for (; tile0 < B; tile0 += tile_stride) {
      const int env = tile0 + lane;
      const bool valid = env < B;
      const int n_before = valid ? min(next_count, K) : 0, t_now = valid ? next_moves : 0;
      if (tile0 + tile_stride + lane < B) {
        next_count = io.env_task_count[tile0 + tile_stride + lane];
        next_moves = io.num_moves[tile0 + tile_stride + lane];
      }
      const bool admits =
          valid && (MODE == kRsStep || (MODE == kRsEntryRefresh && (entry_mask == nullptr || entry_mask[env])));
      const int t_entry = (MODE == kRsStep) ? t_now + 1 : t_now;  // rideshare.py:307 vs :212
      // rows of the time-sorted schedule that enter at t_entry: [schedule_index[t], schedule_index[t + 1])
      int lo = S, hi = S;
      if (admits && t_entry >= 0 && t_entry <= p.schedule_horizon) {
        if (index_words > 0) {
          lo = index_copy[t_entry];
          hi = index_copy[t_entry + 1];
        } else {
          lo = io.schedule_index[t_entry];
          hi = io.schedule_index[t_entry + 1];
        }
      }
      // shared memory this environment needs: its live rows and the rows that may enter, in whole 16-byte pieces
      // (at least one piece, so that every environment of a pass has a copy to issue)
      const uint32_t need = valid ? max(16u, (uint32_t(min(K, n_before + (hi - lo)) * kCols * 4) + 15u) & ~15u) : 0u;
      const uint32_t bytes_in = max(16u, (uint32_t(n_before * kCols * 4) + 15u) & ~15u);
      int* const global_rows = io.passengers + size_t(tile0) * size_t(table_words);  // of the tile's first environment

      // ------------------------------------------------------------------ drivers and their actions
      // (requested before the tables are staged: these loads fly while the bulk copies do)
      const uint32_t agent_at = uint32_t(env) * uint32_t(A);
      int agent_y[MAXA], agent_x[MAXA], act_k[MAXA], act_id[MAXA];
      float cumulative[MAXA];
#pragma unroll
      for (int a = 0; a < MAXA; ++a) {
        agent_y[a] = agent_x[a] = act_k[a] = 0;
        act_id[a] = -100;
        cumulative[a] = 0.f;
      }
      if (valid) {
        if (even_agents) {  // two drivers per 16-byte load
#pragma unroll
          for (int j = 0; j < MAXA / 2; ++j) {
            if (2 * j < A) {
              const int4 at = reinterpret_cast<const int4*>(io.agents)[(agent_at >> 1) + j];
              agent_y[2 * j] = at.x, agent_x[2 * j] = at.y, agent_y[2 * j + 1] = at.z, agent_x[2 * j + 1] = at.w;
              if (MODE == kRsStep) {
                const int4 act = reinterpret_cast<const int4*>(io.actions)[(agent_at >> 1) + j];
                act_k[2 * j] = act.x, act_id[2 * j] = act.y, act_k[2 * j + 1] = act.z, act_id[2 * j + 1] = act.w;
              }
            }
          }
        } else {
#pragma unroll
          for (int a = 0; a < MAXA; ++a) {
            if (a < A) {
              const int2 at = reinterpret_cast<const int2*>(io.agents)[agent_at + a];
              agent_y[a] = at.x, agent_x[a] = at.y;
              if (MODE == kRsStep) {
                const int2 act = reinterpret_cast<const int2*>(io.actions)[agent_at + a];
                act_k[a] = act.x, act_id[a] = act.y;
              }
            }
          }
        }
        if (MODE == kRsStep) {
          if (quad_agents) {
#pragma unroll
            for (int j = 0; j < MAXA / 4; ++j) {
              if (4 * j < A) {
                const float4 sum = reinterpret_cast<const float4*>(io.cumulative_rewards)[(agent_at >> 2) + j];
                cumulative[4 * j] = sum.x, cumulative[4 * j + 1] = sum.y, cumulative[4 * j + 2] = sum.z, cumulative[4 * j + 3] = sum.w;
              }
            }
          } else {
#pragma unroll
            for (int a = 0; a < MAXA; ++a)
              if (a < A) cumulative[a] = io.cumulative_rewards[agent_at + a];
          }
        }
      }

      for (uint32_t pending = __ballot_sync(kFullMask, valid); pending != 0u;) {
        // the environments of this pass: a prefix of the waiting ones whose rows fit in the warp's buffer (never empty:
        // one table always fits); when the tile needs several passes they are cut into pieces of similar size
        const bool waiting = (pending >> lane) & 1u;
        const uint32_t mine = waiting ? need : 0u;
        uint32_t scan = mine;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const uint32_t below = __shfl_up_sync(kFullMask, scan, d);
          if (lane >= d) scan += below;
        }
        const uint32_t total = __shfl_sync(kFullMask, scan, 31);
        uint32_t limit = warp_bytes;
        if (total > warp_bytes) {
          const uint32_t passes = (total + warp_bytes - 1u) / warp_bytes;
          limit = min(warp_bytes, (total + passes - 1u) / passes + one_table);
        }
        const bool now = waiting && scan <= limit;
        const uint32_t batch = __ballot_sync(kFullMask, now);
        const uint32_t offset = scan - mine;  // of this environment's rows in the warp's buffer (a multiple of 16)
        int* const rows = buffer_words + (offset >> 2);

        // ---------------------------------------------------------------- stage the live rows (one bulk copy each)
        const uint32_t load_bytes = now ? bytes_in : 0u;
        const uint32_t total_in = __reduce_add_sync(kFullMask, load_bytes);
        if (FRZ_RS_ABLATE != 2) {
          if (elect_one()) mbarrier_expect_bytes(barrier, total_in);
          // the pass's environments are consecutive lanes; everything but the two shuffled words is warp-uniform
          const int first = __ffs(int(batch)) - 1, last = first + __popc(batch);
          const uint32_t table_at = buffer + offset;
          const char* const tile_rows = reinterpret_cast<const char*>(global_rows);
#pragma unroll 4
          for (int e = first; e < last; ++e) {
            const uint32_t to = __shfl_sync(kFullMask, table_at, e), bytes = __shfl_sync(kFullMask, load_bytes, e);
            if (elect_one()) bulk_load(to, tile_rows + uint32_t(e) * (table_words * 4u), bytes, barrier);
          }
          mbarrier_wait(barrier, phase);
          phase ^= 1u;
        }

        int n_rows = n_before;
        if (now && FRZ_RS_ABLATE != 1) {
          int fare_won[MAXA];
          float move_cost[MAXA];
          // what this step changes: `dirty` = rows of the NEW table whose contents differ from what global memory holds at
          // that index (only those rows and their observation rows are written back); old_list = the drivers' task
          // lists before the step = what task_mask holds
          Mask dirty = 0, old_list[MAXA];
#pragma unroll
          for (int a = 0; a < MAXA; ++a) fare_won[a] = 0, move_cost[a] = 0.f, old_list[a] = 0;

          // ------------------------------------------------------------------ row sets (rideshare.py:374-386)
          // in_state[s] = rows whose passenger is unaccepted / accepted / riding, own[a] = rows associated with driver a;
          // read from the table once, then kept up to date through every edit of the step
          Mask in_state[3] = {0, 0, 0}, own[MAXA];
#pragma unroll
          for (int a = 0; a < MAXA; ++a) own[a] = 0;
          for (int r = 0; r < n_before; ++r) {
            const int state = rows[r * kCols + cState], assoc = rows[r * kCols + cAssoc];
            const Mask bit = Mask(1) << r;
#pragma unroll
            for (int cls = 0; cls < 3; ++cls) in_state[cls] |= state == cls ? bit : Mask(0);
#pragma unroll
            for (int a = 0; a < MAXA; ++a) own[a] |= assoc == a ? bit : Mask(0);
          }

          if (MODE == kRsStep) {

            // ---------------------------------------------------------------- decode + movement
            // (rideshare.py:255-300, transitions/movement.py:57-116)
            int target[MAXA], distance2[MAXA], move_y[MAXA], move_x[MAXA], fare_target[MAXA];
#pragma unroll
            for (int a = 0; a < MAXA; ++a) {
              target[a] = -1, distance2[a] = INT_MAX, move_y[a] = move_x[a] = 0, fare_target[a] = 0;
              if (a < A) {
                const bool noop = act_id[a] == -1, acts = act_id[a] == 0 || act_id[a] == 1 || act_id[a] == 2;
                // the reference only resolves targets of agents that have a task in SOME environment (rideshare.py:276)
                old_list[a] = in_state[0] | own[a];  // what task_mask holds for this driver
                if (!noop && ((agents_with_tasks >> a) & 1u)) {
                  const Mask list = old_list[a];
                  if (act_k[a] >= 0 && act_k[a] < mask_count(list)) target[a] = mask_select(list, act_k[a]);
                  else if (acts) faults |= FRZ_FAULT_BAD_TASK_INDEX;
                }
                if (target[a] >= 0 && acts) {
                  const int* row = rows + target[a] * kCols;
                  const bool drop = act_id[a] == 2;
                  const int goal_y = drop ? row[cDestY] : row[cY], goal_x = drop ? row[cDestX] : row[cX];
                  fare_target[a] = row[cFare];
                  // squared distance agent -> goal before moving (passenger_state.py:48-49)
                  distance2[a] = squared(agent_y[a] - goal_y, agent_x[a] - goal_x);
                  if (fast) {
                    move_y[a] = goal_y - agent_y[a];
                    move_x[a] = goal_x - agent_x[a];
                  } else {
                    // first argmin over stay, N, E, S, W [, NW, NE, SE, SW] of the squared distance after the move,
                    // written as its difference to staying: |v - m|^2 - |v|^2 = |m|^2 - 2 v.m with v = goal - agent
                    const int vy = goal_y - agent_y[a], vx = goal_x - agent_x[a];
                    int best = 0;
                    const auto consider = [&](int dy, int dx) {  // strict <: earlier directions win ties
                      const int change = dy * dy + dx * dx - 2 * (vy * dy + vx * dx);
                      if (change < best) best = change, move_y[a] = dy, move_x[a] = dx;
                    };
                    consider(-1, 0), consider(0, 1), consider(1, 0), consider(0, -1);
                    if (diagonal) consider(-1, -1), consider(-1, 1), consider(1, 1), consider(1, -1);
                  }
                  move_cost[a] = diagonal ? __fsqrt_rn(float(squared(move_y[a], move_x[a])))
                                          : float(abs(move_y[a]) + abs(move_x[a]));
                }
                agent_y[a] += move_y[a];
                agent_x[a] += move_x[a];
              }
            }
            // riding passengers travel with their driver; association -1 wraps to the last agent like the tensor index
            for (Mask m = in_state[2]; m != 0; m &= m - 1) {
              int* row = rows + mask_first(m) * kCols;
              int driver = row[cAssoc];
              driver = driver < 0 ? driver + A : driver;
              int dy = 0, dx = 0;
#pragma unroll
              for (int a = 0; a < MAXA; ++a)
                if (driver == a) dy = move_y[a], dx = move_x[a];
              if ((dy | dx) != 0) {
                row[cY] += dy;
                row[cX] += dx;
                dirty |= m & (~m + 1);
              }
            }

            // ---------------------------------------------------------------- accept conflicts (passenger_state.py:50-74)
            int claim[MAXA];
#pragma unroll
            for (int a = 0; a < MAXA; ++a) claim[a] = (act_id[a] == 0 && target[a] >= 0) ? target[a] : -1;
            {
              bool duplicated[MAXA], any = false;
#pragma unroll
              for (int a = 0; a < MAXA; ++a) {
                duplicated[a] = false;
#pragma unroll
                for (int b = 0; b < MAXA; ++b)
                  if (b != a && claim[a] >= 0 && claim[a] == claim[b]) duplicated[a] = true;
                any |= duplicated[a];
              }
              if (any) {
                // among ALL duplicated claims of the environment only the closest claimant (first on ties) survives
                int closest = INT_MAX, keeper = -1;
#pragma unroll
                for (int a = 0; a < MAXA; ++a)
                  if (duplicated[a] && distance2[a] < closest) closest = distance2[a], keeper = a;
#pragma unroll
                for (int a = 0; a < MAXA; ++a)
                  if (duplicated[a] && a != keeper) claim[a] = -1;
              }
            }
            // ---------------------------------------------------------------- apply: accepts, then picks, then exits
#pragma unroll
            for (int a = 0; a < MAXA; ++a) {
              if (claim[a] >= 0) {
                int* row = rows + claim[a] * kCols;
                row[cState] = 1;
                row[cAccepted] = t_now;
                row[cAssoc] = a;
                const Mask bit = Mask(1) << claim[a];
                dirty |= bit;
                in_state[0] &= ~bit, in_state[2] &= ~bit, in_state[1] |= bit;
#pragma unroll
                for (int b = 0; b < MAXA; ++b) own[b] = b == a ? (own[b] | bit) : (own[b] & ~bit);
              }
            }
#pragma unroll
            for (int a = 0; a < MAXA; ++a) {
              if (act_id[a] == 1 && target[a] >= 0 && distance2[a] == 0) {  // passenger_state.py:89-92 (< 1e-6)
                int* row = rows + target[a] * kCols;
                row[cState] = 2;
                row[cPicked] = t_now;
                const Mask bit = Mask(1) << target[a];
                dirty |= bit;
                in_state[0] &= ~bit, in_state[1] &= ~bit, in_state[2] |= bit;
              }
            }
            Mask leaving = 0;
#pragma unroll
            for (int a = 0; a < MAXA; ++a) {
              if (act_id[a] == 2 && target[a] >= 0 && distance2[a] == 0) {  // passenger_exit.py:40-45 (== 0)
                fare_won[a] = fare_target[a];
                leaving |= Mask(1) << target[a];
              }
            }
            // ---------------------------------------------------------------- exit: order-preserving compaction
            if (leaving != 0) {
              const int first_gap = mask_first(leaving);
              int kept = first_gap;
              for (int r = first_gap + 1; r < n_before; ++r) {
                if (!((leaving >> r) & 1u)) {
#pragma unroll
                  for (int c = 0; c < kCols; ++c) rows[kept * kCols + c] = rows[r * kCols + c];
                  ++kept;
                }
              }
              n_rows = kept;
              // rows below the first gap stay where they were; everything from there on moved
              dirty = (dirty & mask_below(Mask(0), first_gap)) | (mask_below(Mask(0), kept) & ~mask_below(Mask(0), first_gap));
              // the row sets lose the leaving rows' positions (from the highest one down, so positions stay valid)
              for (Mask gone = leaving; gone != 0;) {
                const int at = mask_last(gone);
                gone ^= Mask(1) << at;
                const Mask low = mask_below(Mask(0), at);
#pragma unroll
                for (int cls = 0; cls < 3; ++cls) in_state[cls] = (in_state[cls] & low) | ((in_state[cls] >> 1) & ~low);
#pragma unroll
                for (int a = 0; a < MAXA; ++a) own[a] = (own[a] & low) | ((own[a] >> 1) & ~low);
              }
            }
          }

          // ------------------------------------------------------------------ entry (passenger_entry.py:25-72)
          {
            const int64_t global_env = p.env_offset + env;
            for (int r = lo; r < hi; ++r) {
              const int* s = io.schedule + r * 7;
              const int batch = s[1];
              if (batch == -1 || batch == global_env) {
                if (n_rows < K) {
                  int* row = rows + n_rows * kCols;
                  row[cBatch] = batch_base + env;  // index in the caller's batch (a slice starts at batch_base)
                  row[cY] = s[2], row[cX] = s[3], row[cDestY] = s[4], row[cDestX] = s[5], row[cFare] = s[6];
                  row[cState] = 0, row[cAssoc] = -1, row[cEntered] = t_entry, row[cAccepted] = -1, row[cPicked] = -1;
                  dirty |= Mask(1) << n_rows;
                  in_state[0] |= Mask(1) << n_rows;
                  ++n_rows;
                } else {
                  faults |= FRZ_FAULT_TABLE_FULL;
                }
              }
            }
          }

          // ------------------------------------------------------------------ write back what changed
          // Only the rows this step touched go back to global memory, together with their task observation rows
          // (rideshare.py:398-416): riding passengers that moved, accepted / picked passengers, rows that moved up behind
          // an exit, rows that entered.  A refresh or reset writes every live row.  (The other rows of the table, of
          // task_obs and of task_mask already hold these values: they are functions of the table alone.)
          if (FRZ_RS_ABLATE != 3) {
            int* const table_out = global_rows + size_t(lane) * size_t(table_words);
            int4* const obs = reinterpret_cast<int4*>(io.task_obs) + size_t(env) * size_t(K) * 2u;
            for (Mask m = MODE == kRsStep ? dirty : mask_below(Mask(0), n_rows); m != 0; m &= m - 1) {
              const int r = mask_first(m);
              const int* row = rows + r * kCols;
              const int batch = row[cBatch], y = row[cY], x = row[cX], dest_y = row[cDestY], dest_x = row[cDestX], fare = row[cFare];
              const int state = row[cState], assoc = row[cAssoc], entered = row[cEntered], accepted = row[cAccepted];
              const int picked = row[cPicked];
              obs[2 * r] = make_int4(y, x, dest_y, dest_x);
              obs[2 * r + 1] = make_int4(state == 1 ? assoc : FRZ_PAD, state == 2 ? assoc : FRZ_PAD, fare, entered);
              if (MODE == kRsStep || admits) {
                // the 11 words of the row as five 8-byte stores and one word (rows start on alternating 8-byte phases)
                int* out = table_out + r * kCols;
                if (r & 1) {
                  out[0] = batch;
                  reinterpret_cast<int2*>(out + 1)[0] = make_int2(y, x);
                  reinterpret_cast<int2*>(out + 1)[1] = make_int2(dest_y, dest_x);
                  reinterpret_cast<int2*>(out + 1)[2] = make_int2(fare, state);
                  reinterpret_cast<int2*>(out + 1)[3] = make_int2(assoc, entered);
                  reinterpret_cast<int2*>(out + 1)[4] = make_int2(accepted, picked);
                } else {
                  reinterpret_cast<int2*>(out)[0] = make_int2(batch, y);
                  reinterpret_cast<int2*>(out)[1] = make_int2(x, dest_y);
                  reinterpret_cast<int2*>(out)[2] = make_int2(dest_x, fare);
                  reinterpret_cast<int2*>(out)[3] = make_int2(state, assoc);
                  reinterpret_cast<int2*>(out)[4] = make_int2(entered, accepted);
                  out[10] = picked;
                }
              }
            }
            // padding of the observation rows that just became free (every row past the table on a refresh)
            const int4 pad = make_int4(FRZ_PAD, FRZ_PAD, FRZ_PAD, FRZ_PAD);
            const int pad_to = MODE == kRsStep ? n_before : K;
            for (int r = n_rows; r < pad_to; ++r) obs[2 * r] = pad, obs[2 * r + 1] = pad;
          }

          // ------------------------------------------------------------------ rewards shared by the drivers
          float shared = 0.f;
          if (MODE == kRsStep && (p.flags & FRZ_RS_WAITING_COSTS)) {
            // `global[idx] += v` with duplicate indices keeps ONE write per statement: the last row of the class
            int elapsed_unaccepted = 0;
#pragma unroll
            for (int cls = 0; cls < 3; ++cls) {
              if (in_state[cls] != 0) {
                const int when = rows[mask_last(in_state[cls]) * kCols + (cls == 0 ? cEntered : (cls == 1 ? cAccepted : cPicked))];
                const int elapsed = t_now - when;
                shared = __fadd_rn(shared, __fmul_rn(elapsed >= p.wait_limit[cls] ? 1.f : 0.f, p.general_wait_cost));
                if (cls == 0) elapsed_unaccepted = elapsed;
              }
            }
            if (in_state[0] != 0)
              shared = __fadd_rn(shared, __fmul_rn(elapsed_unaccepted >= p.long_wait_time ? 1.f : 0.f, p.long_wait_cost));
            const int free_slots = A * p.pool_limit - n_rows;
            const float unserved = __fmul_rn(mask_count(in_state[0]) >= free_slots ? 1.f : 0.f, -0.5f);
            shared = __fadd_rn(shared, __fmul_rn(unserved, float(free_slots)));
          }

          // ------------------------------------------------------------------ per driver: counts, task mask, rewards
          int n_tasks[MAXA];
          float reward[MAXA];
          int4 self[MAXA];
#pragma unroll
          for (int a = 0; a < MAXA; ++a) {
            n_tasks[a] = 0, reward[a] = 0.f, self[a] = make_int4(0, 0, 0, 0);
            if (a < A) {
              const int associated = mask_count(own[a]);
              const Mask members = in_state[0] | own[a];
              n_tasks[a] = mask_count(members);
              if (n_tasks[a] > 0) agent_bits |= 1u << a;
              self[a] = make_int4(agent_y[a], agent_x[a], mask_count(own[a] & in_state[1]), mask_count(own[a] & in_state[2]));
              // task mask [A, K] bytes: the 16-row (4-row) pieces whose membership changed; nibble x 0x204081 spreads
              // four bits over four bytes
              const Mask changed = MODE == kRsStep ? (members ^ old_list[a]) : ~Mask(0);
              if (changed != 0 && FRZ_RS_ABLATE != 3) {
                uint32_t* const mask_row = reinterpret_cast<uint32_t*>(io.task_mask + (size_t(agent_at) + a) * size_t(K));
                if ((K & 15) == 0) {
#pragma unroll
                  for (int q = 0; q < (WIDE ? 4 : 2); ++q) {
                    if (16 * q < K && (uint32_t(changed >> (16 * q)) & 0xffffu) != 0u) {
                      const uint32_t part = uint32_t(members >> (16 * q));
                      reinterpret_cast<uint4*>(mask_row)[q] =
                          make_uint4(((part & 0xfu) * 0x00204081u) & 0x01010101u, (((part >> 4) & 0xfu) * 0x00204081u) & 0x01010101u,
                                     (((part >> 8) & 0xfu) * 0x00204081u) & 0x01010101u,
                                     (((part >> 12) & 0xfu) * 0x00204081u) & 0x01010101u);
                    }
                  }
                } else {
                  for (int q = 0; 4 * q < K; ++q)
                    if ((uint32_t(changed >> (4 * q)) & 0xfu) != 0u)
                      mask_row[q] = ((uint32_t(members >> (4 * q)) & 0xfu) * 0x00204081u) & 0x01010101u;
                }
              }
              if (MODE == kRsStep) {  // rideshare.py:309-363
                float value = associated > p.pool_limit ? p.pool_limit_cost : 0.f;
                value = __fadd_rn(value, __fmul_rn(act_id[a] == -1 ? 1.f : 0.f, p.noop_cost));
                value = __fadd_rn(value, __fmul_rn(act_id[a] == 0 ? 1.f : 0.f, p.accept_cost));
                value = __fadd_rn(value, fare_won[a] > 0 ? __fadd_rn(float(fare_won[a]), -p.drop_cost) : 0.f);
                float move_reward = __fmul_rn(move_cost[a], p.move_cost);
                // (x / 1 = x and 0 / n = 0 exactly: the division runs only where it changes the value)
                if ((p.flags & FRZ_RS_VARIABLE_MOVE_COST) && associated > 0 && move_cost[a] != 0.f)
                  move_reward = __fdiv_rn(move_reward, float(associated + 1));
                value = __fadd_rn(value, move_reward);
                reward[a] = __fadd_rn(value, shared);
              }
            }
          }

          // ------------------------------------------------------------------ publish
          if (quad_agents) {  // four drivers per 16-byte store
#pragma unroll
            for (int j = 0; j < MAXA / 4; ++j) {
              if (4 * j < A) {
                reinterpret_cast<int4*>(io.agent_task_count)[(agent_at >> 2) + j] =
                    make_int4(n_tasks[4 * j], n_tasks[4 * j + 1], n_tasks[4 * j + 2], n_tasks[4 * j + 3]);
                if (MODE == kRsStep) {
                  reinterpret_cast<float4*>(io.rewards)[(agent_at >> 2) + j] =
                      make_float4(reward[4 * j], reward[4 * j + 1], reward[4 * j + 2], reward[4 * j + 3]);
                  reinterpret_cast<float4*>(io.cumulative_rewards)[(agent_at >> 2) + j] =
                      make_float4(__fadd_rn(cumulative[4 * j], reward[4 * j]), __fadd_rn(cumulative[4 * j + 1], reward[4 * j + 1]),
                                  __fadd_rn(cumulative[4 * j + 2], reward[4 * j + 2]),
                                  __fadd_rn(cumulative[4 * j + 3], reward[4 * j + 3]));
                }
              }
            }
          } else {
#pragma unroll
            for (int a = 0; a < MAXA; ++a) {
              if (a < A) {
                io.agent_task_count[agent_at + a] = n_tasks[a];
                if (MODE == kRsStep) {
                  io.rewards[agent_at + a] = reward[a];
                  io.cumulative_rewards[agent_at + a] = __fadd_rn(cumulative[a], reward[a]);
                }
              }
            }
          }
#pragma unroll
          for (int a = 0; a < MAXA; ++a)
            if (a < A) reinterpret_cast<int4*>(io.self_obs)[agent_at + a] = self[a];
          if (MODE == kRsStep) {
            if (even_agents) {
#pragma unroll
              for (int j = 0; j < MAXA / 2; ++j)
                if (2 * j < A)
                  reinterpret_cast<int4*>(io.agents)[(agent_at >> 1) + j] =
                      make_int4(agent_y[2 * j], agent_x[2 * j], agent_y[2 * j + 1], agent_x[2 * j + 1]);
            } else {
#pragma unroll
              for (int a = 0; a < MAXA; ++a)
                if (a < A) reinterpret_cast<int2*>(io.agents)[agent_at + a] = make_int2(agent_y[a], agent_x[a]);
            }
            const int moves = t_now + 1;
            const bool truncated = moves >= p.max_steps;
            io.num_moves[env] = moves;
            io.truncated[env] = truncated;
            alive_bits |= 1u | (truncated ? 0u : 2u);  // rideshare never terminates (rideshare.py:252)
          } else {  // refresh: the done flags as a reset, a restore or a hand edit left them
            alive_bits |= (io.terminated[env] ? 0u : 1u) | (io.truncated[env] ? 0u : 2u);
          }
          io.env_task_count[env] = n_rows;
        }

        // this pass's generic accesses to the buffer are ordered before the next pass's bulk copies into it
        fence_async_shared();
        __syncwarp();
        pending &= ~batch;
      }
    }
  }
  finish_launch(control, alive_bits, faults, agent_bits,
                skip ? kPublishNothing : (MODE == kRsStep ? kPublishStep : kPublishRefresh));
}

__global__ void rideshare_restore_kernel(const FrzRideshareParams p, const FrzRideshareBuffers io, const int B,
                                         const uint8_t* __restrict__ env_mask) {
  const int A = p.num_agents, K = p.capacity;
  // items per environment: table words, or driver coordinates when the table is shorter than those (a one-row
  // schedule with many drivers) -- every driver and every reward must be reached
  const int table_words = K * kCols;
  const int per_env = table_words > 2 * A ? table_words : 2 * A;
  const size_t total = size_t(B) * per_env;
  for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += size_t(gridDim.x) * blockDim.x) {
    const int env = int(i / per_env), j = int(i % per_env);
    if (env_mask != nullptr && !env_mask[env]) continue;
    if (j < table_words) io.passengers[size_t(env) * table_words + j] = io.init_passengers[size_t(env) * table_words + j];
    if (j < 2 * A) io.agents[size_t(env) * 2 * A + j] = io.init_agents[size_t(env) * 2 * A + j];
    if (j < A) {
      io.rewards[size_t(env) * A + j] = 0.f;
      io.cumulative_rewards[size_t(env) * A + j] = 0.f;
    }
    if (j == 0) {
      io.env_task_count[env] = io.init_count[env];
      io.terminated[env] = 0;
      io.truncated[env] = 0;
      io.num_moves[env] = 0;
    }
  }
}

// Uniform over [task 0 .. task n-1, noop]; the action id of a task is the passenger's state (0 accept / 1 pick /
// 2 drop), which is the only id the reference's action space offers for it (spaces/actions.py:10-50).
__global__ void rideshare_sample_kernel(const FrzRideshareParams p, const FrzRideshareBuffers io, const int B,
                                        const uint64_t sampler_seed) {
  const int A = p.num_agents, K = p.capacity;
  const Philox philox(sampler_seed);
  const uint64_t step = io.control->step;
  const int total = B * A;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int env = i / A, agent = i - env * A;
    const int n = io.agent_task_count[i];
    const uint64_t genv = uint64_t(p.env_offset + env);
    const uint4 r = philox(uint32_t(genv), uint32_t(step), 0xC0000000u | uint32_t(agent), uint32_t(step >> 32) ^ uint32_t(genv >> 32));
    const int k = min(int(u01(r.x) * float(n + 1)), n);
    int ident = -1;
    if (k < n) {
      const uint8_t* mask = io.task_mask + size_t(i) * K;
      int seen = 0;
      for (int row = 0; row < K; ++row) {
        if (mask[row]) {
          if (seen == k) {
            const int* obs = io.task_obs + (size_t(env) * K + row) * FRZ_RS_TASK_COLUMNS;
            ident = obs[5] != FRZ_PAD ? 2 : (obs[4] != FRZ_PAD ? 1 : 0);
            break;
          }
          ++seen;
        }
      }
    }
    reinterpret_cast<int2*>(const_cast<int32_t*>(io.actions))[i] = make_int2(k, ident);
  }
}

int rideshare_validate(const FrzRideshareParams* p, const FrzRideshareBuffers* io, int B, const char* what) {
  if (p == nullptr || io == nullptr || io->control == nullptr || io->passengers == nullptr || io->agents == nullptr ||
      (p->schedule_rows > 0 && (io->schedule == nullptr || io->schedule_index == nullptr))) {
    set_error("%s: NULL params / buffers", what);
    return FRZ_ERR_NULL;
  }
  if (B <= 0 || p->num_agents < 1 || p->num_agents > FRZ_MAX_AGENTS || p->capacity < 1 ||
      p->capacity > FRZ_MAX_PASSENGERS || p->schedule_rows < 0 ||
      uint64_t(B) * uint64_t(p->capacity) * FRZ_RS_PASSENGER_COLUMNS >= (1ull << 32)) {  // 32-bit element indices
    set_error("%s: unsupported shape B=%d agents=%d capacity=%d schedule=%d", what, B, p->num_agents, p->capacity,
              p->schedule_rows);
    return FRZ_ERR_SHAPE;
  }
  return FRZ_OK;
}

// Lanes per environment and rows per lane: the smallest group that holds the drivers and keeps at most 4 rows per lane.
template <int G, int PPL, int MODE>
int rideshare_launch_geometry(const FrzRideshareParams* p, const FrzRideshareBuffers* io, int B, cudaStream_t s,
                              const uint8_t* entry_mask, int batch_base) {
  constexpr int groups_per_cta = (kRsThreads / 32) * (32 / G);
  const size_t smem = size_t(groups_per_cta) * p->capacity * kCols * sizeof(int);  // one table buffer per group
  auto kernel = rideshare_step_kernel<G, PPL, MODE>;
  if (smem > 48 * 1024 && cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)) != cudaSuccess)
    return check_launch("rideshare shared memory");
  const int ctas_per_sm = resident_ctas(kernel, kRsThreads, smem);
  const int grid = persistent_grid((B + groups_per_cta - 1) / groups_per_cta, ctas_per_sm);
  kernel<<<grid, kRsThreads, smem, s>>>(*p, *io, B, entry_mask, batch_base);
  return check_launch("rideshare_step_kernel");
}

// The tiled kernel: one thread per environment, a one-warp CTA per tile of 32 environments (persistent grid).
template <int MAXA, bool WIDE, int MODE>
int rideshare_launch_tiles(const FrzRideshareParams* p, const FrzRideshareBuffers* io, int B, cudaStream_t s,
                           const uint8_t* entry_mask, int batch_base) {
  const int K = p->capacity;
  const uint32_t one_table = (uint32_t(K * kCols * 4) + 15u) & ~15u;
  const uint32_t typical = (uint32_t(32 * std::min(K, kTileRowBudget) * kCols * 4) + 15u) & ~15u;
  const uint32_t warp_bytes = std::max(one_table, typical);
  // schedule_index travels to shared memory when it is short enough (an entry per step of the schedule's horizon)
  const int index_words = p->schedule_rows > 0 && p->schedule_horizon + 2 <= kTileIndexWords ? p->schedule_horizon + 2 : 0;
  const size_t smem = size_t(kTileWarps) * warp_bytes + 8 * kTileWarps + 4 * size_t(index_words);
  auto kernel = rideshare_tile_kernel<MAXA, WIDE, MODE>;
  if (smem > 48 * 1024 && cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)) != cudaSuccess)
    return check_launch("rideshare shared memory");
  cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  const int ctas_per_sm = resident_ctas(kernel, kTileThreads, smem);
  // every CTA steps the same number of tiles (+-1): the fewest rounds the resident CTAs need, then as many CTAs as
  // those rounds take
  const int tiles = (B + 31) / 32;
  const int resident = sm_count() * ctas_per_sm;
  const int rounds = (tiles + resident - 1) / resident;
  const int grid = (tiles + rounds - 1) / rounds;
  kernel<<<grid, kTileThreads, smem, s>>>(*p, *io, B, entry_mask, batch_base, warp_bytes, index_words);
  return check_launch("rideshare_tile_kernel");
}

template <int MODE>
int rideshare_launch_mode(const FrzRideshareParams* p, const FrzRideshareBuffers* io, int B, cudaStream_t s,
                          const uint8_t* entry_mask, int batch_base) {
  const int K = p->capacity, A = p->num_agents;
  // One thread per environment needs enough environments to fill the GPU with warps (a tile of 32 takes one warp
  // through a long dependent chain); smaller batches keep a group of lanes per environment.  Bulk copies need 16-byte
  // aligned tables.
  const bool tiles = (p->flags & FRZ_RS_KERNEL_TILES) || (!(p->flags & FRZ_RS_KERNEL_GROUPS) && B >= kTileMinimumBatch);
  if (A <= 8 && (K & 3) == 0 && tiles) {
    if (A <= 4) return K <= 32 ? rideshare_launch_tiles<4, false, MODE>(p, io, B, s, entry_mask, batch_base)
                               : rideshare_launch_tiles<4, true, MODE>(p, io, B, s, entry_mask, batch_base);
    return K <= 32 ? rideshare_launch_tiles<8, false, MODE>(p, io, B, s, entry_mask, batch_base)
                   : rideshare_launch_tiles<8, true, MODE>(p, io, B, s, entry_mask, batch_base);
  }
  if (A <= 8 && K <= 8) return rideshare_launch_geometry<8, 1, MODE>(p, io, B, s, entry_mask, batch_base);
  if (A <= 8 && K <= 16) return rideshare_launch_geometry<8, 2, MODE>(p, io, B, s, entry_mask, batch_base);
  if (A <= 8 && K <= 32) return rideshare_launch_geometry<8, 4, MODE>(p, io, B, s, entry_mask, batch_base);
  if (A <= 16 && K <= 32) return rideshare_launch_geometry<16, 2, MODE>(p, io, B, s, entry_mask, batch_base);
  if (A <= 16) return rideshare_launch_geometry<16, 4, MODE>(p, io, B, s, entry_mask, batch_base);
  if (K <= 32) return rideshare_launch_geometry<32, 1, MODE>(p, io, B, s, entry_mask, batch_base);
  return rideshare_launch_geometry<32, 2, MODE>(p, io, B, s, entry_mask, batch_base);
}

int rideshare_launch(const FrzRideshareParams* p, const FrzRideshareBuffers* io, int B, int mode, void* stream,
                     const uint8_t* entry_mask = nullptr, int batch_base = 0) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (mode == kRsStep) return rideshare_launch_mode<kRsStep>(p, io, B, s, entry_mask, batch_base);
  if (mode == kRsRefresh) return rideshare_launch_mode<kRsRefresh>(p, io, B, s, entry_mask, batch_base);
  return rideshare_launch_mode<kRsEntryRefresh>(p, io, B, s, entry_mask, batch_base);
}

}  // namespace
}  // namespace frz

extern "C" {

int frz_rideshare_step(const FrzRideshareParams* params, const FrzRideshareBuffers* io, int32_t parallel_envs,
                       void* stream) {
  const int status = frz::rideshare_validate(params, io, parallel_envs, "frz_rideshare_step");
  if (status != FRZ_OK) return status;
  if (io->actions == nullptr) {
    frz::set_error("frz_rideshare_step: actions is NULL");
    return FRZ_ERR_NULL;
  }
  return frz::rideshare_launch(params, io, parallel_envs, frz::kRsStep, stream);
}

int frz_rideshare_step_host(const FrzRideshareParams* params, const FrzRideshareBuffers* io, int32_t parallel_envs,
                            const FrzHostStep* host, void* stream) {
  const int status = frz::rideshare_validate(params, io, parallel_envs, "frz_rideshare_step_host");
  if (status != FRZ_OK) return status;
  if (io->actions == nullptr || io->rewards == nullptr) {
    frz::set_error("frz_rideshare_step_host: actions / rewards is NULL");
    return FRZ_ERR_NULL;
  }
  const size_t A = size_t(params->num_agents), K = size_t(params->capacity);
  const frz::HostArrays arrays{io->actions, io->rewards, io->terminated, io->truncated, io->control, params->num_agents,
                                 params, sizeof(FrzRideshareParams), io, sizeof(FrzRideshareBuffers)};
  return frz::run_host_pipeline(
      "frz_rideshare_step_host", host, arrays, parallel_envs, static_cast<cudaStream_t>(stream),
      [&](int first, int count, FrzControl* control, cudaStream_t slice_stream) {
        FrzRideshareParams p = *params;
        p.env_offset += first;  // schedule rows name global environment indices
        FrzRideshareBuffers slice = *io;
        const size_t e = size_t(first);
        slice.agents += e * A * 2;
        slice.passengers += e * K * FRZ_RS_PASSENGER_COLUMNS;
        slice.actions += e * A * 2;
        slice.rewards += e * A;
        slice.cumulative_rewards += e * A;
        slice.terminated += e;
        slice.truncated += e;
        slice.num_moves += e;
        slice.env_task_count += e;
        slice.agent_task_count += e * A;
        slice.task_mask += e * A * K;
        slice.self_obs += e * A * 4;
        slice.task_obs += e * K * FRZ_RS_TASK_COLUMNS;
        slice.control = control;
        return frz::rideshare_launch(&p, &slice, count, frz::kRsStep, slice_stream, nullptr, first);
      });
}

int frz_rideshare_refresh(const FrzRideshareParams* params, const FrzRideshareBuffers* io, int32_t parallel_envs,
                          void* stream) {
  const int status = frz::rideshare_validate(params, io, parallel_envs, "frz_rideshare_refresh");
  if (status != FRZ_OK) return status;
  return frz::rideshare_launch(params, io, parallel_envs, frz::kRsRefresh, stream);
}

int frz_rideshare_reset(const FrzRideshareParams* params, const FrzRideshareBuffers* io, int32_t parallel_envs,
                        const uint8_t* env_mask, void* stream) {
  int status = frz::rideshare_validate(params, io, parallel_envs, "frz_rideshare_reset");
  if (status != FRZ_OK) return status;
  if (io->init_agents == nullptr || io->init_passengers == nullptr || io->init_count == nullptr) {
    frz::set_error("frz_rideshare_reset: initial state is NULL");
    return FRZ_ERR_NULL;
  }
  const size_t total = size_t(parallel_envs) * params->capacity * FRZ_RS_PASSENGER_COLUMNS;
  const int grid = frz::persistent_grid(int((total + 255) / 256), 8);
  frz::rideshare_restore_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(*params, *io, parallel_envs, env_mask);
  status = frz::check_launch("rideshare_restore_kernel");
  if (status != FRZ_OK) return status;
  // only the environments being reset admit their t = 0 passengers; the others are merely re-published
  return frz::rideshare_launch(params, io, parallel_envs, frz::kRsEntryRefresh, stream, env_mask);
}

int frz_rideshare_sample_actions(const FrzRideshareParams* params, const FrzRideshareBuffers* io, int32_t parallel_envs,
                                 uint64_t sampler_seed, void* stream) {
  const int status = frz::rideshare_validate(params, io, parallel_envs, "frz_rideshare_sample_actions");
  if (status != FRZ_OK) return status;
  const int total = parallel_envs * params->num_agents;
  const int grid = frz::persistent_grid((total + 255) / 256, 8);
  frz::rideshare_sample_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(*params, *io, parallel_envs, sampler_seed);
  return frz::check_launch("rideshare_sample_kernel");
}

}  // extern "C"
