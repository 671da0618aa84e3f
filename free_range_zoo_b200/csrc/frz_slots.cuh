// The row mapping and reductions shared by the kernels that work on rows of action slots (frz_policy.cu samples from
// them, frz_logprob.cu recomputes their log-probabilities).  Both must map a row and add its terms in exactly the same
// way: that is what makes the recomputed log-probability of a sampled slot the same bits as the sampler's.
//
// A group of G lanes serves a row; slot t belongs to lane t % G, in round t / G, so a round's loads of a group are
// consecutive elements.  G is 1 for C <= 16, else the smallest group that leaves at most 4 slots per lane, up to a warp
// (9 slots per lane for C <= 288).
#pragma once

#include "frz_common.cuh"

namespace frz {

constexpr int kMaxRowSlots = 32 * 9;

template <int G_, int PER_>
struct RowMapping {
  static constexpr int G = G_, PER = PER_;
};

// calls f(RowMapping<G, PER>{}) for the mapping of C (1 <= C <= kMaxRowSlots) and returns its result
template <class F>
inline int with_row_mapping(int C, F&& f) {
  if (C <= 16) return f(RowMapping<1, 16>{});
  if (C <= 32) return f(RowMapping<8, 4>{});
  if (C <= 64) return f(RowMapping<16, 4>{});
  if (C <= 128) return f(RowMapping<32, 4>{});
  return f(RowMapping<32, 9>{});
}

// the G-lane group's bits of a warp-wide predicate
template <int G>
__device__ __forceinline__ uint32_t group_ballot(bool predicate, int base) {
  const uint32_t all = __ballot_sync(kFullMask, predicate);
  return G == 32 ? all : (all >> base) & ((1u << G) - 1u);
}

// the softmax term of a slot given the row's max m: 0 for an illegal slot, exactly 1 at the max
__device__ __forceinline__ float slot_term(bool legal, float l, float m) {
  return legal ? (l == m ? 1.f : expf(l - m)) : 0.f;
}

// one round of the running sum in slot order: returns S + the group's inclusive scan of x at this lane, and adds the
// round's total to S (the same additions at every lane of the group)
template <int G>
__device__ __forceinline__ float running_sum(float x, int glane, float& S) {
#pragma unroll
  for (int o = 1; o < G; o <<= 1) {
    const float y = __shfl_up_sync(kFullMask, x, o, G);
    if (glane >= o) x += y;
  }
  const float running = S + x;
  S += __shfl_sync(kFullMask, x, G - 1, G);
  return running;
}

}  // namespace frz
