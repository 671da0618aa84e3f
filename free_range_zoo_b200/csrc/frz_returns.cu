// GAE advantages and returns of a recorded rollout (frz_advantages, include/frz_returns.h).
//
// A column's T steps are cut into S = min(32, ceil(T / 16)) segments of L = ceil(T / S) steps.  S and L depend on T
// only, which is what keeps a column's bits independent of B, A and the grid.  A CTA covers 32 * G consecutive columns
// with S * G warps: warp (g, s), lane j owns column c0 + 32 g + j for the steps of segment s, so the loads of one step by
// a warp are 32 consecutive elements.
//   phase 1  walk the segment backwards composing the affine map A_start = P + Q * A_end (P <- delta + c P, Q <- c Q);
//            while L <= 16 (T <= 512) the step's delta, v and done bit stay in registers
//   combine  (P, Q) of every segment through shared memory; segment s starts phase 2 from A_end = the composition of the
//            later segments, applied last to first (at most 31 steps, always in the same order)
//   phase 2  walk again from that carry writing A and R.  With L > 16 the step terms are re-read and recomputed by the
//            same operations (same bits); phase 1 has just read them, so they mostly come from L2.
#include <cuda_bf16.h>

#include <algorithm>
#include <cmath>

#include "frz_common.cuh"
#include "frz_returns.h"

namespace frz {
namespace {

constexpr int kMaxSegments = 32;
constexpr int kStepsPerSegment = 16;  // target L, and the most steps phase 1 keeps in registers
constexpr int kTargetWarps = 8;       // S * G when S < 8
constexpr int kMaxThreads = kMaxSegments * 32;

struct Launch {
  FrzAdvantages gae;
  int64_t columns;  // B * A
  int32_t segments, length;  // S, L
  int32_t groups;            // G: 32-column groups per CTA
  float gl;                  // gamma * lambda
};

__device__ __forceinline__ float widen(const float* p, int64_t i) { return p[i]; }
__device__ __forceinline__ float widen(const __nv_bfloat16* p, int64_t i) { return __bfloat162float(p[i]); }

// delta of step t (element `row`, flags at `flag`) given v = v[t] and v_next = v[t + 1] (next_values at T - 1)
template <class V, bool FINAL>
__device__ __forceinline__ float step_delta(const Launch& L, int64_t row, int64_t flag, float v, float v_next,
                                            bool& done) {
  const bool term = L.gae.terminated[flag] != 0, trunc = L.gae.truncated[flag] != 0;
  done = term || trunc;
  float nv = v_next;
  if (term)
    nv = 0.f;
  else if (trunc)
    nv = FINAL ? widen(static_cast<const V*>(L.gae.final_values), row) : 0.f;
  return (L.gae.rewards[row] + L.gae.gamma * nv) - v;
}

template <class V, bool FINAL, bool CACHED>
__global__ void __launch_bounds__(kMaxThreads) advantages_kernel(const Launch L) {
  __shared__ float s_p[kMaxThreads], s_q[kMaxThreads];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int S = L.segments, s = warp % S, g = warp / S;
  const int64_t C = L.columns;
  const int64_t col = (int64_t(blockIdx.x) * L.groups + g) * 32 + lane;
  const bool active = col < C;
  const int T = L.gae.T, start = s * L.length, end = min(T, start + L.length), len = end - start;
  const int64_t env = active ? col / L.gae.A : 0, B = L.gae.B;
  const V* values = static_cast<const V*>(L.gae.values);
  const float gl = L.gl;

  // phase 1
  float P = 0.f, Q = 1.f;
  float delta[CACHED ? kStepsPerSegment : 1], v_at[CACHED ? kStepsPerSegment : 1];
  uint32_t done_bits = 0u;
  if (active) {
    float v_next = end == T ? widen(static_cast<const V*>(L.gae.next_values), col) : widen(values, int64_t(end) * C + col);
    if (CACHED) {
#pragma unroll
      for (int k = kStepsPerSegment - 1; k >= 0; --k) {
        if (k < len) {
          const int t = start + k;
          const int64_t row = int64_t(t) * C + col;
          const float v = widen(values, row);
          bool done;
          const float d = step_delta<V, FINAL>(L, row, int64_t(t) * B + env, v, v_next, done);
          const float c = done ? 0.f : gl;
          P = d + c * P;
          Q = c * Q;
          delta[k] = d;
          v_at[k] = v;
          done_bits |= uint32_t(done) << k;
          v_next = v;
        }
      }
    } else {
#pragma unroll 4
      for (int t = end - 1; t >= start; --t) {
        const int64_t row = int64_t(t) * C + col;
        const float v = widen(values, row);
        bool done;
        const float d = step_delta<V, FINAL>(L, row, int64_t(t) * B + env, v, v_next, done);
        const float c = done ? 0.f : gl;
        P = d + c * P;
        Q = c * Q;
        v_next = v;
      }
    }
  }

  // combine: A_end of segment s = P_{s+1} + Q_{s+1} (P_{s+2} + Q_{s+2} (... P_{S-1}))
  s_p[threadIdx.x] = P;
  s_q[threadIdx.x] = Q;
  __syncthreads();
  float carry = 0.f;
  for (int k = S - 1; k > s; --k) {
    const int i = (g * S + k) * 32 + lane;
    carry = s_p[i] + s_q[i] * carry;
  }
  if (!active) return;

  // phase 2
  float* advantages = L.gae.advantages;
  float* returns = L.gae.returns;
  if (CACHED) {
#pragma unroll
    for (int k = kStepsPerSegment - 1; k >= 0; --k) {
      if (k < len) {
        const int64_t row = int64_t(start + k) * C + col;
        const float c = (done_bits >> k & 1u) ? 0.f : gl;
        carry = delta[k] + c * carry;
        __stcs(advantages + row, carry);
        if (returns != nullptr) __stcs(returns + row, carry + v_at[k]);
      }
    }
  } else {
    float v_next = end == T ? widen(static_cast<const V*>(L.gae.next_values), col) : widen(values, int64_t(end) * C + col);
#pragma unroll 4
    for (int t = end - 1; t >= start; --t) {
      const int64_t row = int64_t(t) * C + col;
      const float v = widen(values, row);
      bool done;
      const float d = step_delta<V, FINAL>(L, row, int64_t(t) * B + env, v, v_next, done);
      const float c = done ? 0.f : gl;
      carry = d + c * carry;
      __stcs(advantages + row, carry);
      if (returns != nullptr) __stcs(returns + row, carry + v);
      v_next = v;
    }
  }
}

template <class V, bool FINAL>
void launch_typed(const Launch& launch, int grid, int threads, cudaStream_t stream) {
  if (launch.length <= kStepsPerSegment)
    advantages_kernel<V, FINAL, true><<<grid, threads, 0, stream>>>(launch);
  else
    advantages_kernel<V, FINAL, false><<<grid, threads, 0, stream>>>(launch);
}

bool unit_interval(float x) { return std::isfinite(x) && x >= 0.f && x <= 1.f; }

}  // namespace
}  // namespace frz

extern "C" {

int frz_advantages(const FrzAdvantages* gae, void* stream) {
  using namespace frz;
  const char* what = "frz_advantages";
  if (gae == nullptr) {
    set_error("%s: NULL argument block", what);
    return FRZ_ERR_NULL;
  }
  if (gae->rewards == nullptr || gae->values == nullptr || gae->next_values == nullptr || gae->terminated == nullptr ||
      gae->truncated == nullptr || gae->advantages == nullptr) {
    set_error("%s: NULL rewards / values / next_values / terminated / truncated / advantages", what);
    return FRZ_ERR_NULL;
  }
  if (gae->T < 1 || gae->B < 1 || gae->A < 1 || int64_t(gae->B) * gae->A > INT32_MAX) {
    set_error("%s: unsupported shape T=%d B=%d A=%d", what, gae->T, gae->B, gae->A);
    return FRZ_ERR_SHAPE;
  }
  if (gae->value_type != FRZ_VALUES_F32 && gae->value_type != FRZ_VALUES_BF16) {
    set_error("%s: unknown value type %d", what, gae->value_type);
    return FRZ_ERR_UNSUPPORTED;
  }
  if (!unit_interval(gae->gamma) || !unit_interval(gae->lambda)) {
    set_error("%s: gamma=%g and lambda=%g must be finite and in [0, 1]", what, double(gae->gamma), double(gae->lambda));
    return FRZ_ERR_UNSUPPORTED;
  }
  Launch launch;
  launch.gae = *gae;
  launch.columns = int64_t(gae->B) * gae->A;
  launch.segments = std::min(kMaxSegments, (gae->T + kStepsPerSegment - 1) / kStepsPerSegment);
  launch.length = (gae->T + launch.segments - 1) / launch.segments;
  launch.groups = std::max(1, kTargetWarps / launch.segments);
  launch.gl = gae->gamma * gae->lambda;
  const int64_t per_cta = int64_t(32) * launch.groups;
  const int grid = int((launch.columns + per_cta - 1) / per_cta);
  const int threads = 32 * launch.segments * launch.groups;
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  const bool final = gae->final_values != nullptr;
  if (gae->value_type == FRZ_VALUES_BF16) {
    if (final)
      launch_typed<__nv_bfloat16, true>(launch, grid, threads, s);
    else
      launch_typed<__nv_bfloat16, false>(launch, grid, threads, s);
  } else {
    if (final)
      launch_typed<float, true>(launch, grid, threads, s);
    else
      launch_typed<float, false>(launch, grid, threads, s);
  }
  return check_launch("advantages_kernel");
}

}  // extern "C"
