// Log-probabilities and entropies of chosen slots under the masked softmax, and their gradient (frz_slot_log_prob,
// frz_slot_log_prob_backward, include/frz_logprob.h).
//
// The row mapping of frz_slots.cuh, as in the sampler (frz_policy.cu): a group of G lanes per row, slot t at lane t % G
// in round t / G, so a round's loads and gradient stores of a group are consecutive elements.
//   load     legality of the lane's slots (mask bytes, or a bit of the row's packed word), the legal logits, their group
//            max m (the sampler's shuffle order); the row is bad if a legal logit is NaN / +inf or m is -inf
//   sums     S by the sampler's running sum (same terms, same additions), so log S and the log-probability of a slot are
//            the sampler's bits; sum e_i (l_i - m) per lane in slot order, then over the group by a butterfly (the same
//            bits at every lane); entropy = log S - that / S
//   forward  the lane owning the chosen slot writes log_prob and entropy (lane 0 of the group when the slot is illegal)
//   backward every lane writes the gradient of its slots, 0 on illegal ones
// Each row's work depends only on its inputs and C: the same bits alone or in any batch.
#include <cuda_bf16.h>

#include <algorithm>

#include "frz_common.cuh"
#include "frz_logprob.h"
#include "frz_slots.cuh"

namespace frz {
namespace {

constexpr int kLogProbThreads = 256;

__device__ __forceinline__ float load_logit(const float* p) { return *p; }
__device__ __forceinline__ float load_logit(const __nv_bfloat16* p) { return __bfloat162float(*p); }
__device__ __forceinline__ void store_grad(float* p, float g) { *p = g; }
__device__ __forceinline__ void store_grad(__nv_bfloat16* p, float g) { *p = __float2bfloat16_rn(g); }

// one row as the lanes of its group hold it
template <int PER>
struct Row {
  uint32_t legal;  // bit j: slot j * G + glane is legal
  float l[PER];    // legal logits, -inf elsewhere
  float e[PER];    // exp(l - m), 0 on illegal slots
  float m, log_S, S, entropy;
  bool bad;
};

template <int G, int PER, class T, bool BITS>
__device__ __forceinline__ void load_row(const FrzSlotLogProb& P, int64_t row, bool active, int glane, int base,
                                         Row<PER>& r) {
  const int C = P.slots;
  const T* logits = static_cast<const T*>(P.logits) + row * P.row_stride;
  r.legal = 0u;
  r.m = -INFINITY;
  bool bad = false;
#pragma unroll
  for (int j = 0; j < PER; ++j) {
    const int t = j * G + glane;
    bool ok = false;
    if (active && t < C) {
      if (BITS) {
        // slots j * G .. j * G + G - 1 share word (j * G) / 32 (G divides 32)
        const uint32_t* words = static_cast<const uint32_t*>(P.legal) + row * ((C + 31) / 32);
        ok = (words[j * G / 32] >> (j * G % 32 + glane) & 1u) != 0u;
      } else {
        ok = static_cast<const uint8_t*>(P.legal)[row * C + t] != 0;
      }
    }
    r.legal |= uint32_t(ok) << j;
    r.l[j] = -INFINITY;
    if (ok) {
      r.l[j] = load_logit(logits + t);
      bad |= r.l[j] != r.l[j] || r.l[j] == INFINITY;
      r.m = fmaxf(r.m, r.l[j]);
    }
  }
#pragma unroll
  for (int o = G / 2; o >= 1; o >>= 1) r.m = fmaxf(r.m, __shfl_xor_sync(kFullMask, r.m, o, G));
  r.bad = group_ballot<G>(bad, base) != 0u || r.m == -INFINITY;
  float S = 0.f, weighted = 0.f;
#pragma unroll
  for (int j = 0; j < PER; ++j) {
    r.e[j] = slot_term(r.legal >> j & 1u, r.l[j], r.m);
    running_sum<G>(r.e[j], glane, S);
    if (r.e[j] != 0.f) weighted += r.e[j] * (r.l[j] - r.m);
  }
#pragma unroll
  for (int o = G / 2; o >= 1; o >>= 1) weighted += __shfl_xor_sync(kFullMask, weighted, o, G);
  r.S = S;
  r.log_S = logf(S);
  r.entropy = r.log_S - weighted / S;
}

// whole warps iterate together (ballots and shuffles need every lane); rows past the end are inactive
#define FRZ_FOR_EACH_ROW(P, G)                                                                                    \
  constexpr int kRowsPerWarp = 32 / G;                                                                            \
  const int lane = threadIdx.x & 31, glane = lane & (G - 1), base = lane - glane;                                \
  const int64_t warps = int64_t(gridDim.x) * (kLogProbThreads / 32);                                             \
  for (int64_t first = (int64_t(blockIdx.x) * (kLogProbThreads / 32) + (threadIdx.x >> 5)) * kRowsPerWarp;      \
       first < P.rows; first += warps * kRowsPerWarp)

template <int G, int PER, class T, bool BITS>
__global__ void __launch_bounds__(kLogProbThreads) slot_log_prob_kernel(const FrzSlotLogProb P) {
  FRZ_FOR_EACH_ROW(P, G) {
    const int64_t row = first + lane / G;
    const bool active = row < P.rows;
    const int s = active ? P.slot[row] : -1;
    Row<PER> r;
    load_row<G, PER, T, BITS>(P, row, active, glane, base, r);
    bool mine = false;
    float chosen = 0.f;
#pragma unroll
    for (int j = 0; j < PER; ++j) {
      if (j * G + glane == s && (r.legal >> j & 1u)) {
        mine = true;
        chosen = r.l[j];
      }
    }
    const bool found = group_ballot<G>(mine, base) != 0u;
    if (active && (mine || (!found && glane == 0))) {
      const float nan = __int_as_float(0x7fc00000);
      P.log_prob[row] = r.bad ? nan : (found ? (chosen - r.m) - r.log_S : -INFINITY);
      if (P.entropy != nullptr) P.entropy[row] = r.bad ? nan : r.entropy;
    }
  }
}

template <int G, int PER, class T, bool BITS>
__global__ void __launch_bounds__(kLogProbThreads) slot_log_prob_backward_kernel(const FrzSlotLogProb P) {
  FRZ_FOR_EACH_ROW(P, G) {
    const int64_t row = first + lane / G;
    const bool active = row < P.rows;
    const int s = active ? P.slot[row] : -1;
    const float g_lp = active && P.grad_log_prob != nullptr ? P.grad_log_prob[row] : 0.f;
    const float g_h = active && P.grad_entropy != nullptr ? P.grad_entropy[row] : 0.f;
    Row<PER> r;
    load_row<G, PER, T, BITS>(P, row, active, glane, base, r);
    if (!active) continue;
    T* grad = static_cast<T*>(P.grad_logits) + row * P.slots;
#pragma unroll
    for (int j = 0; j < PER; ++j) {
      const int t = j * G + glane;
      if (t < P.slots) {
        float g = 0.f;
        if (r.legal >> j & 1u) {
          if (r.bad) {
            g = __int_as_float(0x7fc00000);
          } else {
            const float p = r.e[j] / r.S;
            g = g_lp * ((t == s ? 1.f : 0.f) - p);
            if (p != 0.f) g = g - g_h * (p * (((r.l[j] - r.m) - r.log_S) + r.entropy));
          }
        }
        store_grad(grad + t, g);
      }
    }
  }
}

#undef FRZ_FOR_EACH_ROW

template <int G, int PER, bool BACKWARD, class T, bool BITS>
void launch_typed(const FrzSlotLogProb& P, cudaStream_t stream) {
  const int64_t work_ctas = (P.rows * G + kLogProbThreads - 1) / kLogProbThreads;
  const int grid = persistent_grid(int(std::min<int64_t>(work_ctas, INT32_MAX)), 2048 / kLogProbThreads);
  if (BACKWARD)
    slot_log_prob_backward_kernel<G, PER, T, BITS><<<grid, kLogProbThreads, 0, stream>>>(P);
  else
    slot_log_prob_kernel<G, PER, T, BITS><<<grid, kLogProbThreads, 0, stream>>>(P);
}

template <int G, int PER, bool BACKWARD>
void launch(const FrzSlotLogProb& P, cudaStream_t stream) {
  const bool bits = P.legal_type == FRZ_MASK_BITS;
  if (P.logits_type == FRZ_LOGITS_BF16) {
    if (bits)
      launch_typed<G, PER, BACKWARD, __nv_bfloat16, true>(P, stream);
    else
      launch_typed<G, PER, BACKWARD, __nv_bfloat16, false>(P, stream);
  } else {
    if (bits)
      launch_typed<G, PER, BACKWARD, float, true>(P, stream);
    else
      launch_typed<G, PER, BACKWARD, float, false>(P, stream);
  }
}

bool aligned(const void* p, size_t bytes) { return reinterpret_cast<uintptr_t>(p) % bytes == 0; }

template <bool BACKWARD>
int run(const FrzSlotLogProb* P, void* stream) {
  const char* what = BACKWARD ? "frz_slot_log_prob_backward" : "frz_slot_log_prob";
  if (P == nullptr) {
    set_error("%s: NULL argument block", what);
    return FRZ_ERR_NULL;
  }
  if (P->logits == nullptr || P->legal == nullptr || P->slot == nullptr ||
      (BACKWARD ? P->grad_logits == nullptr : P->log_prob == nullptr)) {
    set_error(BACKWARD ? "%s: NULL logits / legal / slot / grad_logits" : "%s: NULL logits / legal / slot / log_prob",
              what);
    return FRZ_ERR_NULL;
  }
  if (P->rows < 1 || P->slots < 1 || P->slots > FRZ_SLOT_LOG_PROB_MAX_SLOTS) {
    set_error("%s: unsupported shape rows=%lld slots=%d", what, static_cast<long long>(P->rows), P->slots);
    return FRZ_ERR_SHAPE;
  }
  if (P->row_stride < P->slots) {
    set_error("%s: row_stride=%d < slots=%d", what, P->row_stride, P->slots);
    return FRZ_ERR_SHAPE;
  }
  if (P->logits_type != FRZ_LOGITS_F32 && P->logits_type != FRZ_LOGITS_BF16) {
    set_error("%s: unknown logits type %d", what, P->logits_type);
    return FRZ_ERR_UNSUPPORTED;
  }
  if (P->legal_type != FRZ_MASK_BYTES && P->legal_type != FRZ_MASK_BITS) {
    set_error("%s: unknown legal type %d", what, P->legal_type);
    return FRZ_ERR_UNSUPPORTED;
  }
  const size_t logit_bytes = P->logits_type == FRZ_LOGITS_BF16 ? 2 : 4;
  const bool ok = aligned(P->logits, logit_bytes) && aligned(P->legal, P->legal_type == FRZ_MASK_BITS ? 4 : 1) &&
                  aligned(P->slot, 4) &&
                  (BACKWARD ? aligned(P->grad_log_prob, 4) && aligned(P->grad_entropy, 4) &&
                                  aligned(P->grad_logits, logit_bytes)
                            : aligned(P->log_prob, 4) && aligned(P->entropy, 4));
  if (!ok) {
    set_error("%s: a pointer is not aligned to its element type", what);
    return FRZ_ERR_SHAPE;
  }
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  with_row_mapping(P->slots, [&](auto map) {
    using M = decltype(map);
    launch<M::G, M::PER, BACKWARD>(*P, s);
    return 0;
  });
  return check_launch(BACKWARD ? "slot_log_prob_backward_kernel" : "slot_log_prob_kernel");
}

}  // namespace
}  // namespace frz

extern "C" {

int frz_slot_log_prob(const FrzSlotLogProb* args, void* stream) { return frz::run<false>(args, stream); }

int frz_slot_log_prob_backward(const FrzSlotLogProb* args, void* stream) { return frz::run<true>(args, stream); }

}  // extern "C"
