/*
 * frz_returns.h -- GAE advantages and value targets of a recorded rollout, on the device (additive to the C ABI of
 * frz.h).  Domain-agnostic: it reads only the arrays a rollout records, not an environment.
 *
 * A rollout of T steps, B environments and A agents; a column is one (b, a) pair.  Arrays are contiguous:
 *   rewards       f32 [T, B, A]   r[t]: the reward step t returned
 *   values        [T, B, A]       v[t]: the value of the observation BEFORE step t
 *   next_values   [B, A]          the value of the observation after step T-1
 *   final_values  [T, B, A]       the value of the final observation of step t, or NULL; read only where
 *                                 trunc[t] && !term[t]
 *   terminated    u8 [T, B]       term[t] / trunc[t]: the episode ended at step t (the flags the step returned; with
 *   truncated     u8 [T, B]       autoreset the step's own flags, the observation after it belonging to the restart)
 * values, next_values and final_values share one type, f32 or bf16 (value_type); bf16 is widened on load.  Flags are
 * tested against zero.  Outputs are f32 [T, B, A].
 *
 *   nv[t]    = 0               if term[t]
 *            = final_v[t]      if trunc[t] && !term[t]    (0 when final_values is NULL: truncation as termination)
 *            = v[t+1]          otherwise, t < T-1
 *            = next_v          otherwise, t = T-1
 *   c[t]     = gamma * lambda * (1 - (term[t] | trunc[t]))
 *   delta[t] = (r[t] + gamma * nv[t]) - v[t]
 *   A[t]     = delta[t] + c[t] * A[t+1],   A[T] = 0      -> advantages
 *   R[t]     = A[t] + v[t]                               -> returns (optional)
 *
 * Under same-step autoreset the observation after a finished step belongs to the restarted episode, so v[t+1] never
 * bootstraps it.  Without autoreset the done flags of a finished environment stay set on every later step, each of which
 * is then its own one-step terminated episode.
 *
 * Invariance: a column's outputs depend only on T, gamma, lambda and that column's inputs -- never on B, A or the launch
 * geometry -- so a column computed alone and in any batch gives the same bits.  NaN / inf inputs propagate as in the
 * literal recurrence (0 * NaN is NaN, also across an episode boundary).
 *
 * One launch, no host read: capturable.  No fault bits.  Reported through frz_last_error before any launch:
 * FRZ_ERR_NULL for a missing required pointer, FRZ_ERR_SHAPE for T, B or A < 1 or B * A > INT32_MAX,
 * FRZ_ERR_UNSUPPORTED for an unknown value_type or a gamma / lambda that is not finite or outside [0, 1].
 */
#ifndef FRZ_RETURNS_H_
#define FRZ_RETURNS_H_

#include "frz.h"

#ifdef __cplusplus
extern "C" {
#endif

#define FRZ_VALUES_F32 0
#define FRZ_VALUES_BF16 1

typedef struct {
  int32_t T, B, A;
  int32_t value_type;          /* FRZ_VALUES_* */
  float gamma, lambda;
  const float* rewards;        /* f32 [T, B, A] */
  const void* values;          /* [T, B, A] of value_type */
  const void* next_values;     /* [B, A] of value_type */
  const void* final_values;    /* [T, B, A] of value_type, or NULL */
  const uint8_t* terminated;   /* [T, B] */
  const uint8_t* truncated;    /* [T, B] */
  float* advantages;           /* f32 [T, B, A] out */
  float* returns;              /* f32 [T, B, A] out, or NULL */
} FrzAdvantages;

int frz_advantages(const FrzAdvantages* gae, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FRZ_RETURNS_H_ */
