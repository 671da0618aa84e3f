/*
 * frz_logprob.h -- log-probabilities and entropies of chosen action slots under the masked softmax, and their gradient
 * with respect to the logits, on the device (additive to the C ABI of frz.h).  Domain-agnostic: it reads only arrays a
 * rollout records (the logits of a policy, the legal mask frz_<domain>_policy_actions wrote and the chosen slots).
 *
 * R rows of C slots (1 <= C <= 288).  Per row, with sums over the LEGAL slots only:
 *   m   = max legal logit,  e_i = exp(l_i - m),  S = sum e_i,  p_i = e_i / S
 *   log_prob = (l_s - m) - log S                           (s = slot[row])
 *   entropy  = log S - (1 / S) sum e_i (l_i - m)           (a legal slot with e_i = 0, a -inf logit, adds 0)
 *   backward, legal slot i:
 *     grad_i = g_lp ([i = s] - p_i) - g_H p_i ((l_i - m - log S) + entropy)      (g_lp [i = s] where p_i = 0)
 *   and exactly 0 on illegal slots.  Logits of illegal slots are never read.
 * A chosen slot that is illegal or outside [0, C) has log_prob = -inf (as a masked log_softmax gives) and [i = s] = 0
 * for every legal i.  A row with NaN or +inf in a legal slot, no legal slot, or every legal logit -inf has NaN log_prob
 * and entropy, and NaN gradient on its legal slots.
 *
 * The row mapping and the reductions are the sampler's (frz_policy.h, FRZ_POLICY_SAMPLE): the same lanes per row and
 * slots per lane for each C, m by the same group max, S by the same running sum with the same terms (exactly 1 at the
 * max).  So for the same logits and mask, the log_prob of a sampled slot is the same bits as the one the sampler
 * returned (a first-epoch probability ratio of exactly 1), and equal logits over n legal slots give log_prob = -logf(n)
 * and entropy = logf(n) exactly.  A row's outputs depend only on its own inputs and C: the same bits alone or in any
 * batch, with either mask format, with or without the entropy.
 *
 * The backward recomputes m, S and the entropy from the logits, and writes the whole gradient row in one pass; nothing
 * is kept between the two calls.  Offsets are 64-bit.  One launch each, no host read, no fault bits: capturable.
 * Reported through frz_last_error before any launch: FRZ_ERR_NULL for a missing required pointer, FRZ_ERR_SHAPE for
 * rows < 1, C outside [1, 288], row_stride < C or a pointer not aligned to its element, FRZ_ERR_UNSUPPORTED for an
 * unknown logits or mask type.
 */
#ifndef FRZ_LOGPROB_H_
#define FRZ_LOGPROB_H_

#include "frz_policy.h"

#ifdef __cplusplus
extern "C" {
#endif

#define FRZ_MASK_BYTES 0 /* legal: u8 / bool [R, C], nonzero = legal */
#define FRZ_MASK_BITS 1  /* legal: u32 [R, ceil(C / 32)], the packed layout of frz_policy.h (FRZ_POLICY_PACKED_LEGAL) */

#define FRZ_SLOT_LOG_PROB_MAX_SLOTS 288

typedef struct {
  int64_t rows;                /* R >= 1 */
  int32_t slots;               /* C, 1 .. FRZ_SLOT_LOG_PROB_MAX_SLOTS */
  int32_t row_stride;          /* elements between consecutive rows of logits, >= C */
  int32_t logits_type;         /* FRZ_LOGITS_F32 / FRZ_LOGITS_BF16 (frz_policy.h) */
  int32_t legal_type;          /* FRZ_MASK_* */
  const void* logits;          /* [R, row_stride], the first C of each row used */
  const void* legal;           /* FRZ_MASK_BYTES: u8 [R, C]; FRZ_MASK_BITS: u32 [R, ceil(C / 32)] */
  const int32_t* slot;         /* [R] chosen slots */
  float* log_prob;             /* forward out [R] */
  float* entropy;              /* forward out [R], or NULL */
  const float* grad_log_prob;  /* backward in [R], or NULL (= 0) */
  const float* grad_entropy;   /* backward in [R], or NULL (= 0) */
  void* grad_logits;           /* backward out, contiguous [R, C], of logits_type */
} FrzSlotLogProb;

/* forward: log_prob (and entropy unless NULL); grad_* and grad_logits are ignored */
int frz_slot_log_prob(const FrzSlotLogProb* args, void* stream);
/* backward: grad_logits from grad_log_prob and grad_entropy; log_prob and entropy are ignored */
int frz_slot_log_prob_backward(const FrzSlotLogProb* args, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FRZ_LOGPROB_H_ */
