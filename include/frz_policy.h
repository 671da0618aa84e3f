/*
 * frz_policy.h -- policy actions on the device from logits over a fixed-width action layout (additive to the C ABI of
 * frz.h).
 *
 * The engine's action table holds, per environment and agent, a (choice index, action id) pair whose encoding differs
 * by domain: the choice index counts only the choices the agent has in that environment, and the id depends on the
 * choice (a rideshare task's id is its passenger's state).  A learned policy instead scores a fixed number C of SLOTS
 * per agent, aligned with the rows of the padded task observations:
 *
 *   domain          C               slot t < T (T = task capacity)                 extra slots
 *   wildfire        H*W + 1         act on env-local task t (row t of task_obs)    H*W: noop
 *   rideshare       K + 1           act on table row t, with the id the            K: noop
 *                                   passenger's state requires (0 / 1 / 2)
 *   cybersecurity   N + 3           attack / move to node t                        N: noop, N+1: patch,
 *                   (every agent)                                                  N+2: monitor (never for attackers)
 *
 * Legality and decoding: for environment b and agent a the legal slots correspond one to one, in increasing slot
 * order, to the choices of the reference's action space of (b, a) -- wildfire: the set bits of action_mask (every live
 * task with show_bad_actions) then the noop; rideshare: the set bits of task_mask then the noop; cybersecurity: the
 * nodes if the agent may act on them, the noop, and for a defender that may act patch (hidden at the home node unless
 * show_bad_actions) and monitor.  The slot that maps to choice k decodes to (k, id of choice k).  The noop is always
 * legal.  Agents are in the order of the [B, A, 2] action table.
 *
 * One call, one launch, for B = parallel_envs environments and A agents (rows = B * A):
 *   FRZ_POLICY_SAMPLE  slot[row] ~ softmax of the logits restricted to the legal slots, by inverse CDF: m = max over
 *                      legal slots, S = sum exp(l - m) in slot order, u = the uniform frz_<domain>_sample_actions draws
 *                      for the row (Philox(sampler_seed; global env, step, 0xC0000000 | agent), word 0), and the chosen
 *                      slot is the first legal slot whose running sum exceeds u * S (the last legal slot if rounding
 *                      leaves none).  log_prob[row] = (l - m) - log(S).  With equal logits every term is exactly 1, so
 *                      the choice is exactly the one frz_<domain>_sample_actions makes with the same seed.  The decoded
 *                      action is written to io->actions.
 *   FRZ_POLICY_DECODE  io->actions[row] <- the decoded action of the caller's slot[row] (logits are not read).
 *   FRZ_POLICY_LEGAL   legal[row, t] <- 1 iff slot t is legal (nothing else is written).
 * legal (optional in the first two modes) receives the same mask.  bf16 logits are widened to f32 on load.
 *
 * Faults (bits of FrzControl.error_word; the row is decoded as the noop): FRZ_FAULT_BAD_LOGITS when a legal slot's logit
 * is NaN or +inf or every legal logit is -inf (its log_prob is NaN), FRZ_FAULT_ILLEGAL_SLOT when a DECODE slot is out of
 * [0, C) or illegal.  Logits of illegal slots are never read.
 *
 * No host read: capturable.  NULL pointers and shape errors are reported through frz_last_error before any launch.
 */
#ifndef FRZ_POLICY_H_
#define FRZ_POLICY_H_

#include "frz.h"

#ifdef __cplusplus
extern "C" {
#endif

#define FRZ_FAULT_BAD_LOGITS 0x10u    /* NaN / +inf logit in a legal slot, or every legal logit -inf */
#define FRZ_FAULT_ILLEGAL_SLOT 0x20u  /* FRZ_POLICY_DECODE: slot outside [0, C) or not legal */

#define FRZ_POLICY_SAMPLE 0
#define FRZ_POLICY_DECODE 1
#define FRZ_POLICY_LEGAL 2

#define FRZ_LOGITS_F32 0
#define FRZ_LOGITS_BF16 1

typedef struct {
  int32_t mode;          /* FRZ_POLICY_* */
  int32_t logits_type;   /* FRZ_LOGITS_* */
  const void* logits;    /* device [B, A, row_stride], the first `slots` of each row used (SAMPLE) */
  int32_t slots;         /* C of the configuration (checked) */
  int32_t row_stride;    /* elements between consecutive rows of logits, >= slots */
  int32_t* slot;         /* device int32 [B, A]: out (SAMPLE), in (DECODE) */
  float* log_prob;       /* device f32 [B, A] out (SAMPLE), or NULL */
  uint8_t* legal;        /* device u8 [B, A, slots] out, or NULL (required for LEGAL) */
  uint64_t sampler_seed; /* Philox key of SAMPLE, as for frz_<domain>_sample_actions */
} FrzPolicyActions;

int frz_wildfire_policy_actions(const FrzWildfireParams* params, const FrzWildfireBuffers* io, int32_t parallel_envs,
                                const FrzPolicyActions* policy, void* stream);
int frz_rideshare_policy_actions(const FrzRideshareParams* params, const FrzRideshareBuffers* io,
                                 int32_t parallel_envs, const FrzPolicyActions* policy, void* stream);
int frz_cyber_policy_actions(const FrzCyberParams* params, const FrzCyberBuffers* io, int32_t parallel_envs,
                             const FrzPolicyActions* policy, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FRZ_POLICY_H_ */
