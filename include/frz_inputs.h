/*
 * frz_inputs.h -- policy inputs on the device: the observations of every environment and agent encoded into fixed-width
 * float rows whose task rows line up with the action slots of frz_policy.h (additive to the C ABI of frz.h).
 *
 * One call writes two arrays, f32 or bf16 (output_type), for B = parallel_envs environments and A agents in the order of
 * the [B, A, 2] action table:
 *   agent [B, A, Fa]      the agent's own self columns, then the observed columns of every agent of its `others` view,
 *                         in the view's order (the other agents of the same kind, ascending); the shorter cybersecurity
 *                         kind is zero-padded to Fa
 *   tasks [B, V, T, Ft]   row t = padded task row t = action slot t.  Column 0 is a flag: 1 iff row t is a live task
 *                         (t < env_task_count[b]) that view v may see; then the source columns of the row.  A row with
 *                         flag 0 is all zeros and its source row is never read.  V = 1 when every agent sees the same
 *                         tasks (the policy broadcasts over agents), V = A when views differ.
 *
 *   domain          Fa                                          T      V   Ft: flag + source columns
 *   wildfire        4 + (A-1) * popcount(observed)              H*W    1   5: y, x, fire type, intensity
 *   rideshare       4 + (A-1) * popcount(observed) = 4 A        K      1   9: y, x, dest_y, dest_x, accepted_by,
 *                                                                                riding_by, fare, entered
 *   cybersecurity   max over the kinds with agents of           N      A   3: state, criticality; flag 0 for a
 *                   own columns + (kind size - 1) * observed                  defender under partial observability whose
 *                   (attackers 2 own columns, defenders 3)                    monitored byte is 0
 *
 * Every output column is an affine map of the engine's value v, computed in f32 as float(v + offset) * scale (integer
 * sources add the offset as integers, float sources in f32); bf16 outputs round that f32 once, to nearest even.  A column
 * whose `pad_is_none` bit is set reads FRZ_PAD ("nobody") as -1 first, so with offset 1 it maps to exactly 0.  There is
 * no clamping.  The scales and offsets are the caller's (the Python domains derive them from the bounds of
 * observation_space); the library only knows which source column feeds which output.
 *
 * Sources (the Frz<Domain>Buffers fields): self_obs (wildfire f32, rideshare int32) / attacker_self / defender_self,
 * task_obs, env_task_count and, for cybersecurity with FRZ_INPUTS_PARTIALLY_OBSERVABLE, monitored.  Pointing those fields at
 * copies (e.g. the final observations an autoreset keeps) encodes the copies.
 *
 * One launch, no host read: capturable.  NULL pointers, an unknown output type, B <= 0 and widths that do not match the
 * configuration are reported through frz_last_error before any launch.  No fault bits.
 */
#ifndef FRZ_INPUTS_H_
#define FRZ_INPUTS_H_

#include "frz.h"

#ifdef __cplusplus
extern "C" {
#endif

#define FRZ_INPUTS_F32 0
#define FRZ_INPUTS_BF16 1
#define FRZ_INPUTS_MAX_COLUMNS 8
/* cybersecurity constructed with partially_observable=True: a defender's view hides the task rows unless it monitored */
#define FRZ_INPUTS_PARTIALLY_OBSERVABLE 0x1u

/* The normalisation of one source array's columns. */
typedef struct {
  float scale[FRZ_INPUTS_MAX_COLUMNS];
  int32_t offset[FRZ_INPUTS_MAX_COLUMNS];
  int32_t columns;       /* columns of the source array (checked) */
  uint32_t observed;     /* self arrays: bit c = column c of the other agents is in the `others` view */
  uint32_t pad_is_none;  /* bit c = FRZ_PAD in column c means "none" and is read as -1 */
  int32_t reserved;
} FrzInputColumns;

typedef struct {
  void* agent;            /* device [B, A, agent_width] of output_type */
  void* tasks;            /* device [B, views, task_rows, task_width] of output_type */
  int32_t output_type;    /* FRZ_INPUTS_* */
  int32_t agent_width;    /* Fa (checked) */
  int32_t task_width;     /* Ft (checked) */
  int32_t views;          /* V (checked) */
  int32_t task_rows;      /* T (checked) */
  uint32_t flags;         /* FRZ_INPUTS_PARTIALLY_OBSERVABLE */
  FrzInputColumns self_columns[2]; /* [0] self_obs (cybersecurity: attacker_self), [1] cybersecurity defender_self */
  FrzInputColumns task_columns;    /* task_obs */
} FrzPolicyInputs;

int frz_wildfire_policy_inputs(const FrzWildfireParams* params, const FrzWildfireBuffers* io, int32_t parallel_envs,
                               const FrzPolicyInputs* inputs, void* stream);
int frz_rideshare_policy_inputs(const FrzRideshareParams* params, const FrzRideshareBuffers* io,
                                int32_t parallel_envs, const FrzPolicyInputs* inputs, void* stream);
int frz_cyber_policy_inputs(const FrzCyberParams* params, const FrzCyberBuffers* io, int32_t parallel_envs,
                            const FrzPolicyInputs* inputs, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FRZ_INPUTS_H_ */
