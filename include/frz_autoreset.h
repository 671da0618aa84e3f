/*
 * frz_autoreset.h -- same-step autoreset of finished environments (additive to the C ABI of frz.h).
 *
 * A training loop keeps one batch stepping for millions of steps; once every environment is finished a step is a
 * no-op (FrzControl.alive), and restarting only the finished ones through frz_<domain>_reset costs a host-built mask
 * and a refresh pass over the whole batch.  frz_autoreset runs after a step, on the same stream (so also inside a CUDA
 * graph), and restarts exactly the environments the step finished, with work proportional to their number plus one
 * pass over the batch's done flags.
 *
 * A restart is a list of row copies: every restarted environment's rows go back to what the last full reset left
 * there.  State rows come from the caller's init_* arrays; observation, mask and count rows from a snapshot the caller
 * took right after that reset (the refresh of a reset depends on the restored state alone, so the snapshot is what a
 * refresh of the restored state would write); AEC fields such as the done flags and the cumulative rewards are zeroed.
 * The library knows row descriptors only, never domains.
 *
 * A learner that bootstraps a truncated episode from the value of its last observation needs that observation after
 * the restart has overwritten it.  A row with a `keep` array has its current bytes copied there before it is restored:
 * the lane that restores a word loads the old word first, so the copy costs no launch and no ordering, and moves the
 * row's bytes once more for finished environments only.
 *
 * One call, for B = parallel_envs environments:
 *  1. scan (one pass over B): done[b] = terminated[b] | truncated[b]; step_terminated / step_truncated / done receive
 *     copies of the flags the step produced (the live flags are zeroed by the restart); for finished environments
 *     episode_return[b] = cumulative_rewards[b] and episode_length[b] = num_moves[b] (other rows are left as they
 *     are); the finished indices are compacted into finished[0 .. *finished_count) in no particular order.  The
 *     batch-wide flags of FrzControl are republished as a refresh would: alive = 3 (after the restart no environment
 *     is finished) and agents_with_tasks = OR over agents with a task, from agent_task_count of the environments that
 *     did not finish and reset_agent_task_count of those that did.  The step counter is left alone: restarted
 *     environments keep drawing with the global step counter, as after frz_<domain>_reset.
 *  2. restore: every row of every listed environment is copied from src (or zeroed), after its current value has
 *     been copied to keep where the row has one.
 * No host read: capturable.
 */
#ifndef FRZ_AUTORESET_H_
#define FRZ_AUTORESET_H_

#include "frz.h"

#ifdef __cplusplus
extern "C" {
#endif

#define FRZ_AUTORESET_MAX_ROWS 32

/* One per-environment array restored by a restart: keep[b] <- dst[b] (if keep), then dst[b] <- src[b] (or zeros),
   `bytes` bytes per environment. */
typedef struct {
  void* dst;              /* device [B, bytes] */
  const void* src;        /* device [B, bytes], or NULL: zero the row */
  int64_t bytes;          /* > 0 */
  void* keep;             /* device [B, bytes], or NULL: before a finished environment's row is restored, its current
                             bytes are copied to keep[b] */
} FrzAutoresetRow;

typedef struct {
  const uint8_t* terminated;             /* device [B]: the done flags the step wrote (restored by a row, normally
                                            zeroed) */
  const uint8_t* truncated;              /* device [B] */
  uint8_t* step_terminated;              /* device [B] out: copy of terminated */
  uint8_t* step_truncated;               /* device [B] out: copy of truncated */
  uint8_t* done;                         /* device [B] out: terminated | truncated */
  const float* cumulative_rewards;       /* device [B, A], read before the rows are restored */
  float* episode_return;                 /* device [B, A] out, written where done */
  const int32_t* num_moves;              /* device [B] */
  int32_t* episode_length;               /* device [B] out, written where done */
  const int32_t* agent_task_count;       /* device [B, A], or NULL: the domain publishes no agents_with_tasks (0) */
  const int32_t* reset_agent_task_count; /* device [B, A]: the counts a restart restores (NULL with the previous) */
  FrzControl* control;
  int32_t* finished;                     /* device scratch int32 [B]: compacted indices of the finished environments */
  int32_t* finished_count;               /* device int32 [1] */
  uint32_t* scratch;                     /* device uint32 [2], zero before the first call; every call leaves it zero */
  const FrzAutoresetRow* rows;           /* host array of row_count descriptors (copied into the launch) */
  int32_t row_count;                     /* <= FRZ_AUTORESET_MAX_ROWS */
  int32_t num_agents;                    /* A, 1 .. FRZ_MAX_AGENTS */
} FrzAutoreset;

/* Restart every environment of `parallel_envs` that is terminated or truncated (two launches on `stream`). */
int frz_autoreset(const FrzAutoreset* autoreset, int32_t parallel_envs, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FRZ_AUTORESET_H_ */
