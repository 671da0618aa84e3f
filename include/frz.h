/*
 * frz.h -- C ABI of libfrz.so, the B200 (sm_100a) batched environment-step engine for free-range-zoo.
 *
 * The reference has no FFI: its "plugin" boundary is the set of BatchedAECEnv hooks
 *   step_environment()   free_range_zoo/utils/env.py:197-201
 *   update_actions()     free_range_zoo/utils/env.py:273-276
 *   update_observations()free_range_zoo/utils/env.py:278-281
 * plus the AEC bookkeeping of BatchedAECEnv.step (utils/env.py:203-242).  Each frz_<domain>_step below replaces the
 * bodies of those hooks for one domain with ONE fused kernel launch; frz_<domain>_reset replaces
 * BatchedAECEnv.reset / reset_batches (utils/env.py:95-189) on the device side.
 *
 * Conventions
 *  - Plain C, no torch types.  Every pointer inside a Frz*Buffers struct is a DEVICE pointer owned by the caller
 *    (a torch tensor's data_ptr()); the library allocates nothing, frees nothing and keeps no device state (the one
 *    exception: the timing-disabled CUDA events of frz_<domain>_step_host, owned by a FrzHostPipeline handle).
 *  - Every call works on the CURRENT CUDA device (cudaSetDevice by the caller): buffers, stream and control block must
 *    belong to it.  Launch geometry (SM count, resident CTAs) is queried per device.
 *  - frz_<domain>_buffer_bytes() gives the size of every array of a Frz*Buffers struct, so a C caller can allocate
 *    them without reading the Python host code.
 *  - Every call only enqueues work on the caller's cudaStream_t (passed as void*): no synchronisation, no
 *    allocation, no host read-back -> capturable in a CUDA graph.  The step counter / seed / done flags live in the
 *    device-side FrzControl block and are advanced by the kernels themselves, so graph replays need no new arguments.
 *  - Return value: FRZ_OK or a FrzStatus error; the message is available from frz_last_error() (thread-local).
 *    Data-dependent faults (the reference's ValueErrors, e.g. cybersecurity.py:341-363) set bits in
 *    FrzControl.error_word on the device and are read lazily by the host, never on the step path.
 *  - Layouts are environment-major ("[B, ...]", B = parallel_envs) with the reference's dtypes
 *    (int32 / float32 / uint8 for bool), so state tensors are directly the reference's State fields.
 */
#ifndef FRZ_H_
#define FRZ_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FRZ_ABI_VERSION 4

#define FRZ_MAX_AGENTS 32      /* agents per environment (one warp lane each) */
#define FRZ_MAX_EQUIPMENT 8    /* wildfire equipment states */
#define FRZ_MAX_CAPACITIES 8   /* wildfire tank sizes */
#define FRZ_MAX_CELLS 256      /* wildfire H*W */
#define FRZ_MAX_NODES 32       /* cybersecurity subnetworks */
#define FRZ_MAX_NET_STATES 16  /* cybersecurity states per subnetwork */
#define FRZ_MAX_PASSENGERS 64  /* rideshare passengers simultaneously tracked per environment */
#define FRZ_PAD (-100)         /* padding value of padded observations (the reference pads with -100) */

typedef enum {
  FRZ_OK = 0,
  FRZ_ERR_NULL = 1,        /* a required pointer is NULL */
  FRZ_ERR_SHAPE = 2,       /* B <= 0 or a size outside the compiled limits */
  FRZ_ERR_CUDA = 3,        /* cudaGetLastError() after the launch */
  FRZ_ERR_UNSUPPORTED = 4
} FrzStatus;

/* bits of FrzControl.error_word (data-dependent faults found on the device) */
#define FRZ_FAULT_BAD_TASK_INDEX 0x1u  /* action[:,0] is not a valid index into the agent's task list */
#define FRZ_FAULT_BAD_NODE 0x2u        /* cybersecurity: attack / move target outside [0, N) (cybersecurity.py:341,357) */
#define FRZ_FAULT_ABSENT_ACTED 0x4u    /* cybersecurity: non-present agent acted with show_bad_actions=False (:345,362) */
#define FRZ_FAULT_TABLE_FULL 0x8u      /* rideshare: more passengers present than FrzRideshareParams.capacity */

/* Device-resident control block (64 bytes). */
typedef struct {
  uint64_t seed;        /* Philox key */
  uint64_t step;        /* number of executed environment steps since the last full reset (Philox counter) */
  uint32_t ctas_done;   /* scratch: CTAs of the running launch that have finished */
  uint32_t alive_acc;   /* scratch: bit0 = some env not terminated, bit1 = some env not truncated (this launch) */
  uint32_t alive;       /* the same two bits as of the previous launch; 0 in a bit => BatchedAECEnv.step early-out
                           (utils/env.py:212) => the whole launch is a no-op */
  uint32_t error_word;  /* FRZ_FAULT_* bits, sticky until cleared by the host */
  uint32_t agents_with_tasks_acc; /* scratch: bit a = agent a has >= 1 task in some env (this launch) */
  uint32_t agents_with_tasks;     /* the same as of the previous launch: the reference skips an agent's whole action
                                     decode when it has no task in ANY environment (wildfire.py:434) */
  uint32_t reserved[6];
} FrzControl;

/* ----------------------------------------------------------------------------------------------- wildfire */

/* bits of FrzWildfireParams.flags: StochasticConfiguration (structures/configuration.py:271-322), reward switches
 * (:15-56) and the show_bad_actions constructor flag (wildfire.py:176-178) */
#define FRZ_WF_STOCH_SUPPRESSANT_DECREASE 0x0001u
#define FRZ_WF_STOCH_REFILL 0x0002u
#define FRZ_WF_STOCH_TANK_SWITCH 0x0004u
#define FRZ_WF_CRITICAL_ERROR 0x0008u
#define FRZ_WF_STOCH_DEGRADE 0x0010u
#define FRZ_WF_STOCH_REPAIR 0x0020u
#define FRZ_WF_STOCH_FIRE_INCREASE 0x0040u
#define FRZ_WF_STOCH_FIRE_DECREASE 0x0080u
#define FRZ_WF_SPECIAL_BURNOUT 0x0100u
#define FRZ_WF_FIRE_FUEL 0x0200u
#define FRZ_WF_BURNOUT_SCALED 0x0400u
#define FRZ_WF_LOCALIZE_PUTOUTS 0x0800u
#define FRZ_WF_SHOW_BAD_ACTIONS 0x1000u
/* Grids of at most 32 cells with at most 8 agents have two step kernels -- a group of eight lanes per environment, and
 * one thread per environment -- with identical results and identical random streams.  The second one is chosen for
 * tiny grids (at most 16 cells, at most 4 agents) from 49 152 environments up; these two bits force one of them
 * whatever the grid and batch size (tests, kernel timing). */
#define FRZ_WF_KERNEL_TILES 0x2000u
#define FRZ_WF_KERNEL_GROUPS 0x4000u

/* WildfireConfiguration flattened once at construction (passed by value to the kernel). */
typedef struct {
  int32_t height, width, num_agents;
  int32_t num_fire_states;       /* S: burned out = S-1, almost burned out = S-2 (fire_increase.py:25-26) */
  int32_t num_equipment_states;  /* E */
  int32_t num_capacities;
  int32_t max_steps;             /* truncation horizon (utils/env.py:230-233); INT32_MAX = none */
  uint32_t flags;
  int64_t env_offset;            /* global index of local env 0 (multi-GPU shard) -> RNG stream invariant to sharding */
  float p_increase, p_burnout, p_decrease, decrease_bonus;
  float p_random_ignition;       /* fire_random_spread_weight (configuration.py:365-371) */
  float spread_lut[16];          /* fp32 conv sum per lit-neighbour pattern, bit0 N, bit1 W, bit2 E, bit3 S */
  float p_suppressant_decrease, p_refill, p_repair, p_degrade, p_critical, p_tank_switch;
  float capacity_cum[FRZ_MAX_CAPACITIES];    /* cumsum(capacity_probabilities) (capacity.py:28) */
  float capacity_value[FRZ_MAX_CAPACITIES];  /* possible_capacities */
  float equipment_capacity_bonus[FRZ_MAX_EQUIPMENT]; /* equipment_states[:,0] */
  float equipment_power_bonus[FRZ_MAX_EQUIPMENT];    /* equipment_states[:,1]; the range column is folded into range_mask */
  float bad_attack_penalty, burnout_penalty, termination_reward, termination_kappa;
  int32_t agent_y[FRZ_MAX_AGENTS], agent_x[FRZ_MAX_AGENTS];
  float agent_power[FRZ_MAX_AGENTS];         /* fire_reduction_power */
} FrzWildfireParams;

typedef struct {
  /* WildfireState (structures/state.py:11-33), updated in place */
  int32_t* fires;       /* [B, H*W] */
  int32_t* intensity;   /* [B, H*W] */
  int32_t* fuel;        /* [B, H*W] */
  float* suppressants;  /* [B, A] */
  float* capacity;      /* [B, A] */
  int32_t* equipment;   /* [B, A] */
  /* copies restored by frz_wildfire_reset (State.save_initial, utils/state.py:36-38) */
  const int32_t* init_fires;
  const int32_t* init_intensity;
  const int32_t* init_fuel;
  const float* init_suppressants;
  const float* init_capacity;
  const int32_t* init_equipment;
  /* AEC runtime (utils/env.py:129-160) */
  const int32_t* actions;      /* [B, A, 2]  (agent-local task index, action id; id -1 = refill/noop) */
  float* rewards;              /* [B, A] */
  float* cumulative_rewards;   /* [B, A] */
  uint8_t* terminated;         /* [B] */
  uint8_t* truncated;          /* [B] */
  int32_t* num_moves;          /* [B] */
  int32_t* num_burnouts;       /* [B]  (wildfire.py:360,580) */
  int32_t* burnouts;           /* [B]  infos['burnouts'] (wildfire.py:581) */
  int32_t* putouts;            /* [B]  infos['putouts'] (wildfire.py:582) */
  /* what update_actions / update_observations produce (wildfire.py:587-717) */
  int32_t* env_task_count;     /* [B] */
  int32_t* agent_task_count;   /* [B, A] */
  uint8_t* action_mask;        /* [B, A, mask_stride]: 1 iff env-local task t can be fought by the agent */
  float* self_obs;             /* [B, A, 4] (y, x, power, suppressant) */
  int32_t* task_obs;           /* [B, H*W, 4] (y, x, fires, intensity) in row-major lit order, padded with FRZ_PAD */
  /* static tables */
  const float* cell_reward;    /* [H*W] reward_config.fire_rewards */
  const int32_t* cell_ignition;/* [H*W] fire_config.ignition_temp */
  const uint32_t* range_mask;  /* [A, E, mask_words] bit c set iff cell c is within the agent's Chebyshev range when
                                  its equipment is in state e (wildfire.py:606-616, utils/in_range_check.py:5-23) */
  const uint32_t* cell_agents; /* [E, H*W] the same relation transposed: bit a set iff agent a reaches cell c in state e */
  /* randomness */
  FrzControl* control;
  const float* field_uniforms; /* nullable: injected uniforms [3, B, H, W] (wildfire.py:409) instead of Philox */
  const float* agent_uniforms; /* nullable: injected uniforms [5, B, A]    (wildfire.py:410) */
  int32_t mask_stride;         /* row stride of action_mask in bytes: H*W rounded up to a multiple of 4 */
  int32_t mask_words;          /* ceil(H*W / 32) */
} FrzWildfireBuffers;

/* One full environment step for all B envs: action decode, the seven transitions in the reference order, rewards,
 * termination, num_moves/truncation, reward accumulation, observations, task counts and action masks.
 * Replaces wildfire.py:400-717 + utils/env.py:215-237. */
int frz_wildfire_step(const FrzWildfireParams* params, const FrzWildfireBuffers* io, int32_t parallel_envs, void* stream);

/* Recompute observations / counts / masks from the current state without stepping (what reset() does through
 * update_observations + update_actions, wildfire.py:368-371). */
int frz_wildfire_refresh(const FrzWildfireParams* params, const FrzWildfireBuffers* io, int32_t parallel_envs,
                         void* stream);

/* Restore the saved initial state and zero the AEC fields of the envs selected by env_mask (uint8 [B], device;
 * NULL = all), then refresh.  Replaces utils/env.py:163-189 + wildfire.py:376-397. */
int frz_wildfire_reset(const FrzWildfireParams* params, const FrzWildfireBuffers* io, int32_t parallel_envs,
                       const uint8_t* env_mask, void* stream);

/* Uniform random legal actions written into io->actions (caller side of the path: replaces
 * env.action_space(agent).sample_nested(), wildfire.py:720-734 + spaces/actions.py:10-41). */
int frz_wildfire_sample_actions(const FrzWildfireParams* params, const FrzWildfireBuffers* io, int32_t parallel_envs,
                                uint64_t sampler_seed, void* stream);

/* ----------------------------------------------------------------------------------------------- cybersecurity */

#define FRZ_CY_STOCHASTIC_STATE 0x1u   /* StochasticConfiguration.network_state (configuration.py:240-253) */
#define FRZ_CY_SHOW_BAD_ACTIONS 0x2u   /* constructor flag (cybersecurity.py:164-168) */
#define FRZ_CY_MAX_LUT_BITS 12

/* CybersecurityConfiguration flattened once at construction.  Agents are indexed attackers first, then defenders,
 * exactly like the reference's presence tensor (structures/state.py:13-27). */
typedef struct {
  int32_t num_nodes, num_attackers, num_defenders, num_states;
  int32_t max_steps;
  uint32_t flags;
  int64_t env_offset;
  int32_t lut_bits;      /* num_attackers + num_defenders when score_lut is provided, else 0 (tanhf in-kernel) */
  float temperature;
  float patch_reward, bad_action_penalty;
  float power[FRZ_MAX_AGENTS];          /* threat of attacker a / mitigation of defender d, agent-indexed */
  float persist[FRZ_MAX_AGENTS];        /* presence.py:35-60 */
  float returns[FRZ_MAX_AGENTS];
  float state_rewards[FRZ_MAX_NET_STATES];
  float criticality[FRZ_MAX_NODES];     /* adj_matrix.sum(1) as float (configuration.py:215-217, cybersecurity.py:399) */
} FrzCyberParams;

typedef struct {
  /* CybersecurityState (structures/state.py:13-27), updated in place */
  int32_t* network_state;  /* [B, N] */
  int32_t* location;       /* [B, D]  -1 = home node */
  uint8_t* presence;       /* [B, Att+D] */
  const int32_t* init_network_state;
  const int32_t* init_location;
  const uint8_t* init_presence;
  /* AEC runtime */
  const int32_t* actions;     /* [B, Att+D, 2] (node, action id: 0 attack/move, -1 noop, -2 patch, -3 monitor) */
  float* rewards;             /* [B, Att+D] */
  float* cumulative_rewards;  /* [B, Att+D] */
  uint8_t* terminated;        /* [B] (never set: cybersecurity.py:299) */
  uint8_t* truncated;         /* [B] */
  int32_t* num_moves;         /* [B] */
  /* update_actions / update_observations (cybersecurity.py:414-526) */
  int32_t* env_task_count;    /* [B] = N */
  int32_t* agent_task_count;  /* [B, Att+D] = N * presence */
  float* attacker_self;       /* [B, Att, 2] (threat, presence) */
  float* defender_self;       /* [B, D, 3] (mitigation, presence, location) */
  int32_t* task_obs;          /* [B, N, 2] (state, criticality) -- the reference's task_store */
  uint8_t* monitored;         /* [B, D] 1 iff the defender's last action was monitor (-3): with partial observability
                                 a defender only sees task_obs after monitoring (cybersecurity.py:497,510-511) */
  /* static */
  const float* score_lut;     /* nullable: [2^(Att+D)] tanh((patches-attacks)/T) for every (attacker set | defender set
                                 << Att) acting on one node, evaluated on the host with the reference's own tanh */
  /* randomness */
  FrzControl* control;
  const float* network_uniforms; /* nullable: injected [1, B, N]      (cybersecurity.py:304-309) */
  const float* agent_uniforms;   /* nullable: injected [1, B, Att+D]  (cybersecurity.py:310-315) */
} FrzCyberBuffers;

/* One fused step: action decode, movement, presence, subnetwork transitions, rewards, num_moves / truncation,
 * observations and task counts.  Replaces cybersecurity.py:296-526 + utils/env.py:215-237. */
int frz_cyber_step(const FrzCyberParams* params, const FrzCyberBuffers* io, int32_t parallel_envs, void* stream);
int frz_cyber_refresh(const FrzCyberParams* params, const FrzCyberBuffers* io, int32_t parallel_envs, void* stream);
/* Restore initial rows (env_mask uint8 [B] on device, NULL = all), zero AEC fields, mark "not monitored", refresh.
 * Replaces utils/env.py:163-189 + cybersecurity.py:274-293. */
int frz_cyber_reset(const FrzCyberParams* params, const FrzCyberBuffers* io, int32_t parallel_envs,
                    const uint8_t* env_mask, void* stream);
/* Uniform random legal actions (replaces action_space(agent).sample_nested(), spaces/actions.py:11-99). */
int frz_cyber_sample_actions(const FrzCyberParams* params, const FrzCyberBuffers* io, int32_t parallel_envs,
                             uint64_t sampler_seed, void* stream);

/* ----------------------------------------------------------------------------------------------- rideshare */

#define FRZ_RS_FAST_TRAVEL 0x1u          /* AgentConfiguration.use_fast_travel (configuration.py:83-110) */
#define FRZ_RS_DIAGONAL_TRAVEL 0x2u      /* AgentConfiguration.use_diagonal_travel */
#define FRZ_RS_VARIABLE_MOVE_COST 0x4u   /* RewardConfiguration.use_variable_move_cost */
#define FRZ_RS_WAITING_COSTS 0x8u        /* RewardConfiguration.use_waiting_costs */
/* Which of the two step kernels runs is normally decided by the batch size (one thread per environment from 24 576
 * environments up, a group of lanes per environment below).  These two bits force one of them -- results are identical;
 * they exist so that both kernels can be tested and timed at any batch size.  The tiled kernel serves tables with a
 * multiple of four rows and at most eight drivers; other shapes always take the group kernel. */
#define FRZ_RS_KERNEL_TILES 0x100u
#define FRZ_RS_KERNEL_GROUPS 0x200u
#define FRZ_RS_PASSENGER_COLUMNS 11      /* (batch, y, x, dest_y, dest_x, fare, state, assoc, entered, accepted, picked) */
#define FRZ_RS_TASK_COLUMNS 8            /* (y, x, dest_y, dest_x, accepted_by, riding_by, fare, entered) */

/* RideshareConfiguration flattened once at construction. */
typedef struct {
  int32_t num_agents;
  int32_t capacity;        /* K: rows of the per-environment passenger table (<= FRZ_MAX_PASSENGERS) */
  int32_t schedule_rows;   /* S */
  int32_t schedule_horizon;/* latest entry step named by the schedule (-1 when it is empty) */
  int32_t pool_limit;
  int32_t max_steps;
  uint32_t flags;
  int64_t env_offset;      /* global index of local env 0: schedule rows name global environment indices */
  int32_t wait_limit[3];   /* RewardConfiguration.wait_limit: unaccepted / accepted / riding */
  int32_t long_wait_time;
  float move_cost, drop_cost, noop_cost, accept_cost, pool_limit_cost, general_wait_cost, long_wait_cost;
} FrzRideshareParams;

typedef struct {
  /* RideshareState (structures/state.py:11-22).  The reference keeps one flat table [N_total, 11] sorted by
   * environment; here environment b owns rows passengers[b, 0 : env_task_count[b]] in the same order (rows beyond
   * the count are undefined). */
  int32_t* agents;           /* [B, A, 2] (y, x) */
  int32_t* passengers;       /* [B, K, 11] */
  const int32_t* init_agents;        /* [B, A, 2] */
  const int32_t* init_passengers;    /* [B, K, 11] table before the t = 0 entry (normally empty) */
  const int32_t* init_count;         /* [B] */
  const int32_t* schedule;   /* [S, 7] (t, batch | -1, y, x, dest_y, dest_x, fare), stably sorted by t */
  const int32_t* schedule_index; /* [schedule_horizon + 2]: index[t] = first schedule row with entry step >= t, so the
                                    rows entering at step t are [index[t], index[t + 1]); index[horizon + 1] = S */
  /* AEC runtime */
  const int32_t* actions;    /* [B, A, 2] (agent-local task index, action id: 0 accept, 1 pick, 2 drop, -1 noop) */
  float* rewards;            /* [B, A] */
  float* cumulative_rewards; /* [B, A] */
  uint8_t* terminated;       /* [B] (never set: rideshare.py:252) */
  uint8_t* truncated;        /* [B] */
  int32_t* num_moves;        /* [B] */
  /* update_actions / update_observations (rideshare.py:368-467) */
  int32_t* env_task_count;   /* [B] passengers present == valid rows of the table */
  int32_t* agent_task_count; /* [B, A] */
  uint8_t* task_mask;        /* [B, A, K] 1 iff table row p is in the agent's task list (unaccepted or its own) */
  int32_t* self_obs;         /* [B, A, 4] (y, x, #accepted, #riding) */
  int32_t* task_obs;         /* [B, K, 8] one row per passenger in table order, padded with FRZ_PAD */
  FrzControl* control;
} FrzRideshareBuffers;

/* One fused step: action decode, movement, passenger state / exit / entry transitions, rewards, num_moves /
 * truncation, observations, task lists.  Replaces rideshare.py:249-467 + env/transitions/*.py + utils/env.py:215-237. */
int frz_rideshare_step(const FrzRideshareParams* params, const FrzRideshareBuffers* io, int32_t parallel_envs,
                       void* stream);
int frz_rideshare_refresh(const FrzRideshareParams* params, const FrzRideshareBuffers* io, int32_t parallel_envs,
                          void* stream);
/* Restore agents + the pre-entry table of the envs selected by env_mask (NULL = all), zero their AEC fields, let the
 * t = 0 passengers enter (rideshare.py:212) and refresh.  The reference raises NotImplementedError for the partial
 * form (rideshare.py:231-246); it is implemented here to the evident intent. */
int frz_rideshare_reset(const FrzRideshareParams* params, const FrzRideshareBuffers* io, int32_t parallel_envs,
                        const uint8_t* env_mask, void* stream);
/* Uniform random legal actions: task k with id = passenger state, or noop (spaces/actions.py:10-50). */
int frz_rideshare_sample_actions(const FrzRideshareParams* params, const FrzRideshareBuffers* io, int32_t parallel_envs,
                                 uint64_t sampler_seed, void* stream);

/* ----------------------------------------------------------------------------------------------- host-buffer step */

/* The same step for callers whose actions live in HOST memory and who read rewards / done flags on the host -- what
 * a rollout loop around the reference's `env.step(actions)` does when the policy runs on the CPU
 * (utils/conversions.py:39-99: actions in, rewards / terminations / truncations out).  The batch is cut into `chunks`
 * contiguous slices of environments; slice i is uploaded, stepped and downloaded on streams[i], so its kernel overlaps
 * the upload of slice i+1 and the download of slice i-1 (PCIe is full duplex) instead of the three waiting for each
 * other.  Environments are independent and the Philox counters are keyed by the global environment index, so the
 * result is bit-identical to frz_<domain>_step on the whole batch.  The call only enqueues work: the main stream
 * (last argument) waits for every slice before it continues, so synchronising it makes the host buffers readable.
 * Injected uniforms (parity mode) are not supported on this path. */
#define FRZ_MAX_CHUNKS 16

/* Events of the pipelined host step: one handle per caller (environment object / host thread) and device, so that two
 * environments -- or two devices in one process -- never share an event.  Created on the current device. */
typedef struct FrzHostPipeline FrzHostPipeline;
int frz_host_pipeline_create(FrzHostPipeline** out);
int frz_host_pipeline_destroy(FrzHostPipeline* pipeline);

#define FRZ_HOST_ACTIONS_I32 0  /* actions: int32 [B, A, 2], the device layout */
#define FRZ_HOST_ACTIONS_I16 1  /* actions: int16 [B, A, 2] -- half the upload; widened on the device (every task index
                                   and action id of the three domains fits: <= 256 tasks, ids in [-3, 2]) */
#define FRZ_HOST_ACTIONS_I8 2   /* actions: int8 [B, A, 2] -- a quarter of the upload, for configurations with at most
                                   127 tasks per environment (grids of <= 127 cells, every rideshare / cybersecurity
                                   shape); where several GPUs share a PCIe uplink the upload is what a host-driven
                                   step waits for */

typedef struct {
  const void* actions;         /* HOST, page-locked: [B, A, 2] in `action_format` */
  float* rewards;              /* HOST, page-locked: [B, A] */
  uint8_t* terminated;         /* HOST, page-locked: [B] */
  uint8_t* truncated;          /* HOST, page-locked: [B] */
  FrzControl* chunk_controls;  /* DEVICE scratch owned by the caller: `chunks` control blocks (64 bytes each) */
  void* const* streams;        /* `chunks` cudaStream_t of the caller, one per slice */
  int32_t chunks;              /* 1 .. FRZ_MAX_CHUNKS */
  int32_t action_format;       /* FRZ_HOST_ACTIONS_* */
  int16_t* packed_actions;     /* DEVICE scratch [B, A, 2] int16, required for FRZ_HOST_ACTIONS_I16 / _I8 */
  FrzHostPipeline* pipeline;   /* NULL = per-thread, per-device events kept by the library */
} FrzHostStep;

/* Which Philox call feeds which draw in the one-thread-per-environment kernel of a small grid (pure host logic, for
 * tests): returns the number of calls n (<= 24) or -FrzStatus; call i uses streams[i] as its third counter word, its
 * word j feeds slot destinations[4 i + j]: c = increase / decrease of cell c, H*W + c = spread of cell c,
 * 2 H*W + 4 a + j = word j of agent a, -1 = unused.  The table restates the word assignment of the group kernel for the
 * same grid, which is why the two kernels draw identical trajectories. */
int frz_wildfire_tile_random_layout(const FrzWildfireParams* params, uint32_t* streams, int8_t* destinations);
int frz_wildfire_step_host(const FrzWildfireParams* params, const FrzWildfireBuffers* io, int32_t parallel_envs,
                           const FrzHostStep* host, void* stream);
/* How frz_<domain>_step_host cuts a batch: writes bounds[0] = 0 < ... < bounds[n] = parallel_envs (room for
 * FRZ_MAX_CHUNKS + 1 entries) and returns n <= chunks, or -FrzStatus.  Inner boundaries are multiples of 1024
 * environments; the first slice is half as long as the others (no kernel can start before it has been uploaded). */
int frz_host_slices(int32_t parallel_envs, int32_t chunks, int32_t* bounds);
int frz_cyber_step_host(const FrzCyberParams* params, const FrzCyberBuffers* io, int32_t parallel_envs,
                        const FrzHostStep* host, void* stream);
int frz_rideshare_step_host(const FrzRideshareParams* params, const FrzRideshareBuffers* io, int32_t parallel_envs,
                            const FrzHostStep* host, void* stream);

/* ----------------------------------------------------------------------------------------------- observation download */

/* The step publishes observations as padded arrays -- task_obs [B, capacity, columns], action / task masks
 * [B, agents, capacity] -- of which only the first counts[b] rows per environment are live; the reference hands the
 * same data to a policy as jagged nested tensors, i.e. a packed value buffer + offsets (wildfire.py:669-717,
 * rideshare.py:398-467, `obs['tasks']`, `agent_action_mapping`).  A caller that reads observations on the HOST wants
 * that packed buffer: the PCIe link is the slowest hop of a host-driven step, so the live rows are compacted on the
 * device and each array then leaves with ONE cudaMemcpyAsync of exactly offsets[B] * groups * row_bytes bytes.
 *
 * One padded array: src = [B, groups, capacity] rows of row_bytes bytes, environment b owns rows 0 .. counts[b]-1 of
 * each of its `groups` row blocks; in dst environment b's block g starts at row offsets[b] * groups + g * counts[b]. */
typedef struct {
  const void* src;      /* device */
  void* dst;            /* device, room for parallel_envs * groups * capacity rows */
  int32_t row_bytes, capacity, groups;
  int32_t reserved;
} FrzGatherArray;

/* offsets[0 .. B] <- exclusive prefix sum of counts (offsets[B] = all live rows), then every array is compacted.
 * scratch = device int32 [(B + 1023) / 1024 + 1].  Only enqueues work on `stream`; allocates nothing. */
int frz_gather_live_rows(const int32_t* counts, int32_t parallel_envs, int32_t* offsets, int32_t* scratch,
                         const FrzGatherArray* arrays, int32_t array_count, void* stream);

/* ----------------------------------------------------------------------------------------------- common */

int frz_version(void);
const char* frz_last_error(void);
/* (re)initialise a control block on the device: seed, step = 0, alive = 3, error_word = 0 */
int frz_control_init(FrzControl* control, uint64_t seed, void* stream);
/* Restore the random stream of a checkpoint: (seed, step) are all the generator state there is -- every draw is
 * Philox(seed; global env, step, event) -- so this is the engine's load_state_dict (the reference pickles one
 * torch.Generator state per environment: utils/random_generator.py:148-176).  Clears error_word.  The published flags
 * (alive, agents_with_tasks) are left as they are: restore the state arrays (done flags included), call this, then run
 * frz_<domain>_refresh, which recomputes both flags from the restored arrays.  frz_<domain>_refresh and
 * frz_<domain>_reset publish both flags the same way, so a step after a reset or a hand edit of the state sees the done
 * flags it left. */
int frz_control_restore(FrzControl* control, uint64_t seed, uint64_t step, void* stream);

/* Size in bytes of the array behind field `field` of Frz<Domain>Buffers (its name as spelled in the struct, e.g.
 * "fires", "action_mask", "task_obs") for `parallel_envs` environments of this configuration; -1 for an unknown
 * name.  (wildfire: mask_stride = H*W rounded up to a multiple of 4; rideshare: rows per table = params->capacity.) */
int64_t frz_wildfire_buffer_bytes(const FrzWildfireParams* params, int32_t parallel_envs, const char* field);
int64_t frz_cyber_buffer_bytes(const FrzCyberParams* params, int32_t parallel_envs, const char* field);
int64_t frz_rideshare_buffer_bytes(const FrzRideshareParams* params, int32_t parallel_envs, const char* field);

#ifdef __cplusplus
}
#endif
#endif /* FRZ_H_ */
