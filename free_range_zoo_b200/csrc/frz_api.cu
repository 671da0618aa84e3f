// Library-wide entry points of libfrz.so: version, thread-local error string, control-block initialisation.
#include <cstdarg>
#include <cstdio>
#include <cstring>

#include "frz_common.cuh"
#include "frz_host.cuh"

namespace frz {

static thread_local char g_error[512] = "";

void set_error(const char* fmt, ...) {
  va_list args;
  va_start(args, fmt);
  vsnprintf(g_error, sizeof(g_error), fmt, args);
  va_end(args);
}

int check_launch(const char* what) {
  const cudaError_t err = cudaGetLastError();
  if (err == cudaSuccess) return FRZ_OK;
  set_error("%s: %s", what, cudaGetErrorString(err));
  return FRZ_ERR_CUDA;
}

namespace {
__global__ void control_init_kernel(FrzControl* control, uint64_t seed) {
  control->seed = seed;
  control->step = 0;
  control->ctas_done = 0;
  control->alive_acc = 0;
  control->alive = 3u;
  control->error_word = 0;
  control->agents_with_tasks_acc = 0;
  control->agents_with_tasks = 0;
}

// a checkpoint's random stream: every draw is Philox(seed; env, step, event), so (seed, step) is the whole state.  The
// published flags are left to the refresh that follows (they depend on the restored state arrays); faults recorded
// before the restore belong to the abandoned run.
__global__ void control_restore_kernel(FrzControl* control, uint64_t seed, uint64_t step) {
  control->seed = seed;
  control->step = step;
  control->ctas_done = 0;
  control->alive_acc = 0;
  control->error_word = 0;
  control->agents_with_tasks_acc = 0;
}

// every chunk block starts the step as a copy of the main block (seed, step counter, published flags)
__global__ void control_broadcast_kernel(const FrzControl* main_block, FrzControl* chunk_blocks, int count) {
  const int i = threadIdx.x;
  if (i >= count) return;
  FrzControl block = *main_block;
  block.ctas_done = 0;
  block.alive_acc = 0;
  block.agents_with_tasks_acc = 0;
  block.error_word = 0;
  chunk_blocks[i] = block;
}

// the main block ends the step with what one launch over the whole batch would have published: the flags are ORs over
// the slices, the step counter is the slices' common one
__global__ void control_merge_kernel(FrzControl* main_block, const FrzControl* chunk_blocks, int count) {
  unsigned alive = 0, agents = 0, faults = 0;
  for (int i = 0; i < count; ++i) {
    alive |= chunk_blocks[i].alive;
    agents |= chunk_blocks[i].agents_with_tasks;
    faults |= chunk_blocks[i].error_word;
  }
  if (chunk_blocks[0].step != main_block->step) {  // the slices stepped (no "every environment is done" early-out)
    main_block->alive = alive;
    main_block->agents_with_tasks = agents;
    main_block->step = chunk_blocks[0].step;
  }
  main_block->error_word |= faults;
}
}  // namespace

int control_broadcast(FrzControl* main_block, FrzControl* chunk_blocks, int count, cudaStream_t stream) {
  control_broadcast_kernel<<<1, 32, 0, stream>>>(main_block, chunk_blocks, count);
  return check_launch("control_broadcast_kernel");
}

int control_merge(FrzControl* main_block, FrzControl* chunk_blocks, int count, cudaStream_t stream) {
  control_merge_kernel<<<1, 1, 0, stream>>>(main_block, chunk_blocks, count);
  return check_launch("control_merge_kernel");
}

}  // namespace frz

// (FrzHostPipeline is defined in frz_common.cuh; events: [0] = "broadcast done", then "slice i uploaded" and "slice i
// finished")

namespace frz {

namespace {
bool create_events(FrzHostPipeline* pipeline) {
  pipeline->device = current_device();
  for (auto& event : pipeline->events)
    if (cudaEventCreateWithFlags(&event, cudaEventDisableTiming) != cudaSuccess) return false;
  return true;
}

// four packed action words (short4 / char4) -> four int32
template <class Packed4, class Scalar>
__global__ void widen_actions_kernel(const Packed4* __restrict__ packed, int4* __restrict__ actions, size_t quads,
                                     const Scalar* __restrict__ tail_in, int32_t* __restrict__ tail_out, int tail) {
  for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < quads; i += size_t(gridDim.x) * blockDim.x) {
    const Packed4 v = packed[i];
    actions[i] = make_int4(v.x, v.y, v.z, v.w);
  }
  if (blockIdx.x == 0 && int(threadIdx.x) < tail) tail_out[threadIdx.x] = tail_in[threadIdx.x];
}
}  // namespace

cudaEvent_t* pipeline_events(FrzHostPipeline* pipeline) {
  if (pipeline != nullptr) {
    if (pipeline->device != current_device()) {
      set_error("FrzHostPipeline was created on device %d, the current device is %d", pipeline->device, current_device());
      return nullptr;
    }
    return pipeline->events;
  }
  // no handle: one set of events per host thread and device (events belong to the device they were created on)
  static thread_local FrzHostPipeline* per_device[kMaxDevices] = {};
  const int device = current_device();
  if (device < 0 || device >= kMaxDevices) {
    set_error("device ordinal %d outside [0, %d)", device, kMaxDevices);
    return nullptr;
  }
  if (per_device[device] == nullptr) {
    FrzHostPipeline* created = new FrzHostPipeline;
    if (!create_events(created)) {
      delete created;
      check_launch("pipeline events");
      return nullptr;
    }
    per_device[device] = created;
  }
  return per_device[device]->events;
}

int widen_actions(const void* packed, int element_bytes, int32_t* actions, size_t count, cudaStream_t stream) {
  const size_t quads = count / 4;  // (both arrays start 16-byte aligned: slices begin on multiples of 1024 environments)
  const int tail = int(count % 4);
  const size_t blocks = (quads + 255) / 256;
  const int grid = persistent_grid(int(blocks < 1 ? 1 : (blocks > (1u << 20) ? (1u << 20) : blocks)), 8);
  int4* const out = reinterpret_cast<int4*>(actions);
  if (element_bytes == 2) {
    const int16_t* in = static_cast<const int16_t*>(packed);
    widen_actions_kernel<<<grid, 256, 0, stream>>>(reinterpret_cast<const short4*>(in), out, quads, in + 4 * quads,
                                                   actions + 4 * quads, tail);
  } else {
    const int8_t* in = static_cast<const int8_t*>(packed);
    widen_actions_kernel<<<grid, 256, 0, stream>>>(reinterpret_cast<const char4*>(in), out, quads, in + 4 * quads,
                                                   actions + 4 * quads, tail);
  }
  return check_launch("widen_actions_kernel");
}

}  // namespace frz

extern "C" {

int frz_version(void) { return FRZ_ABI_VERSION; }

const char* frz_last_error(void) { return frz::g_error; }

int frz_host_slices(int32_t parallel_envs, int32_t chunks, int32_t* bounds) {
  if (bounds == nullptr) {
    frz::set_error("frz_host_slices: bounds is NULL");
    return -FRZ_ERR_NULL;
  }
  if (parallel_envs <= 0 || chunks < 1 || chunks > FRZ_MAX_CHUNKS) {
    frz::set_error("frz_host_slices: parallel_envs=%d chunks=%d", parallel_envs, chunks);
    return -FRZ_ERR_SHAPE;
  }
  return frz::slice_bounds(parallel_envs, chunks, bounds);
}

namespace {
struct FieldSize {
  const char* name;
  int64_t bytes;
};
int64_t lookup_field(const FieldSize* fields, size_t count, const char* field, const char* what) {
  if (field != nullptr)
    for (size_t i = 0; i < count; ++i)
      if (std::strcmp(fields[i].name, field) == 0) return fields[i].bytes;
  frz::set_error("%s: unknown buffer field '%s'", what, field == nullptr ? "(null)" : field);
  return -1;
}
}  // namespace

int64_t frz_wildfire_buffer_bytes(const FrzWildfireParams* p, int32_t parallel_envs, const char* field) {
  if (p == nullptr || parallel_envs <= 0) {
    frz::set_error("frz_wildfire_buffer_bytes: NULL params or parallel_envs <= 0");
    return -1;
  }
  const int64_t B = parallel_envs, HW = int64_t(p->height) * p->width, A = p->num_agents, E = p->num_equipment_states;
  const int64_t stride = (HW + 3) / 4 * 4, words = (HW + 31) / 32;
  const FieldSize fields[] = {
      {"fires", 4 * B * HW}, {"intensity", 4 * B * HW}, {"fuel", 4 * B * HW}, {"suppressants", 4 * B * A},
      {"capacity", 4 * B * A}, {"equipment", 4 * B * A}, {"init_fires", 4 * B * HW}, {"init_intensity", 4 * B * HW},
      {"init_fuel", 4 * B * HW}, {"init_suppressants", 4 * B * A}, {"init_capacity", 4 * B * A},
      {"init_equipment", 4 * B * A}, {"actions", 8 * B * A}, {"rewards", 4 * B * A}, {"cumulative_rewards", 4 * B * A},
      {"terminated", B}, {"truncated", B}, {"num_moves", 4 * B}, {"num_burnouts", 4 * B}, {"burnouts", 4 * B},
      {"putouts", 4 * B}, {"env_task_count", 4 * B}, {"agent_task_count", 4 * B * A}, {"action_mask", B * A * stride},
      {"self_obs", 16 * B * A}, {"task_obs", 16 * B * HW}, {"cell_reward", 4 * HW}, {"cell_ignition", 4 * HW},
      {"range_mask", 4 * A * E * words}, {"cell_agents", 4 * E * HW}, {"control", int64_t(sizeof(FrzControl))},
      {"field_uniforms", 4 * 3 * B * HW}, {"agent_uniforms", 4 * 5 * B * A}};
  return lookup_field(fields, sizeof(fields) / sizeof(fields[0]), field, "frz_wildfire_buffer_bytes");
}

int64_t frz_cyber_buffer_bytes(const FrzCyberParams* p, int32_t parallel_envs, const char* field) {
  if (p == nullptr || parallel_envs <= 0) {
    frz::set_error("frz_cyber_buffer_bytes: NULL params or parallel_envs <= 0");
    return -1;
  }
  const int64_t B = parallel_envs, N = p->num_nodes, att = p->num_attackers, dfd = p->num_defenders, n = att + dfd;
  const FieldSize fields[] = {
      {"network_state", 4 * B * N}, {"location", 4 * B * dfd}, {"presence", B * n}, {"init_network_state", 4 * B * N},
      {"init_location", 4 * B * dfd}, {"init_presence", B * n}, {"actions", 8 * B * n}, {"rewards", 4 * B * n},
      {"cumulative_rewards", 4 * B * n}, {"terminated", B}, {"truncated", B}, {"num_moves", 4 * B},
      {"env_task_count", 4 * B}, {"agent_task_count", 4 * B * n}, {"attacker_self", 8 * B * att},
      {"defender_self", 12 * B * dfd}, {"task_obs", 8 * B * N}, {"monitored", B * dfd},
      {"score_lut", p->lut_bits > 0 ? int64_t(4) << p->lut_bits : 0}, {"control", int64_t(sizeof(FrzControl))},
      {"network_uniforms", 4 * B * N}, {"agent_uniforms", 4 * B * n}};
  return lookup_field(fields, sizeof(fields) / sizeof(fields[0]), field, "frz_cyber_buffer_bytes");
}

int64_t frz_rideshare_buffer_bytes(const FrzRideshareParams* p, int32_t parallel_envs, const char* field) {
  if (p == nullptr || parallel_envs <= 0) {
    frz::set_error("frz_rideshare_buffer_bytes: NULL params or parallel_envs <= 0");
    return -1;
  }
  const int64_t B = parallel_envs, A = p->num_agents, K = p->capacity, S = p->schedule_rows;
  const FieldSize fields[] = {
      {"agents", 8 * B * A}, {"passengers", 4 * B * K * FRZ_RS_PASSENGER_COLUMNS}, {"init_agents", 8 * B * A},
      {"init_passengers", 4 * B * K * FRZ_RS_PASSENGER_COLUMNS}, {"init_count", 4 * B}, {"schedule", 4 * S * 7},
      {"schedule_index", 4 * (int64_t(p->schedule_horizon) + 2)}, {"actions", 8 * B * A}, {"rewards", 4 * B * A},
      {"cumulative_rewards", 4 * B * A}, {"terminated", B}, {"truncated", B}, {"num_moves", 4 * B},
      {"env_task_count", 4 * B}, {"agent_task_count", 4 * B * A}, {"task_mask", B * A * K}, {"self_obs", 16 * B * A},
      {"task_obs", 4 * B * K * FRZ_RS_TASK_COLUMNS}, {"control", int64_t(sizeof(FrzControl))}};
  return lookup_field(fields, sizeof(fields) / sizeof(fields[0]), field, "frz_rideshare_buffer_bytes");
}

int frz_host_pipeline_create(FrzHostPipeline** out) {
  if (out == nullptr) {
    frz::set_error("frz_host_pipeline_create: out is NULL");
    return FRZ_ERR_NULL;
  }
  FrzHostPipeline* pipeline = new FrzHostPipeline;
  if (!frz::create_events(pipeline)) {
    delete pipeline;
    return frz::check_launch("frz_host_pipeline_create");
  }
  *out = pipeline;
  return FRZ_OK;
}

int frz_host_pipeline_destroy(FrzHostPipeline* pipeline) {
  if (pipeline == nullptr) return FRZ_OK;
  for (auto& event : pipeline->events) cudaEventDestroy(event);
  if (pipeline->exec != nullptr) cudaGraphExecDestroy(pipeline->exec);
  if (pipeline->graph != nullptr) cudaGraphDestroy(pipeline->graph);
  delete pipeline;
  return FRZ_OK;
}

int frz_control_restore(FrzControl* control, uint64_t seed, uint64_t step, void* stream) {
  if (control == nullptr) {
    frz::set_error("frz_control_restore: control is NULL");
    return FRZ_ERR_NULL;
  }
  frz::control_restore_kernel<<<1, 1, 0, static_cast<cudaStream_t>(stream)>>>(control, seed, step);
  return frz::check_launch("control_restore_kernel");
}

int frz_control_init(FrzControl* control, uint64_t seed, void* stream) {
  if (control == nullptr) {
    frz::set_error("frz_control_init: control is NULL");
    return FRZ_ERR_NULL;
  }
  frz::control_init_kernel<<<1, 1, 0, static_cast<cudaStream_t>(stream)>>>(control, seed);
  return frz::check_launch("control_init_kernel");
}

}  // extern "C"
