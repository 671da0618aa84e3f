// Policy inputs: observations encoded into the fixed-width agent / task rows of include/frz_inputs.h
// (frz_<domain>_policy_inputs).
//
// One streaming launch over a persistent grid.  Both outputs are walked by element, VEC consecutive elements per thread
// (16 bytes of output: 4 f32 or 8 bf16), task block first, then agent block; a thread decomposes its first element's
// index once and advances the (row, column) counters for the others, so Ft, a compile-time constant per domain, is the
// only divisor in the inner loop.  Stores are 16-byte vectors when the output is 16-byte aligned, scalars otherwise (a
// caller's `out` slice may start anywhere).  The per-column tables live in shared memory (see Tables).
//   task element (b, v, t, c)  c = 0: the flag; c > 0: task_obs[b, t, c - 1], loaded only when t < env_task_count[b]
//                              and view v sees the tasks (cybersecurity: a hidden defender view reads nothing)
//   agent element (b, a, f)    a gather from the self table of a's kind through the host-built table (rank, column)[f]:
//                              rank -1 = a itself, r >= 0 = the r-th other agent of a's kind, kNone = zero padding
#include <cuda_bf16.h>

#include "frz_common.cuh"
#include "frz_inputs.h"

namespace frz {
namespace {

constexpr int kInputThreads = 256;
constexpr int kMaxAgentWidth = 4 + (FRZ_MAX_AGENTS - 1) * 4;  // four own columns, all four observed, 32 agents
constexpr int8_t kNone = -2;

// the two self tables (index 1 only for cybersecurity defenders) and the gather table of the agent block
struct AgentSource {
  const void* table[2];
  int32_t first[2];   // action-table index of the kind's first agent (first[1] = A when there is one kind)
  int32_t count[2];   // agents of the kind
  int8_t rank[2][kMaxAgentWidth];
  int8_t column[2][kMaxAgentWidth];
};

struct Launch {
  FrzPolicyInputs in;
  AgentSource agents;
  const int32_t* task_obs;       // [B, T, task_columns.columns]
  const int32_t* env_task_count; // [B]
  const uint8_t* monitored;      // [B, A - hidden_from]; NULL = every view sees the tasks
  int32_t hidden_from;           // first view that monitored may hide
  int32_t A;
  int64_t task_elements, agent_elements;
};

__device__ __forceinline__ float to_float(float v, int32_t offset) { return v + float(offset); }
__device__ __forceinline__ float to_float(int32_t v, int32_t offset) { return float(v + offset); }

template <class Out>
struct Vec;
template <>
struct Vec<float> {
  static constexpr int kCount = 4;
  __device__ __forceinline__ static void store(float* p, const float* v) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  }
  __device__ __forceinline__ static float cast(float v) { return v; }
};
template <>
struct Vec<__nv_bfloat16> {
  static constexpr int kCount = 8;
  __device__ __forceinline__ static void store(__nv_bfloat16* p, const float* v) {
    uint4 packed;
    uint32_t* words = reinterpret_cast<uint32_t*>(&packed);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const __nv_bfloat162 pair = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
      words[i] = *reinterpret_cast<const uint32_t*>(&pair);
    }
    *reinterpret_cast<uint4*>(p) = packed;
  }
  __device__ __forceinline__ static __nv_bfloat16 cast(float v) { return __float2bfloat16_rn(v); }
};

// q = x / d, r = x % d for 64-bit x (32-bit arithmetic whenever x fits)
__device__ __forceinline__ void divmod(int64_t x, int32_t d, int64_t& q, int32_t& r) {
  if (x <= int64_t(UINT32_MAX)) {
    const uint32_t q32 = uint32_t(x) / uint32_t(d);
    q = q32;
    r = int32_t(uint32_t(x) - q32 * uint32_t(d));
  } else {
    q = x / d;
    r = int32_t(x - q * d);
  }
}

template <class Out>
__device__ __forceinline__ void store_group(Out* out, int64_t first, int64_t total, const float* v) {
  constexpr int N = Vec<Out>::kCount;
  if (first + N <= total && (reinterpret_cast<uintptr_t>(out) & 15u) == 0u) {
    Vec<Out>::store(out + first, v);
  } else {
#pragma unroll
    for (int i = 0; i < N; ++i)
      if (first + i < total) out[first + i] = Vec<Out>::cast(v[i]);
  }
}

// The column tables, copied once per block to shared memory: lanes of a warp index them with different columns, which
// a constant-bank (kernel parameter) load would serialise.  [0] / [1] the self kinds, [2] the task columns.
struct Tables {
  float scale[3][FRZ_INPUTS_MAX_COLUMNS];
  int32_t offset[3][FRZ_INPUTS_MAX_COLUMNS];
  int8_t rank[2][kMaxAgentWidth];
  int8_t column[2][kMaxAgentWidth];
};

// whether view v of environment b sees the tasks (cybersecurity: a defender's monitored byte)
__device__ __forceinline__ bool view_sees(const Launch& L, int64_t b, int v) {
  return L.monitored == nullptr || v < L.hidden_from ||
         L.monitored[b * (L.A - L.hidden_from) + (v - L.hidden_from)] != 0;
}

// the N task elements from `first` on: (b, v, t, c) counters advanced in row-major order; the environment's count and
// the view's visibility are reloaded only when the row moves to another view
template <int Ft, class Out>
__device__ __forceinline__ void task_group(const Launch& L, const Tables& S, int64_t first) {
  constexpr int N = Vec<Out>::kCount;
  const int T = L.in.task_rows, V = L.in.views, source = L.in.task_columns.columns;
  const uint32_t pad_is_none = L.in.task_columns.pad_is_none;
  int64_t bvt;
  int32_t c, t, v;
  divmod(first, Ft, bvt, c);
  int64_t bv, b;
  divmod(bvt, T, bv, t);
  divmod(bv, V, b, v);
  int count = 0;
  if (first < L.task_elements) count = view_sees(L, b, v) ? L.env_task_count[b] : 0;
  float value[N];
#pragma unroll
  for (int i = 0; i < N; ++i) {
    float x = 0.f;
    if (t < count) {  // (count is 0 past the end)
      if (c == 0) {
        x = 1.f;
      } else {
        const int k = c - 1;
        int32_t raw = L.task_obs[(b * T + t) * source + k];
        if ((pad_is_none >> k & 1u) && raw == FRZ_PAD) raw = -1;
        x = to_float(raw, S.offset[2][k]) * S.scale[2][k];
      }
    }
    value[i] = x;
    if (++c == Ft) {
      c = 0;
      if (++t == T) {
        t = 0;
        if (++v == V) {
          v = 0;
          ++b;
        }
        count = first + i + 1 < L.task_elements && view_sees(L, b, v) ? L.env_task_count[b] : 0;
      }
    }
  }
  store_group(static_cast<Out*>(L.in.tasks), first, L.task_elements, value);
}

// the N agent elements from `first` on: (b, a, f) counters advanced in row-major order
template <class Self, class Out>
__device__ __forceinline__ void agent_group(const Launch& L, const Tables& S, int64_t first) {
  constexpr int N = Vec<Out>::kCount;
  const AgentSource& G = L.agents;
  const int Fa = L.in.agent_width, A = L.A, split = G.first[1];
  const Self* const tables[2] = {static_cast<const Self*>(G.table[0]), static_cast<const Self*>(G.table[1])};
  int64_t row, b;
  int32_t f, a;
  divmod(first, Fa, row, f);
  divmod(row, A, b, a);
  float value[N];
#pragma unroll
  for (int i = 0; i < N; ++i) {
    float x = 0.f;
    if (first + i < L.agent_elements) {
      const int kind = a >= split;
      const int rank = S.rank[kind][f];
      if (rank != kNone) {
        const int k = S.column[kind][f];
        const int local = kind ? a - split : a;
        const int count = kind ? G.count[1] : G.count[0];
        const int columns = kind ? L.in.self_columns[1].columns : L.in.self_columns[0].columns;
        const int src = rank < 0 ? local : (rank < local ? rank : rank + 1);
        const Self raw = (kind ? tables[1] : tables[0])[(b * count + src) * columns + k];
        x = to_float(raw, S.offset[kind][k]) * S.scale[kind][k];
      }
    }
    value[i] = x;
    if (++f == Fa) {
      f = 0;
      if (++a == A) {
        a = 0;
        ++b;
      }
    }
  }
  store_group(static_cast<Out*>(L.in.agent), first, L.agent_elements, value);
}

template <int Ft, class Self, class Out>
__global__ void __launch_bounds__(kInputThreads) inputs_kernel(const __grid_constant__ Launch L) {
  constexpr int N = Vec<Out>::kCount;
  __shared__ Tables S;
  for (int i = threadIdx.x; i < 3 * FRZ_INPUTS_MAX_COLUMNS; i += kInputThreads) {
    const int kind = i / FRZ_INPUTS_MAX_COLUMNS, k = i % FRZ_INPUTS_MAX_COLUMNS;
    const FrzInputColumns& cols = kind < 2 ? L.in.self_columns[kind] : L.in.task_columns;
    S.scale[kind][k] = cols.scale[k];
    S.offset[kind][k] = cols.offset[k];
  }
  for (int i = threadIdx.x; i < 2 * kMaxAgentWidth; i += kInputThreads) {
    S.rank[i / kMaxAgentWidth][i % kMaxAgentWidth] = L.agents.rank[i / kMaxAgentWidth][i % kMaxAgentWidth];
    S.column[i / kMaxAgentWidth][i % kMaxAgentWidth] = L.agents.column[i / kMaxAgentWidth][i % kMaxAgentWidth];
  }
  __syncthreads();
  const int64_t task_groups = (L.task_elements + N - 1) / N;
  const int64_t groups = task_groups + (L.agent_elements + N - 1) / N;
  for (int64_t g = int64_t(blockIdx.x) * kInputThreads + threadIdx.x; g < groups;
       g += int64_t(gridDim.x) * kInputThreads) {
    if (g < task_groups)
      task_group<Ft, Out>(L, S, g * N);
    else
      agent_group<Self, Out>(L, S, (g - task_groups) * N);
  }
}

template <int Ft, class Self>
int launch(const Launch& L, cudaStream_t stream) {
  const int N = L.in.output_type == FRZ_INPUTS_BF16 ? Vec<__nv_bfloat16>::kCount : Vec<float>::kCount;
  const int64_t groups = (L.task_elements + N - 1) / N + (L.agent_elements + N - 1) / N;
  const int64_t work_ctas = (groups + kInputThreads - 1) / kInputThreads;
  const int grid = persistent_grid(int(work_ctas < INT32_MAX ? work_ctas : INT32_MAX), 2048 / kInputThreads);
  if (L.in.output_type == FRZ_INPUTS_BF16)
    inputs_kernel<Ft, Self, __nv_bfloat16><<<grid, kInputThreads, 0, stream>>>(L);
  else
    inputs_kernel<Ft, Self, float><<<grid, kInputThreads, 0, stream>>>(L);
  return check_launch("inputs_kernel");
}

// the agent-block width of one kind of `count` agents with `own` self columns (0 for an empty kind)
int kind_width(int count, int own, uint32_t observed) {
  return count < 1 ? 0 : own + (count - 1) * __builtin_popcount(observed);
}

// the gather table of one kind: its own columns, then the observed columns of each other agent, then zero padding
void fill_gather(AgentSource& S, int kind, int count, int own, uint32_t observed, int width) {
  int f = 0;
  for (int k = 0; k < own; ++k, ++f) {
    S.rank[kind][f] = -1;
    S.column[kind][f] = int8_t(k);
  }
  for (int r = 0; r < count - 1; ++r)
    for (int k = 0; k < own; ++k)
      if (observed >> k & 1u) {
        S.rank[kind][f] = int8_t(r);
        S.column[kind][f] = int8_t(k);
        ++f;
      }
  for (; f < width; ++f) {
    S.rank[kind][f] = kNone;
    S.column[kind][f] = 0;
  }
}

// argument checks shared by the three domains; fills `L` (the sources are set by the caller)
int check_inputs(const FrzPolicyInputs* in, int B, int A, int task_rows, int task_columns, int views,
                 const int own[2], const int count[2], const char* what, Launch* L) {
  if (in == nullptr || in->agent == nullptr || in->tasks == nullptr) {
    set_error("%s: NULL inputs block / agent / tasks", what);
    return FRZ_ERR_NULL;
  }
  if (in->output_type != FRZ_INPUTS_F32 && in->output_type != FRZ_INPUTS_BF16) {
    set_error("%s: unknown output type %d", what, in->output_type);
    return FRZ_ERR_UNSUPPORTED;
  }
  if (B <= 0 || A < 1 || A > FRZ_MAX_AGENTS) {
    set_error("%s: unsupported shape B=%d agents=%d", what, B, A);
    return FRZ_ERR_SHAPE;
  }
  const FrzInputColumns* self = in->self_columns;
  for (int kind = 0; kind < 2; ++kind) {
    if (count[kind] > 0 && (self[kind].columns != own[kind] || (self[kind].observed >> own[kind]) != 0u)) {
      set_error("%s: self columns %d (observed 0x%x), but this configuration has %d", what, self[kind].columns,
                self[kind].observed, own[kind]);
      return FRZ_ERR_SHAPE;
    }
  }
  if (in->task_columns.columns != task_columns) {
    set_error("%s: task columns %d, but this configuration has %d", what, in->task_columns.columns, task_columns);
    return FRZ_ERR_SHAPE;
  }
  const int widths[2] = {kind_width(count[0], own[0], self[0].observed), kind_width(count[1], own[1], self[1].observed)};
  const int Fa = widths[0] > widths[1] ? widths[0] : widths[1];
  if (in->agent_width != Fa || in->task_width != task_columns + 1 || in->views != views ||
      in->task_rows != task_rows) {
    set_error("%s: widths Fa=%d Ft=%d V=%d T=%d, but this configuration has %d %d %d %d", what, in->agent_width,
              in->task_width, in->views, in->task_rows, Fa, task_columns + 1, views, task_rows);
    return FRZ_ERR_SHAPE;
  }
  L->in = *in;
  L->A = A;
  L->agents.first[0] = 0;
  L->agents.first[1] = count[0];
  for (int kind = 0; kind < 2; ++kind) {
    L->agents.count[kind] = count[kind];
    fill_gather(L->agents, kind, count[kind], own[kind], self[kind].observed, Fa);
  }
  L->task_elements = int64_t(B) * views * task_rows * (task_columns + 1);
  L->agent_elements = int64_t(B) * A * Fa;
  L->monitored = nullptr;
  L->hidden_from = A;
  return FRZ_OK;
}

}  // namespace
}  // namespace frz

extern "C" {

int frz_wildfire_policy_inputs(const FrzWildfireParams* params, const FrzWildfireBuffers* io, int32_t parallel_envs,
                               const FrzPolicyInputs* inputs, void* stream) {
  using namespace frz;
  const char* what = "frz_wildfire_policy_inputs";
  if (params == nullptr || io == nullptr) {
    set_error("%s: NULL params / buffers", what);
    return FRZ_ERR_NULL;
  }
  const int cells = params->height * params->width;
  if (params->height < 1 || params->width < 1 || cells > FRZ_MAX_CELLS) {
    set_error("%s: unsupported grid %dx%d", what, params->height, params->width);
    return FRZ_ERR_SHAPE;
  }
  const int own[2] = {4, 0}, count[2] = {params->num_agents, 0};
  Launch L;
  int status = check_inputs(inputs, parallel_envs, params->num_agents, cells, 4, 1, own, count, what, &L);
  if (status != FRZ_OK) return status;
  if (io->self_obs == nullptr || io->task_obs == nullptr || io->env_task_count == nullptr) {
    set_error("%s: NULL self_obs / task_obs / env_task_count", what);
    return FRZ_ERR_NULL;
  }
  L.agents.table[0] = io->self_obs;
  L.agents.table[1] = nullptr;
  L.task_obs = io->task_obs;
  L.env_task_count = io->env_task_count;
  return frz::launch<5, float>(L, static_cast<cudaStream_t>(stream));
}

int frz_rideshare_policy_inputs(const FrzRideshareParams* params, const FrzRideshareBuffers* io,
                                int32_t parallel_envs, const FrzPolicyInputs* inputs, void* stream) {
  using namespace frz;
  const char* what = "frz_rideshare_policy_inputs";
  if (params == nullptr || io == nullptr) {
    set_error("%s: NULL params / buffers", what);
    return FRZ_ERR_NULL;
  }
  if (params->capacity < 1 || params->capacity > FRZ_MAX_PASSENGERS) {
    set_error("%s: unsupported capacity %d", what, params->capacity);
    return FRZ_ERR_SHAPE;
  }
  const int own[2] = {4, 0}, count[2] = {params->num_agents, 0};
  Launch L;
  int status = check_inputs(inputs, parallel_envs, params->num_agents, params->capacity, FRZ_RS_TASK_COLUMNS, 1, own,
                            count, what, &L);
  if (status != FRZ_OK) return status;
  if (io->self_obs == nullptr || io->task_obs == nullptr || io->env_task_count == nullptr) {
    set_error("%s: NULL self_obs / task_obs / env_task_count", what);
    return FRZ_ERR_NULL;
  }
  L.agents.table[0] = io->self_obs;
  L.agents.table[1] = nullptr;
  L.task_obs = io->task_obs;
  L.env_task_count = io->env_task_count;
  return frz::launch<9, int32_t>(L, static_cast<cudaStream_t>(stream));
}

int frz_cyber_policy_inputs(const FrzCyberParams* params, const FrzCyberBuffers* io, int32_t parallel_envs,
                            const FrzPolicyInputs* inputs, void* stream) {
  using namespace frz;
  const char* what = "frz_cyber_policy_inputs";
  if (params == nullptr || io == nullptr) {
    set_error("%s: NULL params / buffers", what);
    return FRZ_ERR_NULL;
  }
  if (params->num_nodes < 1 || params->num_nodes > FRZ_MAX_NODES || params->num_attackers < 0 ||
      params->num_defenders < 0) {
    set_error("%s: unsupported network N=%d attackers=%d defenders=%d", what, params->num_nodes, params->num_attackers,
              params->num_defenders);
    return FRZ_ERR_SHAPE;
  }
  const int A = params->num_attackers + params->num_defenders;
  const int own[2] = {2, 3}, count[2] = {params->num_attackers, params->num_defenders};
  Launch L;
  int status = check_inputs(inputs, parallel_envs, A, params->num_nodes, 2, A, own, count, what, &L);
  if (status != FRZ_OK) return status;
  const bool hidden = (inputs->flags & FRZ_INPUTS_PARTIALLY_OBSERVABLE) != 0u && params->num_defenders > 0;
  if ((params->num_attackers > 0 && io->attacker_self == nullptr) ||
      (params->num_defenders > 0 && io->defender_self == nullptr) || io->task_obs == nullptr ||
      io->env_task_count == nullptr || (hidden && io->monitored == nullptr)) {
    set_error("%s: NULL attacker_self / defender_self / task_obs / env_task_count / monitored", what);
    return FRZ_ERR_NULL;
  }
  L.agents.table[0] = io->attacker_self;
  L.agents.table[1] = io->defender_self;
  L.task_obs = io->task_obs;
  L.env_task_count = io->env_task_count;
  if (hidden) {
    L.monitored = io->monitored;
    L.hidden_from = params->num_attackers;
  }
  return frz::launch<3, float>(L, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
