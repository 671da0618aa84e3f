"""ctypes binding of libfrz.so (the C ABI declared in include/frz.h).

There is deliberately no fallback: if the CUDA library has not been built (``python -c "import __graft_entry__ as g;
g.build()"`` or ``make -C free_range_zoo_b200/csrc``) importing an environment raises.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# FRZ_LIBRARY selects an alternative build of the same library (kernel tuning experiments); never a fallback
LIBRARY_PATH = os.environ.get('FRZ_LIBRARY') or os.path.join(_HERE, 'csrc', 'libfrz.so')

MAX_AGENTS = 32
MAX_EQUIPMENT = 8
MAX_CAPACITIES = 8
MAX_CELLS = 256
MAX_NODES = 32
MAX_NET_STATES = 16
MAX_PASSENGERS = 64
PAD = -100

FAULT_NAMES = {
    0x1: 'action[:, 0] is not a valid index into the agent\'s task list',
    0x2: 'cybersecurity attack / movement target outside [0, num_nodes)',
    0x4: 'a non-present cybersecurity agent acted while show_bad_actions=False',
    0x8: 'rideshare passenger table overflow',
    0x10: 'policy logits are NaN or +inf in a legal slot, or -inf in every legal slot (decoded as the noop)',
    0x20: 'a policy slot is out of range or not legal (decoded as the noop)',
}


class Control(C.Structure):
    _fields_ = [('seed', C.c_uint64), ('step', C.c_uint64), ('ctas_done', C.c_uint32), ('alive_acc', C.c_uint32),
                ('alive', C.c_uint32), ('error_word', C.c_uint32), ('agents_with_tasks_acc', C.c_uint32),
                ('agents_with_tasks', C.c_uint32), ('reserved', C.c_uint32 * 6)]


# bits of WildfireParams.flags (include/frz.h)
WF_FLAGS = dict(suppressant_decrease=0x0001, suppressant_refill=0x0002, tank_switch=0x0004, critical_error=0x0008,
                degrade=0x0010, repair=0x0020, fire_increase=0x0040, fire_decrease=0x0080,
                special_burnout_probability=0x0100, fire_fuel=0x0200)
WF_BURNOUT_SCALED = 0x0400
WF_LOCALIZE_PUTOUTS = 0x0800
WF_SHOW_BAD_ACTIONS = 0x1000
WF_KERNEL_TILES, WF_KERNEL_GROUPS = 0x2000, 0x4000


class WildfireParams(C.Structure):
    _fields_ = [
        ('height', C.c_int32), ('width', C.c_int32), ('num_agents', C.c_int32), ('num_fire_states', C.c_int32),
        ('num_equipment_states', C.c_int32), ('num_capacities', C.c_int32), ('max_steps', C.c_int32),
        ('flags', C.c_uint32), ('env_offset', C.c_int64),
        ('p_increase', C.c_float), ('p_burnout', C.c_float), ('p_decrease', C.c_float), ('decrease_bonus', C.c_float),
        ('p_random_ignition', C.c_float), ('spread_lut', C.c_float * 16),
        ('p_suppressant_decrease', C.c_float), ('p_refill', C.c_float), ('p_repair', C.c_float),
        ('p_degrade', C.c_float), ('p_critical', C.c_float), ('p_tank_switch', C.c_float),
        ('capacity_cum', C.c_float * MAX_CAPACITIES), ('capacity_value', C.c_float * MAX_CAPACITIES),
        ('equipment_capacity_bonus', C.c_float * MAX_EQUIPMENT), ('equipment_power_bonus', C.c_float * MAX_EQUIPMENT),
        ('bad_attack_penalty', C.c_float), ('burnout_penalty', C.c_float), ('termination_reward', C.c_float),
        ('termination_kappa', C.c_float),
        ('agent_y', C.c_int32 * MAX_AGENTS), ('agent_x', C.c_int32 * MAX_AGENTS), ('agent_power', C.c_float * MAX_AGENTS),
    ]


_WF_POINTERS = ('fires', 'intensity', 'fuel', 'suppressants', 'capacity', 'equipment', 'init_fires', 'init_intensity',
                'init_fuel', 'init_suppressants', 'init_capacity', 'init_equipment', 'actions', 'rewards',
                'cumulative_rewards', 'terminated', 'truncated', 'num_moves', 'num_burnouts', 'burnouts', 'putouts',
                'env_task_count', 'agent_task_count', 'action_mask', 'self_obs', 'task_obs', 'cell_reward',
                'cell_ignition', 'range_mask', 'cell_agents', 'control', 'field_uniforms', 'agent_uniforms')


class WildfireBuffers(C.Structure):
    _fields_ = [(name, C.c_void_p) for name in _WF_POINTERS] + [('mask_stride', C.c_int32), ('mask_words', C.c_int32)]


CY_STOCHASTIC_STATE = 0x1
CY_SHOW_BAD_ACTIONS = 0x2
CY_MAX_LUT_BITS = 12


class CyberParams(C.Structure):
    _fields_ = [
        ('num_nodes', C.c_int32), ('num_attackers', C.c_int32), ('num_defenders', C.c_int32), ('num_states', C.c_int32),
        ('max_steps', C.c_int32), ('flags', C.c_uint32), ('env_offset', C.c_int64), ('lut_bits', C.c_int32),
        ('temperature', C.c_float), ('patch_reward', C.c_float), ('bad_action_penalty', C.c_float),
        ('power', C.c_float * MAX_AGENTS), ('persist', C.c_float * MAX_AGENTS), ('returns', C.c_float * MAX_AGENTS),
        ('state_rewards', C.c_float * MAX_NET_STATES), ('criticality', C.c_float * MAX_NODES),
    ]


_CY_POINTERS = ('network_state', 'location', 'presence', 'init_network_state', 'init_location', 'init_presence',
                'actions', 'rewards', 'cumulative_rewards', 'terminated', 'truncated', 'num_moves', 'env_task_count',
                'agent_task_count', 'attacker_self', 'defender_self', 'task_obs', 'monitored', 'score_lut', 'control',
                'network_uniforms', 'agent_uniforms')


class CyberBuffers(C.Structure):
    _fields_ = [(name, C.c_void_p) for name in _CY_POINTERS]


RS_FAST_TRAVEL = 0x1
RS_DIAGONAL_TRAVEL = 0x2
RS_VARIABLE_MOVE_COST = 0x4
RS_WAITING_COSTS = 0x8
RS_KERNEL_TILES, RS_KERNEL_GROUPS = 0x100, 0x200
RS_PASSENGER_COLUMNS = 11
RS_TASK_COLUMNS = 8


class RideshareParams(C.Structure):
    _fields_ = [
        ('num_agents', C.c_int32), ('capacity', C.c_int32), ('schedule_rows', C.c_int32), ('schedule_horizon', C.c_int32),
        ('pool_limit', C.c_int32),
        ('max_steps', C.c_int32), ('flags', C.c_uint32), ('env_offset', C.c_int64), ('wait_limit', C.c_int32 * 3),
        ('long_wait_time', C.c_int32), ('move_cost', C.c_float), ('drop_cost', C.c_float), ('noop_cost', C.c_float),
        ('accept_cost', C.c_float), ('pool_limit_cost', C.c_float), ('general_wait_cost', C.c_float),
        ('long_wait_cost', C.c_float),
    ]


_RS_POINTERS = ('agents', 'passengers', 'init_agents', 'init_passengers', 'init_count', 'schedule', 'schedule_index', 'actions',
                'rewards', 'cumulative_rewards', 'terminated', 'truncated', 'num_moves', 'env_task_count',
                'agent_task_count', 'task_mask', 'self_obs', 'task_obs', 'control')


class RideshareBuffers(C.Structure):
    _fields_ = [(name, C.c_void_p) for name in _RS_POINTERS]


MAX_CHUNKS = 16


class HostStep(C.Structure):
    """FrzHostStep: page-locked host buffers, per-slice control blocks (device) and streams of the pipelined host step."""
    _fields_ = [('actions', C.c_void_p), ('rewards', C.c_void_p), ('terminated', C.c_void_p), ('truncated', C.c_void_p),
                ('chunk_controls', C.c_void_p), ('streams', C.POINTER(C.c_void_p)), ('chunks', C.c_int32),
                ('action_format', C.c_int32), ('packed_actions', C.c_void_p), ('pipeline', C.c_void_p)]


class GatherArray(C.Structure):
    """FrzGatherArray: one padded [B, groups, capacity, row_bytes] array and where its live rows are packed to."""
    _fields_ = [('src', C.c_void_p), ('dst', C.c_void_p), ('row_bytes', C.c_int32), ('capacity', C.c_int32),
                ('groups', C.c_int32), ('reserved', C.c_int32)]


class ObsArray(C.Structure):
    """FrzObsArray (include/frz_obs.h): one array of the compact observation download."""
    _fields_ = [('src', C.c_void_p), ('dst', C.c_void_p), ('host', C.c_void_p), ('kind', C.c_int32), ('src_type', C.c_int32),
                ('dst_type', C.c_int32), ('groups', C.c_int32), ('capacity', C.c_int32), ('src_columns', C.c_int32),
                ('column_first', C.c_int32), ('columns', C.c_int32)]


class ObsDownload(C.Structure):
    """FrzObsDownload (include/frz_obs.h): counts, host offsets, device scratch and the arrays of one download."""
    _fields_ = [('counts', C.c_void_p), ('offsets', C.c_void_p), ('host_offsets', C.c_void_p), ('scan', C.c_void_p),
                ('scratch', C.c_void_p),
                ('status', C.c_void_p), ('arrays', C.POINTER(ObsArray)), ('array_count', C.c_int32),
                ('mask_groups', C.c_int32)]


class AutoresetRow(C.Structure):
    """FrzAutoresetRow (include/frz_autoreset.h): one per-environment array a restart restores (src NULL = zeros),
    its pre-restart bytes copied to ``keep`` first unless that is NULL."""
    _fields_ = [('dst', C.c_void_p), ('src', C.c_void_p), ('bytes', C.c_int64), ('keep', C.c_void_p)]


AUTORESET_MAX_ROWS = 32


class Autoreset(C.Structure):
    """FrzAutoreset (include/frz_autoreset.h): flags, episode statistics, scratch and rows of the same-step autoreset."""
    _fields_ = [(name, C.c_void_p) for name in (
        'terminated', 'truncated', 'step_terminated', 'step_truncated', 'done', 'cumulative_rewards', 'episode_return',
        'num_moves', 'episode_length', 'agent_task_count', 'reset_agent_task_count', 'control', 'finished',
        'finished_count', 'scratch')] + [('rows', C.POINTER(AutoresetRow)), ('row_count', C.c_int32),
                                         ('num_agents', C.c_int32)]


class PolicyActions(C.Structure):
    """FrzPolicyActions (include/frz_policy.h): mode, logits and outputs of one policy-actions launch."""
    _fields_ = [('mode', C.c_int32), ('logits_type', C.c_int32), ('logits', C.c_void_p), ('slots', C.c_int32),
                ('row_stride', C.c_int32), ('slot', C.c_void_p), ('log_prob', C.c_void_p), ('legal', C.c_void_p),
                ('sampler_seed', C.c_uint64)]


POLICY_SAMPLE, POLICY_DECODE, POLICY_LEGAL = 0, 1, 2
POLICY_PACKED_LEGAL = 0x100
LOGITS_F32, LOGITS_BF16 = 0, 1

INPUTS_MAX_COLUMNS = 8


class InputColumns(C.Structure):
    """FrzInputColumns (include/frz_inputs.h): per-column scale / offset of one source array of the policy inputs."""
    _fields_ = [('scale', C.c_float * INPUTS_MAX_COLUMNS), ('offset', C.c_int32 * INPUTS_MAX_COLUMNS),
                ('columns', C.c_int32), ('observed', C.c_uint32), ('pad_is_none', C.c_uint32), ('reserved', C.c_int32)]


class PolicyInputs(C.Structure):
    """FrzPolicyInputs (include/frz_inputs.h): outputs, widths and column tables of one policy-inputs launch."""
    _fields_ = [('agent', C.c_void_p), ('tasks', C.c_void_p), ('output_type', C.c_int32), ('agent_width', C.c_int32),
                ('task_width', C.c_int32), ('views', C.c_int32), ('task_rows', C.c_int32), ('flags', C.c_uint32),
                ('self_columns', InputColumns * 2), ('task_columns', InputColumns)]


INPUTS_F32, INPUTS_BF16 = 0, 1
INPUTS_PARTIALLY_OBSERVABLE = 0x1


class Advantages(C.Structure):
    """FrzAdvantages (include/frz_returns.h): sizes, discounts, inputs and outputs of one GAE launch.  (``lambda`` is a
    Python keyword: set it with ``setattr``.)"""
    _fields_ = [('T', C.c_int32), ('B', C.c_int32), ('A', C.c_int32), ('value_type', C.c_int32), ('gamma', C.c_float),
                ('lambda', C.c_float), ('rewards', C.c_void_p), ('values', C.c_void_p), ('next_values', C.c_void_p),
                ('final_values', C.c_void_p), ('terminated', C.c_void_p), ('truncated', C.c_void_p),
                ('advantages', C.c_void_p), ('returns', C.c_void_p)]


VALUES_F32, VALUES_BF16 = 0, 1


class SlotLogProb(C.Structure):
    """FrzSlotLogProb (include/frz_logprob.h): rows, logits, mask, chosen slots, outputs and incoming gradients of one
    masked log-probability / entropy launch (forward or backward)."""
    _fields_ = [('rows', C.c_int64), ('slots', C.c_int32), ('row_stride', C.c_int32), ('logits_type', C.c_int32),
                ('legal_type', C.c_int32), ('logits', C.c_void_p), ('legal', C.c_void_p), ('slot', C.c_void_p),
                ('log_prob', C.c_void_p), ('entropy', C.c_void_p), ('grad_log_prob', C.c_void_p),
                ('grad_entropy', C.c_void_p), ('grad_logits', C.c_void_p)]


MASK_BYTES, MASK_BITS = 0, 1
SLOT_LOG_PROB_MAX_SLOTS = 288

OBS_DENSE, OBS_ROWS, OBS_MASK_BITS = 0, 1, 2
OBS_I32, OBS_I16, OBS_I8, OBS_U8, OBS_F32 = 0, 1, 2, 3, 4
HOST_ACTIONS_I32, HOST_ACTIONS_I16, HOST_ACTIONS_I8 = 0, 1, 2
ABI_VERSION = 4


_lib = None


def library() -> C.CDLL:
    """Load libfrz.so once; raise (never fall back) when it is missing or has the wrong ABI."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIBRARY_PATH):
        raise RuntimeError(f'{LIBRARY_PATH} is missing: the B200 engine has no CPU fallback. '
                           'Build it with `python -c "import __graft_entry__ as g; g.build()"`.')
    lib = C.CDLL(LIBRARY_PATH)
    lib.frz_version.restype = C.c_int
    lib.frz_last_error.restype = C.c_char_p
    lib.frz_control_init.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p]
    for name in ('frz_wildfire_step', 'frz_wildfire_refresh'):
        getattr(lib, name).argtypes = [C.POINTER(WildfireParams), C.POINTER(WildfireBuffers), C.c_int32, C.c_void_p]
    lib.frz_wildfire_reset.argtypes = [C.POINTER(WildfireParams), C.POINTER(WildfireBuffers), C.c_int32, C.c_void_p,
                                       C.c_void_p]
    lib.frz_wildfire_sample_actions.argtypes = [C.POINTER(WildfireParams), C.POINTER(WildfireBuffers), C.c_int32,
                                                C.c_uint64, C.c_void_p]
    for name in ('frz_cyber_step', 'frz_cyber_refresh'):
        getattr(lib, name).argtypes = [C.POINTER(CyberParams), C.POINTER(CyberBuffers), C.c_int32, C.c_void_p]
    lib.frz_cyber_reset.argtypes = [C.POINTER(CyberParams), C.POINTER(CyberBuffers), C.c_int32, C.c_void_p, C.c_void_p]
    lib.frz_cyber_sample_actions.argtypes = [C.POINTER(CyberParams), C.POINTER(CyberBuffers), C.c_int32, C.c_uint64,
                                             C.c_void_p]
    for name in ('frz_rideshare_step', 'frz_rideshare_refresh'):
        getattr(lib, name).argtypes = [C.POINTER(RideshareParams), C.POINTER(RideshareBuffers), C.c_int32, C.c_void_p]
    lib.frz_rideshare_reset.argtypes = [C.POINTER(RideshareParams), C.POINTER(RideshareBuffers), C.c_int32, C.c_void_p,
                                        C.c_void_p]
    lib.frz_rideshare_sample_actions.argtypes = [C.POINTER(RideshareParams), C.POINTER(RideshareBuffers), C.c_int32,
                                                 C.c_uint64, C.c_void_p]
    for name, params, buffers in (('frz_wildfire_step_host', WildfireParams, WildfireBuffers),
                                  ('frz_cyber_step_host', CyberParams, CyberBuffers),
                                  ('frz_rideshare_step_host', RideshareParams, RideshareBuffers)):
        getattr(lib, name).argtypes = [C.POINTER(params), C.POINTER(buffers), C.c_int32, C.POINTER(HostStep), C.c_void_p]
    lib.frz_host_slices.argtypes = [C.c_int32, C.c_int32, C.POINTER(C.c_int32)]
    lib.frz_wildfire_tile_random_layout.argtypes = [C.POINTER(WildfireParams), C.POINTER(C.c_uint32), C.POINTER(C.c_int8)]
    lib.frz_gather_live_rows.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.POINTER(GatherArray), C.c_int32,
                                         C.c_void_p]
    lib.frz_observe_compact.argtypes = [C.POINTER(ObsDownload), C.c_int32, C.c_void_p]
    lib.frz_autoreset.argtypes = [C.POINTER(Autoreset), C.c_int32, C.c_void_p]
    for name, params, buffers in (('frz_wildfire_policy_actions', WildfireParams, WildfireBuffers),
                                  ('frz_cyber_policy_actions', CyberParams, CyberBuffers),
                                  ('frz_rideshare_policy_actions', RideshareParams, RideshareBuffers)):
        getattr(lib, name).argtypes = [C.POINTER(params), C.POINTER(buffers), C.c_int32, C.POINTER(PolicyActions),
                                       C.c_void_p]
    for name, params, buffers in (('frz_wildfire_policy_inputs', WildfireParams, WildfireBuffers),
                                  ('frz_cyber_policy_inputs', CyberParams, CyberBuffers),
                                  ('frz_rideshare_policy_inputs', RideshareParams, RideshareBuffers)):
        getattr(lib, name).argtypes = [C.POINTER(params), C.POINTER(buffers), C.c_int32, C.POINTER(PolicyInputs),
                                       C.c_void_p]
    lib.frz_advantages.argtypes = [C.POINTER(Advantages), C.c_void_p]
    for name in ('frz_slot_log_prob', 'frz_slot_log_prob_backward'):
        getattr(lib, name).argtypes = [C.POINTER(SlotLogProb), C.c_void_p]
    if lib.frz_version() != ABI_VERSION:
        raise RuntimeError(f'libfrz.so ABI version {lib.frz_version()} != {ABI_VERSION}; rebuild the library')
    lib.frz_control_restore.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p]
    lib.frz_host_pipeline_create.argtypes = [C.POINTER(C.c_void_p)]
    lib.frz_host_pipeline_destroy.argtypes = [C.c_void_p]
    for name, params in (('frz_wildfire_buffer_bytes', WildfireParams), ('frz_cyber_buffer_bytes', CyberParams),
                         ('frz_rideshare_buffer_bytes', RideshareParams)):
        getattr(lib, name).argtypes = [C.POINTER(params), C.c_int32, C.c_char_p]
        getattr(lib, name).restype = C.c_int64
    _lib = lib
    return lib


def host_slices(parallel_envs: int, chunks: int):
    """Boundaries of the slices ``frz_<domain>_step_host`` cuts a batch into (include/frz.h: frz_host_slices)."""
    bounds = (C.c_int32 * (MAX_CHUNKS + 1))()
    count = library().frz_host_slices(parallel_envs, chunks, bounds)
    if count < 0:
        check(-count, 'frz_host_slices')
    return list(bounds[:count + 1])


def check(status: int, what: str = '') -> None:
    if status != 0:
        message = library().frz_last_error().decode()
        raise RuntimeError(f'libfrz {what} failed (status {status}): {message}')


def stream_handle(device: torch.device) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def pointer(tensor: torch.Tensor | None) -> int | None:
    return None if tensor is None else tensor.data_ptr()


def exported_symbols(header: str = 'frz.h'):
    """Every extern "C" symbol an include/ header declares (used by the CPU-side ABI tests)."""
    import re
    header = os.path.join(os.path.dirname(_HERE), 'include', header)
    text = open(header).read()
    return sorted(set(re.findall(r'\b(frz_[a-z_]+)\s*\(', text)))
