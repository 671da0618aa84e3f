"""Policy inputs without a GPU: the C ABI of include/frz_inputs.h, argument errors reported before any launch, the
shapes of the presets and the scales of the schema."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from free_range_zoo_b200 import _lib, presets
from free_range_zoo_b200.envs.cybersecurity.env import cybersecurity
from free_range_zoo_b200.envs.rideshare.env import rideshare
from free_range_zoo_b200.envs.wildfire.env import wildfire

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ENTRIES = ['frz_cyber_policy_inputs', 'frz_rideshare_policy_inputs', 'frz_wildfire_policy_inputs']


@pytest.fixture(scope='module')
def lib():
    if not os.path.exists(_lib.LIBRARY_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return _lib.library()


def test_the_declared_symbols_are_exported_from_the_new_header_only(lib):
    declared = _lib.exported_symbols('frz_inputs.h')
    assert declared == ENTRIES
    for name in declared:
        assert hasattr(lib, name)
    others = set()
    for header in ('frz.h', 'frz_obs.h', 'frz_autoreset.h', 'frz_policy.h'):
        others |= set(_lib.exported_symbols(header))
    assert not set(declared) & others


def test_ctypes_mirror_matches_the_c_layout(tmp_path):
    constants = dict(FRZ_INPUTS_F32=_lib.INPUTS_F32, FRZ_INPUTS_BF16=_lib.INPUTS_BF16,
                     FRZ_INPUTS_MAX_COLUMNS=_lib.INPUTS_MAX_COLUMNS,
                     FRZ_INPUTS_PARTIALLY_OBSERVABLE=_lib.INPUTS_PARTIALLY_OBSERVABLE)
    structs = dict(FrzPolicyInputs=_lib.PolicyInputs, FrzInputColumns=_lib.InputColumns)
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "frz_inputs.h"', 'int main(void) {']
    lines += [f'  printf("{name} %u\\n", (unsigned)({name}));' for name in constants]
    for struct, mirror in structs.items():
        lines.append(f'  printf("{struct} %zu\\n", sizeof({struct}));')
        for field, _ in mirror._fields_:
            lines.append(f'  printf("{struct}.{field} %zu\\n", offsetof({struct}, {field}));')
    lines += ['  return 0;', '}']
    source = tmp_path / 'probe.c'
    source.write_text('\n'.join(lines))
    binary = tmp_path / 'probe'
    subprocess.run(['gcc', '-I', os.path.join(ROOT, 'include'), str(source), '-o', str(binary)], check=True)
    layout = dict(line.split() for line in subprocess.run([str(binary)], capture_output=True, text=True,
                                                          check=True).stdout.splitlines())
    for name, value in constants.items():
        assert int(layout[name]) == value, name
    for struct, mirror in structs.items():
        assert int(layout[struct]) == ctypes.sizeof(mirror), struct
        for field, _ in mirror._fields_:
            assert int(layout[f'{struct}.{field}']) == getattr(mirror, field).offset, field
        # no implicit padding
        assert sum(ctypes.sizeof(kind) for _, kind in mirror._fields_) == ctypes.sizeof(mirror), struct
    # no new fault bits
    assert max(_lib.FAULT_NAMES) == 0x20


def _domains():
    """(entry, params, buffers with every pointer a domain may read set to a dummy address, layout arguments)."""
    dummy = ctypes.create_string_buffer(4096)
    address = ctypes.addressof(dummy)
    wf = wildfire.flatten_configuration(presets.wildfire_large(), 10, False)[0]
    wf_io = _lib.WildfireBuffers(**{name: address for name in _lib._WF_POINTERS})
    rs = rideshare.flatten_configuration(presets.rideshare_c2(), 10, 4)[0]
    rs_io = _lib.RideshareBuffers(**{name: address for name in _lib._RS_POINTERS})
    cy = cybersecurity.flatten_configuration(presets.cyber_c3(), 10, False)[0]
    cy_io = _lib.CyberBuffers(**{name: address for name in _lib._CY_POINTERS})
    A_rs, K = int(rs.num_agents), int(rs.capacity)
    A_cy = int(cy.num_attackers) + int(cy.num_defenders)
    # (name, params, io, self column counts, observed bits, task columns, Fa, V, T, the io field every call needs)
    return dummy, [
        ('frz_wildfire_policy_inputs', wf, wf_io, (4, 0), (0b11, 0), 4, 4 + 9 * 2, 1, 100, 'task_obs'),
        ('frz_rideshare_policy_inputs', rs, rs_io, (4, 0), (0b1111, 0), 8, 4 * A_rs, 1, K, 'self_obs'),
        ('frz_cyber_policy_inputs', cy, cy_io, (2, 3), (0b1, 0b1), 2, None, A_cy, int(cy.num_nodes), 'task_obs')]


@pytest.mark.parametrize('index', range(3))
def test_null_type_width_and_shape_errors_are_reported_without_a_gpu(lib, index):
    dummy, domains = _domains()
    name, params, io, own, observed, task_columns, Fa, V, T, needed = domains[index]
    if Fa is None:  # cybersecurity: the wider of the two kinds
        counts = (int(params.num_attackers), int(params.num_defenders))
        Fa = max(o + (n - 1) * bin(m).count('1') for o, m, n in zip(own, observed, counts) if n > 0)
    entry = getattr(lib, name)
    address = ctypes.addressof(dummy)

    def block(**fields):
        b = _lib.PolicyInputs(agent=address, tasks=address, output_type=_lib.INPUTS_F32, agent_width=Fa,
                              task_width=task_columns + 1, views=V, task_rows=T)
        for kind in range(2):
            b.self_columns[kind].columns, b.self_columns[kind].observed = own[kind], observed[kind]
        b.task_columns.columns = task_columns
        for field, value in fields.items():
            setattr(b, field, value)
        return b

    def call(B=4, params_=params, io_=io, block_=None, **fields):
        return entry(params_, io_, B, ctypes.byref(block_ if block_ is not None else block(**fields)), None)

    assert entry(params, io, 4, None, None) == 1  # FRZ_ERR_NULL
    assert b'NULL' in lib.frz_last_error()
    assert entry(None, io, 4, ctypes.byref(block()), None) == 1
    assert call(io_=None) == 1
    assert call(agent=None) == 1
    assert call(tasks=None) == 1
    saved = getattr(io, needed)
    setattr(io, needed, None)
    assert call() == 1 and needed.encode() in lib.frz_last_error()
    setattr(io, needed, saved)
    assert call(output_type=2) == 4 and b'output type' in lib.frz_last_error()  # FRZ_ERR_UNSUPPORTED
    assert call(B=0) == 2 and b'unsupported shape' in lib.frz_last_error()  # FRZ_ERR_SHAPE
    assert call(B=-3) == 2
    for field, value in (('agent_width', Fa + 1), ('agent_width', Fa - 1), ('task_width', task_columns + 2),
                         ('views', V + 1), ('task_rows', T - 1)):
        assert call(**{field: value}) == 2 and b'widths' in lib.frz_last_error(), field
    wrong = block()
    wrong.task_columns.columns = task_columns + 1
    assert call(block_=wrong) == 2 and b'task columns' in lib.frz_last_error()
    wrong = block()
    wrong.self_columns[0].observed = 1 << own[0]  # a column the self table does not have
    assert call(block_=wrong) == 2 and b'self columns' in lib.frz_last_error()
    if name == 'frz_cyber_policy_inputs':  # monitored is needed only under partial observability
        saved = io.monitored
        io.monitored = None
        assert call(flags=_lib.INPUTS_PARTIALLY_OBSERVABLE) == 1 and b'monitored' in lib.frz_last_error()
        io.monitored = saved


def _env(config, **flags):
    """An environment object with only ``_params`` and the observe flags set (the constructor allocates device
    buffers); ``config`` is kept for the schema."""
    name = type(config).__module__
    if 'wildfire' in name:
        env_class, params = wildfire.raw_env, wildfire.flatten_configuration(config, 10, False)[0]
        defaults = dict(observe_other_power=False, observe_other_suppressant=False)
    elif 'rideshare' in name:
        env_class, params = rideshare.raw_env, rideshare.flatten_configuration(config, 10, 4)[0]
        defaults = {}
    else:
        env_class, params = cybersecurity.raw_env, cybersecurity.flatten_configuration(config, 10, False)[0]
        defaults = dict(observe_other_power=True, observe_other_presence=False, observe_other_location=False,
                        partially_observable=True)
    env = env_class.__new__(env_class)
    env._params = params
    for key, value in dict(defaults, **flags).items():
        setattr(env, key, value)
    return env


WILDFIRE_16 = lambda: presets.wildfire_large(height=16, width=16, num_agents=32, seed=12)  # noqa: E731


@pytest.mark.parametrize('config,flags,shapes', [
    (presets.wildfire_large, {}, {'agent': (10, 4 + 9 * 2), 'tasks': (1, 100, 5)}),
    (presets.wildfire_large, dict(observe_other_power=True), {'agent': (10, 4 + 9 * 3), 'tasks': (1, 100, 5)}),
    (presets.wildfire_large, dict(observe_other_power=True, observe_other_suppressant=True),
     {'agent': (10, 4 + 9 * 4), 'tasks': (1, 100, 5)}),
    (presets.wildfire_3x3, {}, None),
    (WILDFIRE_16, dict(observe_other_suppressant=True), {'agent': (32, 4 + 31 * 3), 'tasks': (1, 256, 5)}),
    (lambda: presets.wildfire_large(num_agents=1), dict(observe_other_power=True), {'agent': (1, 4), 'tasks': (1, 100, 5)}),
    (presets.rideshare_c2, {}, None),
    (lambda: presets.rideshare_synthetic(drivers=1, rows=16, horizon=10), {}, None),
    (presets.cyber_c3, {}, None),
    (presets.cyber_c3, dict(observe_other_power=False, observe_other_presence=True, observe_other_location=True), None),
    (presets.cyber_c3, dict(observe_other_power=False), None),
])
def test_policy_input_shapes_of_the_presets(config, flags, shapes):
    configuration = config()
    env = _env(configuration, **flags)
    p = env._params
    if shapes is None:  # derived from the configuration's own sizes
        if isinstance(env, wildfire.raw_env):
            A, HW = int(p.num_agents), int(p.height) * int(p.width)
            shapes = {'agent': (A, 4 + (A - 1) * 2), 'tasks': (1, HW, 5)}
        elif isinstance(env, rideshare.raw_env):
            A = int(p.num_agents)
            shapes = {'agent': (A, 4 * A), 'tasks': (1, int(p.capacity), 9)}
        else:
            n_att, n_def = int(p.num_attackers), int(p.num_defenders)
            att = 2 + (n_att - 1) * (int(env.observe_other_power) + int(env.observe_other_presence))
            dfn = 3 + (n_def - 1) * (int(env.observe_other_power) + int(env.observe_other_presence) +
                                     int(env.observe_other_location))
            widths = [w for w, n in ((att, n_att), (dfn, n_def)) if n > 0]
            shapes = {'agent': (n_att + n_def, max(widths)), 'tasks': (n_att + n_def, int(p.num_nodes), 3)}
    assert env.policy_input_shapes == shapes
    assert env.policy_input_shapes['tasks'][1] == env.action_slots - (3 if isinstance(env, cybersecurity.raw_env) else 1)


def _f32(x):
    return float(np.float32(x))


@pytest.mark.parametrize('config,max_steps', [(presets.wildfire_large, 10), (WILDFIRE_16, 10), (presets.rideshare_c2, 10),
                                               (presets.rideshare_c2, None), (presets.cyber_c3, 10)])
def test_the_schema_scales_are_one_over_the_published_bounds(config, max_steps):
    configuration = config()
    env = _env(configuration, observe_other_power=True)
    env.config = configuration
    H, W = int(getattr(configuration, 'grid_height', 0)), int(getattr(configuration, 'grid_width', 0))
    # the bounds the constructor publishes (the attributes observation_space reads)
    if isinstance(env, wildfire.raw_env):
        fc, ac = configuration.fire_config, configuration.agent_config
        env.agent_observation_bounds = (H, W, ac.max_fire_reduction_power, ac.suppressant_states)
        env.fire_observation_bounds = (H, W, fc.max_fire_type, fc.num_fire_states)
    elif isinstance(env, rideshare.raw_env):
        A = int(env._params.num_agents)
        env.agent_observation_bounds = (H, W, configuration.agent_config.pool_limit, configuration.agent_config.pool_limit)
        env.passenger_observation_bounds = (H, W, H, W, A, A, configuration.max_fare, max_steps)
    block = env._policy_inputs_block()
    own = lambda kind: [(_f32(block.self_columns[kind].scale[c]), block.self_columns[kind].offset[c])  # noqa: E731
                        for c in range(block.self_columns[kind].columns)]
    tasks = [(_f32(block.task_columns.scale[c]), block.task_columns.offset[c]) for c in range(block.task_columns.columns)]
    inverse = lambda high: _f32(1.0 / float(high))  # noqa: E731
    if isinstance(env, wildfire.raw_env):
        assert own(0) == [(inverse(h), 0) for h in env.agent_observation_bounds]
        assert tasks == [(inverse(h), 0) for h in env.fire_observation_bounds]
        assert block.task_columns.pad_is_none == 0
        assert block.self_columns[0].observed == 0b111  # y, x and the observed power
    elif isinstance(env, rideshare.raw_env):
        assert own(0) == [(inverse(h), 0) for h in env.agent_observation_bounds]
        assert tasks == [(inverse(H), 0), (inverse(W), 0), (inverse(H), 0), (inverse(W), 0), (inverse(A + 1), 1),
                         (inverse(A + 1), 1), (inverse(configuration.max_fare), 0),
                         (1.0 if max_steps is None else inverse(max_steps), 0)]
        assert block.task_columns.pad_is_none == 0b110000
    else:
        threat, presence = configuration.attacker_observation_bounds
        mitigation, _, location = configuration.defender_observation_bounds
        assert own(0) == [(inverse(threat), 0), (inverse(presence), 0)]
        assert own(1) == [(inverse(mitigation), 0), (1.0, 0), (inverse(location + 1), 1)]
        criticality = max(abs(int(v)) for v in np.asarray(configuration.network_config.adj_matrix).sum(1))
        assert tasks == [(inverse(configuration.network_observation_bounds[0]), 0), (inverse(criticality), 0)]
        assert block.flags == _lib.INPUTS_PARTIALLY_OBSERVABLE


def test_missing_or_non_positive_bounds_scale_by_one():
    from free_range_zoo_b200.utils.env import input_column
    assert input_column(None) == (1.0, 0)
    assert input_column(0) == (1.0, 0)
    assert input_column(-3) == (1.0, 0)
    assert input_column(None, none=True) == (1.0, 1)
    assert input_column(4) == (0.25, 0)
    assert input_column(3, none=True) == (0.25, 1)
