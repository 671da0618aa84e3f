"""Policy actions without a GPU: the C ABI of include/frz_policy.h, argument errors reported before any launch, and the
slot count of every preset."""
import ctypes
import os
import subprocess

import pytest

from free_range_zoo_b200 import _lib, presets
from free_range_zoo_b200.envs.cybersecurity.env import cybersecurity
from free_range_zoo_b200.envs.rideshare.env import rideshare
from free_range_zoo_b200.envs.wildfire.env import wildfire

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ENTRIES = ['frz_cyber_policy_actions', 'frz_rideshare_policy_actions', 'frz_wildfire_policy_actions']


@pytest.fixture(scope='module')
def lib():
    if not os.path.exists(_lib.LIBRARY_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return _lib.library()


def test_the_declared_symbols_are_exported(lib):
    declared = _lib.exported_symbols('frz_policy.h')
    assert declared == ENTRIES
    for name in declared:
        assert hasattr(lib, name)
    others = set()
    for header in ('frz.h', 'frz_obs.h', 'frz_autoreset.h'):
        others |= set(_lib.exported_symbols(header))
    assert not set(declared) & others


def test_ctypes_mirror_matches_the_c_layout(tmp_path):
    constants = dict(FRZ_FAULT_BAD_LOGITS=0x10, FRZ_FAULT_ILLEGAL_SLOT=0x20, FRZ_POLICY_SAMPLE=_lib.POLICY_SAMPLE,
                     FRZ_POLICY_DECODE=_lib.POLICY_DECODE, FRZ_POLICY_LEGAL=_lib.POLICY_LEGAL,
                     FRZ_LOGITS_F32=_lib.LOGITS_F32, FRZ_LOGITS_BF16=_lib.LOGITS_BF16)
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "frz_policy.h"', 'int main(void) {']
    lines += [f'  printf("{name} %u\\n", (unsigned)({name}));' for name in constants]
    lines.append('  printf("FrzPolicyActions %zu\\n", sizeof(FrzPolicyActions));')
    for field, _ in _lib.PolicyActions._fields_:
        lines.append(f'  printf("FrzPolicyActions.{field} %zu\\n", offsetof(FrzPolicyActions, {field}));')
    lines += ['  return 0;', '}']
    source = tmp_path / 'probe.c'
    source.write_text('\n'.join(lines))
    binary = tmp_path / 'probe'
    subprocess.run(['gcc', '-I', os.path.join(ROOT, 'include'), str(source), '-o', str(binary)], check=True)
    layout = dict(line.split() for line in subprocess.run([str(binary)], capture_output=True, text=True,
                                                          check=True).stdout.splitlines())
    for name, value in constants.items():
        assert int(layout[name]) == value, name
    assert int(layout['FrzPolicyActions']) == ctypes.sizeof(_lib.PolicyActions)
    for field, _ in _lib.PolicyActions._fields_:
        assert int(layout[f'FrzPolicyActions.{field}']) == getattr(_lib.PolicyActions, field).offset, field
    # no implicit padding
    assert sum(ctypes.sizeof(kind) for _, kind in _lib.PolicyActions._fields_) == ctypes.sizeof(_lib.PolicyActions)
    # the two fault bits follow the engine's and are named for check_errors()
    assert {0x10, 0x20} <= set(_lib.FAULT_NAMES) and max(set(_lib.FAULT_NAMES) - {0x10, 0x20}) == 0x8


def _domains():
    """(entry, params, buffers with every pointer a domain may read set to a dummy address, C)."""
    dummy = ctypes.create_string_buffer(4096)
    address = ctypes.addressof(dummy)
    wf = wildfire.flatten_configuration(presets.wildfire_large(), 10, False)[0]
    wf_io = _lib.WildfireBuffers(**{name: address for name in _lib._WF_POINTERS})
    wf_io.mask_stride = 100
    rs = rideshare.flatten_configuration(presets.rideshare_c2(), 10, 4)[0]
    rs_io = _lib.RideshareBuffers(**{name: address for name in _lib._RS_POINTERS})
    cy = cybersecurity.flatten_configuration(presets.cyber_c3(), 10, False)[0]
    cy_io = _lib.CyberBuffers(**{name: address for name in _lib._CY_POINTERS})
    return dummy, [('frz_wildfire_policy_actions', wf, wf_io, 101), ('frz_rideshare_policy_actions', rs, rs_io, 33),
                   ('frz_cyber_policy_actions', cy, cy_io, 6)]


@pytest.mark.parametrize('index', range(3))
def test_null_shape_mode_and_dtype_errors_are_reported_without_a_gpu(lib, index):
    dummy, domains = _domains()
    name, params, io, C = domains[index]
    entry = getattr(lib, name)
    address = ctypes.addressof(dummy)

    def call(B=4, params_=params, io_=io, **fields):
        block = _lib.PolicyActions(mode=_lib.POLICY_SAMPLE, logits_type=_lib.LOGITS_F32, logits=address, slots=C,
                                   row_stride=C, slot=address, log_prob=address, legal=None, sampler_seed=1)
        for field, value in fields.items():
            setattr(block, field, value)
        return entry(params_, io_, B, ctypes.byref(block), None)

    assert entry(params, io, 4, None, None) == 1  # FRZ_ERR_NULL
    assert b'NULL' in lib.frz_last_error()
    assert entry(None, io, 4, None, None) == 1
    assert call(io_=None) == 1
    assert call(logits=None) == 1
    assert call(slot=None) == 1
    assert call(mode=_lib.POLICY_DECODE, slot=None) == 1
    assert call(mode=_lib.POLICY_LEGAL) == 1  # LEGAL needs `legal`
    saved = io.actions
    io.actions = None
    assert call() == 1 and call(mode=_lib.POLICY_DECODE) == 1
    io.actions = saved
    assert call(mode=3) == 4 and b'mode' in lib.frz_last_error()  # FRZ_ERR_UNSUPPORTED
    assert call(logits_type=2) == 4 and b'logits type' in lib.frz_last_error()
    assert call(slots=C + 1) == 2 and b'slots' in lib.frz_last_error()  # FRZ_ERR_SHAPE
    assert call(slots=C - 1) == 2
    assert call(row_stride=C - 1) == 2 and b'row_stride' in lib.frz_last_error()
    assert call(B=0) == 2 and b'unsupported' in lib.frz_last_error()


@pytest.mark.parametrize('config,slots', [
    (presets.wildfire_large, 101), (presets.wildfire_3x3, 10),
    (lambda: presets.wildfire_large(height=16, width=16, num_agents=32, seed=12), 257),
    (presets.rideshare_c2, 33), (presets.cyber_c3, 6)])
def test_action_slots_of_the_presets(config, slots):
    configuration = config()
    name = type(configuration).__module__
    if 'wildfire' in name:
        env_class, params = wildfire.raw_env, wildfire.flatten_configuration(configuration, 10, False)[0]
    elif 'rideshare' in name:
        env_class, params = rideshare.raw_env, rideshare.flatten_configuration(configuration, 10, 4)[0]
    else:
        env_class, params = cybersecurity.raw_env, cybersecurity.flatten_configuration(configuration, 10, False)[0]
    env = env_class.__new__(env_class)  # (the constructor allocates device buffers)
    env._params = params
    assert env.action_slots == slots
