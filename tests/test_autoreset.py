"""Autoreset without a GPU: every buffer a domain binds has exactly one decision about what a restart does with it, the
C ABI of include/frz_autoreset.h, argument errors, and the constructor's refusal of the logging tap."""
import ctypes
import os
import subprocess

import pytest
import torch

from free_range_zoo_b200 import _lib, presets
from free_range_zoo_b200.envs.cybersecurity.env import cybersecurity
from free_range_zoo_b200.envs.rideshare.env import rideshare
from free_range_zoo_b200.envs.wildfire.env import wildfire

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STRUCTS = {'FrzAutoresetRow': _lib.AutoresetRow, 'FrzAutoreset': _lib.Autoreset}
DOMAINS = {'wildfire': (wildfire.raw_env, _lib._WF_POINTERS), 'rideshare': (rideshare.raw_env, _lib._RS_POINTERS),
           'cybersecurity': (cybersecurity.raw_env, _lib._CY_POINTERS)}


@pytest.fixture(scope='module')
def lib():
    if not os.path.exists(_lib.LIBRARY_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return _lib.library()


@pytest.mark.parametrize('domain', sorted(DOMAINS))
def test_every_bound_buffer_has_exactly_one_restart_decision(domain):
    """``_bound`` binds one tensor per pointer of the domain's buffer struct; each is restored from its init_* copy,
    restored from the reset snapshot, zeroed, overwritten by every step, or static -- never two of these, never none."""
    env_class, pointers = DOMAINS[domain]
    rows = env_class._autoreset_rows()
    groups = [set(rows.init), set(rows.snapshot), set(rows.zero), set(rows.overwritten), set(rows.static)]
    assert sum(len(group) for group in groups) == len(set().union(*groups)), 'a buffer is in two groups'
    assert set().union(*groups) == set(pointers), 'buffers without a decision / decisions about unknown buffers'
    assert len(rows.snapshot) == len(set(rows.snapshot)) and len(rows.zero) == len(set(rows.zero))
    for target, source in rows.init.items():
        assert source == f'init_{target}' and source in rows.static, (target, source)
    for name in ('terminated', 'truncated', 'num_moves', 'cumulative_rewards'):
        assert name in rows.zero, name
    assert 'rewards' in rows.overwritten
    assert ('agent_task_count' in rows.snapshot) and rows.agents_with_tasks == (domain != 'cybersecurity')
    assert len(rows.init) + len(rows.snapshot) + len(rows.zero) <= _lib.AUTORESET_MAX_ROWS


def test_the_declared_symbol_is_exported(lib):
    declared = _lib.exported_symbols('frz_autoreset.h')
    assert declared == ['frz_autoreset']
    assert hasattr(lib, 'frz_autoreset')
    assert not set(declared) & (set(_lib.exported_symbols('frz.h')) | set(_lib.exported_symbols('frz_obs.h')))


def test_ctypes_mirrors_match_the_c_layout(tmp_path):
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "frz_autoreset.h"', 'int main(void) {',
             '  printf("FRZ_AUTORESET_MAX_ROWS %d\\n", FRZ_AUTORESET_MAX_ROWS);']
    for c_name, mirror in STRUCTS.items():
        lines.append(f'  printf("{c_name} %zu\\n", sizeof({c_name}));')
        for field, _ in mirror._fields_:
            lines.append(f'  printf("{c_name}.{field} %zu\\n", offsetof({c_name}, {field}));')
    lines += ['  return 0;', '}']
    source = tmp_path / 'probe.c'
    source.write_text('\n'.join(lines))
    binary = tmp_path / 'probe'
    subprocess.run(['gcc', '-I', os.path.join(ROOT, 'include'), str(source), '-o', str(binary)],
                   check=True)
    layout = dict(line.split() for line in subprocess.run([str(binary)], capture_output=True, text=True,
                                                          check=True).stdout.splitlines())
    assert int(layout['FRZ_AUTORESET_MAX_ROWS']) == _lib.AUTORESET_MAX_ROWS
    for c_name, mirror in STRUCTS.items():
        assert int(layout[c_name]) == ctypes.sizeof(mirror), c_name
        for field, _ in mirror._fields_:
            assert int(layout[f'{c_name}.{field}']) == getattr(mirror, field).offset, f'{c_name}.{field}'
    for mirror in STRUCTS.values():  # no implicit padding: the fields tile the structures exactly
        assert sum(ctypes.sizeof(kind) for _, kind in mirror._fields_) == ctypes.sizeof(mirror)


def test_null_and_shape_errors_are_reported_without_a_gpu(lib):
    assert lib.frz_autoreset(None, 4, None) == 1  # FRZ_ERR_NULL
    assert b'NULL' in lib.frz_last_error()
    block = _lib.Autoreset()
    assert lib.frz_autoreset(ctypes.byref(block), 4, None) == 1
    dummy = ctypes.create_string_buffer(256)
    address = ctypes.addressof(dummy)
    for name in ('terminated', 'truncated', 'step_terminated', 'step_truncated', 'done', 'cumulative_rewards',
                 'episode_return', 'num_moves', 'episode_length', 'control', 'finished', 'finished_count', 'scratch'):
        setattr(block, name, address)
    block.num_agents = 2
    block.agent_task_count = address  # without the snapshot counts
    assert lib.frz_autoreset(ctypes.byref(block), 4, None) == 1
    block.reset_agent_task_count = address
    rows = (_lib.AutoresetRow * 2)()
    block.row_count = 2  # rows missing
    assert lib.frz_autoreset(ctypes.byref(block), 4, None) == 1
    block.rows = rows
    assert lib.frz_autoreset(ctypes.byref(block), 4, None) == 1  # a row without a destination
    for row in rows:
        row.dst, row.bytes = address, 8
    rows[1].bytes = 0
    assert lib.frz_autoreset(ctypes.byref(block), 4, None) == 2  # FRZ_ERR_SHAPE
    rows[1].bytes = 4
    for change in (dict(parallel_envs=0), dict(num_agents=0), dict(num_agents=33),
                   dict(row_count=_lib.AUTORESET_MAX_ROWS + 1), dict(row_count=-1)):
        B = change.pop('parallel_envs', 4)
        saved = {name: getattr(block, name) for name in change}
        for name, value in change.items():
            setattr(block, name, value)
        assert lib.frz_autoreset(ctypes.byref(block), B, None) == 2, change
        assert b'unsupported' in lib.frz_last_error()
        for name, value in saved.items():
            setattr(block, name, value)


@pytest.mark.parametrize('domain,config', [('wildfire', presets.wildfire_large), ('rideshare', presets.rideshare_c2),
                                           ('cybersecurity', presets.cyber_c3)])
def test_autoreset_refuses_a_log_directory(domain, config, tmp_path):
    """A restart happens on the device inside the step, out of the logging tap's sight (before any device work)."""
    with pytest.raises(ValueError, match='log_directory'):
        DOMAINS[domain][0](configuration=config(), parallel_envs=2, max_steps=5, device=torch.device('cuda', 0),
                           autoreset=True, log_directory=str(tmp_path))
