"""Compact observation format without a GPU: type selection from configuration bounds, ``unpack()`` of synthetic
downloads against a numpy construction, the mask byte offsets, and the C ABI of include/frz_obs.h."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

from free_range_zoo_b200 import _lib, presets
from free_range_zoo_b200.envs.cybersecurity.env import cybersecurity
from free_range_zoo_b200.envs.rideshare.env import rideshare
from free_range_zoo_b200.envs.wildfire.env import wildfire
from free_range_zoo_b200.utils import compact

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STRUCTS = {'FrzObsArray': _lib.ObsArray, 'FrzObsDownload': _lib.ObsDownload}


@pytest.fixture(scope='module')
def lib():
    if not os.path.exists(_lib.LIBRARY_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return _lib.library()


# ------------------------------------------------------------------------------------------------ type selection


def test_narrow_types():
    assert [compact.narrow_dtype(b) for b in (0, 127, 128, 32767, 32768, 2**31 - 1)] == \
        [torch.int8, torch.int8, torch.int16, torch.int16, torch.int32, torch.int32]
    assert compact.count_dtype(255) == torch.uint8 and compact.count_dtype(256) == torch.int16


def test_wildfire_types_follow_the_grid():
    assert wildfire.compact_bounds(presets.wildfire_large()) == dict(task_obs=9, agent_task_count=100)
    assert compact.narrow_dtype(wildfire.compact_bounds(presets.wildfire_3x3())['task_obs']) == torch.int8
    wide = wildfire.compact_bounds(presets.wildfire_large(height=1, width=256, num_agents=4))
    assert wide['task_obs'] == 255 and compact.narrow_dtype(wide['task_obs']) == torch.int16  # x runs to 255
    assert compact.count_dtype(256) == torch.int16  # a 1x256 grid can have 256 tasks


def test_rideshare_types_follow_grid_fares_and_horizon():
    config = presets.rideshare_c2()
    params = rideshare.flatten_configuration(config, 100, 4)[0]
    bounds = rideshare.compact_bounds(config, params, 100)
    assert bounds['task_obs'] == 100 and compact.narrow_dtype(bounds['task_obs']) == torch.int8  # padding -100, 100 steps
    assert compact.narrow_dtype(bounds['self_obs']) == torch.int8
    assert compact.narrow_dtype(rideshare.compact_bounds(config, params, 1000)['task_obs']) == torch.int16
    assert compact.narrow_dtype(rideshare.compact_bounds(config, params, None)['task_obs']) == torch.int32
    schedule = presets.synthetic_schedule(8, 10, 10, 10, seed=1)
    schedule[0, 6] = 40000  # one fare beyond int16
    fares = presets._rideshare(None, height=10, width=10, starts=[[0, 0]], pool_limit=2, diagonal=False, fast=False,
                               schedule=schedule, reward={})
    fare_params = rideshare.flatten_configuration(fares, 50, 4)[0]
    assert compact.narrow_dtype(rideshare.compact_bounds(fares, fare_params, 50)['task_obs']) == torch.int32


def test_cybersecurity_types():
    params = cybersecurity.flatten_configuration(presets.cyber_c3(), 100, False)[0]
    bounds = cybersecurity.compact_bounds(params)
    assert bounds['agent_task_count'] == 3 and compact.narrow_dtype(bounds['task_obs']) == torch.int8


# ------------------------------------------------------------------------------------------------ unpack


def synthetic_download(counts, groups, capacity, columns, dtype, rng):
    """A schema with one row array, one mask and one dense array over random padded arrays, its compact download
    encoded in numpy, and the packed arrays gather_observations() would return."""
    B = len(counts)
    task_obs = torch.from_numpy(rng.integers(-100, 100, (B, capacity, columns), dtype=np.int32))
    masks = torch.from_numpy(rng.integers(0, 2, (B, groups, capacity), dtype=np.uint8))
    self_obs = torch.from_numpy(rng.random((B, groups, 4), dtype=np.float32))
    fill = torch.from_numpy(rng.random((groups, 4), dtype=np.float32))
    schema = compact.Schema(capacity=capacity, mask_groups=groups, arrays=[
        compact.rows('task_obs', task_obs, bound=100 if dtype == torch.int8 else 1000),
        compact.mask('action_mask', masks, groups=groups),
        compact.dense('self_obs', self_obs, columns=(3, 1), fill=fill),
    ])
    offsets = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    rows = np.concatenate([task_obs.numpy()[b, :counts[b]] for b in range(B)] + [np.zeros((0, columns), np.int32)])
    bits = []
    for b in range(B):
        entries = masks.numpy()[b, :, :counts[b]].reshape(-1)  # bit g * counts[b] + t
        bits.append(np.packbits(entries, bitorder='little'))
    buffers = {
        'counts': torch.from_numpy(np.asarray(counts, dtype=np.uint8)),
        'task_obs': torch.from_numpy(rows.reshape(-1)).to(dtype),
        'action_mask': torch.from_numpy(np.concatenate(bits + [np.zeros(0, np.uint8)])),
        'self_obs': self_obs[:, :, 3].contiguous().view(-1),
    }
    observations = compact.CompactObservations(schema, buffers['counts'], torch.from_numpy(offsets), buffers)
    full_self = fill.expand(B, groups, 4).clone()
    full_self[:, :, 3] = self_obs[:, :, 3]
    packed_mask = np.concatenate([masks.numpy()[b, g, :counts[b]] for b in range(B) for g in range(groups)]
                                 + [np.zeros(0, np.uint8)])
    want = dict(task_obs=torch.from_numpy(rows), action_mask=torch.from_numpy(packed_mask), self_obs=full_self)
    return observations, offsets, want


@pytest.mark.parametrize('groups', [1, 3, 10])
@pytest.mark.parametrize('dtype', [torch.int8, torch.int16])
def test_unpack_rebuilds_the_packed_arrays(groups, dtype):
    rng = np.random.default_rng(groups)
    capacity = 13
    counts = rng.integers(0, capacity + 1, 40)
    counts[:3] = [0, capacity, 0]  # empty and full environments
    observations, offsets, want = synthetic_download(counts, groups, capacity, 4, dtype, rng)
    got = observations.unpack()
    assert np.array_equal(got['counts'].numpy(), counts) and got['counts'].dtype == torch.int32
    assert np.array_equal(got['offsets'].numpy(), offsets) and got['total'] == int(offsets[-1])
    for name, tensor in want.items():
        assert got[name].dtype == tensor.dtype and got[name].shape == tensor.shape, name
        assert torch.equal(got[name], tensor), name
    assert observations['self_obs'].shape == (40, groups)
    assert observations['task_obs'].dtype == dtype and observations['task_obs'].shape == (int(offsets[-1]), 4)
    row_bytes = 4 * torch.empty(0, dtype=dtype).element_size()
    assert observations.bytes == 40 + 4 * 41 + int(offsets[-1]) * row_bytes + \
        int(compact.mask_offsets(counts, groups)[-1]) + 40 * groups * 4


def test_unpack_of_a_batch_without_live_rows():
    rng = np.random.default_rng(0)
    observations, offsets, want = synthetic_download(np.zeros(5, np.int64), 2, 4, 4, torch.int8, rng)
    got = observations.unpack()
    assert got['total'] == 0 and got['task_obs'].shape == (0, 4) and got['action_mask'].shape == (0, )


def test_mask_offsets():
    counts = np.array([0, 1, 7, 8, 3, 0, 25])
    assert compact.mask_offsets(counts, 1).tolist() == [0, 0, 1, 2, 3, 4, 4, 8]
    assert compact.mask_offsets(counts, 10).tolist() == [0, 0, 2, 11, 21, 25, 25, 57]
    # byte-aligned per environment: the offsets of a batch are the concatenation of any slicing's
    first, second = compact.mask_offsets(counts[:3], 10), compact.mask_offsets(counts[3:], 10)
    assert np.array_equal(np.concatenate([first, first[-1] + second[1:]]), compact.mask_offsets(counts, 10))


def test_a_column_selection_needs_fill_values():
    with pytest.raises(ValueError, match='other columns'):
        compact.dense('self_obs', torch.zeros((2, 3, 4)), columns=(3, 1))
    with pytest.raises(ValueError, match='uint8'):
        compact.mask('action_mask', torch.zeros((2, 3, 4), dtype=torch.int32), groups=3)


# ------------------------------------------------------------------------------------------------ C ABI


def test_every_declared_symbol_is_exported(lib):
    declared = _lib.exported_symbols('frz_obs.h')
    assert declared == ['frz_observe_compact']
    assert all(hasattr(lib, name) for name in declared)
    assert not set(declared) & set(_lib.exported_symbols('frz.h'))


def test_ctypes_mirrors_match_the_c_layout(tmp_path):
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "frz_obs.h"', 'int main(void) {']
    for c_name, mirror in STRUCTS.items():
        lines.append(f'  printf("{c_name} %zu\\n", sizeof({c_name}));')
        for field, _ in mirror._fields_:
            lines.append(f'  printf("{c_name}.{field} %zu\\n", offsetof({c_name}, {field}));')
    lines += ['  return 0;', '}']
    source = tmp_path / 'probe.c'
    source.write_text('\n'.join(lines))
    binary = tmp_path / 'probe'
    subprocess.run(['gcc', '-I', os.path.join(ROOT, 'include'), str(source), '-o', str(binary)], check=True)
    layout = dict(line.split() for line in subprocess.run([str(binary)], capture_output=True, text=True,
                                                          check=True).stdout.splitlines())
    for c_name, mirror in STRUCTS.items():
        assert int(layout[c_name]) == ctypes.sizeof(mirror), c_name
        for field, _ in mirror._fields_:
            assert int(layout[f'{c_name}.{field}']) == getattr(mirror, field).offset, f'{c_name}.{field}'
    # no implicit padding: the fields tile the structures exactly
    for mirror in STRUCTS.values():
        assert sum(ctypes.sizeof(kind) for _, kind in mirror._fields_) == ctypes.sizeof(mirror)


def test_null_and_shape_errors_are_reported_without_a_gpu(lib):
    assert lib.frz_observe_compact(None, 4, None) == 1  # FRZ_ERR_NULL
    assert b'NULL' in lib.frz_last_error()
    block = _lib.ObsDownload()
    assert lib.frz_observe_compact(ctypes.byref(block), 4, None) == 1
    dummy = ctypes.create_string_buffer(256)
    address = ctypes.addressof(dummy)
    block.counts = block.offsets = block.scan = block.scratch = block.status = address
    assert lib.frz_observe_compact(ctypes.byref(block), 0, None) == 2  # FRZ_ERR_SHAPE
    arrays = (_lib.ObsArray * 1)()
    block.arrays, block.array_count, block.mask_groups = ctypes.cast(arrays, ctypes.POINTER(_lib.ObsArray)), 1, 2
    assert lib.frz_observe_compact(ctypes.byref(block), 4, None) == 1  # the array's pointers are NULL
    a = arrays[0]
    a.src, a.dst = address, address
    a.kind, a.src_type, a.dst_type, a.groups, a.capacity, a.src_columns, a.column_first, a.columns = \
        _lib.OBS_ROWS, _lib.OBS_I32, _lib.OBS_I8, 1, 8, 4, 0, 4
    bad = [dict(kind=7), dict(src_type=_lib.OBS_F32), dict(dst_type=_lib.OBS_F32), dict(capacity=0), dict(groups=0),
           dict(column_first=2), dict(columns=0),
           dict(kind=_lib.OBS_MASK_BITS, src_type=_lib.OBS_U8, dst_type=_lib.OBS_U8, groups=3, src_columns=1, columns=1),
           dict(kind=_lib.OBS_DENSE, groups=2), dict(capacity=1 << 28)]
    good = {name: getattr(a, name) for name, _ in _lib.ObsArray._fields_ if name not in ('src', 'dst')}
    for change in bad:
        for name, value in {**good, **change}.items():
            setattr(a, name, value)
        assert lib.frz_observe_compact(ctypes.byref(block), 4, None) == 2, change
        assert b'unsupported' in lib.frz_last_error()
