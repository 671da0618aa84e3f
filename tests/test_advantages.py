"""GAE advantages without a GPU: the C ABI of include/frz_returns.h, argument errors reported before any launch, and the
argument checks of ``utils.returns.advantages``."""
import ctypes
import math
import os
import subprocess

import pytest
import torch

from free_range_zoo_b200 import _lib
from free_range_zoo_b200.utils.returns import advantages

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def lib():
    if not os.path.exists(_lib.LIBRARY_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return _lib.library()


def test_the_declared_symbol_is_exported_from_the_new_header_only(lib):
    declared = _lib.exported_symbols('frz_returns.h')
    assert declared == ['frz_advantages']
    assert hasattr(lib, 'frz_advantages')
    others = set()
    for header in ('frz.h', 'frz_obs.h', 'frz_autoreset.h', 'frz_policy.h', 'frz_inputs.h'):
        others |= set(_lib.exported_symbols(header))
    assert not set(declared) & others


def test_ctypes_mirror_matches_the_c_layout(tmp_path):
    constants = dict(FRZ_VALUES_F32=_lib.VALUES_F32, FRZ_VALUES_BF16=_lib.VALUES_BF16)
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "frz_returns.h"', 'int main(void) {']
    lines += [f'  printf("{name} %u\\n", (unsigned)({name}));' for name in constants]
    lines.append('  printf("FrzAdvantages %zu\\n", sizeof(FrzAdvantages));')
    for field, _ in _lib.Advantages._fields_:
        lines.append(f'  printf("FrzAdvantages.{field} %zu\\n", offsetof(FrzAdvantages, {field}));')
    lines += ['  return 0;', '}']
    source = tmp_path / 'probe.c'
    source.write_text('\n'.join(lines))
    binary = tmp_path / 'probe'
    subprocess.run(['gcc', '-I', os.path.join(ROOT, 'include'), str(source), '-o', str(binary)], check=True)
    layout = dict(line.split() for line in subprocess.run([str(binary)], capture_output=True, text=True,
                                                          check=True).stdout.splitlines())
    for name, value in constants.items():
        assert int(layout[name]) == value, name
    assert int(layout['FrzAdvantages']) == ctypes.sizeof(_lib.Advantages)
    for field, _ in _lib.Advantages._fields_:
        assert int(layout[f'FrzAdvantages.{field}']) == getattr(_lib.Advantages, field).offset, field
    # no implicit padding
    assert sum(ctypes.sizeof(kind) for _, kind in _lib.Advantages._fields_) == ctypes.sizeof(_lib.Advantages)
    # no new fault bits
    assert max(_lib.FAULT_NAMES) == 0x20


def test_null_shape_type_and_discount_errors_are_reported_without_a_gpu(lib):
    dummy = ctypes.create_string_buffer(4096)
    address = ctypes.addressof(dummy)

    def call(**fields):
        block = _lib.Advantages(T=4, B=3, A=2, value_type=_lib.VALUES_F32, gamma=0.99, rewards=address, values=address,
                                next_values=address, final_values=None, terminated=address, truncated=address,
                                advantages=address, returns=None)
        setattr(block, 'lambda', 0.95)
        for field, value in fields.items():
            setattr(block, field, value)
        return lib.frz_advantages(ctypes.byref(block), None)

    assert lib.frz_advantages(None, None) == 1  # FRZ_ERR_NULL
    assert b'NULL' in lib.frz_last_error()
    for field in ('rewards', 'values', 'next_values', 'terminated', 'truncated', 'advantages'):
        assert call(**{field: None}) == 1, field
        assert field.encode() in lib.frz_last_error()
    for field in ('T', 'B', 'A'):  # FRZ_ERR_SHAPE
        assert call(**{field: 0}) == 2 and b'shape' in lib.frz_last_error(), field
        assert call(**{field: -1}) == 2, field
    assert call(B=1 << 16, A=1 << 15) == 2  # B * A > INT32_MAX
    assert call(value_type=2) == 4 and b'value type' in lib.frz_last_error()  # FRZ_ERR_UNSUPPORTED
    assert call(value_type=-1) == 4
    for field in ('gamma', 'lambda'):
        for value in (-0.01, 1.01, math.inf, -math.inf, math.nan):
            assert call(**{field: value}) == 4 and field.encode() in lib.frz_last_error(), (field, value)
    # NULL beats the other errors; final_values and returns are optional (not launched here: T = 0)
    assert call(rewards=None, T=0, value_type=7) == 1
    assert call(T=0, final_values=address, returns=address) == 2


def _inputs(T=5, B=3, A=2, dtype=torch.float32):
    return dict(rewards=torch.zeros((T, B, A)), values=torch.zeros((T, B, A), dtype=dtype),
                terminated=torch.zeros((T, B), dtype=torch.bool), truncated=torch.zeros((T, B), dtype=torch.uint8),
                next_values=torch.zeros((B, A), dtype=dtype), final_values=torch.zeros((T, B, A), dtype=dtype))


@pytest.mark.parametrize('field,value,match', [
    ('rewards', torch.zeros((5, 3)), 'rewards'),
    ('rewards', torch.zeros((0, 3, 2)), 'rewards'),
    ('rewards', torch.zeros((5, 3, 2), dtype=torch.float64), 'rewards'),
    ('rewards', torch.zeros((5, 2, 3)).transpose(1, 2), 'rewards must be contiguous'),
    ('values', torch.zeros((5, 3, 2), dtype=torch.float16), 'values'),
    ('values', torch.zeros((5, 3, 3)), 'values'),
    ('values', torch.zeros((5, 3, 4))[..., ::2], 'values must be contiguous'),
    ('next_values', torch.zeros((3, 2), dtype=torch.bfloat16), 'next_values'),
    ('next_values', torch.zeros((2, 3)), 'next_values'),
    ('final_values', torch.zeros((5, 3, 2), dtype=torch.bfloat16), 'final_values'),
    ('final_values', torch.zeros((4, 3, 2)), 'final_values'),
    ('terminated', torch.zeros((5, 3), dtype=torch.int32), 'terminated'),
    ('terminated', torch.zeros((5, 3, 1), dtype=torch.bool), 'terminated'),
    ('truncated', torch.zeros((3, 5), dtype=torch.bool).t(), 'truncated must be contiguous'),
    ('truncated', torch.zeros((5, 4), dtype=torch.bool), 'truncated'),
    ('gamma', 1.5, 'gamma'),
    ('gamma', math.nan, 'gamma'),
    ('lam', -0.1, 'lam'),
    ('lam', math.inf, 'lam'),
    ('rewards', torch.zeros((5, 3, 2)), 'must be on the CUDA device'),  # everything valid, but on the host
])
def test_the_wrapper_rejects_bad_arguments_with_value_error(field, value, match):
    kwargs = _inputs()
    kwargs[field] = value
    with pytest.raises(ValueError, match=match):
        advantages(**kwargs)


def test_the_wrapper_rejects_bad_and_aliased_outputs():
    kwargs = _inputs()
    good = torch.zeros((5, 3, 2))
    for out, match in [((good, ), 'pair'), ((good[:, :, :1], None), 'out advantages'),
                       ((good, torch.zeros((5, 3, 2), dtype=torch.bfloat16)), 'out returns'),
                       ((torch.zeros((5, 3, 4))[..., ::2], None), 'contiguous'),
                       ((kwargs['rewards'], None), 'shares storage with an input'),
                       ((good, kwargs['final_values']), 'shares storage with an input'),
                       ((good, good), 'share storage'),
                       ((good, torch.zeros((10, 3, 2))[5:]), 'must be on the CUDA device')]:
        with pytest.raises(ValueError, match=match):
            advantages(**kwargs, out=out)
    # a view of an input's storage is refused too
    wide = torch.zeros((2, 5, 3, 2))
    kwargs['rewards'] = wide[0]
    with pytest.raises(ValueError, match='shares storage'):
        advantages(**kwargs, out=(wide[1], None))
