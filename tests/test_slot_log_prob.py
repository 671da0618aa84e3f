"""Masked slot log-probabilities without a GPU: the C ABI of include/frz_logprob.h, argument errors reported before any
launch, the packed-legal flag of include/frz_policy.h, and the argument checks of ``utils.policy``."""
import ctypes
import os
import subprocess

import pytest
import torch

from free_range_zoo_b200 import _lib, presets
from free_range_zoo_b200.envs.wildfire.env import wildfire
from free_range_zoo_b200.utils.policy import legal_words, slot_log_prob, unpack_legal

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OTHER_HEADERS = ('frz.h', 'frz_obs.h', 'frz_autoreset.h', 'frz_policy.h', 'frz_inputs.h', 'frz_returns.h')


@pytest.fixture(scope='module')
def lib():
    if not os.path.exists(_lib.LIBRARY_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return _lib.library()


def pack_legal(mask: torch.Tensor) -> torch.Tensor:
    """The packed int32 [..., W] mask of a bool [..., C] mask, by the definition in include/frz_policy.h."""
    C = mask.shape[-1]
    padded = torch.zeros(mask.shape[:-1] + (32 * legal_words(C), ), dtype=torch.int64, device=mask.device)
    padded[..., :C] = mask.to(torch.int64)
    weights = torch.tensor([1 << b for b in range(32)], dtype=torch.int64, device=mask.device)
    words = (padded.reshape(mask.shape[:-1] + (-1, 32)) * weights).sum(-1)
    return torch.where(words >= 1 << 31, words - (1 << 32), words).to(torch.int32)


def test_the_declared_symbols_are_exported_from_the_new_header_only(lib):
    declared = _lib.exported_symbols('frz_logprob.h')
    assert declared == ['frz_slot_log_prob', 'frz_slot_log_prob_backward']
    for name in declared:
        assert hasattr(lib, name)
    others = set()
    for header in OTHER_HEADERS:
        others |= set(_lib.exported_symbols(header))
    assert not set(declared) & others
    assert len(_lib.exported_symbols('frz.h')) == 27 and lib.frz_version() == 4


def test_ctypes_mirror_matches_the_c_layout(tmp_path):
    constants = dict(FRZ_MASK_BYTES=_lib.MASK_BYTES, FRZ_MASK_BITS=_lib.MASK_BITS,
                     FRZ_SLOT_LOG_PROB_MAX_SLOTS=_lib.SLOT_LOG_PROB_MAX_SLOTS,
                     FRZ_POLICY_PACKED_LEGAL=_lib.POLICY_PACKED_LEGAL, FRZ_LOGITS_F32=_lib.LOGITS_F32,
                     FRZ_LOGITS_BF16=_lib.LOGITS_BF16)
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "frz_logprob.h"', 'int main(void) {']
    lines += [f'  printf("{name} %u\\n", (unsigned)({name}));' for name in constants]
    lines.append('  printf("FrzSlotLogProb %zu\\n", sizeof(FrzSlotLogProb));')
    for field, _ in _lib.SlotLogProb._fields_:
        lines.append(f'  printf("FrzSlotLogProb.{field} %zu\\n", offsetof(FrzSlotLogProb, {field}));')
    lines += ['  return 0;', '}']
    source = tmp_path / 'probe.c'
    source.write_text('\n'.join(lines))
    binary = tmp_path / 'probe'
    subprocess.run(['gcc', '-I', os.path.join(ROOT, 'include'), str(source), '-o', str(binary)], check=True)
    layout = dict(line.split() for line in subprocess.run([str(binary)], capture_output=True, text=True,
                                                          check=True).stdout.splitlines())
    for name, value in constants.items():
        assert int(layout[name]) == value, name
    assert int(layout['FrzSlotLogProb']) == ctypes.sizeof(_lib.SlotLogProb)
    for field, _ in _lib.SlotLogProb._fields_:
        assert int(layout[f'FrzSlotLogProb.{field}']) == getattr(_lib.SlotLogProb, field).offset, field
    # no implicit padding
    assert sum(ctypes.sizeof(kind) for _, kind in _lib.SlotLogProb._fields_) == ctypes.sizeof(_lib.SlotLogProb)


@pytest.mark.parametrize('backward', [False, True])
def test_null_shape_type_and_alignment_errors_are_reported_without_a_gpu(lib, backward):
    dummy = ctypes.create_string_buffer(4096)
    address = (ctypes.addressof(dummy) + 15) // 16 * 16
    entry = lib.frz_slot_log_prob_backward if backward else lib.frz_slot_log_prob

    def call(**fields):
        block = _lib.SlotLogProb(rows=4, slots=101, row_stride=101, logits_type=_lib.LOGITS_F32,
                                 legal_type=_lib.MASK_BITS, logits=address, legal=address, slot=address,
                                 log_prob=address, entropy=None, grad_log_prob=None, grad_entropy=None,
                                 grad_logits=address)
        for field, value in fields.items():
            setattr(block, field, value)
        # rows = 0 keeps every call that passes the checks from launching (it fails the shape check instead)
        return entry(ctypes.byref(block), None)

    assert entry(None, None) == 1  # FRZ_ERR_NULL
    assert b'NULL' in lib.frz_last_error()
    required = ('logits', 'legal', 'slot') + (('grad_logits', ) if backward else ('log_prob', ))
    for field in required:
        assert call(**{field: None}) == 1, field
        assert field.encode() in lib.frz_last_error()
    # the pointers the other direction needs are not required
    optional = ('log_prob', 'entropy') if backward else ('grad_logits', 'grad_log_prob', 'grad_entropy')
    for field in optional:
        assert call(rows=0, **{field: None}) == 2, field
    for fields in (dict(rows=0), dict(rows=-1), dict(slots=0), dict(slots=289, row_stride=289), dict(slots=-3)):
        assert call(**fields) == 2 and b'shape' in lib.frz_last_error(), fields  # FRZ_ERR_SHAPE
    assert call(row_stride=100) == 2 and b'row_stride' in lib.frz_last_error()
    assert call(logits_type=2) == 4 and b'logits type' in lib.frz_last_error()  # FRZ_ERR_UNSUPPORTED
    assert call(legal_type=2) == 4 and b'legal type' in lib.frz_last_error()
    assert call(legal_type=-1) == 4
    for field in ('legal', 'slot', 'logits') + (('grad_log_prob', 'grad_entropy') if backward else
                                                ('log_prob', 'entropy')):
        assert call(**{field: address + 2}) == 2 and b'aligned' in lib.frz_last_error(), field
    assert call(logits_type=_lib.LOGITS_BF16, logits=address + 1) == 2
    if backward:
        assert call(grad_logits=address + 2) == 2 and b'aligned' in lib.frz_last_error()
        assert call(logits_type=_lib.LOGITS_BF16, logits=address + 2, grad_logits=address + 1) == 2
    # NULL beats the other errors
    assert call(logits=None, rows=0, logits_type=9) == 1


def test_the_packed_legal_flag_and_its_alignment_are_checked_without_a_gpu(lib):
    dummy = ctypes.create_string_buffer(4096)
    address = (ctypes.addressof(dummy) + 15) // 16 * 16
    params = wildfire.flatten_configuration(presets.wildfire_large(), 10, False)[0]
    io = _lib.WildfireBuffers(**{name: address for name in _lib._WF_POINTERS})
    io.mask_stride = 100

    def call(B=4, **fields):
        block = _lib.PolicyActions(mode=_lib.POLICY_LEGAL | _lib.POLICY_PACKED_LEGAL, logits_type=_lib.LOGITS_F32,
                                   logits=address, slots=101, row_stride=101, slot=address, log_prob=address,
                                   legal=address, sampler_seed=1)
        for field, value in fields.items():
            setattr(block, field, value)
        return lib.frz_wildfire_policy_actions(params, io, B, ctypes.byref(block), None)

    for mode in (_lib.POLICY_SAMPLE, _lib.POLICY_DECODE, _lib.POLICY_LEGAL):
        # the flag is accepted with every mode (B = 0: rejected at the shape check, after the mode check)
        assert call(B=0, mode=mode | _lib.POLICY_PACKED_LEGAL) == 2 and b'unsupported shape' in lib.frz_last_error()
        for offset in (1, 2, 3):
            assert call(mode=mode | _lib.POLICY_PACKED_LEGAL, legal=address + offset) == 2
            assert b'aligned' in lib.frz_last_error()
        # a byte mask has no alignment requirement
        assert call(B=0, mode=mode, legal=address + 1) == 2 and b'unsupported shape' in lib.frz_last_error()
    for mode in (3, 3 | _lib.POLICY_PACKED_LEGAL, 0x200, -1):
        assert call(mode=mode) == 4 and b'mode' in lib.frz_last_error(), mode
    assert call(mode=_lib.POLICY_LEGAL | _lib.POLICY_PACKED_LEGAL, legal=None) == 1


@pytest.mark.parametrize('C', [1, 2, 16, 31, 32, 33, 64, 65, 101, 257, 288])
def test_unpack_legal_round_trips(C):
    generator = torch.Generator().manual_seed(C)
    mask = torch.rand((3, 5, C), generator=generator) < 0.5
    mask[0, 0] = True
    mask[0, 1] = False
    bits = pack_legal(mask)
    assert bits.shape == (3, 5, legal_words(C)) and bits.dtype == torch.int32
    assert torch.equal(unpack_legal(bits, C), mask)
    # slot t is bit t % 32 of word t / 32
    t = C - 1
    assert bool((int(bits[0, 0, t // 32]) >> (t % 32)) & 1)


def test_unpack_legal_rejects_bad_words():
    with pytest.raises(ValueError, match='int32'):
        unpack_legal(torch.zeros((2, 4), dtype=torch.int64), 101)
    with pytest.raises(ValueError, match='W = ceil'):
        unpack_legal(torch.zeros((2, 3), dtype=torch.int32), 101)


def _inputs(lead=(3, 4), C=33, dtype=torch.float32):
    return dict(logits=torch.zeros(lead + (C, ), dtype=dtype), slots=torch.zeros(lead, dtype=torch.int32),
                legal=torch.ones(lead + (C, ), dtype=torch.bool))


@pytest.mark.parametrize('field,value,match', [
    ('logits', torch.zeros((3, 4, 33), dtype=torch.float16), 'logits must be torch.float32 or torch.bfloat16'),
    ('logits', torch.zeros((3, 4, 33), dtype=torch.float64), 'logits'),
    ('logits', torch.zeros(()), 'logits'),
    ('logits', torch.zeros((3, 4, 0)), 'logits must have 1 <= C <= 288'),
    ('logits', torch.zeros((3, 4, 289)), 'logits must have 1 <= C <= 288'),
    ('logits', torch.zeros((3, 33, 4)).transpose(1, 2), 'logits rows must be evenly spaced'),
    ('logits', torch.zeros((3, 4, 66))[..., ::2], 'logits rows must be evenly spaced'),
    ('logits', torch.zeros((4, 3, 33)).transpose(0, 1), 'logits rows must be evenly spaced'),
    ('logits', torch.zeros((3, 5, 40))[:, :4, :33], 'logits rows must be evenly spaced'),
    ('slots', torch.zeros((3, 4), dtype=torch.int64), 'slots must be an int32'),
    ('slots', torch.zeros((3, 5), dtype=torch.int32), 'slots must have shape'),
    ('slots', torch.zeros((4, 3), dtype=torch.int32).t(), 'slots must be contiguous'),
    ('legal', torch.ones((3, 4, 33), dtype=torch.float32), 'legal must be a bool / uint8'),
    ('legal', torch.ones((3, 4, 32), dtype=torch.bool), r'C = 33 slots'),
    ('legal', torch.ones((3, 4, 1), dtype=torch.int32), r'W = ceil\(33 / 32\) = 2 words'),
    ('legal', torch.ones((3, 4, 33), dtype=torch.int32), r'W = ceil\(33 / 32\) = 2 words'),
    ('legal', torch.ones((3, 33, 4), dtype=torch.bool).transpose(1, 2), 'legal must be contiguous'),
    ('logits', torch.zeros((3, 4, 33)), 'logits must be on the CUDA device'),  # everything valid, but on the host
])
def test_the_wrapper_rejects_bad_arguments_with_value_error(field, value, match):
    kwargs = _inputs()
    kwargs[field] = value
    with pytest.raises(ValueError, match=match):
        slot_log_prob(**kwargs)


def test_the_wrapper_accepts_strided_row_views_before_the_device_check():
    """A [..., :C] view of a wider tensor and size-1 leading dimensions pass the layout checks (and stop at the device
    check, on the host)."""
    for logits in (torch.zeros((3, 4, 40))[..., :33], torch.zeros((1, 4, 1, 33)), torch.zeros((33, ))):
        kwargs = _inputs(lead=tuple(logits.shape[:-1]))
        kwargs['logits'] = logits
        with pytest.raises(ValueError, match='must be on the CUDA device'):
            slot_log_prob(**kwargs)
