"""Log-probabilities and entropies of chosen action slots under the masked softmax, with gradients, on the device
(include/frz_logprob.h); and the packed legal masks of include/frz_policy.h."""
from __future__ import annotations

import ctypes
from typing import Optional, Tuple

import torch
from torch.autograd.function import once_differentiable

from free_range_zoo_b200 import _lib


def legal_words(slots: int) -> int:
    """W = ceil(C / 32): the int32 words per row of a packed legal mask of C slots."""
    return (int(slots) + 31) // 32


def unpack_legal(bits: torch.Tensor, slots: int) -> torch.Tensor:
    """bool [..., C] from a packed legal mask int32 [..., W] (bit t % 32 of word t / 32 is slot t), e.g. to mask a greedy
    ``logits.masked_fill(~unpack_legal(bits, C), -inf).argmax(-1)``."""
    if not isinstance(bits, torch.Tensor) or bits.dtype != torch.int32 or bits.dim() < 1:
        raise ValueError('bits must be an int32 tensor [..., W]')
    if bits.shape[-1] != legal_words(slots):
        raise ValueError(f'bits must have W = ceil({slots} / 32) = {legal_words(slots)} words per row, '
                         f'not {bits.shape[-1]}')
    t = torch.arange(slots, device=bits.device)
    return (bits[..., t // 32] >> (t % 32).to(torch.int32)) & 1 != 0


def _row_stride(logits: torch.Tensor) -> Optional[int]:
    """Elements between consecutive rows of ``logits [..., C]`` when its rows are evenly spaced with unit stride along
    C (a contiguous tensor or a ``[..., :C]`` view of one), else None."""
    C = logits.shape[-1]
    if logits.numel() == 0:
        return C
    if C > 1 and logits.stride(-1) != 1:
        return None
    row_stride, expected = None, None
    for size, stride in zip(reversed(logits.shape[:-1]), reversed(logits.stride()[:-1])):
        if size == 1:
            continue
        if row_stride is None:
            row_stride = expected = stride
        if stride != expected:
            return None
        expected = stride * size
    return C if row_stride is None else row_stride


def _block(logits: torch.Tensor, slots: torch.Tensor, legal: torch.Tensor, row_stride: int) -> _lib.SlotLogProb:
    return _lib.SlotLogProb(
        rows=slots.numel(), slots=logits.shape[-1], row_stride=row_stride,
        logits_type=_lib.LOGITS_BF16 if logits.dtype == torch.bfloat16 else _lib.LOGITS_F32,
        legal_type=_lib.MASK_BITS if legal.dtype == torch.int32 else _lib.MASK_BYTES,
        logits=logits.data_ptr(), legal=legal.data_ptr(), slot=slots.data_ptr())


class _SlotLogProb(torch.autograd.Function):

    @staticmethod
    def forward(ctx, logits, slots, legal, row_stride, entropy):
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(logits, slots, legal)
        ctx.row_stride = row_stride
        log_prob = torch.empty(slots.shape, dtype=torch.float32, device=logits.device)
        ent = torch.empty(slots.shape, dtype=torch.float32, device=logits.device) if entropy else None
        if slots.numel() > 0:
            block = _block(logits, slots, legal, row_stride)
            block.log_prob, block.entropy = log_prob.data_ptr(), _lib.pointer(ent)
            with torch.cuda.device(logits.device):
                _lib.check(_lib.library().frz_slot_log_prob(ctypes.byref(block), _lib.stream_handle(logits.device)),
                           'frz_slot_log_prob')
        return (log_prob, ent) if entropy else log_prob

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_log_prob, grad_entropy=None):
        logits, slots, legal = ctx.saved_tensors
        grad = torch.empty(logits.shape, dtype=logits.dtype, device=logits.device)
        if slots.numel() == 0:
            return grad, None, None, None, None
        grad_log_prob = None if grad_log_prob is None else grad_log_prob.float().contiguous()
        grad_entropy = None if grad_entropy is None else grad_entropy.float().contiguous()
        block = _block(logits, slots, legal, ctx.row_stride)
        block.grad_log_prob, block.grad_entropy = _lib.pointer(grad_log_prob), _lib.pointer(grad_entropy)
        block.grad_logits = grad.data_ptr()
        with torch.cuda.device(logits.device):
            _lib.check(_lib.library().frz_slot_log_prob_backward(ctypes.byref(block),
                                                                 _lib.stream_handle(logits.device)),
                       'frz_slot_log_prob_backward')
        return grad, None, None, None, None


def slot_log_prob(logits: torch.Tensor, slots: torch.Tensor, legal: torch.Tensor, entropy: bool = True
                  ) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """Log-probability of the chosen slots and entropy of the softmax over the legal slots, differentiable in
    ``logits``, in one fused launch each way on the current stream (no host read: capturable in a CUDA graph).

    - ``logits`` f32 or bf16 [..., C] on a CUDA device, 1 <= C <= 288; rows evenly spaced with unit stride along C (a
      contiguous tensor, or a ``[..., :C]`` view of a wider one), as for ``sample_actions_from_logits``;
    - ``slots`` int32 [...], contiguous: the chosen slots (e.g. the ``slots`` the sampler returned);
    - ``legal`` contiguous: bool or uint8 [..., C], or the packed int32 [..., W] mask (W = ``legal_words(C)``) that
      ``legal_actions(packed=True)`` and ``sample_actions_from_logits(legal_out=...)`` write.

    Per row, over the legal slots only, with m the max legal logit and S = sum exp(l - m)::

        log_prob = (l_s - m) - log S                      (-inf when slot s is illegal or outside [0, C))
        entropy  = log S - sum exp(l_i - m) (l_i - m) / S   (a -inf legal logit adds 0, not NaN)

    A row with NaN or +inf in a legal slot, no legal slot, or only -inf legal logits gives NaN (and a NaN gradient on
    its legal slots).  Illegal slots are never read and get a gradient of exactly 0.

    The reductions are the sampler's, so ``log_prob`` equals, bit for bit, the ``log_prob`` that
    ``sample_actions_from_logits`` returned for the same logits (a first-epoch ratio ``exp(new - old)`` of exactly 1),
    and a row gives the same bits alone or in any batch, with either mask format.

    Returns ``(log_prob, entropy)``, f32 [...]; ``entropy`` is None when ``entropy=False``.  The gradient with respect
    to ``logits`` is contiguous, in the dtype of ``logits`` (bf16 rounded once), computed in one pass that recomputes
    the softmax from the logits; nothing but the inputs is kept for it.  Double backward is not supported.
    """
    if not isinstance(logits, torch.Tensor) or logits.dim() < 1:
        raise ValueError('logits must be a [..., C] tensor')
    if logits.dtype not in (torch.float32, torch.bfloat16):
        raise ValueError(f'logits must be torch.float32 or torch.bfloat16, not {logits.dtype}')
    C, lead = logits.shape[-1], tuple(logits.shape[:-1])
    if not 1 <= C <= _lib.SLOT_LOG_PROB_MAX_SLOTS:
        raise ValueError(f'logits must have 1 <= C <= {_lib.SLOT_LOG_PROB_MAX_SLOTS} slots, not {C}')
    row_stride = _row_stride(logits)
    if row_stride is None:
        raise ValueError('logits rows must be evenly spaced with unit stride along the slots (a contiguous tensor, or a '
                         '[..., :C] view of one)')
    if not isinstance(slots, torch.Tensor) or slots.dtype != torch.int32:
        raise ValueError(f'slots must be an int32 tensor of shape {lead}')
    if tuple(slots.shape) != lead:
        raise ValueError(f'slots must have shape {lead}, not {tuple(slots.shape)}')
    if not slots.is_contiguous():
        raise ValueError('slots must be contiguous')
    if not isinstance(legal, torch.Tensor) or legal.dtype not in (torch.bool, torch.uint8, torch.int32):
        raise ValueError('legal must be a bool / uint8 [..., C] or a packed int32 [..., W] tensor')
    width = legal_words(C) if legal.dtype == torch.int32 else C
    if tuple(legal.shape) != lead + (width, ):
        what = f'W = ceil({C} / 32) = {width} words' if legal.dtype == torch.int32 else f'C = {C} slots'
        raise ValueError(f'legal must have shape {lead + (width, )} ({what} per row), not {tuple(legal.shape)}')
    if not legal.is_contiguous():
        raise ValueError('legal must be contiguous')
    for name, tensor in (('logits', logits), ('slots', slots), ('legal', legal)):
        if tensor.device.type != 'cuda' or tensor.device != logits.device:
            raise ValueError(f'{name} must be on the CUDA device of logits, not {tensor.device}')
    if row_stride > 0x7FFFFFFF:
        raise ValueError('logits row stride does not fit in 32 bits')
    out = _SlotLogProb.apply(logits, slots, legal, row_stride, bool(entropy))
    return out if entropy else (out, None)
