"""GAE advantages and value targets of a recorded rollout, computed on the device (include/frz_returns.h)."""
from __future__ import annotations

import ctypes
import math
import numbers
from typing import Optional, Tuple

import torch

from free_range_zoo_b200 import _lib


def _check(name: str, tensor, shape, dtypes) -> None:
    if not isinstance(tensor, torch.Tensor):
        raise ValueError(f'{name} must be a tensor')
    if tensor.dtype not in dtypes:
        raise ValueError(f'{name} must be {" or ".join(str(d) for d in dtypes)}, not {tensor.dtype}')
    if tuple(tensor.shape) != tuple(shape):
        raise ValueError(f'{name} must have shape {tuple(shape)}, not {tuple(tensor.shape)}')
    if not tensor.is_contiguous():
        raise ValueError(f'{name} must be contiguous')


def advantages(rewards: torch.Tensor, values: torch.Tensor, terminated: torch.Tensor, truncated: torch.Tensor,
               next_values: torch.Tensor, final_values: Optional[torch.Tensor] = None, gamma: float = 0.99,
               lam: float = 0.95, out: Optional[Tuple[torch.Tensor, torch.Tensor]] = None
               ) -> Tuple[torch.Tensor, torch.Tensor]:
    """Generalised advantage estimates and returns of a rollout of T steps, B environments and A agents, in one launch
    on the current stream with no host read (capturable in a CUDA graph together with the rollout).

    Inputs, contiguous and on one CUDA device:

    - ``rewards`` f32 [T, B, A]: ``r[t]``, the rewards step t returned (``env.reward_table`` after the step);
    - ``values`` f32 or bf16 [T, B, A]: ``v[t]``, the value of the observation *before* step t;
    - ``terminated``, ``truncated`` bool or uint8 [T, B]: the episode ended at step t (``env.terminated`` /
      ``env.truncated`` after the step; with ``autoreset=True`` these are the step's own flags);
    - ``next_values`` [B, A], dtype of ``values``: the value of the observation after step T-1;
    - ``final_values`` [T, B, A], dtype of ``values``, or None: the value of the final observation of step t (e.g. of
      ``policy_inputs(final=True)`` after the step); read only where ``truncated[t] and not terminated[t]``.

    The recurrence, per column (b, a), in f32 (bf16 values are widened on load)::

        nv[t]    = 0             if terminated[t]
                 = final_v[t]    if truncated[t] and not terminated[t]   (0 without final_values)
                 = v[t+1]        otherwise, t < T-1
                 = next_v        otherwise, t = T-1
        c[t]     = gamma * lam * (1 - (terminated[t] | truncated[t]))
        delta[t] = (r[t] + gamma * nv[t]) - v[t]
        A[t]     = delta[t] + c[t] * A[t+1],   A[T] = 0
        R[t]     = A[t] + v[t]

    With same-step autoreset (``autoreset=True``), step t returns the rewards and flags of the finishing episode and the
    observation after it belongs to the restarted one, so ``v[t+1]`` never bootstraps a finished step; a truncated step
    bootstraps from its final observation (``keep_final_observations=True``), a terminated one from 0, and termination
    wins when both flags are set.  Without autoreset the done flags of a finished environment stay set, so each later
    step counts as its own one-step terminated episode: use ``autoreset=True`` for training.

    A column's results depend only on T, gamma, lam and its own inputs, never on B or A: the same column gives the same
    bits alone or in any batch.  NaN inputs propagate.

    Returns ``(advantages, returns)``, f32 [T, B, A], newly allocated unless ``out=(advantages, returns)`` gives
    contiguous f32 tensors of that shape, which must not share storage with an input or with each other.
    ``out=(advantages, None)`` skips the returns and returns ``(advantages, None)``.
    """
    if not isinstance(rewards, torch.Tensor) or rewards.dim() != 3:
        raise ValueError('rewards must be a [T, B, A] tensor')
    T, B, A = rewards.shape
    if min(T, B, A) < 1:
        raise ValueError(f'rewards must have T, B, A >= 1, not {tuple(rewards.shape)}')
    _check('rewards', rewards, (T, B, A), (torch.float32, ))
    _check('values', values, (T, B, A), (torch.float32, torch.bfloat16))
    _check('next_values', next_values, (B, A), (values.dtype, ))
    if final_values is not None:
        _check('final_values', final_values, (T, B, A), (values.dtype, ))
    _check('terminated', terminated, (T, B), (torch.bool, torch.uint8))
    _check('truncated', truncated, (T, B), (torch.bool, torch.uint8))
    for name, x in (('gamma', gamma), ('lam', lam)):
        if not (isinstance(x, numbers.Real) and math.isfinite(x) and 0.0 <= x <= 1.0):
            raise ValueError(f'{name} must be a finite number in [0, 1], not {x!r}')
    inputs = {'rewards': rewards, 'values': values, 'next_values': next_values, 'terminated': terminated,
              'truncated': truncated}
    if final_values is not None:
        inputs['final_values'] = final_values
    outputs = {}
    if out is not None:
        if not isinstance(out, (tuple, list)) or len(out) != 2:
            raise ValueError('out must be a pair (advantages, returns)')
        outputs = {name: tensor for name, tensor in zip(('out advantages', 'out returns'), out)
                   if tensor is not None or name == 'out advantages'}
        for name, tensor in outputs.items():
            _check(name, tensor, (T, B, A), (torch.float32, ))
        storages = {x.untyped_storage().data_ptr() for x in inputs.values()}
        for name, tensor in outputs.items():
            if tensor.untyped_storage().data_ptr() in storages:
                raise ValueError(f'{name} shares storage with an input')
        if len(outputs) == 2 and out[0].untyped_storage().data_ptr() == out[1].untyped_storage().data_ptr():
            raise ValueError('out advantages and out returns share storage')
    device = rewards.device
    for name, tensor in dict(inputs, **outputs).items():
        if tensor.device.type != 'cuda' or tensor.device != device:
            raise ValueError(f'{name} must be on the CUDA device of rewards, not {tensor.device}')
    out = (torch.empty((T, B, A), dtype=torch.float32, device=device),
           torch.empty((T, B, A), dtype=torch.float32, device=device)) if out is None else tuple(out)
    block = _lib.Advantages(T=T, B=B, A=A, gamma=float(gamma),
                            value_type=_lib.VALUES_BF16 if values.dtype == torch.bfloat16 else _lib.VALUES_F32,
                            rewards=rewards.data_ptr(), values=values.data_ptr(), next_values=next_values.data_ptr(),
                            final_values=_lib.pointer(final_values), terminated=terminated.data_ptr(),
                            truncated=truncated.data_ptr(), advantages=out[0].data_ptr(), returns=_lib.pointer(out[1]))
    setattr(block, 'lambda', float(lam))
    with torch.cuda.device(device):
        _lib.check(_lib.library().frz_advantages(ctypes.byref(block), _lib.stream_handle(device)), 'frz_advantages')
    return out
