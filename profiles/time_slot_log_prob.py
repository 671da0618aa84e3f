"""Cost of masked slot log-probabilities and entropies with their gradient (``utils.policy.slot_log_prob``,
include/frz_logprob.h) against the torch expression a training script writes instead.

    python profiles/time_slot_log_prob.py [--out profiles/r8_slot_log_prob.json] [--reps 20]

Workloads are the rows a policy update recomputes: wildfire C4 (65 536 environments x 10 agents, C = 101) for one step
(655 360 rows) and for a minibatch of 8 steps (5 242 880 rows, whose logits exceed the 126 MB L2), and rideshare C2 at
its saturating batch (524 288 x 4 = 2 097 152 rows, C = 33).  Logits are seeded normals (f32 and bf16), masks seeded
with density 0.5 plus the noop, slots a legal slot per row.

Per variant:
  fused      one frz_slot_log_prob launch (forward, with entropy) and one frz_slot_log_prob_backward launch (both
             incoming gradients), with the bool mask and with the packed mask; CUDA events around each launch
  torch      ``log_softmax(logits.float().masked_fill(~legal, -inf))``, the gather of the chosen slot, and the NaN-safe
             entropy ``-(exp(logp) * logp.masked_fill(~legal, 0)).sum(-1)``; forward alone, and forward + backward
             (``torch.autograd.grad`` with both incoming gradients), on the bool mask
Before every timed launch a 256 MB buffer is overwritten so that inputs come from HBM, not L2.  Algorithmic bytes come
from the shapes (logits, mask, slots and outputs for the forward; logits, mask, slots, incoming gradients and the
gradient for the backward).  The HBM peak is a 2 GB device-to-device copy measured in the same run, as are the card's
name and power limit.  Peak memory is the most allocated during forward + backward through the public API, above the
inputs.  Results are compared with the torch expression (max abs difference where both are finite).
"""
import argparse
import ctypes
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'profiles'))

from time_policy_actions import copy_peak_gbs, gpu_description, timed_launches  # noqa: E402

WORKLOADS = [('wildfire_c4_1step', 655360, 101), ('wildfire_c4_8steps', 5242880, 101),
             ('rideshare_c2', 2097152, 33)]


def inputs(torch, R, C, dtype):
    gen = torch.Generator(device='cuda').manual_seed(R + C)
    logits = (torch.randn((R, C), generator=gen, device='cuda') * 2.0).to(dtype)
    legal = torch.rand((R, C), generator=gen, device='cuda') < 0.5
    legal[:, -1] = True
    slots = torch.rand((R, C), generator=gen, device='cuda').masked_fill(~legal, -1.0).argmax(-1).to(torch.int32)
    return logits, legal, slots


def torch_forward(torch, logits, legal, slots):
    logp = torch.log_softmax(logits.float().masked_fill(~legal, float('-inf')), -1)
    lp = logp.gather(-1, slots.long()[:, None])[:, 0]
    entropy = -(logp.exp() * logp.masked_fill(~legal, 0.0)).sum(-1)
    return lp, entropy


def algorithmic_bytes(R, C, element, packed):
    mask = R * 4 * ((C + 31) // 32) if packed else R * C
    logits = R * C * element
    forward = logits + mask + R * 4 + 2 * R * 4
    backward = logits + mask + R * 4 + 2 * R * 4 + logits
    return dict(forward=forward, backward=backward, mask=mask)


def measure(name, R, C, reps, peak):
    import torch

    from free_range_zoo_b200 import _lib
    from free_range_zoo_b200.utils.policy import slot_log_prob
    from tests.test_slot_log_prob import pack_legal
    lib = _lib.library()
    flush = torch.zeros(1 << 26, dtype=torch.float32, device='cuda')  # 256 MB
    stream = _lib.stream_handle(torch.device('cuda'))
    row = dict(workload=name, rows=R, slots=C, variants={})
    for dtype, key in ((torch.float32, 'f32'), (torch.bfloat16, 'bf16')):
        logits, legal, slots = inputs(torch, R, C, dtype)
        bits = pack_legal(legal)
        g_lp = torch.randn((R, ), device='cuda')
        g_h = torch.randn((R, ), device='cuda')
        lp = torch.empty((R, ), device='cuda')
        ent = torch.empty((R, ), device='cuda')
        grad = torch.empty((R, C), dtype=dtype, device='cuda')
        # the torch expression, forward and forward + backward
        x = logits.detach().requires_grad_(True)
        forward = lambda: torch_forward(torch, logits, legal, slots)  # noqa: E731

        def both():
            out = torch_forward(torch, x, legal, slots)
            return torch.autograd.grad(out, x, (g_lp, g_h))[0]

        torch_fwd_us, torch_fwd_all = timed_launches(torch, forward, flush, reps)
        torch_both_us, torch_both_all = timed_launches(torch, both, flush, reps)
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        want_grad = both()
        torch.cuda.synchronize()
        torch_peak = torch.cuda.max_memory_allocated() - base
        want_lp, want_h = forward()
        for mask, mask_key in ((legal, 'bytes'), (bits, 'packed')):
            packed = mask_key == 'packed'
            block = _lib.SlotLogProb(
                rows=R, slots=C, row_stride=C, logits_type=_lib.LOGITS_BF16 if dtype == torch.bfloat16 else
                _lib.LOGITS_F32, legal_type=_lib.MASK_BITS if packed else _lib.MASK_BYTES, logits=logits.data_ptr(),
                legal=mask.data_ptr(), slot=slots.data_ptr(), log_prob=lp.data_ptr(), entropy=ent.data_ptr(),
                grad_log_prob=g_lp.data_ptr(), grad_entropy=g_h.data_ptr(), grad_logits=grad.data_ptr())
            fwd = lambda: _lib.check(lib.frz_slot_log_prob(ctypes.byref(block), stream))  # noqa: E731
            bwd = lambda: _lib.check(lib.frz_slot_log_prob_backward(ctypes.byref(block), stream))  # noqa: E731
            fwd_us, fwd_all = timed_launches(torch, fwd, flush, reps)
            bwd_us, bwd_all = timed_launches(torch, bwd, flush, reps)
            torch.cuda.synchronize()
            finite = torch.isfinite(want_lp)
            difference = dict(log_prob=float((lp - want_lp)[finite].abs().max()),
                              entropy=float((ent - want_h).abs().max()),
                              gradient=float((grad.float() - want_grad.float()).abs().max()))
            # peak memory through the public API
            y = logits.detach().requires_grad_(True)
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            out = slot_log_prob(y, slots, mask)
            torch.autograd.grad(out, y, (g_lp, g_h))
            torch.cuda.synchronize()
            fused_peak = torch.cuda.max_memory_allocated() - base
            del out
            bytes_ = algorithmic_bytes(R, C, logits.element_size(), packed)
            fwd_gbs = bytes_['forward'] / (fwd_us * 1e-6) / 1e9
            bwd_gbs = bytes_['backward'] / (bwd_us * 1e-6) / 1e9
            row['variants'][f'{key}_{mask_key}'] = dict(
                forward_us=fwd_us, forward_us_all=fwd_all, backward_us=bwd_us, backward_us_all=bwd_all,
                forward_backward_us=fwd_us + bwd_us, torch_forward_us=torch_fwd_us, torch_forward_us_all=torch_fwd_all,
                torch_forward_backward_us=torch_both_us, torch_forward_backward_us_all=torch_both_all,
                algorithmic_bytes=bytes_, forward_gbs=fwd_gbs, backward_gbs=bwd_gbs,
                forward_fraction_of_copy_peak=fwd_gbs / peak, backward_fraction_of_copy_peak=bwd_gbs / peak,
                speedup_forward=torch_fwd_us / fwd_us, speedup_forward_backward=torch_both_us / (fwd_us + bwd_us),
                peak_allocated_bytes_fused=fused_peak, peak_allocated_bytes_torch=torch_peak,
                max_abs_difference_vs_torch=difference)
        del logits, legal, slots, bits, grad, x, want_grad
        torch.cuda.empty_cache()
    return row


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument('--out', default='')
    parser.add_argument('--reps', type=int, default=20)
    parser.add_argument('--workloads', default=','.join(w[0] for w in WORKLOADS))
    args = parser.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('time_slot_log_prob.py measures on a CUDA device; none is available')
    peak = copy_peak_gbs(torch)
    result = dict(device=gpu_description(), copy_peak_gbs=peak, rows=[])
    print(json.dumps({**result['device'], 'copy_peak_gbs': peak}), flush=True)
    wanted = args.workloads.split(',')
    for name, R, C in WORKLOADS:
        if name in wanted:
            row = measure(name, R, C, args.reps, peak)
            brief = {key: {k: v for k, v in value.items() if not k.endswith('_all') and k != 'algorithmic_bytes'}
                     for key, value in row['variants'].items()}
            print(json.dumps(dict(workload=name, variants=brief)), flush=True)
            result['rows'].append(row)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as handle:
            json.dump(result, handle, indent=1)


if __name__ == '__main__':
    main()
