"""Cost of GAE advantages and returns on the device (``utils.returns.advantages``, include/frz_returns.h).

    python profiles/time_advantages.py [--out profiles/r7_advantages.json] [--reps 50]

Workloads are rollouts of T steps at the sizes the engine's benchmark presets run (B environments x A agents): wildfire
C4 65 536 x 10 at T = 128, wildfire C1 524 288 x 3 at T = 32, the same domain at the 1 024 environments a small run
uses at T = 128, and cybersecurity C3 524 288 x 4 at T = 64.  Each with f32 and bf16 values, with and without final
values.  Inputs are seeded uniforms; each step terminates and truncates an environment with probability 0.5 % each
(episodes of about 100 steps, the benchmark's horizon), so a few steps have both flags.

Per variant:
  kernel     one frz_advantages launch, timed with CUDA events around each launch; before every launch a 256 MB buffer
             is overwritten so that the inputs come from HBM, not L2
  torch      the same recurrence as a reverse loop over T in torch ops, as a user writes it (about eight elementwise
             launches per step), timed the same way eagerly and as a replay of a CUDA graph of the whole loop
Algorithmic bytes come from the shapes: rewards, values, advantages and returns (T x B x A each), next values, both
flag arrays (T x B bytes each) and the final values of the truncated-not-terminated steps only (the kernel reads no
others).  The HBM peak is a device-to-device copy of 2 GB measured in the same run; the card's name and power limit are
read in the same run.  The kernel's results are compared with the torch loop's (max abs difference).
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'profiles'))

from time_policy_actions import copy_peak_gbs, gpu_description, timed_launches  # noqa: E402

WORKLOADS = [('wildfire_c4', 65536, 10, 128), ('wildfire_c1', 524288, 3, 32), ('wildfire_c1_1024', 1024, 3, 128),
             ('cyber_c3', 524288, 4, 64)]
GAMMA, LAM, DONE_PROBABILITY = 0.99, 0.95, 0.005


def inputs(torch, B, A, T, dtype, final):
    gen = torch.Generator(device='cuda').manual_seed(B + T)
    uniform = lambda *shape: torch.rand(shape, generator=gen, device='cuda') * 2 - 1  # noqa: E731
    flags = lambda: torch.rand((T, B), generator=gen, device='cuda') < DONE_PROBABILITY  # noqa: E731
    return dict(rewards=uniform(T, B, A), values=uniform(T, B, A).to(dtype), terminated=flags(), truncated=flags(),
                next_values=uniform(B, A).to(dtype), final_values=uniform(T, B, A).to(dtype) if final else None)


def torch_loop(torch, x, adv, ret):
    """The recurrence of include/frz_returns.h as a reverse loop in torch ops."""
    r, v, term, trunc = x['rewards'], x['values'], x['terminated'], x['truncated']
    final = x['final_values']
    gl = GAMMA * LAM
    a = torch.zeros_like(r[0])
    for t in range(r.shape[0] - 1, -1, -1):
        following = (x['next_values'] if t == r.shape[0] - 1 else v[t + 1]).float()
        bootstrap = final[t].float() if final is not None else torch.zeros_like(following)
        nv = torch.where(term[t, :, None], 0.0, torch.where(trunc[t, :, None], bootstrap, following))
        delta = (r[t] + GAMMA * nv) - v[t].float()
        c = gl * (~(term[t] | trunc[t])).float()[:, None]
        a = delta + c * a
        adv[t].copy_(a)
    torch.add(adv, v.float(), out=ret)


def captured(torch, body):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        body()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        body()
    return graph


def algorithmic_bytes(x):
    T, B, A = x['rewards'].shape
    vb = x['values'].element_size()
    bytes_ = dict(rewards=T * B * A * 4, values=T * B * A * vb, outputs=2 * T * B * A * 4, next_values=B * A * vb,
                  flags=2 * T * B)
    if x['final_values'] is not None:
        bootstrapped = int((x['truncated'] & ~x['terminated']).sum())
        bytes_['final_values'] = bootstrapped * A * vb
    bytes_['total'] = sum(bytes_.values())
    return bytes_


def measure(name, B, A, T, reps, peak):
    import torch

    from free_range_zoo_b200.utils.returns import advantages
    flush = torch.zeros(1 << 26, dtype=torch.float32, device='cuda')  # 256 MB
    row = dict(workload=name, parallel_envs=B, agents=A, steps=T, variants={})
    for dtype, key in ((torch.float32, 'f32'), (torch.bfloat16, 'bf16')):
        for final in (False, True):
            x = inputs(torch, B, A, T, dtype, final)
            out = (torch.empty((T, B, A), device='cuda'), torch.empty((T, B, A), device='cuda'))
            ref = (torch.empty((T, B, A), device='cuda'), torch.empty((T, B, A), device='cuda'))
            kernel = lambda: advantages(**x, gamma=GAMMA, lam=LAM, out=out)  # noqa: E731
            eager = lambda: torch_loop(torch, x, *ref)  # noqa: E731
            kernel_us, kernel_all = timed_launches(torch, kernel, flush, reps)
            eager_us, eager_all = timed_launches(torch, eager, flush, max(5, reps // 5))
            graph = captured(torch, eager)
            graph_us, graph_all = timed_launches(torch, graph.replay, flush, max(5, reps // 5))
            kernel()
            graph.replay()
            torch.cuda.synchronize()
            difference = max(float((out[0] - ref[0]).abs().max()), float((out[1] - ref[1]).abs().max()))
            bytes_ = algorithmic_bytes(x)
            gbs = bytes_['total'] / (kernel_us * 1e-6) / 1e9
            row['variants'][f'{key}{"_final" if final else ""}'] = dict(
                kernel_us=kernel_us, kernel_us_all=kernel_all, torch_eager_us=eager_us, torch_eager_us_all=eager_all,
                torch_graph_us=graph_us, torch_graph_us_all=graph_all, algorithmic_bytes=bytes_, kernel_gbs=gbs,
                fraction_of_copy_peak=gbs / peak, speedup_over_torch_graph=graph_us / kernel_us,
                speedup_over_torch_eager=eager_us / kernel_us, max_abs_difference_vs_torch=difference)
            del graph, x, out, ref
            torch.cuda.empty_cache()
    return row


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument('--out', default='')
    parser.add_argument('--reps', type=int, default=50)
    parser.add_argument('--workloads', default=','.join(w[0] for w in WORKLOADS))
    args = parser.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('time_advantages.py measures on a CUDA device; none is available')
    peak = copy_peak_gbs(torch)
    result = dict(device=gpu_description(), copy_peak_gbs=peak, rows=[])
    print(json.dumps({**result['device'], 'copy_peak_gbs': peak}), flush=True)
    wanted = args.workloads.split(',')
    for name, B, A, T in WORKLOADS:
        if name in wanted:
            row = measure(name, B, A, T, args.reps, peak)
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
