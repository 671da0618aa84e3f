"""Cost of sampling policy actions from logits on the device (``sample_actions_from_logits``, include/frz_policy.h).

    python profiles/time_policy_actions.py [--out r5_policy_actions.json] [--reps 50]

Per workload and logits type (f32, bf16):
  fused      one frz_<domain>_policy_actions launch in SAMPLE mode, timed with CUDA events around each launch; before
             every launch a 256 MB buffer is overwritten so that the logits and masks come from HBM, not L2 (the
             126 MB L2 would otherwise hold the smaller workloads' working sets)
  torch      the same pass as torch ops, as a user writes it without the engine's kernel: masked_fill, log_softmax,
             inverse-CDF sampling (torch.rand, cumsum, searchsorted), gather of the log-probability and the decode of
             the chosen slot to (choice index, action id) through ``action_space(agent)`` per agent.  The legal mask is
             handed to it precomputed (untimed), which favours it.  Timed the same way, with the same L2 flush.
Algorithmic bytes come from the shapes: logits, the legality inputs the kernel reads (wildfire action_mask rows,
rideshare task_mask rows + the chosen task row's two state columns, cybersecurity task counts and defender locations)
and the outputs (action pair, slot, log-probability: 16 bytes per agent).  The HBM peak is a device-to-device copy of
2 GB measured in the same run.

Env-steps/s of a CUDA graph of 10 x [sample_actions_from_logits -> step] (fixed f32 logits) next to 10 x
[sample_actions -> step], replayed back to back.
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = [('wildfire_c4', 'wildfire', 'wildfire_large', {}, 65536),
             ('wildfire_c1', 'wildfire', 'wildfire_3x3', {}, 524288),
             ('rideshare_c2', 'rideshare', 'rideshare_c2', {}, 524288),
             ('cyber_c3', 'cybersecurity', 'cyber_c3', dict(show_bad_actions=False, partially_observable=True), 524288)]
MAX_STEPS, SEED, SAMPLER, GRAPH_STEPS = 100, 2026, 2026, 10


def gpu_description():
    import torch
    info = {'gpu': torch.cuda.get_device_name(0)}
    try:
        info['power_limit'] = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'],
                                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        info['power_limit'] = 'unknown'
    return info


def make(domain, preset, kwargs, B):
    import torch

    from free_range_zoo_b200 import presets
    module = importlib.import_module(f'free_range_zoo_b200.envs.{domain}_v0')
    env = module.parallel_env(parallel_envs=B, max_steps=MAX_STEPS, configuration=getattr(presets, preset)(),
                              device=torch.device('cuda:0'), **kwargs)
    return env.unwrapped


def copy_peak_gbs(torch):
    source = torch.empty(1 << 31, dtype=torch.uint8, device='cuda')
    target = torch.empty_like(source)
    target.copy_(source)
    times = []
    for _ in range(10):
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        target.copy_(source)
        stop.record()
        stop.synchronize()
        times.append(start.elapsed_time(stop))
    return 2 * source.numel() / (statistics.median(times) * 1e-3) / 1e9


def timed_launches(torch, body, flush, reps):
    """Median microseconds of `body` over `reps` launches, L2 overwritten before each."""
    body()
    times = []
    for _ in range(reps):
        flush.add_(1)
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        body()
        stop.record()
        stop.synchronize()
        times.append(1e3 * start.elapsed_time(stop))
    return statistics.median(times), times


def kernel_bytes(raw, domain, element):
    B, A, C = raw.parallel_envs, len(raw.agents), raw.action_slots
    rows = B * A
    logits = rows * C * element
    if domain == 'wildfire':
        inputs = B * raw.environment_task_count.element_size() if raw.show_bad_actions else rows * raw._mask_stride
    elif domain == 'rideshare':
        inputs = rows * raw._capacity + rows * 8
    else:
        inputs = rows * 4 + B * raw._n_def * 4
    return dict(logits=logits, inputs=inputs, outputs=rows * 16, total=logits + inputs + rows * 16)


def torch_composition(torch, raw, logits, legal):
    """The pass in torch ops (see the module docstring): returns (slots, log_prob, actions)."""
    masked = logits.float().masked_fill(~legal, float('-inf'))
    log_p = torch.log_softmax(masked, dim=2)
    cdf = torch.cumsum(log_p.exp(), dim=2)
    u = torch.rand(cdf.shape[:2], device=cdf.device).unsqueeze(2) * cdf[..., -1:]
    slots = torch.searchsorted(cdf, u, right=True).clamp(max=legal.shape[2] - 1)
    log_prob = log_p.gather(2, slots).squeeze(2)
    k = (torch.cumsum(legal, dim=2, dtype=torch.int32) - 1).gather(2, slots).squeeze(2)
    ids = torch.stack([raw.action_space(agent).starts.gather(1, k[:, a:a + 1].long()).squeeze(1)
                       for a, agent in enumerate(raw.agents)], dim=1)
    return slots.squeeze(2), log_prob, torch.stack([k, ids.to(torch.int32)], dim=2)


def graph_rate(torch, raw, body, windows=5, replays=10):
    raw.reset(seed=SEED)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        body()
        raw.step_all(None)
    torch.cuda.current_stream().wait_stream(side)
    raw.reset(seed=SEED)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(GRAPH_STEPS):
            body()
            raw.step_all(None)
    rates = []
    for _ in range(windows):
        raw.reset(seed=SEED)  # (max_steps = 100 = the steps of one window: every environment stays live)
        torch.cuda.synchronize()
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        for _ in range(replays):
            graph.replay()
        stop.record()
        stop.synchronize()
        rates.append(raw.parallel_envs * GRAPH_STEPS * replays / (start.elapsed_time(stop) * 1e-3))
    return rates


def measure(name, domain, preset, kwargs, B, reps, peak):
    import torch
    raw = make(domain, preset, kwargs, B)
    raw.reset(seed=SEED)
    A, C = len(raw.agents), raw.action_slots
    flush = torch.zeros(1 << 26, dtype=torch.float32, device='cuda')  # 256 MB
    generator = torch.Generator(device='cuda').manual_seed(7)
    logits32 = torch.randn((B, A, C), device='cuda', generator=generator) * 2
    legal = raw.legal_actions().clone()
    row = dict(workload=name, parallel_envs=B, agents=A, slots=C, kernels={})
    for dtype, element in ((torch.float32, 4), (torch.bfloat16, 2)):
        logits = logits32.to(dtype)
        key = 'f32' if dtype == torch.float32 else 'bf16'
        fused_us, fused_all = timed_launches(torch, lambda: raw.sample_actions_from_logits(logits, SAMPLER), flush, reps)
        torch_us, torch_all = timed_launches(torch, lambda: torch_composition(torch, raw, logits, legal), flush,
                                             max(5, reps // 5))
        bytes_ = kernel_bytes(raw, domain, element)
        row['kernels'][key] = dict(
            fused_us=fused_us, fused_us_all=fused_all, torch_us=torch_us, torch_us_all=torch_all,
            algorithmic_bytes=bytes_, fused_gbs=bytes_['total'] / (fused_us * 1e-6) / 1e9,
            roofline_us=bytes_['total'] / (peak * 1e9) * 1e6,
            fraction_of_copy_peak=bytes_['total'] / (fused_us * 1e-6) / 1e9 / peak,
            speedup_over_torch=torch_us / fused_us)
    fixed = logits32.clone()
    row['graph_env_steps_per_s'] = dict(
        policy=graph_rate(torch, raw, lambda: raw.sample_actions_from_logits(fixed, SAMPLER)),
        uniform=graph_rate(torch, raw, lambda: raw.sample_actions(SAMPLER)))
    del raw, flush, logits32, legal
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
        raise SystemExit('time_policy_actions.py measures on a CUDA device; none is available')
    peak = copy_peak_gbs(torch)
    result = dict(device=gpu_description(), copy_peak_gbs=peak, rows=[])
    print(json.dumps({**result['device'], 'copy_peak_gbs': peak}), flush=True)
    wanted = args.workloads.split(',')
    for name, domain, preset, kwargs, B in WORKLOADS:
        if name in wanted:
            row = measure(name, domain, preset, kwargs, B, args.reps, peak)
            brief = {key: {k: v for k, v in value.items() if not k.endswith('_all')} for key, value in row['kernels'].items()}
            print(json.dumps(dict(workload=name, kernels=brief, graph={k: statistics.median(v) for k, v in
                                                                        row['graph_env_steps_per_s'].items()})),
                  flush=True)
            result['rows'].append(row)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as handle:
            json.dump(result, handle, indent=1)


if __name__ == '__main__':
    main()
