"""Cost of the same-step autoreset (``autoreset=True``, include/frz_autoreset.h) per workload.

    python profiles/time_autoreset.py [--out r4_autoreset.json] [--windows 5] [--graph-steps 10]

Four variants of one engine over whole episodes of ``max_steps`` = 100 steps (the horizon of every named workload),
actions sampled on the device:
  off       ``autoreset=False``: ``capture_graph(sample=True, steps=K)`` replays
  on        ``autoreset=True``: the same replays, the autoreset launches captured after every step
  final     ``autoreset=True, keep_final_observations=True``: as ``on``, the restore also keeps the final observations
  explicit  ``autoreset=False`` with ``reset_batches(finished)`` after every step (eager: the index list needs the host)
Each window resets the engine (untimed), then times one episode with CUDA events; windows alternate between the
variants.  env-steps/s = B x max_steps / episode time (the nominal step count: after every environment of an ``off``
batch has terminated, its remaining steps are no-ops).

The autoreset launches alone, inside a graph of 20 back-to-back calls: on a step where no environment finished, and
where every environment is truncated (the graph sets every truncated flag before each call; the same graph without the
autoreset is subtracted), for ``on`` and for ``final``.  The working sets are smaller than L2 at C4 and larger at the
524 288-environment workloads.
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
             ('rideshare_c2', 'rideshare', 'rideshare_c2', {}, 524288),
             ('cyber_c3', 'cybersecurity', 'cyber_c3', dict(show_bad_actions=False, partially_observable=True), 524288),
             ('wildfire_c1', 'wildfire', 'wildfire_3x3', {}, 524288)]
MAX_STEPS, SEED, SAMPLER, REPS = 100, 2026, 2026, 20


def gpu_description():
    import torch
    info = {'gpu': torch.cuda.get_device_name(0)}
    try:
        info['power_limit'] = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'],
                                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        info['power_limit'] = 'unknown'
    return info


def make(domain, preset, kwargs, B, autoreset, keep=False):
    import torch

    from free_range_zoo_b200 import presets
    module = importlib.import_module(f'free_range_zoo_b200.envs.{domain}_v0')
    env = module.parallel_env(parallel_envs=B, max_steps=MAX_STEPS, configuration=getattr(presets, preset)(),
                              device=torch.device('cuda:0'), autoreset=autoreset,
                              keep_final_observations=keep, **kwargs)
    return env.unwrapped


def timed(torch, body):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    body()
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop)


def episode(torch, raw, variant, graph_steps):
    """Milliseconds of one episode from a fresh reset."""
    raw.reset(seed=SEED)
    if variant == 'explicit':
        def body():
            for _ in range(MAX_STEPS):
                raw.sample_actions(SAMPLER)
                raw.step_all()
                raw.reset_batches(raw.finished.nonzero().flatten())
    else:
        def body():
            for _ in range(MAX_STEPS // graph_steps):
                raw.replay()
    return timed(torch, body)


def autoreset_launch_us(torch, raw, every_truncated):
    """Microseconds of one frz_autoreset call inside a graph of REPS calls (minus the flag fill when it is on)."""
    raw.reset(seed=SEED)
    graphs = {}
    for name, launch in (('with', True), ('without', False))[:2 if every_truncated else 1]:
        graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):  # warm-up outside capture
            raw._autoreset_launch()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        with torch.cuda.graph(graph):
            for _ in range(REPS):
                if every_truncated:
                    raw._truncated.fill_(1)
                if launch:
                    raw._autoreset_launch()
        graphs[name] = graph
    samples = {name: [] for name in graphs}
    for _ in range(5):
        for name, graph in graphs.items():
            graph.replay()
            samples[name].append(timed(torch, graph.replay))
    baseline = statistics.median(samples['without']) if every_truncated else 0.0
    return 1e3 * (statistics.median(samples['with']) - baseline) / REPS


def measure(name, domain, preset, kwargs, B, windows, graph_steps):
    import torch
    engines = {'off': make(domain, preset, kwargs, B, False), 'on': make(domain, preset, kwargs, B, True),
               'final': make(domain, preset, kwargs, B, True, keep=True), 'explicit': make(domain, preset, kwargs, B, False)}
    for variant in ('off', 'on', 'final'):
        engines[variant].reset(seed=SEED)
        engines[variant].capture_graph(sample=True, sampler_seed=SAMPLER, steps=graph_steps)
    for variant, raw in engines.items():  # warm-up episode
        episode(torch, raw, variant, graph_steps)
    times = {variant: [] for variant in engines}
    for _ in range(windows):
        for variant, raw in engines.items():
            times[variant].append(episode(torch, raw, variant, graph_steps))
    rate = {variant: [B * MAX_STEPS / (ms * 1e-3) for ms in values] for variant, values in times.items()}
    median = {variant: statistics.median(values) for variant, values in times.items()}
    on, final = engines['on'], engines['final']
    row = dict(workload=name, parallel_envs=B, max_steps=MAX_STEPS, graph_steps=graph_steps, windows=windows,
               episode_ms=times, env_steps_per_s=rate,
               env_steps_per_s_median={variant: B * MAX_STEPS / (ms * 1e-3) for variant, ms in median.items()},
               autoreset_overhead_pct=100.0 * (median['on'] / median['off'] - 1.0),
               final_overhead_pct=100.0 * (median['final'] / median['on'] - 1.0),
               explicit_step_ms=median['explicit'] / MAX_STEPS, off_step_ms=median['off'] / MAX_STEPS,
               autoreset_us_nothing_finished=autoreset_launch_us(torch, on, False),
               autoreset_us_every_env_truncated=autoreset_launch_us(torch, on, True),
               final_us_nothing_finished=autoreset_launch_us(torch, final, False),
               final_us_every_env_truncated=autoreset_launch_us(torch, final, True),
               snapshot_bytes_per_env=sum(t.numel() * t.element_size() for t in on._reset_snapshot.values()) // B,
               final_bytes_per_env=sum(t.numel() * t.element_size() for t in final._final_buffers.values()) // B)
    del engines, on, final
    torch.cuda.empty_cache()
    return row


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument('--out', default='')
    parser.add_argument('--windows', type=int, default=5)
    parser.add_argument('--graph-steps', type=int, default=10)
    parser.add_argument('--workloads', default=','.join(w[0] for w in WORKLOADS))
    args = parser.parse_args()
    if MAX_STEPS % args.graph_steps:
        raise SystemExit('--graph-steps must divide max_steps = 100')
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('time_autoreset.py measures on a CUDA device; none is available')
    result = dict(device=gpu_description(), rows=[])
    print(json.dumps(result['device']), flush=True)
    wanted = args.workloads.split(',')
    for name, domain, preset, kwargs, B in WORKLOADS:
        if name in wanted:
            row = measure(name, domain, preset, kwargs, B, args.windows, args.graph_steps)
            print(json.dumps(row), flush=True)
            result['rows'].append(row)
    if args.out:
        with open(args.out, 'w') as handle:
            json.dump(result, handle, indent=1)


if __name__ == '__main__':
    main()
