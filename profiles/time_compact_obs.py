"""Host-driven step with and without observations: ``step_host`` without observations, with ``observations=True`` (the
packed int32 / byte-mask download) and with ``observations='compact'`` (utils/compact.py), per workload; plus the
compact format downloaded the other way, ``compact_copy_engine``: encoded into the same device staging, then the host
reads the live sizes and issues one ``cudaMemcpyAsync`` per array (the alternative to the shipped mapped-memory flush).

    python profiles/time_compact_obs.py [--out r3_compact_obs.json] [--steps 24] [--window 4] [--trace DIR]

One seeded rollout is recorded per workload (actions sampled on the device, copied to page-locked host memory), then
every leg replays it from the same reset: a warm-up window, then the median over windows of ``--window`` steps (each
``step_host`` call ends in a stream synchronisation).  Bytes per step are counted from the tensors that were copied.
``unpack()`` (host CPU work a policy pays to get the packed form back) is timed separately and is not part of a leg.
"""
import argparse
import ctypes
import importlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = [('wildfire_c4', 65536), ('rideshare_c2', 524288), ('wildfire_c1', 524288), ('cyber_c3', 524288)]


def gpu_description():
    import torch
    info = {'gpu': torch.cuda.get_device_name(0)}
    try:
        limit = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'],
                               capture_output=True, text=True, timeout=30).stdout.strip()
        info['power_limit'] = limit
    except (OSError, subprocess.SubprocessError):
        info['power_limit'] = 'unknown'
    return info


def copy_engine_download(raw):
    """The compact download with copy-engine transfers: encode into the staging only (no host pointers), download the
    fixed-size arrays and the live totals, synchronise, then copy exactly the live rows / mask bytes and synchronise."""
    import torch

    from free_range_zoo_b200 import _lib
    from free_range_zoo_b200.utils import compact
    download = raw._compact_download()
    if not hasattr(download, 'staged_block'):
        arrays = (_lib.ObsArray * download.block.array_count)()
        ctypes.memmove(arrays, download.descriptors, ctypes.sizeof(arrays))
        for a in arrays:
            a.host = None
        block = _lib.ObsDownload.from_buffer_copy(download.block)
        block.host_offsets = None
        block.arrays = ctypes.cast(arrays, ctypes.POINTER(_lib.ObsArray))
        download.staged_block, download.staged_arrays = block, arrays
        download.totals = torch.zeros(2, dtype=torch.int32).pin_memory()
    B = raw.parallel_envs
    stream = torch.cuda.current_stream(raw.device)
    _lib.check(raw._lib.frz_observe_compact(ctypes.byref(download.staged_block), B, raw._stream()), 'frz_observe_compact')
    download.offsets.copy_(download.device_offsets, non_blocking=True)
    download.totals.copy_(download.scan[2 * B:2 * B + 2], non_blocking=True)
    kinds = {array.name: array for array in download.schema.arrays}
    for name, staged in download.staging.items():
        if name == 'counts' or kinds[name].kind == 'dense':
            download.buffers[name].copy_(staged, non_blocking=True)
    stream.synchronize()
    rows, mask_bytes = int(download.totals[0]), int(download.totals[1])
    for name, staged in download.staging.items():
        array = kinds.get(name)
        if array is None or array.kind == 'dense':
            continue
        live = rows * array.groups * array.columns if array.kind == 'rows' else mask_bytes
        if live:
            download.buffers[name][:live].copy_(staged[:live], non_blocking=True)
    stream.synchronize()
    return compact.CompactObservations(download.schema, download.buffers['counts'], download.offsets, download.buffers,
                                       mask_bytes)


def trace(workload, B, steps, out_dir):
    """torch.profiler over a few compact steps (a run of its own): per-kernel / per-copy device time."""
    import torch

    import bench
    from free_range_zoo_b200 import presets
    spec = bench.WORKLOADS[workload]
    module = importlib.import_module(f'free_range_zoo_b200.envs.{spec["domain"]}_v0')
    env = module.parallel_env(parallel_envs=B, max_steps=100, device=torch.device('cuda', 0),
                              configuration=getattr(presets, spec['preset'])(**spec.get('preset_kwargs', {})),
                              **spec['kwargs'])
    raw = env.unwrapped
    actions = torch.empty((B, len(raw.agents), 2), dtype=torch.int32).pin_memory()
    env.reset(seed=bench.SEED)
    for t in range(steps):
        raw.sample_actions(bench.SAMPLER)
        actions.copy_(raw._actions)
        torch.cuda.synchronize()
        if t == steps // 2:
            profiler = torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU,
                                                          torch.profiler.ProfilerActivity.CUDA])
            profiler.__enter__()
        raw.step_host(actions, observations='compact')
    profiler.__exit__(None, None, None)
    table = profiler.key_averages().table(sort_by='self_device_time_total', row_limit=25)
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, f'{workload}_compact_profile.txt'), 'w') as handle:
        handle.write(f'{B} envs, {steps - steps // 2} step_host(observations="compact") calls\n' + table)
    print(table)


def measure(workload, B, steps, window):
    import torch

    import bench
    from free_range_zoo_b200 import presets
    spec = bench.WORKLOADS[workload]
    module = importlib.import_module(f'free_range_zoo_b200.envs.{spec["domain"]}_v0')
    # (max_steps = 100 > the rollout: no environment is truncated, and rideshare's entry-step bound stays narrow)
    env = module.parallel_env(parallel_envs=B, max_steps=100, device=torch.device('cuda', 0),
                              configuration=getattr(presets, spec['preset'])(**spec.get('preset_kwargs', {})),
                              **spec['kwargs'])
    raw = env.unwrapped
    A = len(raw.agents)
    actions = torch.empty((steps, B, A, 2), dtype=torch.int32).pin_memory()
    env.reset(seed=bench.SEED)
    for t in range(steps):
        raw.sample_actions(bench.SAMPLER)
        actions[t].copy_(raw._actions)
        raw.step_all()
    torch.cuda.synchronize()
    up = actions[0].numel() * actions.element_size()
    rows = []
    for leg, mode in (('no_observations', False), ('observations', True), ('compact', 'compact'),
                      ('compact_copy_engine', 'copy_engine')):
        env.reset(seed=bench.SEED)
        times, moved, unpack = [], [], []
        for start in range(0, steps - window + 1, window):
            begin = time.perf_counter()
            for t in range(start, start + window):
                if mode == 'copy_engine':
                    result = raw.step_host(actions[t]) + (copy_engine_download(raw), )
                    mode_bytes = 'compact'
                else:
                    result = raw.step_host(actions[t], observations=mode)
                    mode_bytes = mode
                down = result[0].numel() * 4 + 2 * B
                if mode_bytes is True:
                    down += result[3]['bytes']
                elif mode_bytes == 'compact':
                    down += result[3].bytes
                moved.append(down)
            times.append((time.perf_counter() - begin) / window)
            if mode in ('compact', 'copy_engine'):
                begin = time.perf_counter()
                result[3].unpack()
                unpack.append(time.perf_counter() - begin)
        timed = sorted(times[1:])  # the first window is the warm-up (graph capture, first touches)
        per_step = timed[len(timed) // 2]
        row = dict(workload=workload, parallel_envs=B, leg=leg, env_steps_per_s=round(B / per_step, -4),
                   ms_per_step=round(1e3 * per_step, 4), h2d_bytes_per_step=up,
                   d2h_bytes_per_step=int(sum(moved[window:]) / len(moved[window:])), windows=len(timed),
                   window_steps=window, spread_ms=[round(1e3 * timed[0], 4), round(1e3 * timed[-1], 4)])
        if unpack:
            row['unpack_host_ms_per_step'] = round(1e3 * sorted(unpack)[len(unpack) // 2], 3)
        print(json.dumps(row), flush=True)
        rows.append(row)
    del env, raw, actions
    torch.cuda.empty_cache()
    return rows


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument('--out', default='')
    parser.add_argument('--steps', type=int, default=24)
    parser.add_argument('--window', type=int, default=4)
    parser.add_argument('--workloads', default=','.join(name for name, _ in WORKLOADS))
    parser.add_argument('--trace', default='', help='directory: write a torch.profiler table of the compact leg instead')
    args = parser.parse_args()
    if args.trace:
        trace('wildfire_c4', 65536, 12, args.trace)
        trace('wildfire_c1', 524288, 12, args.trace)
        return
    wanted = args.workloads.split(',')
    result = dict(gpu_description(), legs=[])
    for workload, B in WORKLOADS:
        if workload in wanted:
            result['legs'] += measure(workload, B, args.steps, args.window)
    if args.out:
        with open(args.out, 'w') as handle:
            json.dump(result, handle, indent=1)


if __name__ == '__main__':
    main()
