"""Benchmark of the fused environment-step path (BASELINE.json metric: env-steps/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload wildfire_c4] [--impl engine|reference]

A "step" is one environment step of ALL ``parallel_envs`` environments with random legal actions.  At N=1 the default
workload is BASELINE.json configs[3] -- wildfire 10x10 / 10 agents, agent+task+frame openness, parallel_envs=65,536 --
the configuration the headline target (>= 50x the host-CPU path, >= 60 % of HBM roofline) is quoted on.  For N>1
(launched by ``python -m torch.distributed.run``) every rank steps its own shard of ``parallel_envs`` environments (weak
scaling, no step-path collective; the global env index keys the RNG so trajectories do not depend on N); NCCL is used
only for the barrier, the max-over-ranks timing and the episode-statistics all-reduce.

One JSON line is printed by rank 0:
  value            whole-job env-steps/s, inputs resident in HBM, [sample_actions -> step] captured in a CUDA graph.  The
                   window "reset, W warm-up steps, K timed steps (barrier + synchronize on both sides, CUDA events, max
                   over ranks)" is repeated ``--windows`` times on the same seeded rollout; ``value`` is the MEDIAN
                   window, every window is listed in ``windows_ms``
  roofline         the step kernel alone: algorithmic bytes per launch (DESIGN.md section 3) / CUDA-event duration of the
                   launch, against the measured HBM copy bandwidth of MEASURED_PEAKS.json
  e2e              the same metric through the public Parallel API with HOST buffers (``parallel_env.step_host``):
                   page-locked int32 actions H2D + step + rewards / dones D2H + stream sync, every step; upload, kernel
                   and download are pipelined over slices of the batch inside frz_<domain>_step_host
  e2e_i16_actions  the same call with the opt-in int16 action format (half the upload); e2e_i8_actions: int8 (a quarter)
  e2e_full_obs     the same call returning the observations as well (self observations, task counts, the live task rows
                   and action-mask rows, compacted on the device): what a CPU policy needs per step
  cpu_baseline     the UNMODIFIED reference (oracle/_ref, stepped through oracle/ref_driver.py) on all host cores on a
                   bounded sample of the workload, with the numpy oracle port's number beside it
  config.other_workloads   the other named configurations (C1, C2, C3) at their named batch size and at a saturating
                   one: device-resident value, step-kernel time, roofline fraction, end-to-end value (N=1 only)
``--impl reference`` times the reference's own CPU implementation of the path on all host cores, on the same config and
step counts, and prints the same line shape (rank 0 only under torchrun).

``--dump-outputs DIR`` writes what the last timed step of the device-resident path left in the engine's per-environment
buffers (state, actions, rewards, dones, observations, masks) as ``DIR/<name>.npy``, at most 64 MB in all whatever N
(a fixed seeded sample of the environments of every rank, ``DIR/env_index.npy``), so that two builds can be compared
output for output: the inputs are seeded, so they are the same on every run.  ``--steps`` is the number of timed steps
of every GPU leg and of ``--impl reference``; only ``cpu_baseline`` times a bounded sample of its own.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# name: domain, preset, parallel_envs per GPU, env kwargs, a batch size that saturates the GPU (C5 sweep)
WORKLOADS = {
    'wildfire_c4': dict(domain='wildfire', preset='wildfire_large', envs=65536, kwargs={}, saturating=262144),
    'wildfire_c1': dict(domain='wildfire', preset='wildfire_3x3', envs=1024, kwargs={}, saturating=524288),
    'rideshare_c2': dict(domain='rideshare', preset='rideshare_c2', envs=16384, kwargs={}, saturating=524288),
    # the two rideshare step kernels at any batch size (kernel tuning: the dispatcher picks by batch size otherwise)
    'rideshare_c2_tiles': dict(domain='rideshare', preset='rideshare_c2', envs=16384, kwargs={}, engine_kwargs=dict(step_kernel='tiles')),
    'rideshare_c2_groups': dict(domain='rideshare', preset='rideshare_c2', envs=16384, kwargs={}, engine_kwargs=dict(step_kernel='groups')),
    # extra wildfire geometries (kernel tuning; not named by BASELINE.json)
    'wildfire_5x6': dict(domain='wildfire', preset='wildfire_large', envs=262144, kwargs={},
                         preset_kwargs=dict(height=5, width=6, num_agents=6, seed=21)),
    'wildfire_7x8': dict(domain='wildfire', preset='wildfire_large', envs=262144, kwargs={},
                         preset_kwargs=dict(height=7, width=8, num_agents=5, seed=5)),
    'cyber_c3': dict(domain='cybersecurity', preset='cyber_c3', envs=16384,
                     kwargs=dict(show_bad_actions=False, partially_observable=True), saturating=4194304),
}
KERNELS = {'wildfire': 'wildfire_step_kernel', 'rideshare': 'rideshare_tile_kernel / rideshare_step_kernel (by batch size)',
           'cybersecurity': 'cyber_step_tiled_kernel'}
SEED, SAMPLER = 2026, 2026
DUMP_ENVS, DUMP_BYTES = 4096, 64 << 20  # --dump-outputs: at most this many sampled environments, this many bytes


def algorithmic_bytes(domain: str, raw, present: float = 0.0) -> float:
    """ALGORITHMIC bytes per env-step (SURVEY.md section 8d; restated in DESIGN.md section 3): every live tensor read
    once and written once in the reference's dtypes, outputs written once, padded int32 observations, u8 masks."""
    if domain == 'wildfire':
        HW, A = raw.max_y * raw.max_x, len(raw.agents)
        state = 12 * HW + 12 * A
        return 2 * state + 8 * A + 4 * A + 2 * A + 16 + 16 * A + 16 * HW + 4 + A * HW + 4 * A
    if domain == 'cybersecurity':
        N, att, dfd = raw._n_nodes, raw._n_att, raw._n_def
        n = att + dfd
        state = 4 * N + 4 * dfd + n
        return 2 * state + 8 * n + 4 * n + 2 * n + 4 + (8 * att + 12 * dfd) + 8 * N + dfd + n
    A, K = len(raw.agents), raw._capacity  # `present` = measured mean passengers per environment over the timed steps
    return 2 * (8 * A + 44 * present) + 8 * A + 4 * A + 2 + 4 + 16 * A + 32 * present + A * K + 4 * (A + 1)


def measured_peak_gbs():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        return float(json.load(open(path))['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


def ncu_traffic(workload: str, parallel_envs: int):
    """dram__bytes_read.sum + dram__bytes_write.sum of one step-kernel launch, from the committed `ncu --set full`
    capture of this workload (profiles/traffic.json, written by profiles/summarize.py); None when there is none."""
    path = os.path.join(ROOT, 'profiles', 'traffic.json')
    if not os.path.exists(path):
        return None
    entry = json.load(open(path)).get(f'{workload}@{parallel_envs}')
    return None if entry is None else entry['dram_bytes_per_launch']


class ClockSampler:
    """Samples SM clocks / throttle reasons of one GPU through NVML: from a thread of this process every 50 ms (no
    process is forked, nothing is launched on the GPU) and, through ``mark()``, right before and after every timed
    window -- the windows last a few milliseconds, so the boundary samples are what reliably brackets them."""

    def __init__(self, index: int, period: float = 0.05):
        self.index, self.period, self.samples, self._stop, self._thread = index, period, [], threading.Event(), None
        self.handle = self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get('CUDA_VISIBLE_DEVICES')
            if visible and all(part.strip().isdigit() for part in visible.split(',')):
                index = int(visible.split(',')[index])
            self.nvml, self.handle = pynvml, pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception as error:  # pragma: no cover - depends on the driver
            self.error = repr(error)

    def _sample(self):
        n = self.nvml
        clock = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
        reasons = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)) if hasattr(
            n, 'nvmlDeviceGetCurrentClocksEventReasons') else int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
        try:
            power = n.nvmlDeviceGetPowerUsage(self.handle) / 1e3
        except Exception:
            power = 0.0
        self.samples.append((clock, reasons, power))

    def mark(self):
        if self.handle is not None:
            try:
                self._sample()
            except Exception:
                pass

    def _run(self):
        while not self._stop.is_set():
            try:
                self._sample()
            except Exception:
                pass
            self._stop.wait(self.period)

    def __enter__(self):
        if self.handle is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()

    def summary(self):
        if not self.samples:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable: ' + getattr(self, 'error', 'no samples')]}
        n = self.nvml
        busy = sorted(clock for clock, _, power in self.samples)
        names = {'hw_slowdown': getattr(n, 'nvmlClocksThrottleReasonHwSlowdown', 0x8),
                 'hw_thermal_slowdown': getattr(n, 'nvmlClocksThrottleReasonHwThermalSlowdown', 0x40),
                 'sw_thermal_slowdown': getattr(n, 'nvmlClocksThrottleReasonSwThermalSlowdown', 0x20),
                 'sw_power_cap': getattr(n, 'nvmlClocksThrottleReasonSwPowerCap', 0x4)}
        seen = 0
        for _, reasons, _ in self.samples:
            seen |= reasons
        return {'sm_mhz': busy[len(busy) // 2], 'sm_max_mhz': self.max_mhz, 'samples': len(busy), 'source': 'NVML',
                'window': 'every timed region of the run (graph windows, kernel timing, end-to-end legs)',
                'power_w_max': max(power for _, _, power in self.samples),
                'reasons': sorted(name for name, bit in names.items() if seen & bit)}


def pin_to_local_cores(local_rank: int, world: int):
    """One disjoint set of host cores per rank (the ranks of one node otherwise migrate over each other's cores and
    caches while they feed their GPUs); page-locked buffers are allocated afterwards so they are first touched there."""
    try:
        cores = sorted(os.sched_getaffinity(0))
        if world <= 1 or len(cores) < 2 * world:
            return None
        share = len(cores) // world
        mine = cores[local_rank * share:(local_rank + 1) * share]
        os.sched_setaffinity(0, mine)
        return [mine[0], mine[-1]]
    except (AttributeError, OSError):
        return None


# ------------------------------------------------------------------------------------------------ CPU arms


def _oracle_rollout(job):
    """Worker: steps one batch of the numpy oracle port and returns (env-steps executed, seconds inside ``step``);
    action sampling and the generation of the injected uniforms are excluded (SURVEY.md section 8d)."""
    workload, envs, steps, seed = job
    import numpy as np

    from free_range_zoo_b200 import presets
    spec = WORKLOADS[workload]
    config = getattr(presets, spec['preset'])(**spec.get('preset_kwargs', {}))
    rng = np.random.default_rng(seed)
    if spec['domain'] == 'wildfire':
        from oracle.wildfire import WildfireOracle
        oracle = WildfireOracle(config, envs, 1 << 30, **spec['kwargs'])
        oracle.reset()
        H, W, A = oracle.H, oracle.W, oracle.A

        def one_step():
            counts = oracle.agent_task_count
            k = np.minimum((rng.random(counts.shape) * (counts + 1)).astype(np.int64), counts)
            actions = np.stack([k, np.where(k == counts, -1, 0)], axis=2).astype(np.int32)
            uniforms = (rng.random((3, envs, H, W), dtype=np.float32), rng.random((5, envs, A), dtype=np.float32))
            start = time.perf_counter()
            oracle.step(actions, *uniforms)
            return time.perf_counter() - start
    elif spec['domain'] == 'cybersecurity':
        from oracle.cybersecurity import CybersecurityOracle
        oracle = CybersecurityOracle(config, envs, 1 << 30, **spec['kwargs'])
        oracle.reset()

        def one_step():
            n = oracle.n_agents
            count = oracle.agent_task_count
            k = np.minimum((rng.random(count.shape) * (count + 1)).astype(np.int64), count)
            actions = np.stack([k, np.where(k == count, -1, 0)], axis=2).astype(np.int32)  # attack / move or noop
            uniforms = (rng.random((1, envs, oracle.N), dtype=np.float32), rng.random((1, envs, n), dtype=np.float32))
            start = time.perf_counter()
            oracle.step(actions, *uniforms)
            return time.perf_counter() - start
    else:
        from oracle.rideshare import RideshareOracle
        oracle = RideshareOracle(config, envs, 1 << 30)
        oracle.reset()

        def one_step():
            actions = np.zeros((envs, oracle.A, 2), np.int32)
            for b in range(envs):
                for a in range(oracle.A):
                    mine = oracle._task_list(b, a)
                    k = min(int(rng.random() * (len(mine) + 1)), len(mine))
                    actions[b, a] = (k, -1) if k == len(mine) else (k, oracle.tables[b][mine[k]][6])
            start = time.perf_counter()
            oracle.step(actions)
            return time.perf_counter() - start

    one_step()
    return envs * steps, sum(one_step() for _ in range(steps))


def _reference_rollout(job):
    """Worker: steps one batch of the UNMODIFIED reference environment (oracle/_ref under the import shim) on one
    core and returns (env-steps executed, seconds inside ``env.step``)."""
    workload, envs, steps, seed, warmup = job
    import torch
    torch.set_num_threads(1)
    from oracle.ref_driver import timed_rollout
    spec = WORKLOADS[workload]
    return timed_rollout(spec['domain'], spec['preset'], spec.get('preset_kwargs', {}), spec['kwargs'], envs, steps, seed,
                         warmup=warmup)


def _run_workers(worker, jobs, timeout: float = 900.0):
    """One forked process per job.  Only ever called BEFORE this process touches CUDA (a forked child of a process with
    a CUDA context dies when it collects the inherited CUDA objects, and a dead pool worker hangs ``map``); the
    timeout turns any other stall into an error instead of a hang."""
    import multiprocessing as mp
    if len(jobs) == 1:
        return [worker(jobs[0])]
    with mp.get_context('fork').Pool(len(jobs)) as pool:
        return pool.map_async(worker, jobs).get(timeout=timeout)


def cpu_throughput(kind: str, workload: str, processes: int, envs_per_process: int, steps: int, warmup: int = 1):
    """env-steps/s of a CPU implementation of the path: ``processes`` single-threaded workers, each stepping its own
    batch of environments; the slowest worker's time counts (all of them run concurrently)."""
    if kind == 'reference':
        results = _run_workers(_reference_rollout, [(workload, envs_per_process, steps, 100 + i, warmup)
                                                    for i in range(processes)])
    else:
        results = _run_workers(_oracle_rollout, [(workload, envs_per_process, steps, 100 + i) for i in range(processes)])
    executed = sum(count for count, _ in results)
    slowest = max(seconds for _, seconds in results)
    return executed / max(slowest, 1e-9), executed


def reference_available():
    try:
        from oracle import ref_shim
        return ref_shim.reference_root() is not None
    except Exception:
        return False


def cpu_sample_size(workload: str):
    """(envs per process, steps) of the bounded cpu_baseline sample: a few seconds of CPU work per core."""
    return {'wildfire': (1024, 5), 'cybersecurity': (4096, 10), 'rideshare': (1024, 10)}[WORKLOADS[workload]['domain']]


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on all host cores, on the engine arm's
    config (B environments in total, split over one single-threaded process per core) and step counts."""
    if int(os.environ.get('RANK', '0')) != 0:
        return
    spec = WORKLOADS[args.workload]
    cores = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    B = args.parallel_envs or spec['envs']
    K, W = args.steps, max(1, min(args.warmup, 2))
    envs_per_process = max(1, -(-B // cores))
    kind = 'reference' if reference_available() else 'port'
    start = time.perf_counter()
    if kind == 'reference':
        value, executed = cpu_throughput('reference', args.workload, cores, envs_per_process, K, warmup=W)
        source = ('UNMODIFIED reference (oracle/_ref/free_range_zoo, imported under oracle/ref_shim.py), '
                  f'{args.workload}_v0.parallel_env(device="cpu", single_seeding=True, buffer_size=0)')
    else:  # the copy of the reference did not travel: fall back to the numpy restatement and say so
        envs_per_process = min(envs_per_process, cpu_sample_size(args.workload)[0])
        value, executed = cpu_throughput('port', args.workload, cores, envs_per_process, K)
        source = f'numpy oracle port (oracle/{spec["domain"]}.py): oracle/_ref is absent'
    wall = time.perf_counter() - start
    total_envs = cores * envs_per_process
    sample = (f'{cores} single-threaded processes x {envs_per_process} envs = {total_envs} envs x {K} steps of '
              f'{args.workload} ({W} warm-up steps); {source}; env.step() only, action sampling excluded; the slowest '
              'process counts')
    line = {
        'impl': 'reference', 'metric': 'env-steps/sec', 'value': value, 'unit': 'env-steps/s', 'n_gpus': args.gpus,
        'steps': K, 'warmup': W, 'ms_per_step': 1e3 * total_envs / value, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'int32+f32', 'data': 'synthetic',
        'config': {'workload': args.workload, 'domain': spec['domain'], 'preset': spec['preset'],
                   'parallel_envs_per_gpu': B, 'parallel_envs_total': total_envs,
                   'note': 'throughput of one node\'s host cores on one GPU\'s share of the batch; for N > 1 GPUs the '
                           'engine arm steps N x this many environments, the host has the same cores'},
        'cpu_baseline': {'value': value, 'unit': 'env-steps/s', 'cores': cores, 'kind': kind, 'sample': sample},
        'e2e': {'value': value, 'unit': 'env-steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0, 'env_steps_executed': executed, 'wall_s': wall,
    }
    print(json.dumps(line))


def measure_cpu_baseline(workload: str):
    """The ``cpu_baseline`` object of the engine's line: the UNMODIFIED reference (oracle/_ref) on all host cores on a
    bounded sample of the workload, the numpy oracle port beside it (or alone when the reference copy is absent)."""
    domain = WORKLOADS[workload]['domain']
    host_cores = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    envs_per_process, cpu_steps = cpu_sample_size(workload)
    port_value, _ = cpu_throughput('port', workload, host_cores, min(envs_per_process, 1024), cpu_steps)
    if reference_available():
        cpu_value, _ = cpu_throughput('reference', workload, host_cores, envs_per_process, cpu_steps)
        return {'value': cpu_value, 'unit': 'env-steps/s', 'cores': host_cores, 'kind': 'reference',
                'sample': f'{host_cores} single-threaded processes x {envs_per_process} envs x {cpu_steps} steps of '
                          f'{workload}: the UNMODIFIED reference (oracle/_ref) on CPU, env.step() only, action '
                          'sampling excluded',
                'port_value': port_value,
                'port': f'numpy oracle port (oracle/{domain}.py), same processes x steps, step() only'}
    return {'value': port_value, 'unit': 'env-steps/s', 'cores': host_cores, 'kind': 'port',
            'sample': f'{host_cores} processes x {min(envs_per_process, 1024)} envs x {cpu_steps} steps of '
                      f'{workload}, numpy oracle port (oracle/{domain}.py); oracle/_ref is absent'}


# ------------------------------------------------------------------------------------------------ GPU arm


class Harness:
    """One workload on this rank's GPU: the measurements every reported number comes from."""

    def __init__(self, workload, B, device, rank, world, K, W):
        import importlib

        import torch
        import torch.distributed as dist

        from free_range_zoo_b200 import presets
        self.torch, self.dist = torch, dist
        self.workload, self.spec, self.B, self.device, self.rank, self.world, self.K, self.W = (
            workload, WORKLOADS[workload], B, device, rank, world, K, W)
        spec = self.spec
        config = getattr(presets, spec['preset'])(**spec.get('preset_kwargs', {}))
        module = importlib.import_module(f'free_range_zoo_b200.envs.{spec["domain"]}_v0')
        self.env = module.parallel_env(parallel_envs=B, max_steps=1 << 30, configuration=config, device=device,
                                       env_offset=rank * B, **spec['kwargs'], **spec.get('engine_kwargs', {}))
        self.raw = self.env.unwrapped
        self.agents = len(self.raw.agents)
        self.start = torch.cuda.Event(enable_timing=True)
        self.stop = torch.cuda.Event(enable_timing=True)
        self.clocks = None  # ClockSampler of the run (sampled at the boundaries of every timed window)

    def mark(self):
        if self.clocks is not None:
            self.clocks.mark()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.device)

    def max_over_ranks(self, ms: float) -> float:
        if self.world == 1:
            return ms
        t = self.torch.tensor([ms], device=self.device, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    # ---- (1) device-resident throughput: [sample_actions -> step] in a CUDA graph, several steps per graph launch
    def graph_windows(self, windows: int):
        K, W, raw = self.K, self.W, self.raw
        per_replay = max(d for d in (10, 5, 4, 3, 2, 1) if K % d == 0 and W % d == 0)
        self.env.reset(seed=SEED)
        raw.capture_graph(sample=True, sampler_seed=SAMPLER, steps=per_replay)
        times = []
        for _ in range(windows):
            self.env.reset(seed=SEED)
            for _ in range(W // per_replay):
                raw.replay()
            self.mark()
            self.barrier()
            self.start.record()
            for _ in range(K // per_replay):
                raw.replay()
            self.stop.record()
            self.barrier()
            self.mark()
            times.append(self.max_over_ranks(self.start.elapsed_time(self.stop)))
        return per_replay, times

    def restart(self):
        self.env.reset(seed=SEED)
        for _ in range(self.W):
            self.raw.sample_actions(SAMPLER)
            self.raw.step_environment()
        self.barrier()

    # ---- (2) the step kernel alone, CUDA events on the launching stream
    def kernel_times(self):
        """(eager ms per launch, in-graph ms per launch, mean live tasks per env over the window).  Eager: an event pair
        around each frz_<domain>_step launch.  In graph: R x [sample, step] captured in one CUDA graph minus
        R x [sample] -- back-to-back kernels, no host in between; the roofline fraction uses this one.  Every measurement
        covers the same window of the same seeded rollout (the cost of a step follows the number of live tasks)."""
        torch, K, raw = self.torch, self.K, self.raw
        pairs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
        self.restart()
        tasks_seen = torch.zeros((), dtype=torch.float64, device=self.device)
        for before, after in pairs:
            raw.sample_actions(SAMPLER)
            before.record()
            raw.step_environment()
            after.record()
            tasks_seen += raw.environment_task_count.sum()
        self.barrier()
        eager_ms = sum(b.elapsed_time(a) for b, a in pairs) / K
        mean_tasks = float(tasks_seen.item()) / (K * self.B)
        raw.check_errors()

        def in_graph_ms(with_step: bool) -> float:
            repeats = max(d for d in (10, 5, 4, 3, 2, 1) if K % d == 0)
            torch.cuda.synchronize(self.device)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                for _ in range(repeats):
                    raw.sample_actions(SAMPLER)
                    if with_step:
                        raw.step_environment()
            graph.replay()  # first replay uploads the graph
            self.restart()
            self.start.record()
            for _ in range(K // repeats):
                graph.replay()
            self.stop.record()
            torch.cuda.synchronize(self.device)
            return self.start.elapsed_time(self.stop) / K

        kernel_ms = max(in_graph_ms(True) - in_graph_ms(False), 1e-6)
        raw.check_errors()
        return eager_ms, kernel_ms, mean_tasks

    # ---- (3) end to end through the public Parallel API with host buffers
    def record_actions(self, steps: int):
        """Legal actions for every step of the seeded rollout, recorded from a dry run (the engine is deterministic, so
        they stay legal on replay); page-locked int32 [steps, B, A, 2]."""
        torch, raw = self.torch, self.raw
        recorded = torch.empty((steps, self.B, self.agents, 2), dtype=torch.int32).pin_memory()
        self.env.reset(seed=SEED)
        for t in range(steps):
            raw.sample_actions(SAMPLER)
            recorded[t].copy_(raw._actions, non_blocking=True)
            raw.step_all()
        torch.cuda.synchronize(self.device)
        return recorded

    def host_leg(self, recorded, chunks=None, observations: bool = False, repeats: int = 3):
        """K timed ``step_host`` calls (after W untimed ones) on the recorded actions, the window repeated ``repeats``
        times on the same seeded rollout; returns the median ms per step (max over ranks) and the (H2D, D2H) bytes of one
        step, counted from the tensors that are copied."""
        K, W, raw = self.K, self.W, self.raw
        call = (lambda t: self.env.step_host(recorded[t], chunks, observations=True)) if observations else (
            lambda t: self.env.step_host(recorded[t], chunks))
        windows = []
        for _ in range(max(1, repeats)):
            self.env.reset(seed=SEED)
            for t in range(W):
                call(t)
            self.mark()
            self.barrier()
            d2h_extra = 0
            self.start.record()
            for t in range(W, W + K):
                out = call(t)
                if observations:
                    d2h_extra += out[3]['bytes']
            self.stop.record()
            self.barrier()
            self.mark()
            windows.append(self.max_over_ranks(self.start.elapsed_time(self.stop)) / K)
        ms = sorted(windows)[len(windows) // 2]
        state = raw._host_state
        h2d = recorded[0].numel() * recorded.element_size()
        d2h = state['rewards'].numel() * 4 + state['done'].numel() + d2h_extra // K
        # the host copies are the device's results (checked outside the timed region)
        assert self.torch.equal(state['rewards'], raw._rewards.cpu()) and self.torch.equal(state['done'][0],
                                                                                            raw._terminated.cpu())
        return ms, h2d, d2h, state['chunks']

    def host_wall_clock(self, steps: int, warmup: int):
        """End-to-end time per ``step_host`` call measured with the host's clock, for batches whose recorded rollout
        would not fit in page-locked memory: per step [untimed: sample on device, copy to the host buffer] [timed: the
        step_host call, which returns after the stream synchronised]."""
        torch, raw = self.torch, self.raw
        host_actions = torch.empty((self.B, self.agents, 2), dtype=torch.int32).pin_memory()
        self.env.reset(seed=SEED)
        seconds = 0.0
        for t in range(warmup + steps):
            raw.sample_actions(SAMPLER)
            host_actions.copy_(raw._actions)
            torch.cuda.synchronize(self.device)
            begin = time.perf_counter()
            self.env.step_host(host_actions)
            if t >= warmup:
                seconds += time.perf_counter() - begin
        return 1e3 * seconds / steps


def summarize_workload(name: str, B: int, device, K: int, W: int, e2e: str):
    """Compact record of one of the other named workloads (N=1): device-resident value, kernel time, roofline, e2e."""
    import torch
    h = Harness(name, B, device, 0, 1, K, W)
    per_replay, windows = h.graph_windows(3)
    graph_ms = sorted(windows)[len(windows) // 2]
    eager_ms, kernel_ms, mean_tasks = h.kernel_times()
    bytes_per_env = algorithmic_bytes(h.spec['domain'], h.raw, mean_tasks)
    peak, _ = measured_peak_gbs()
    record = {
        'parallel_envs': B, 'value': B * K / (graph_ms * 1e-3), 'ms_per_step': graph_ms / K,
        'steps_per_graph_launch': per_replay, 'kernel': KERNELS[h.spec['domain']], 'kernel_ms': kernel_ms,
        'kernel_ms_eager_launch': eager_ms, 'algorithmic_bytes_per_env_step': bytes_per_env,
        'roofline_frac': bytes_per_env * B / (kernel_ms * 1e-3) / 1e9 / peak, 'mean_tasks_per_env': mean_tasks,
        'working_set_mb': bytes_per_env * B / 1e6, 'traffic': ncu_traffic(name, B),
    }
    if e2e == 'events':
        ms, h2d, d2h, slices = h.host_leg(h.record_actions(W + K))
        record['e2e'] = {'value': B / (ms * 1e-3), 'ms_per_step': ms, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                         'slices': slices, 'timing': 'CUDA events around K step_host calls'}
    else:
        ms = h.host_wall_clock(K, W)
        record['e2e'] = {'value': B / (ms * 1e-3), 'ms_per_step': ms, 'timing': f'host clock per step_host call, {K} steps'}
    del h
    torch.cuda.empty_cache()
    return record


def dump_outputs(raw, B: int, directory: str, rank: int = 0, world: int = 1, dist=None):
    """Every per-environment buffer the step kernels write as ``<name>.npy``: float32, or float64 for 32- and 64-bit
    integers and doubles so that every value is exact.  The configuration tables bound next to them, the initial-state
    copies, the control block and injected uniforms are left out.  Rows are environments: all ``world * B`` of them, or a
    fixed seeded sample when that would exceed DUMP_ENVS environments or DUMP_BYTES in all; ``env_index.npy`` lists their
    global indices.  Rank r steps environments [r * B, (r + 1) * B); rank 0 gathers the rows and writes the files."""
    import numpy as np
    import torch
    skipped = {'control', 'cell_reward', 'cell_ignition', 'range_mask', 'cell_agents', 'schedule', 'schedule_index',
               'score_lut'}
    arrays = {name: tensor for name, tensor in raw._bound.items() if tensor is not None and name not in skipped
              and not name.startswith('init_') and not name.endswith('_uniforms')}
    wide = {name: tensor.element_size() >= 4 and (not tensor.is_floating_point() or tensor.dtype == torch.float64)
            for name, tensor in arrays.items()}
    env_bytes = 8 + sum(tensor[0].numel() * (8 if wide[name] else 4) for name, tensor in arrays.items())
    total = world * B
    count = min(total, DUMP_ENVS, DUMP_BYTES // env_bytes)
    index = np.arange(total) if count == total else np.sort(np.random.default_rng(SEED).choice(total, count, replace=False))
    mine = index[(index >= rank * B) & (index < (rank + 1) * B)] - rank * B
    rows = torch.from_numpy(mine).to(raw.device)
    values = {name: tensor.index_select(0, rows).cpu().numpy() for name, tensor in arrays.items()}
    if world > 1:
        shards = [None] * world if rank == 0 else None
        dist.gather_object(values, shards, dst=0)
        if rank != 0:
            return
        values = {name: np.concatenate([shard[name] for shard in shards]) for name in arrays}
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, 'env_index.npy'), index.astype(np.float64))
    for name, array in values.items():
        np.save(os.path.join(directory, f'{name}.npy'), array.astype(np.float64 if wide[name] else np.float32))


def run_engine(args):
    import torch
    import torch.distributed as dist

    from free_range_zoo_b200.distributed import all_reduce_statistics, episode_statistics

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    # the CPU arm runs first, while this process has no CUDA context yet (its workers are forked)
    cpu_baseline = measure_cpu_baseline(args.workload) if world == 1 else None
    cores = pin_to_local_cores(local_rank, world)
    torch.cuda.set_device(local_rank)
    device = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=device)

    spec = WORKLOADS[args.workload]
    domain = spec['domain']
    B = args.parallel_envs or spec['envs']
    K, W = args.steps, max(3, args.warmup)
    h = Harness(args.workload, B, device, rank, world, K, W)
    raw = h.raw

    clocks = ClockSampler(local_rank)
    clocks.__enter__()
    h.clocks = clocks
    per_replay, windows = h.graph_windows(max(1, args.windows))
    graph_ms = sorted(windows)[len(windows) // 2]
    value = world * B * K / (graph_ms * 1e-3)
    if args.dump_outputs:
        dump_outputs(raw, B, args.dump_outputs, rank, world, dist)

    eager_ms, kernel_ms, mean_tasks = h.kernel_times()
    bytes_per_env = algorithmic_bytes(domain, raw, mean_tasks)
    peak, peak_kind = measured_peak_gbs()
    achieved = bytes_per_env * B / (kernel_ms * 1e-3) / 1e9

    recorded = h.record_actions(W + K)
    e2e_ms, h2d, d2h, slices = h.host_leg(recorded, args.host_chunks or None)
    packed = recorded.to(torch.int16).pin_memory()
    i16_ms, i16_h2d, i16_d2h, _ = h.host_leg(packed, args.host_chunks or None)
    bytes_ok = int(recorded.max()) <= 127 and int(recorded.min()) >= -128
    if world > 1:  # every rank must take the same legs (their timings are reduced over the ranks)
        flag = torch.tensor([int(bytes_ok)], device=device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        bytes_ok = bool(flag.item())
    tiny = recorded.to(torch.int8).pin_memory() if bytes_ok else None
    if tiny is not None:
        i8_ms, i8_h2d, i8_d2h, _ = h.host_leg(tiny, args.host_chunks or None)
    full = None
    if hasattr(raw, 'gather_observations'):
        full_ms, full_h2d, full_d2h, _ = h.host_leg(recorded, args.host_chunks or None, observations=True)
        full = {'value': world * B / (full_ms * 1e-3), 'unit': 'env-steps/s', 'ms_per_step': full_ms,
                'h2d_bytes_per_step': full_h2d, 'd2h_bytes_per_step': full_d2h,
                'returns': 'rewards, done flags, self observations, task counts, live task rows and action-mask rows'}
    clocks.__exit__()

    # ---- episode statistics: the only collective, off the step path (SURVEY.md section 8e)
    stats = all_reduce_statistics(episode_statistics(raw._cumulative, raw.terminated, raw.truncated, raw.num_moves))

    if rank == 0:
        line = {
            'metric': 'env-steps/sec', 'value': value, 'unit': 'env-steps/s', 'n_gpus': world, 'steps': K, 'warmup': W,
            'ms_per_step': graph_ms / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'int32+f32', 'data': 'synthetic',
            'windows_ms': windows, 'windows_spread': (max(windows) - min(windows)) / graph_ms,
            'config': {
                'workload': args.workload, 'domain': domain, 'preset': spec['preset'], 'parallel_envs_per_gpu': B,
                'parallel_envs_total': world * B, 'agents': h.agents, 'agent_steps_per_s': value * h.agents,
                'actions': 'uniform random legal actions sampled on device (Philox), inside the timed region',
                'steps_per_graph_launch': per_replay,
                'window': f'reset, {W} warm-up steps, {K} timed steps; repeated {len(windows)}x on the same seeded '
                          'rollout, median reported',
                'l2': (f'state+outputs per step = {bytes_per_env * B / 1e6:.0f} MB > 126 MB L2 (inputs larger than L2)'
                       if bytes_per_env * B > 126e6 else
                       f'working set {bytes_per_env * B / 1e6:.1f} MB fits in L2: launch-latency-bound configuration'),
                'parallelism': f'dp{world} (env-batch sharding, no step-path collective)',
                'host_cores_of_rank0': cores,
            },
            'roofline': {
                'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                'traffic': ncu_traffic(args.workload, B),
                'traffic_source': 'ncu --set full capture committed under profiles/ (not re-measured by this run)',
                'peak_kind': peak_kind, 'kernel': KERNELS[domain],
                'kernel_ms': kernel_ms, 'kernel_ms_eager_launch': eager_ms,
                'algorithmic_bytes_per_launch': bytes_per_env * B, 'algorithmic_bytes_per_env_step': bytes_per_env,
                'mean_tasks_per_env': mean_tasks,
            },
            'e2e': {'value': world * B / (e2e_ms * 1e-3), 'unit': 'env-steps/s', 'h2d_bytes_per_step': h2d,
                    'd2h_bytes_per_step': d2h, 'ms_per_step': e2e_ms,
                    'api': 'parallel_env.step_host (frz_<domain>_step_host)', 'slices': slices,
                    'h2d_gbs_per_rank': h2d / (e2e_ms * 1e-3) / 1e9, 'd2h_gbs_per_rank': d2h / (e2e_ms * 1e-3) / 1e9},
            'e2e_i16_actions': {'value': world * B / (i16_ms * 1e-3), 'unit': 'env-steps/s', 'ms_per_step': i16_ms,
                                'h2d_bytes_per_step': i16_h2d, 'd2h_bytes_per_step': i16_d2h,
                                'api': 'parallel_env.step_host with int16 actions (FRZ_HOST_ACTIONS_I16)'},
            'gpu_launches': 2 * K,  # K x [sample kernel, step kernel] in the device-timed region
            'clocks': clocks.summary(),
            'stats': {'env_steps_executed': float(stats[0]), 'terminated_envs': float(stats[1]),
                      'truncated_envs': float(stats[2]), 'cumulative_reward_sum': float(stats[3:].sum())},
        }
        if tiny is not None:
            line['e2e_i8_actions'] = {'value': world * B / (i8_ms * 1e-3), 'unit': 'env-steps/s', 'ms_per_step': i8_ms,
                                      'h2d_bytes_per_step': i8_h2d, 'd2h_bytes_per_step': i8_d2h,
                                      'api': 'parallel_env.step_host with int8 actions (FRZ_HOST_ACTIONS_I8)'}
        if full is not None:
            line['e2e_full_obs'] = full
        del h, raw, recorded, packed, tiny
        torch.cuda.empty_cache()
        if world == 1:
            line['cpu_baseline'] = cpu_baseline
            if not args.skip_other_workloads:
                others = {}
                for name in ('wildfire_c1', 'rideshare_c2', 'cyber_c3', 'wildfire_c4'):
                    named, saturating = WORKLOADS[name]['envs'], WORKLOADS[name]['saturating']
                    if name != args.workload:
                        others[f'{name}@{named}'] = summarize_workload(name, named, device, K, W, 'events')
                    others[f'{name}@{saturating}'] = summarize_workload(name, saturating, device, K, W, 'host clock')
                line['config']['other_workloads'] = others
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument('--gpus', type=int, default=1)
    parser.add_argument('--steps', type=int, default=20)
    parser.add_argument('--warmup', type=int, default=5)
    parser.add_argument('--windows', type=int, default=7, help='repetitions of the timed K-step window (median reported)')
    parser.add_argument('--impl', default='engine', choices=['engine', 'reference'])
    parser.add_argument('--workload', default='wildfire_c4', choices=sorted(WORKLOADS))
    parser.add_argument('--parallel-envs', type=int, default=0, help='override parallel_envs per GPU')
    parser.add_argument('--host-chunks', type=int, default=0,
                        help='slices of the pipelined host-buffer step of the e2e leg (0 = the engine\'s default)')
    parser.add_argument('--skip-other-workloads', action='store_true',
                        help='only the named workload (skips config.other_workloads)')
    parser.add_argument('--dump-outputs', metavar='DIR',
                        help='write the outputs of the last timed step as DIR/<name>.npy (engine only)')
    args = parser.parse_args()
    if args.steps < 1:
        parser.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'engine':
        parser.error('--dump-outputs writes the engine\'s outputs; --impl reference has none to write')
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_engine(args)


if __name__ == '__main__':
    main()
