"""Cost of encoding observations into policy inputs on the device (``policy_inputs``, include/frz_inputs.h).

    python profiles/time_policy_inputs.py [--out r6_policy_inputs.json] [--reps 50]

Per workload and output type (f32, bf16):
  kernel     one frz_<domain>_policy_inputs launch, timed with CUDA events around each launch; before every launch a
             256 MB buffer is overwritten so that the observations come from HBM, not L2 (the 126 MB L2 would otherwise
             hold the smaller workloads' working sets)
  torch      the same encoding as torch ops: the restatement tests/test_policy_inputs_gpu.py checks the kernel against,
             over freshly built observation views (the ``others`` gathers and padded task rows), then the cast to the
             output type.  Timed the same way, with the same L2 flush.
Algorithmic bytes come from the shapes: the outputs, the self observations, the task counts (and cybersecurity's
monitored bytes) and the live task rows, at the mean live row count measured on the timed state.  The HBM peak is a
device-to-device copy of 2 GB measured in the same run.

Env-steps/s of a CUDA graph of 10 x [policy_inputs -> a fixed two-layer MLP -> sample_actions_from_logits -> step]
next to 10 x [sample_actions -> step], replayed back to back.
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from profiles.time_policy_actions import copy_peak_gbs, gpu_description, make, timed_launches  # noqa: E402

WORKLOADS = [('wildfire_c4', 'wildfire', 'wildfire_large', {}, 65536),
             ('wildfire_c1', 'wildfire', 'wildfire_3x3', {}, 524288),
             ('rideshare_c2', 'rideshare', 'rideshare_c2', {}, 524288),
             ('cyber_c3', 'cybersecurity', 'cyber_c3', dict(show_bad_actions=False, partially_observable=True), 524288)]
SEED, SAMPLER, GRAPH_STEPS, WARM_STEPS = 2026, 2026, 10, 3


def kernel_bytes(raw, domain, element):
    B = raw.parallel_envs
    shapes = raw.policy_input_shapes
    A, Fa = shapes['agent']
    V, T, Ft = shapes['tasks']
    outputs = B * (A * Fa + V * T * Ft) * element
    live = float(raw.environment_task_count.float().mean())
    if domain == 'cybersecurity':
        self_obs = raw._attacker_self.numel() * 4 + raw._defender_self.numel() * 4
        counts = B * 4 + raw._monitored.numel()
    else:
        self_obs = raw._self_obs.numel() * 4
        counts = B * 4
    rows = B * live * raw._task_obs.shape[2] * 4
    return dict(outputs=outputs, self_obs=self_obs, counts=counts, live_rows=rows, mean_live_rows=live,
                total=outputs + self_obs + counts + rows)


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

    from tests.test_policy_inputs_gpu import Policy, restate
    raw = make(domain, preset, kwargs, B)
    raw.reset(seed=SEED)
    for t in range(WARM_STEPS):  # a state some steps into the episode
        raw.sample_actions(SAMPLER + t)
        raw.step_all(None)
    flush = torch.zeros(1 << 26, dtype=torch.float32, device='cuda')  # 256 MB
    shapes = raw.policy_input_shapes
    row = dict(workload=name, parallel_envs=B, shapes=shapes, kernels={})

    def torch_encoding(dtype):
        views = raw._observation_views(raw._observation_buffers())
        agent, tasks = restate(raw, views=views)
        return agent.to(dtype), tasks.to(dtype)

    for dtype, element in ((torch.float32, 4), (torch.bfloat16, 2)):
        key = 'f32' if dtype == torch.float32 else 'bf16'
        got = [t.clone() for t in raw.policy_inputs(dtype)]
        want = torch_encoding(dtype)
        assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1]), f'{name} {key}: kernel != torch'
        kernel_us, kernel_all = timed_launches(torch, lambda: raw.policy_inputs(dtype), flush, reps)
        torch_us, torch_all = timed_launches(torch, lambda: torch_encoding(dtype), flush, max(5, reps // 5))
        bytes_ = kernel_bytes(raw, domain, element)
        row['kernels'][key] = dict(
            kernel_us=kernel_us, kernel_us_all=kernel_all, torch_us=torch_us, torch_us_all=torch_all,
            algorithmic_bytes=bytes_, kernel_gbs=bytes_['total'] / (kernel_us * 1e-6) / 1e9,
            roofline_us=bytes_['total'] / (peak * 1e9) * 1e6,
            fraction_of_copy_peak=bytes_['total'] / (kernel_us * 1e-6) / 1e9 / peak,
            speedup_over_torch=torch_us / kernel_us)
    policy = Policy(raw)

    def device_loop():
        agent, tasks = raw.policy_inputs()
        raw.sample_actions_from_logits(policy(agent, tasks), SAMPLER)

    row['graph_env_steps_per_s'] = dict(policy=graph_rate(torch, raw, device_loop),
                                        uniform=graph_rate(torch, raw, lambda: raw.sample_actions(SAMPLER)))
    del raw, flush, policy
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
        raise SystemExit('time_policy_inputs.py measures on a CUDA device; none is available')
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
