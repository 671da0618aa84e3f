"""Pipelined host-buffer step (frz_<domain>_step_host, include/frz.h) == the whole-batch device step, bit for bit.

Two engines with the same seed run the same rollout: one is stepped on the device (``step_all``), the other receives
the same actions from page-locked host memory through ``step_host`` with the batch cut into slices.  Every state
array, every published output and the control block must be identical; the host-side rewards / done flags must equal
the device's.
"""
import importlib

import numpy as np
import pytest
import torch

from free_range_zoo_b200 import presets

pytestmark = pytest.mark.gpu

CASES = [
    ('wildfire', 'wildfire_large', {}, 5000, 3),
    ('wildfire', 'wildfire_large', {}, 3000, 1),
    ('wildfire', 'wildfire_3x3', {}, 4096, 4),
    ('wildfire', 'wildfire_large', {}, 30000, 3),
    ('rideshare', 'rideshare_c2', {}, 4100, 3),
    ('rideshare', 'rideshare_c2', {}, 2500, 2),
    ('cybersecurity', 'cyber_c3', dict(show_bad_actions=False, partially_observable=True), 6000, 5),
    ('cybersecurity', 'cyber_c3', dict(show_bad_actions=False, partially_observable=True), 70000, 16),
]


def make(domain, preset, kwargs, B, max_steps):
    module = importlib.import_module(f'free_range_zoo_b200.envs.{domain}_v0')
    return module.parallel_env(parallel_envs=B, max_steps=max_steps, configuration=getattr(presets, preset)(),
                               device=torch.device('cuda:0'), **kwargs)


def device_arrays(raw):
    """Every tensor the step kernel reads or writes, by the name it has in the Frz*Buffers struct."""
    return {name: tensor for name, tensor in raw._bound.items()
            if tensor is not None and not name.startswith('init_') and name != 'control'}


@pytest.mark.parametrize('dtype', [torch.int32, torch.int16, torch.int8], ids=['i32', 'i16', 'i8'])
@pytest.mark.parametrize('domain,preset,kwargs,B,chunks', CASES)
def test_host_step_equals_device_step(domain, preset, kwargs, B, chunks, dtype):
    steps = 12
    device_env, host_env = make(domain, preset, kwargs, B, 10), make(domain, preset, kwargs, B, 10)
    device_env.reset(seed=11)
    host_env.reset(seed=11)
    reference, raw = device_env.unwrapped, host_env.unwrapped
    A = len(raw.agents)
    host_actions = torch.empty((B, A, 2), dtype=dtype).pin_memory()  # int16 pairs are widened on the device
    for t in range(steps):  # runs past max_steps: the "every environment is done" early-out is covered too
        reference.sample_actions(5)
        host_actions.copy_(reference._actions)
        torch.cuda.synchronize()
        reference.step_all()
        rewards, terminated, truncated = host_env.step_host(host_actions, chunks)
        assert rewards.is_pinned() and rewards.device.type == 'cpu'
        assert torch.equal(rewards, reference._rewards.cpu()), f'step {t}'
        assert torch.equal(terminated, reference.terminated.cpu()) and torch.equal(truncated, reference.truncated.cpu())
        ours, theirs = device_arrays(raw), device_arrays(reference)
        assert ours.keys() == theirs.keys()
        for name in ours:
            if domain == 'rideshare' and name == 'passengers':  # rows beyond the count are undefined
                K = raw._capacity
                valid = (torch.arange(K, device='cuda')[None, :] < raw.environment_task_count[:, None])
                assert torch.equal(ours[name].view(B, K, -1)[valid], theirs[name].view(B, K, -1)[valid]), (name, t)
            else:
                assert torch.equal(ours[name], theirs[name]), (name, t)
        mine, other = raw.control_block(), reference.control_block()
        for field in ('seed', 'step', 'alive', 'agents_with_tasks', 'error_word'):
            assert mine[field] == other[field], (field, t)
    assert reference.control_block()['step'] == 10  # two calls after the horizon were no-ops, on both engines
    raw.check_errors()


def test_host_step_mixes_with_device_steps_and_graphs():
    """The main control block stays authoritative: host steps, eager device steps and graph replays interleave."""
    B = 3072
    a, b = make('wildfire', 'wildfire_large', {}, B, 50), make('wildfire', 'wildfire_large', {}, B, 50)
    a.reset(seed=4)
    b.reset(seed=4)
    ra, rb = a.unwrapped, b.unwrapped
    host_actions = torch.empty((B, len(ra.agents), 2), dtype=torch.int32).pin_memory()
    for t in range(9):
        ra.sample_actions(9)
        ra.step_all()
        rb.sample_actions(9)
        if t % 3 == 1:
            host_actions.copy_(rb._actions)
            torch.cuda.synchronize()
            rb.step_host(host_actions, chunks=2)
        else:
            rb.step_all()
        assert torch.equal(ra.state().fires, rb.state().fires) and torch.equal(ra._rewards, rb._rewards), t
        assert torch.equal(ra._action_mask, rb._action_mask), t


def test_host_step_rejects_unpinned_or_misshaped_actions():
    env = make('cybersecurity', 'cyber_c3', {}, 64, 10)
    env.reset(seed=0)
    raw = env.unwrapped
    A = len(raw.agents)
    with pytest.raises(ValueError):
        raw.step_host(torch.zeros((64, A, 2), dtype=torch.int32))  # not page-locked
    with pytest.raises(ValueError):
        raw.step_host(torch.zeros((64, A), dtype=torch.int32).pin_memory())
    with pytest.raises(ValueError):
        raw.step_host(torch.zeros((64, A, 2), dtype=torch.int64).pin_memory())
    rewards, terminated, truncated = env.step_host(torch.full((64, A, 2), -1, dtype=torch.int32).pin_memory())
    assert rewards.shape == (64, A) and terminated.shape == (64, ) and not np.asarray(truncated).any()


def test_two_environments_keep_their_own_pipeline_events():
    """Each environment owns a FrzHostPipeline handle: host steps of two environments interleave without sharing events."""
    a, b = make('wildfire', 'wildfire_large', {}, 26000, 50), make('wildfire', 'wildfire_large', {}, 26000, 50)
    a.reset(seed=1)
    b.reset(seed=1)
    ra, rb = a.unwrapped, b.unwrapped
    actions = torch.empty((26000, 10, 2), dtype=torch.int32).pin_memory()
    for _ in range(4):
        ra.sample_actions(3)
        actions.copy_(ra._actions)
        torch.cuda.synchronize()
        first = [t.clone() for t in ra.step_host(actions, 3)]
        second = rb.step_host(actions, 2)
        for x, y in zip(first, second):
            assert torch.equal(x, y)
    assert ra._host_events.value != rb._host_events.value
    assert torch.equal(ra.state().fires, rb.state().fires)


@pytest.mark.parametrize('domain,preset,kwargs,chunks', [
    pytest.param('wildfire', 'wildfire_large', {}, None, id='wildfire-wildfire_large-kwargs0'),
    pytest.param('cybersecurity', 'cyber_c3', dict(show_bad_actions=False, partially_observable=True), None,
                 id='cybersecurity-cyber_c3-kwargs1'),
    pytest.param('rideshare', 'rideshare_c2', {}, None, id='rideshare-rideshare_c2'),
    pytest.param('wildfire', 'wildfire_large', {}, 3, id='wildfire-wildfire_large-step_host'),
    pytest.param('rideshare', 'rideshare_c2', {}, 3, id='rideshare-rideshare_c2-step_host'),
])
def test_generator_state_restores_a_checkpoint(domain, preset, kwargs, chunks):
    """generator_state_dict / load_generator_state_dict (reference: RandomGenerator.state_dict / load_state_dict,
    utils/random_generator.py:148-176): state tensors + (seed, step) continue a rollout bit for bit, through the
    device step or (``chunks``) the pipelined host step."""
    B = 700
    env = make(domain, preset, kwargs, B, 100)
    env.reset(seed=77)
    raw = env.unwrapped
    for _ in range(6):
        raw.sample_actions(8)
        raw.step_all()
    checkpoint = {name: tensor.clone() for name, tensor in device_arrays(raw).items()}
    generator = raw.generator_state_dict()
    assert generator['seed'] == 77 and generator['step'] == 6
    for _ in range(5):
        raw.sample_actions(8)
        raw.step_all()
    want = {name: tensor.clone() for name, tensor in device_arrays(raw).items()}

    other = make(domain, preset, kwargs, B, 100)
    other.reset(seed=123)  # a different stream, then the checkpoint is loaded over it
    restored = other.unwrapped
    for name, tensor in checkpoint.items():
        restored._bound[name].copy_(tensor)
    restored.load_generator_state_dict(generator)
    host_actions = torch.empty((B, len(restored.agents), 2), dtype=torch.int32).pin_memory()
    for _ in range(5):
        restored.sample_actions(8)
        if chunks is None:
            restored.step_all()
        else:
            host_actions.copy_(restored._actions)
            torch.cuda.synchronize()
            restored.step_host(host_actions, chunks)
    for name, tensor in want.items():
        if domain == 'rideshare' and name == 'passengers':  # rows beyond the count are undefined
            valid = torch.arange(restored._capacity, device='cuda')[None, :] < restored.environment_task_count[:, None]
            assert torch.equal(restored._bound[name][valid], tensor[valid]), name
        else:
            assert torch.equal(restored._bound[name], tensor), name


def test_capture_graph_does_not_advance_the_environment():
    env = make('wildfire', 'wildfire_3x3', {}, 1500, 100)
    env.reset(seed=5)
    raw = env.unwrapped
    for _ in range(3):
        raw.sample_actions(2)
        raw.step_all()
    before = {name: tensor.clone() for name, tensor in raw._bound.items() if tensor is not None}
    raw.capture_graph(sample=True, sampler_seed=2, steps=2)
    for name, tensor in before.items():
        assert torch.equal(raw._bound[name], tensor), name
    twin = make('wildfire', 'wildfire_3x3', {}, 1500, 100)
    twin.reset(seed=5)
    for _ in range(5):
        twin.unwrapped.sample_actions(2)
        twin.unwrapped.step_all()
    raw.replay()  # two more steps
    torch.cuda.synchronize()
    assert torch.equal(raw.state().fires, twin.unwrapped.state().fires)
    assert torch.equal(raw._cumulative, twin.unwrapped._cumulative)


def expected_packing(raw):
    """The packed observation download rebuilt with plain torch indexing from the padded device arrays."""
    B = raw.parallel_envs
    counts = raw.environment_task_count.cpu().numpy()
    offsets = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    dense, ragged = raw._observation_download()
    want = {name: tensor.cpu() for name, tensor in dense.items()}
    for name, (tensor, groups) in ragged.items():
        host = tensor.cpu()
        pieces = []
        for b in range(B):
            blocks = host[b] if groups > 1 else host[b][None]
            for g in range(groups):
                pieces.append(blocks[g][:counts[b]])
        want[name] = torch.cat(pieces) if pieces else host.new_zeros((0, ) + tuple(host.shape[2:]))
    return counts, offsets, want


@pytest.mark.parametrize('domain,preset,kwargs,B', [
    ('wildfire', 'wildfire_large', {}, 1500),
    ('wildfire', 'wildfire_3x3', {}, 2049),
    ('rideshare', 'rideshare_c2', {}, 1300),
    ('cybersecurity', 'cyber_c3', dict(show_bad_actions=False, partially_observable=True), 3000),
])
def test_gather_observations_packs_the_live_rows(domain, preset, kwargs, B):
    """frz_gather_live_rows: counts, offsets, dense arrays and packed live rows in host memory == the padded device
    arrays, bit for bit, at several points of a rollout (ragged, empty and full environments included)."""
    env = make(domain, preset, kwargs, B, 50)
    env.reset(seed=4)
    raw = env.unwrapped
    for t in range(10):
        raw.sample_actions(9)
        raw.step_all()
        if t % 3:
            continue
        got = raw.gather_observations()
        counts, offsets, want = expected_packing(raw)
        assert np.array_equal(got['counts'].numpy(), counts) and np.array_equal(got['offsets'].numpy(), offsets)
        assert got['total'] == int(offsets[-1])
        moved = got['counts'].numel() * 4 + got['offsets'].numel() * 4
        for name, tensor in want.items():
            assert got[name].is_pinned()
            assert torch.equal(got[name].reshape(tensor.shape), tensor), (name, t)
            moved += tensor.numel() * tensor.element_size()
        assert got['bytes'] == moved  # exactly the live bytes crossed the link


def test_step_host_returns_the_next_observations():
    """step_host(observations=True): the fourth element is the packed observation download of the stepped state."""
    B = 4100
    device_env, host_env = make('wildfire', 'wildfire_large', {}, B, 20), make('wildfire', 'wildfire_large', {}, B, 20)
    device_env.reset(seed=2)
    host_env.reset(seed=2)
    reference, raw = device_env.unwrapped, host_env.unwrapped
    host_actions = torch.empty((B, len(raw.agents), 2), dtype=torch.int32).pin_memory()
    for t in range(6):
        reference.sample_actions(3)
        host_actions.copy_(reference._actions)
        torch.cuda.synchronize()
        reference.step_all()
        rewards, terminated, truncated, observations = host_env.step_host(host_actions, 3, observations=True)
        assert torch.equal(rewards, reference._rewards.cpu())
        counts, offsets, want = expected_packing(reference)
        assert np.array_equal(observations['counts'].numpy(), counts)
        assert np.array_equal(observations['offsets'].numpy(), offsets)
        for name, tensor in want.items():
            assert torch.equal(observations[name].reshape(tensor.shape), tensor), (name, t)


def test_a_fault_in_one_slice_reaches_check_errors():
    """An invalid task index submitted through step_host in ONE slice of the batch: the slice's control block records
    the fault, the merge folds it into the environment's block, check_errors raises (and clears it) -- and the other
    environments stepped normally."""
    B = 30000
    device_env, host_env = make('wildfire', 'wildfire_large', {}, B, 20), make('wildfire', 'wildfire_large', {}, B, 20)
    device_env.reset(seed=6)
    host_env.reset(seed=6)
    reference, raw = device_env.unwrapped, host_env.unwrapped
    reference.sample_actions(1)
    host_actions = torch.empty((B, len(raw.agents), 2), dtype=torch.int32).pin_memory()
    host_actions.copy_(reference._actions)
    torch.cuda.synchronize()
    bad_env = 25000  # inside the last of three slices
    host_actions[bad_env, 0] = torch.tensor([99, 0], dtype=torch.int32)  # fight task 99 of a 10x10 grid with ~15 fires
    reference._actions.copy_(host_actions)
    reference.step_all()
    rewards, _, _ = host_env.step_host(host_actions, 3)
    assert torch.equal(rewards, reference._rewards.cpu())  # identical to the device step, faulty environment included
    with pytest.raises(ValueError, match='not a valid index'):
        raw.check_errors()
    raw.check_errors()  # cleared
    with pytest.raises(ValueError, match='not a valid index'):
        reference.check_errors()
