"""Compact observation download (frz_observe_compact, utils/compact.py) on the device: ``unpack()`` gives back exactly
the packed observations, through ``gather_observations(compact=True)`` and ``step_host(observations='compact')``."""
import importlib

import numpy as np
import pytest
import torch

from free_range_zoo_b200 import presets
from free_range_zoo_b200.utils import compact

pytestmark = pytest.mark.gpu

CYBER = dict(show_bad_actions=False, partially_observable=True)


def make(domain, config, B, max_steps, **kwargs):
    module = importlib.import_module(f'free_range_zoo_b200.envs.{domain}_v0')
    return module.parallel_env(parallel_envs=B, max_steps=max_steps, configuration=config,
                               device=torch.device('cuda:0'), **kwargs)


def explicit_packing(raw):
    """The packed observations built from the padded device arrays with the layout stated per array (masks are
    [B, agents, stride], task rows [B, capacity, columns]) -- correct for one-agent environments too."""
    B = raw.parallel_envs
    counts = raw.environment_task_count.cpu().numpy()
    offsets = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    dense, ragged = raw._observation_download()
    want = {name: tensor.cpu() for name, tensor in dense.items()}
    for name, (tensor, _) in ragged.items():
        host = tensor.cpu()
        blocks = host if name.endswith('mask') else host[:, None]
        pieces = [blocks[b, g, :counts[b]] for b in range(B) for g in range(blocks.shape[1])]
        want[name] = torch.cat(pieces)
    return counts, offsets, want


def assert_unpacks_to(observations, counts, offsets, want, where=''):
    got = observations.unpack()
    assert np.array_equal(got['counts'].numpy(), counts), where
    assert np.array_equal(got['offsets'].numpy(), offsets), where
    assert got['total'] == int(offsets[-1])
    assert set(got) == set(want) | {'counts', 'offsets', 'total', 'bytes'}
    for name, tensor in want.items():
        assert got[name].dtype == tensor.dtype and got[name].shape == tensor.shape, (name, where)
        assert torch.equal(got[name], tensor), (name, where)


def expected_bytes(observations):
    """Bytes of a download computed from the counts and the schema alone."""
    B, total = observations.counts.shape[0], int(observations.counts.to(torch.int64).sum())
    size = observations.counts.element_size() * B + 4 * (B + 1)
    for array in observations.schema.arrays:
        item = torch.empty(0, dtype=array.dtype).element_size()
        if array.kind == 'dense':
            size += B * array.rows * array.columns * item
        elif array.kind == 'rows':
            size += total * array.groups * array.columns * item
        else:
            size += int(compact.mask_offsets(observations.counts.numpy(), array.groups)[-1])
    return size


EQUALS_PACKED = [
    ('wildfire', presets.wildfire_large, {}),
    ('wildfire', presets.wildfire_3x3, dict(step_kernel='tiles')),
    ('wildfire', presets.wildfire_3x3, dict(step_kernel='groups')),
    ('wildfire', presets.wildfire_quirks, dict(step_kernel='tiles')),
    ('wildfire', presets.wildfire_quirks, dict(step_kernel='groups')),
    ('rideshare', presets.rideshare_c2, dict(step_kernel='tiles')),
    ('rideshare', presets.rideshare_c2, dict(step_kernel='groups')),
    ('rideshare', lambda: presets.rideshare_synthetic(drivers=20), {}),
    ('cybersecurity', presets.cyber_c3, CYBER),
    ('cybersecurity', presets.cyber_synthetic, CYBER),
]


@pytest.mark.parametrize('domain,preset,kwargs', EQUALS_PACKED,
                         ids=[f'{d}-{p.__name__}-{k.get("step_kernel", "auto")}' for d, p, k in EQUALS_PACKED])
def test_compact_unpacks_to_the_packed_observations(domain, preset, kwargs):
    """gather_observations(compact=True).unpack() == gather_observations(), bit for bit, through a rollout that
    empties, fills and terminates environments and runs past max_steps."""
    B, max_steps = 3000, 8
    env = make(domain, preset(), B, max_steps, **kwargs)
    env.reset(seed=21)
    raw = env.unwrapped
    for t in range(max_steps + 3):
        observations = raw.gather_observations(compact=True)
        packed = raw.gather_observations()
        got = observations.unpack()
        assert set(got) == set(packed)
        for name, tensor in packed.items():
            if name in ('total', 'bytes'):
                continue
            assert got[name].dtype == tensor.dtype and got[name].shape == tensor.shape, (name, t)
            assert torch.equal(got[name], tensor), (name, t)
        assert got['total'] == packed['total']
        assert observations.bytes == expected_bytes(observations) < packed['bytes']
        raw.sample_actions(3 + t)
        raw.step_all()
    raw.check_errors()


@pytest.mark.parametrize('domain,config,kwargs', [
    ('wildfire', lambda: presets.wildfire_large(num_agents=1), {}),
    ('rideshare', lambda: presets.rideshare_synthetic(drivers=1), {}),
    ('cybersecurity', lambda: presets.cyber_synthetic(attackers=1, defenders=1), CYBER),
], ids=['wildfire', 'rideshare', 'cybersecurity'])
def test_one_agent_environments(domain, config, kwargs):
    B = 2500
    env = make(domain, config(), B, 6, **kwargs)
    env.reset(seed=5)
    raw = env.unwrapped
    assert len(raw.agents) == (2 if domain == 'cybersecurity' else 1)  # (one attacker and one defender)
    for t in range(8):
        counts, offsets, want = explicit_packing(raw)
        assert_unpacks_to(raw.gather_observations(compact=True), counts, offsets, want, f'step {t}')
        raw.sample_actions(t)
        raw.step_all()


def device_arrays(raw):
    return {name: tensor for name, tensor in raw._bound.items()
            if tensor is not None and not name.startswith('init_') and name != 'control'}


def assert_same_device_state(raw, reference, where):
    B = raw.parallel_envs
    ours, theirs = device_arrays(raw), device_arrays(reference)
    for name in ours:
        if name == 'passengers':  # rows beyond the count are undefined
            K = raw._capacity
            valid = torch.arange(K, device='cuda')[None, :] < raw.environment_task_count[:, None]
            assert torch.equal(ours[name].view(B, K, -1)[valid], theirs[name].view(B, K, -1)[valid]), (name, where)
        else:
            assert torch.equal(ours[name], theirs[name]), (name, where)
    mine, other = raw.control_block(), reference.control_block()
    for field in ('seed', 'step', 'alive', 'agents_with_tasks', 'error_word'):
        assert mine[field] == other[field], (field, where)


PIPELINE = [
    ('wildfire', 'wildfire_large', {}, 5000, 3),
    ('wildfire', 'wildfire_large', {}, 3000, 1),
    ('wildfire', 'wildfire_3x3', {}, 4096, 4),
    ('wildfire', 'wildfire_large', {}, 30000, 3),
    ('rideshare', 'rideshare_c2', {}, 4100, 3),
    ('rideshare', 'rideshare_c2', {}, 2500, 2),
    ('cybersecurity', 'cyber_c3', CYBER, 6000, 5),
    ('cybersecurity', 'cyber_c3', CYBER, 70000, 16),
]


@pytest.mark.parametrize('dtype', [torch.int32, torch.int8], ids=['i32', 'i8'])
@pytest.mark.parametrize('domain,preset,kwargs,B,chunks', PIPELINE)
def test_compact_host_step_equals_device_step(domain, preset, kwargs, B, chunks, dtype):
    steps = 12
    device_env = make(domain, getattr(presets, preset)(), B, 10, **kwargs)
    host_env = make(domain, getattr(presets, preset)(), B, 10, **kwargs)
    device_env.reset(seed=11)
    host_env.reset(seed=11)
    reference, raw = device_env.unwrapped, host_env.unwrapped
    host_actions = torch.empty((B, len(raw.agents), 2), dtype=dtype).pin_memory()
    for t in range(steps):  # past max_steps
        reference.sample_actions(5)
        host_actions.copy_(reference._actions)
        torch.cuda.synchronize()
        reference.step_all()
        rewards, terminated, truncated, observations = host_env.step_host(host_actions, chunks, observations='compact')
        assert isinstance(observations, compact.CompactObservations)
        assert rewards.is_pinned() and observations.offsets.is_pinned()
        assert torch.equal(rewards, reference._rewards.cpu()), f'step {t}'
        assert torch.equal(terminated, reference.terminated.cpu()) and torch.equal(truncated, reference.truncated.cpu())
        assert_same_device_state(raw, reference, f'step {t}')
        counts, offsets, want = explicit_packing(reference)
        assert_unpacks_to(observations, counts, offsets, want, f'step {t}')
    raw.check_errors()


def test_switching_observation_modes_and_action_buffers():
    """False / True / 'compact' and two page-locked action buffers alternate on one environment: every result stays
    right.  (The compact download is enqueued after the pipelined step, outside its cached graph; this checks that the
    modes do not disturb each other or the graph's action-buffer patching.)"""
    B = 20000
    device_env, host_env = make('wildfire', presets.wildfire_large(), B, 30), make('wildfire', presets.wildfire_large(), B, 30)
    device_env.reset(seed=3)
    host_env.reset(seed=3)
    reference, raw = device_env.unwrapped, host_env.unwrapped
    buffers = [torch.empty((B, len(raw.agents), 2), dtype=torch.int32).pin_memory() for _ in range(2)]
    modes = [False, True, 'compact', 'compact', True, False, 'compact']
    for t, mode in enumerate(modes):
        reference.sample_actions(7)
        actions = buffers[t % 2]
        actions.copy_(reference._actions)
        torch.cuda.synchronize()
        reference.step_all()
        result = host_env.step_host(actions, 3, observations=mode)
        assert torch.equal(result[0], reference._rewards.cpu()), (t, mode)
        assert_same_device_state(raw, reference, (t, mode))
        counts, offsets, want = explicit_packing(reference)
        if mode == 'compact':
            assert_unpacks_to(result[3], counts, offsets, want, (t, mode))
        elif mode:
            for name, tensor in want.items():
                assert torch.equal(result[3][name].reshape(tensor.shape), tensor), (name, t)
        else:
            assert len(result) == 3
    with pytest.raises(ValueError, match="'compact'"):
        host_env.step_host(buffers[0], 3, observations='packed')


def test_compact_bytes_at_c4():
    """At C4 with 65 536 environments the compact download moves at most 0.3x the bytes of observations=True."""
    B = 65536
    env = make('wildfire', presets.wildfire_large(), B, 100)
    env.reset(seed=1)
    raw = env.unwrapped
    for t in range(3):
        raw.sample_actions(t)
        raw.step_all()
    observations = raw.gather_observations(compact=True)
    packed = raw.gather_observations()
    assert observations.bytes == expected_bytes(observations)
    assert observations.bytes <= 0.3 * packed['bytes'], (observations.bytes, packed['bytes'])
    assert observations['task_obs'].dtype == torch.int8 and observations.counts.dtype == torch.uint8


@pytest.mark.parametrize('domain,preset,kwargs', [('wildfire', presets.wildfire_large, {}),
                                                  ('rideshare', presets.rideshare_c2, {}),
                                                  ('cybersecurity', presets.cyber_c3, CYBER)])
def test_compact_download_leaves_the_device_state_unchanged(domain, preset, kwargs):
    B = 5000
    env = make(domain, preset(), B, 20, **kwargs)
    env.reset(seed=8)
    raw = env.unwrapped
    raw.sample_actions(1)
    raw.step_all()
    before = {name: tensor.clone() for name, tensor in raw._bound.items() if tensor is not None}
    control = raw.control_block()
    raw.gather_observations(compact=True)
    torch.cuda.synchronize()
    for name, tensor in before.items():
        assert torch.equal(raw._bound[name], tensor), name
    assert raw.control_block() == control


def test_a_fault_in_one_slice_reaches_check_errors_on_the_compact_path():
    B = 30000
    device_env, host_env = make('wildfire', presets.wildfire_large(), B, 20), make('wildfire', presets.wildfire_large(), B, 20)
    device_env.reset(seed=6)
    host_env.reset(seed=6)
    reference, raw = device_env.unwrapped, host_env.unwrapped
    reference.sample_actions(1)
    host_actions = torch.empty((B, len(raw.agents), 2), dtype=torch.int32).pin_memory()
    host_actions.copy_(reference._actions)
    torch.cuda.synchronize()
    host_actions[25000, 0] = torch.tensor([99, 0], dtype=torch.int32)  # inside the last of three slices
    reference._actions.copy_(host_actions)
    reference.step_all()
    rewards, _, _, observations = host_env.step_host(host_actions, 3, observations='compact')
    assert torch.equal(rewards, reference._rewards.cpu())
    counts, offsets, want = explicit_packing(reference)
    assert_unpacks_to(observations, counts, offsets, want)
    with pytest.raises(ValueError, match='not a valid index'):
        raw.check_errors()
    raw.check_errors()


def test_a_value_outside_the_configured_bound_is_reported():
    """An initial state from outside the configuration (a fire type the configuration does not have) cannot be
    narrowed: the download says so instead of returning wrapped values."""
    B = 64
    env = make('wildfire', presets.wildfire_large(), B, 10)
    env.reset(seed=0)
    raw = env.unwrapped
    state = raw.state().clone()
    state.fires[:] = 1000  # every cell lit with fire type 1000
    state.intensity[:] = 1
    env.reset(seed=0, options={'initial_state': state})
    with pytest.raises(ValueError, match='outside the bound'):
        raw.gather_observations(compact=True)
    packed = raw.gather_observations()  # the wide download still works
    assert int(packed['task_obs'][:, 2].max()) == 1000


def test_counts_beyond_the_capacity_are_clamped_and_reported():
    """A live-row count above the arrays' capacity (a corrupted count) must not move the packed offsets past the
    buffers: the scan and the encoders clamp alike and the download reports it."""
    B = 4096
    env = make('wildfire', presets.wildfire_large(), B, 10)
    env.reset(seed=0)
    raw = env.unwrapped
    raw.environment_task_count[[0, B - 1]] = 250  # capacity: 100 cells
    with pytest.raises(ValueError, match='outside the bound'):
        raw.gather_observations(compact=True)
    download = raw._compact
    assert int(download.offsets[B]) <= B * 100
    raw.environment_task_count[[0, B - 1]] = 0
    counts, offsets, want = explicit_packing(raw)
    assert_unpacks_to(raw.gather_observations(compact=True), counts, offsets, want)
