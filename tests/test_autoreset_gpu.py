"""Same-step autoreset (``autoreset=True``, include/frz_autoreset.h) against the explicit API and the CPU oracle.

The specification of a step with autoreset is ``step(); reset_batches(finished)`` on an ``autoreset=False`` engine,
whose every step and reset is checked against the oracle here (tests/test_lifecycle_gpu.py's rollouts): the autoreset
engine must return that engine's step outputs (rewards, done flags, infos) and then hold exactly its state,
observations, masks, counts and batch-wide flags after the reset -- bit for bit, from generated states in which
environments finish at different steps.
"""
import importlib

import numpy as np
import pytest
import torch

from free_range_zoo_b200 import distributed, presets
from tests.engine_util import cpu
from tests.test_cyber_gpu import legal_actions
from tests.test_lifecycle_gpu import (CYBER_PO, given, make, rideshare_actions, rideshare_state, setup, wildfire_actions,
                                      wildfire_config, wildfire_state, cyber_state)
from tests.test_philox_parity_gpu import WILDFIRE_GEOMETRIES

pytestmark = pytest.mark.gpu

BATCHES = [1, 31, 129, 2049]
INPUTS = ('actions', 'field_uniforms', 'agent_uniforms', 'network_uniforms', 'control')


def overwritten(raw):
    return set(type(raw)._autoreset_rows().overwritten)


def compare_published(auto, explicit, context):
    """Every array the engines publish or step from, and the control block, bit for bit -- except the step outputs
    that the explicit reset clears and the autoreset leaves as the finishing step wrote them."""
    skip = overwritten(auto) | set(INPUTS)
    for name, tensor in explicit._bound.items():
        if tensor is not None and name not in skip:
            assert torch.equal(auto._bound[name], tensor), f'{context}: {name}'
    a, e = auto.control_block(), explicit.control_block()
    for name in ('step', 'alive', 'agents_with_tasks', 'error_word'):
        assert a[name] == e[name], f'{context}: control.{name} {a[name]} != {e[name]}'
    assert a['alive'] == 3, f'{context}: a batch with autoreset is never idle'


def compare_step_outputs(auto, explicit, context):
    """What the step returned: rewards, done flags and infos of the finishing step, and the finished episodes."""
    assert torch.equal(auto._rewards, explicit._rewards), f'{context}: rewards'
    for name in overwritten(auto) - {'rewards'}:
        assert torch.equal(auto._bound[name], explicit._bound[name]), f'{context}: {name}'
    assert torch.equal(auto.terminated, explicit.terminated) and torch.equal(auto.truncated, explicit.truncated), context
    assert torch.equal(auto.finished, explicit.finished), context
    for agent in auto.agents:
        assert torch.equal(auto.terminations[agent], explicit.terminated), context
        assert torch.equal(auto.truncations[agent], explicit.truncated), context
    stats = auto.episode_statistics
    done = explicit.finished
    assert torch.equal(stats['done'], done) and torch.equal(stats['terminated'], explicit.terminated), context
    assert torch.equal(stats['truncated'], explicit.truncated), context
    assert torch.equal(stats['return'][done], explicit._cumulative[done]), f'{context}: episode return'
    assert torch.equal(stats['length'][done], explicit.num_moves[done]), f'{context}: episode length'


def autoreset_twin(domain, config, B, max_steps, kernel, offset, seed, kwargs, state):
    """An autoreset engine reset into the same initial state as the explicit run."""
    if domain == 'rideshare':
        raw = make(domain, config, B, max_steps, step_kernel=kernel, autoreset=True)
        agents, passengers = state
        raw.reset(seed=seed, options={'initial_state': given(agents=agents, passengers=passengers)})
        return raw
    extra = dict(step_kernel=kernel) if domain == 'wildfire' else {}
    raw = make(domain, config, B, max_steps, env_offset=offset, autoreset=True, **extra, **kwargs)
    raw.reset(seed=seed, options={'initial_state': given(**state)})
    return raw


def generated_state(domain, config, B, max_steps, rng, kwargs):
    """A generated initial state with environments that finish at once (wildfire: nothing lit; cybersecurity: nobody
    present) and, for wildfire, one fully lit environment."""
    if domain == 'wildfire':
        from oracle.wildfire import WildfireOracle
        dead, lit = ([0], [B - 1]) if B > 1 else ((), ())
        return wildfire_state(WildfireOracle(config, B, max_steps, **kwargs), rng, dead=dead, all_lit=lit)
    if domain == 'cybersecurity':
        from oracle.cybersecurity import CybersecurityOracle
        return cyber_state(CybersecurityOracle(config, B, max_steps, **kwargs), rng, absent=[0, B - 1])
    from oracle.rideshare import RideshareOracle
    return rideshare_state(RideshareOracle(config, B, max_steps), config, rng, max_steps + 10)


def run_against_explicit(domain, config, B, kernel='auto', philox=False, kwargs=None, max_steps=5, seed=0):
    kwargs = dict(kwargs or {})
    offset = 3 * B + 5 if philox else 0
    rng = np.random.default_rng(B + 17)
    state = generated_state(domain, config, B, max_steps, rng, kwargs)
    run = setup(domain, config, B, max_steps, rng, kernel=kernel, philox=philox, offset=offset, seed=seed, kwargs=kwargs,
                state=state)
    explicit, o = run.raw, run.oracle
    auto = autoreset_twin(domain, config, B, max_steps, kernel, offset, seed, kwargs, state)
    compare_published(auto, explicit, 'reset')
    actions_of = {'wildfire': wildfire_actions, 'cybersecurity': legal_actions, 'rideshare': rideshare_actions}[domain]
    for t in range(3 * max_steps):
        context = f'{domain} B={B} t={t}'
        if t == 2:  # stagger the horizons: a third of the environments start over here
            mask = np.arange(B) % 3 == 0
            o.reset_batches(mask)
            explicit.reset_batches(np.nonzero(mask)[0].tolist())
            auto.reset_batches(np.nonzero(mask)[0].tolist())
        actions = actions_of(o, run.rng)
        run.step(context, actions=actions)  # the oracle and the explicit engine, checked against each other
        if not philox and domain != 'rideshare':
            auto.inject_uniforms(*explicit._uniforms)
        auto.step_all(torch.from_numpy(actions).cuda())
        compare_step_outputs(auto, explicit, context)
        finished = o.terminated | o.truncated
        stats = auto.episode_statistics
        assert np.array_equal(cpu(stats['length'])[finished], o.num_moves[finished]), context
        assert np.allclose(cpu(stats['return'])[finished], o.cumulative_rewards[finished], rtol=1e-5, atol=1e-4), context
        o.reset_batches(finished)
        explicit.reset_batches(np.nonzero(finished)[0].tolist())
        run.check(f'{context} after reset_batches')
        compare_published(auto, explicit, context)
    auto.check_errors()
    return run, auto


WILDFIRE_CASES = [(spec, BATCHES[i % len(BATCHES)], kernel)
                  for i, (spec, _, geometry) in enumerate(WILDFIRE_GEOMETRIES)
                  for kernel in (['groups', 'tiles'] if geometry[0] == 8 else ['auto'])]


@pytest.mark.parametrize('spec,B,kernel', WILDFIRE_CASES, ids=lambda v: str(v).replace(' ', ''))
def test_wildfire_autoreset_matches_oracle_and_reset_batches(spec, B, kernel):
    run_against_explicit('wildfire', wildfire_config(spec), B, kernel=kernel,
                         kwargs=dict(show_bad_actions=B % 2 == 1 and B > 1))


@pytest.mark.parametrize('B', BATCHES)
@pytest.mark.parametrize('kernel', ['groups', 'tiles'])
def test_rideshare_autoreset_matches_oracle_and_reset_batches(kernel, B):
    run_against_explicit('rideshare', presets.rideshare_c2(), B, kernel=kernel, max_steps=5)


@pytest.mark.parametrize('preset,B,kwargs', [
    ('cyber_c3', 129, CYBER_PO),
    ('cyber_c3', 2049, dict(show_bad_actions=True, partially_observable=False)),
    (('cyber_synthetic', dict(nodes=20, attackers=9, defenders=9)), 31, dict(show_bad_actions=True)),
    (('cyber_synthetic', dict(nodes=32, attackers=16, defenders=16)), 1, dict(show_bad_actions=True)),  # direct kernel
])
def test_cyber_autoreset_matches_oracle_and_reset_batches(preset, B, kwargs):
    config = getattr(presets, preset)() if isinstance(preset, str) else getattr(presets, preset[0])(**preset[1])
    run_against_explicit('cybersecurity', config, B, kwargs=kwargs)


@pytest.mark.parametrize('domain,spec,B,kernel,kwargs', [
    ('wildfire', {}, 129, 'auto', {}),
    ('wildfire', 'wildfire_3x3', 2049, 'tiles', dict(show_bad_actions=True)),
    ('wildfire', 'wildfire_3x3', 31, 'groups', {}),
    ('cybersecurity', 'cyber_c3', 129, 'auto', CYBER_PO),
    ('cybersecurity', 'cyber_c3', 2049, 'auto', dict(show_bad_actions=True, partially_observable=False)),
])
def test_philox_autoreset_equals_reset_batches_with_an_env_offset(domain, spec, B, kernel, kwargs):
    config = wildfire_config(spec) if domain == 'wildfire' else getattr(presets, spec)()
    run_against_explicit(domain, config, B, kernel=kernel, philox=True, kwargs=kwargs, seed=(0xA7 << 36) | B)


def test_distributed_statistics_accept_the_episode_statistics():
    run, auto = run_against_explicit('wildfire', wildfire_config('wildfire_3x3'), 129, kernel='tiles', max_steps=3)
    stats = auto.episode_statistics
    whole = distributed.episode_statistics(stats['return'], stats['terminated'], stats['truncated'], stats['length'])
    assert whole.shape == (3 + len(auto.agents), )
    done = stats['done']
    record = distributed.episode_statistics(stats['return'][done], stats['terminated'][done], stats['truncated'][done],
                                            stats['length'][done])
    assert record[0].item() == stats['length'][done].sum().item()
    assert record[1].item() + record[2].item() >= done.sum().item()


# ------------------------------------------------------------------------------------------------ every stepping path


DOMAINS = {'wildfire': ('wildfire_large', {}), 'rideshare': ('rideshare_c2', {}), 'cybersecurity': ('cyber_c3', CYBER_PO)}


def fresh(domain, B, max_steps, **extra):
    preset, kwargs = DOMAINS[domain]
    module = importlib.import_module(f'free_range_zoo_b200.envs.{domain}_v0')
    env = module.parallel_env(parallel_envs=B, max_steps=max_steps, configuration=getattr(presets, preset)(),
                              device=torch.device('cuda:0'), env_offset=B, autoreset=True, **kwargs, **extra)
    env.reset(seed=23)
    return env


def same_trajectory(raw, reference, context):
    for name, tensor in reference._bound.items():
        if tensor is not None and name not in INPUTS:
            assert torch.equal(raw._bound[name], tensor), f'{context}: {name}'
    for name, tensor in reference.episode_statistics.items():
        assert torch.equal(raw.episode_statistics[name], tensor), f'{context}: episode_statistics[{name}]'
    assert raw.control_block() == reference.control_block(), context


def host_observations_equal(got, want, context):
    for name, value in want.items():
        if isinstance(value, torch.Tensor):
            assert torch.equal(got[name], value), f'{context}: observations[{name}]'


@pytest.mark.parametrize('domain', sorted(DOMAINS))
def test_every_stepping_path_gives_the_same_trajectory(domain):
    B, max_steps, steps = 3000, 4, 12
    reference_env = fresh(domain, B, max_steps)
    reference = reference_env.unwrapped
    paths = {name: fresh(domain, B, max_steps) for name in ('parallel', 'aec', 'host', 'graph')}
    paths['graph'].unwrapped.capture_graph(sample=True, sampler_seed=9, steps=3)
    A = len(reference.agents)
    host_i32 = torch.empty((B, A, 2), dtype=torch.int32).pin_memory()
    host_i8 = torch.empty((B, A, 2), dtype=torch.int8).pin_memory()
    finished_some = False
    for t in range(steps):
        context = f'{domain} t={t}'
        actions = reference.sample_actions(9).clone()
        reference.step_all()
        finished_some |= bool(reference.finished.any())
        # Parallel API with a dict of per-agent actions
        parallel = paths['parallel']
        _, rewards, terminations, truncations, _ = parallel.step({a: actions[:, i] for i, a in enumerate(reference.agents)})
        for i, agent in enumerate(reference.agents):
            assert torch.equal(rewards[agent], reference._rewards[:, i]), context
            assert torch.equal(terminations[agent], reference.terminated), context
            assert torch.equal(truncations[agent], reference.truncated), context
        same_trajectory(parallel.unwrapped, reference, f'{context} parallel')
        # AEC: one agent at a time, the last one advances the batch
        aec = paths['aec'].unwrapped
        for i in range(A):
            aec.step(actions[:, i])
        same_trajectory(aec, reference, f'{context} aec')
        # host buffers: int32 and int8 actions, every observation mode
        host = paths['host'].unwrapped
        buffer = host_i32 if t % 2 == 0 else host_i8
        buffer.copy_(actions)
        torch.cuda.synchronize()
        mode = (False, True, 'compact')[t % 3]
        results = host.step_host(buffer, chunks=3, observations=mode)
        assert torch.equal(results[0], reference._rewards.cpu()), context
        assert torch.equal(results[1], reference.terminated.cpu()) and torch.equal(results[2], reference.truncated.cpu())
        same_trajectory(host, reference, f'{context} host')
        if mode:
            got = results[3].unpack() if mode == 'compact' else results[3]
            host_observations_equal(got, reference.gather_observations(), f'{context} host {mode}')
        # graph replays: three sampled steps each
        if t % 3 == 2:
            graph = paths['graph'].unwrapped
            graph.replay()
            same_trajectory(graph, reference, f'{context} graph')
    assert finished_some, 'no environment finished: the paths never restarted one'


def test_a_reset_with_a_new_initial_state_retakes_the_snapshot():
    """After autoreset steps, ``reset(options={'initial_state': S2})``: later restarts go to S2."""
    from oracle.wildfire import WildfireOracle
    config, B, max_steps = presets.wildfire_large(), 64, 3
    rng = np.random.default_rng(5)
    probe = WildfireOracle(config, B, max_steps)
    first, second = wildfire_state(probe, rng), wildfire_state(probe, rng, all_lit=range(B))
    auto = make('wildfire', config, B, max_steps, autoreset=True, env_offset=B)
    explicit = make('wildfire', config, B, max_steps, env_offset=B)
    for env in (auto, explicit):
        env.reset(seed=4, options={'initial_state': given(**first)})
    for state, steps in ((first, 4), (second, 3 * max_steps)):
        if state is second:
            for env in (auto, explicit):
                env.reset(seed=4, options={'initial_state': given(**state)})
            compare_published(auto, explicit, 'second reset')
        for t in range(steps):
            for env in (auto, explicit):
                env.sample_actions(3)
                env.step_all()
            compare_step_outputs(auto, explicit, f't={t}')
            finished = explicit.finished.clone()
            explicit.reset_batches(finished.nonzero().flatten())
            compare_published(auto, explicit, f't={t}')
            if state is second and bool(finished.any()):
                fires = torch.from_numpy(second['fires']).cuda()
                restarted = finished & (auto.num_moves == 0)
                assert torch.equal(auto.state().fires[restarted], fires[restarted]), 'restarted into the first state'


def test_full_size_wildfire_c4_never_idles():
    """Wildfire C4 at 65 536 environments, on-device sampler, 3 x max_steps steps: the batch never goes idle, episode
    lengths stay within the horizon, returns are the rewards summed in torch, and the run equals the explicit one."""
    B, max_steps = 65536, 100
    config = presets.wildfire_large()
    auto = make('wildfire', config, B, max_steps, autoreset=True)
    explicit = make('wildfire', config, B, max_steps)
    for env in (auto, explicit):
        env.reset(seed=2026)
    summed = torch.zeros_like(auto._rewards)
    episodes = 0
    for t in range(3 * max_steps):
        for env in (auto, explicit):
            env.sample_actions(2026)
            env.step_all()
        summed += auto._rewards
        stats = auto.episode_statistics
        done = stats['done']
        assert auto.control_block()['alive'] == 3, f't={t}'
        if bool(done.any()):
            episodes += int(done.sum())
            assert int(stats['length'][done].max()) <= max_steps and int(stats['length'][done].min()) >= 1, f't={t}'
            assert torch.allclose(stats['return'][done], summed[done], rtol=1e-5, atol=1e-4), f't={t}'
            summed[done] = 0
        compare_step_outputs(auto, explicit, f't={t}')
        explicit.reset_batches(explicit.finished.nonzero().flatten())
        compare_published(auto, explicit, f't={t}')
    assert episodes >= 2 * B, episodes
