"""Final observations of the same-step autoreset (``keep_final_observations=True``) against the explicit API.

The observation a finished episode ended with is what an ``autoreset=False`` engine shows right after the finishing
step, before its ``reset_batches``: the final buffers, the ``final_observations`` views and the host downloads of the
finished environments must equal that engine's live ones bit for bit.  And keeping them must change nothing else: an
engine with the keyword and one without step identically.  The generated states, the staggered horizons and the
explicit twin are those of tests/test_autoreset_gpu.py (whose engines are checked against the oracle there).
"""
import numpy as np
import pytest
import torch

from free_range_zoo_b200 import presets
from tests.test_autoreset_gpu import (BATCHES, DOMAINS, WILDFIRE_CASES, fresh, generated_state, host_observations_equal,
                                      same_trajectory)
from tests.test_lifecycle_gpu import CYBER_PO, given, make, wildfire_config

pytestmark = pytest.mark.gpu


def engine(domain, config, B, max_steps, kernel, offset, seed, kwargs, state, **extra):
    """An engine reset into the generated initial state (``extra``: autoreset / keep_final_observations)."""
    if domain == 'rideshare':
        raw = make(domain, config, B, max_steps, step_kernel=kernel, **extra)
        agents, passengers = state
        raw.reset(seed=seed, options={'initial_state': given(agents=agents, passengers=passengers)})
        return raw
    more = dict(step_kernel=kernel) if domain == 'wildfire' else {}
    raw = make(domain, config, B, max_steps, env_offset=offset, **more, **kwargs, **extra)
    raw.reset(seed=seed, options={'initial_state': given(**state)})
    return raw


def injected_uniforms(domain, raw, rng):
    B = raw.parallel_envs
    if domain == 'wildfire':
        shapes = (3, B, raw.max_y, raw.max_x), (5, B, len(raw.possible_agents))
    else:
        shapes = (1, B, raw._n_nodes), (1, B, len(raw.possible_agents))
    return tuple(torch.from_numpy(rng.random(shape, dtype=np.float32)) for shape in shapes)


def jagged_rows(tensor, b):
    offsets = tensor.offsets()
    return tensor.values()[int(offsets[b]):int(offsets[b + 1])]


def finals_equal_explicit(keep, explicit, done, context):
    """Final buffers and ``final_observations`` of the finished environments == the explicit engine's live ones."""
    for name, tensor in keep._final_buffers.items():
        assert torch.equal(tensor[done], explicit._bound[name][done]), f'{context}: final {name}'
    finished = done.nonzero().flatten().tolist()
    final = keep.final_observations
    for agent in explicit.agents:
        want, got = explicit.observations[agent], final[agent]
        assert list(got.keys()) == list(want.keys()), context
        for key in want.keys():
            w, g = want[key], got[key]
            where = f'{context}: final_observations[{agent}][{key}]'
            assert g.dtype == w.dtype and g.is_nested == w.is_nested, where
            if w.is_nested:  # jagged tasks: environment by environment
                for b in finished:
                    assert torch.equal(jagged_rows(g, b), jagged_rows(w, b)), f'{where} b={b}'
            else:
                assert g.shape == w.shape and torch.equal(g[done], w[done]), where


def downloads_equal_explicit(keep, explicit, done, context):
    """``gather_observations(final=True)`` == the explicit engine's ``gather_observations()`` on the finished
    environments, counts 0 elsewhere; the compact form unpacks to the packed one."""
    B = explicit.parallel_envs
    want = explicit.gather_observations()
    got = keep.gather_observations(final=True)
    d = done.cpu()
    assert torch.equal(got['counts'], torch.where(d, want['counts'], 0)), f'{context}: counts'
    assert got['total'] == int(want['counts'][d].sum()), context
    dense, ragged = explicit._observation_download()
    for name in dense:
        assert torch.equal(got[name][d], want[name][d]), f'{context}: {name}'
    for name, (_, groups) in ragged.items():
        env_of_row = torch.repeat_interleave(torch.arange(B), want['counts'].long() * groups)
        assert torch.equal(got[name], want[name][d[env_of_row]]), f'{context}: {name}'
    host_observations_equal(keep.gather_observations(final=True, compact=True).unpack(), got, f'{context} compact')


def run_final_against_explicit(domain, config, B, kernel='auto', philox=False, kwargs=None, max_steps=5, seed=0):
    kwargs = dict(kwargs or {})
    offset = 3 * B + 5 if philox else 0
    rng = np.random.default_rng(B + 29)
    state = generated_state(domain, config, B, max_steps, rng, kwargs)
    args = (domain, config, B, max_steps, kernel, offset, seed, kwargs, state)
    explicit = engine(*args)
    auto = engine(*args, autoreset=True)
    keep = engine(*args, autoreset=True, keep_final_observations=True)
    for name, tensor in keep._final_buffers.items():  # a full reset: the reset's observations
        assert torch.equal(tensor, explicit._bound[name]), f'reset: final {name}'
    finished_some = False
    for t in range(3 * max_steps):
        context = f'{domain} B={B} t={t}'
        if t == 2:  # stagger the horizons
            restart = np.nonzero(np.arange(B) % 3 == 0)[0].tolist()
            for env in (explicit, auto, keep):
                env.reset_batches(restart)
        explicit.sample_actions(t + 1)
        actions = explicit._actions.clone()
        if not philox and domain != 'rideshare':
            uniforms = injected_uniforms(domain, explicit, rng)
            for env in (explicit, auto, keep):
                env.inject_uniforms(*uniforms)
        explicit.step_all()
        auto.step_all(actions)
        keep.step_all(actions)
        done = explicit.finished.clone()
        assert torch.equal(keep.episode_statistics['done'], done), context
        same_trajectory(keep, auto, f'{context} keep vs no keep')
        finals_equal_explicit(keep, explicit, done, context)
        downloads_equal_explicit(keep, explicit, done, context)
        finished_some |= bool(done.any())
        explicit.reset_batches(done.nonzero().flatten())
    assert finished_some, 'no environment finished'
    keep.check_errors()


@pytest.mark.parametrize('spec,B,kernel', WILDFIRE_CASES, ids=lambda v: str(v).replace(' ', ''))
def test_wildfire_final_observations_equal_the_explicit_engine(spec, B, kernel):
    run_final_against_explicit('wildfire', wildfire_config(spec), B, kernel=kernel,
                               kwargs=dict(show_bad_actions=B % 2 == 1 and B > 1))


@pytest.mark.parametrize('B', BATCHES)
@pytest.mark.parametrize('kernel', ['groups', 'tiles'])
def test_rideshare_final_observations_equal_the_explicit_engine(kernel, B):
    run_final_against_explicit('rideshare', presets.rideshare_c2(), B, kernel=kernel)


@pytest.mark.parametrize('preset,B,kwargs', [
    ('cyber_c3', 129, CYBER_PO),
    ('cyber_c3', 2049, dict(show_bad_actions=True, partially_observable=False)),
    (('cyber_synthetic', dict(nodes=20, attackers=9, defenders=9)), 31, CYBER_PO),
    (('cyber_synthetic', dict(nodes=32, attackers=16, defenders=16)), 1, dict(show_bad_actions=True)),
])
def test_cyber_final_observations_equal_the_explicit_engine(preset, B, kwargs):
    config = getattr(presets, preset)() if isinstance(preset, str) else getattr(presets, preset[0])(**preset[1])
    run_final_against_explicit('cybersecurity', config, B, kwargs=kwargs)


@pytest.mark.parametrize('domain,spec,B,kernel,kwargs', [
    ('wildfire', {}, 129, 'auto', {}),
    ('wildfire', 'wildfire_3x3', 2049, 'tiles', dict(show_bad_actions=True)),
    ('wildfire', 'wildfire_3x3', 31, 'groups', {}),
    ('cybersecurity', 'cyber_c3', 129, 'auto', CYBER_PO),
    ('cybersecurity', 'cyber_c3', 2049, 'auto', dict(show_bad_actions=True, partially_observable=False)),
])
def test_philox_final_observations_with_an_env_offset(domain, spec, B, kernel, kwargs):
    config = wildfire_config(spec) if domain == 'wildfire' else getattr(presets, spec)()
    run_final_against_explicit(domain, config, B, kernel=kernel, philox=True, kwargs=kwargs, seed=(0xF1 << 36) | B)


# ------------------------------------------------------------------------------------------------ every stepping path


def same_finals(raw, reference, context):
    for name, tensor in reference._final_buffers.items():
        assert torch.equal(raw._final_buffers[name], tensor), f'{context}: final {name}'


@pytest.mark.parametrize('domain', sorted(DOMAINS))
def test_every_stepping_path_keeps_the_same_final_observations(domain):
    B, max_steps, steps = 3000, 4, 12
    reference = fresh(domain, B, max_steps, keep_final_observations=True).unwrapped
    plain = fresh(domain, B, max_steps).unwrapped  # the same autoreset without the keyword
    paths = {name: fresh(domain, B, max_steps, keep_final_observations=True) for name in ('parallel', 'aec', 'host', 'graph')}
    paths['graph'].unwrapped.capture_graph(sample=True, sampler_seed=9, steps=3)
    A = len(reference.agents)
    host_i32 = torch.empty((B, A, 2), dtype=torch.int32).pin_memory()
    host_i8 = torch.empty((B, A, 2), dtype=torch.int8).pin_memory()
    finished_some = False
    for t in range(steps):
        context = f'{domain} t={t}'
        actions = reference.sample_actions(9).clone()
        reference.step_all()
        plain.step_all(actions)
        same_trajectory(reference, plain, f'{context} keep vs no keep')
        finished_some |= bool(reference.episode_statistics['done'].any())
        parallel = paths['parallel']
        parallel.step({a: actions[:, i] for i, a in enumerate(reference.agents)})
        same_finals(parallel.unwrapped, reference, f'{context} parallel')
        for agent in reference.agents:  # the wrapper forwards the views
            assert torch.equal(parallel.final_observations[agent]['self'], reference.final_observations[agent]['self'])
        aec = paths['aec'].unwrapped
        for i in range(A):
            aec.step(actions[:, i])
        same_finals(aec, reference, f'{context} aec')
        host = paths['host'].unwrapped
        buffer = host_i32 if t % 2 == 0 else host_i8
        buffer.copy_(actions)
        torch.cuda.synchronize()
        host.step_host(buffer, chunks=3, observations=(False, True, 'compact')[t % 3])
        same_finals(host, reference, f'{context} host')
        host_observations_equal(host.gather_observations(final=True), reference.gather_observations(final=True),
                                f'{context} host download')
        if t % 3 == 2:
            graph = paths['graph'].unwrapped
            graph.replay()
            same_finals(graph, reference, f'{context} graph')
            same_trajectory(graph, reference, f'{context} graph')
    assert finished_some, 'no environment finished'


def test_capture_and_resets_treat_the_final_buffers_as_documented():
    """capture_graph leaves them as they were, reset_batches does not touch them, a full reset sets them to its
    observations; the live and final downloads keep separate cached state."""
    B, max_steps = 512, 3
    raw = fresh('wildfire', B, max_steps, keep_final_observations=True).unwrapped
    for _ in range(max_steps):  # every environment is truncated at the last step
        raw.sample_actions(5)
        raw.step_all()
    assert bool(raw.episode_statistics['done'].all())
    kept = {name: tensor.clone() for name, tensor in raw._final_buffers.items()}
    assert any(not torch.equal(tensor, raw._bound[name]) for name, tensor in kept.items()), 'nothing to tell apart'
    raw.capture_graph(sample=True, steps=2)
    same = {name: torch.equal(tensor, kept[name]) for name, tensor in raw._final_buffers.items()}
    assert all(same.values()), same
    raw.reset_batches(list(range(0, B, 2)))
    assert all(torch.equal(tensor, kept[name]) for name, tensor in raw._final_buffers.items())
    live, final = raw.gather_observations(), raw.gather_observations(final=True)
    # the restarted half no longer counts as finished; the other half still downloads its final rows
    assert torch.equal(final['counts'][0::2], torch.zeros(B // 2, dtype=torch.int32))
    assert final['total'] == int(raw._final_buffers['env_task_count'][1::2].sum())
    cached = (raw._gather, raw._gather_final)
    raw.gather_observations(compact=True), raw.gather_observations(final=True, compact=True)
    compact_cached = (raw._compact, raw._compact_final)
    raw.gather_observations(), raw.gather_observations(final=True, compact=True), raw.gather_observations(final=True)
    raw.gather_observations(compact=True)
    assert (raw._gather, raw._gather_final) == cached and (raw._compact, raw._compact_final) == compact_cached
    assert live['bytes'] > 0
    raw.reset(seed=11)
    for name, tensor in raw._final_buffers.items():
        assert torch.equal(tensor, raw._bound[name]), name


def test_without_the_keyword_nothing_is_kept():
    raw = fresh('wildfire', 64, 3).unwrapped
    assert raw.autoreset and not raw.keep_final_observations
    assert getattr(raw, '_final_buffers', None) is None
    rows = raw._autoreset_block[1]
    assert all(row.keep is None for row in rows)
    with pytest.raises(RuntimeError, match='keep_final_observations'):
        raw.final_observations
    for compact in (False, True):
        with pytest.raises(RuntimeError, match='keep_final_observations'):
            raw.gather_observations(final=True, compact=compact)


def test_full_size_wildfire_c4_final_observations():
    """Wildfire C4 at 65 536 environments, on-device sampler, 3 x max_steps steps: the final observations equal the
    explicit engine's on every step where an environment finished."""
    B, max_steps = 65536, 100
    config = presets.wildfire_large()
    keep = make('wildfire', config, B, max_steps, autoreset=True, keep_final_observations=True)
    explicit = make('wildfire', config, B, max_steps)
    for env in (keep, explicit):
        env.reset(seed=2026)
    steps_with_finals = 0
    for t in range(3 * max_steps):
        for env in (keep, explicit):
            env.sample_actions(2026)
            env.step_all()
        done = explicit.finished.clone()
        assert torch.equal(keep.episode_statistics['done'], done), f't={t}'
        if bool(done.any()):
            steps_with_finals += 1
            for name, tensor in keep._final_buffers.items():
                assert torch.equal(tensor[done], explicit._bound[name][done]), f't={t}: final {name}'
        explicit.reset_batches(done.nonzero().flatten())
    assert steps_with_finals >= 3, steps_with_finals
