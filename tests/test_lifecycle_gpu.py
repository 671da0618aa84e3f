"""How an engine gets into a state -- ``reset(options={'initial_state': ...})``, ``reset_batches``, the refresh launches
behind ``update_actions()`` / ``update_observations()`` and checkpoint restore -- against the CPU oracle, from states
that preset rollouts rarely reach.

Every path republishes the control block's batch-wide flags (``alive``: some environment not terminated / not
truncated, the early return of utils/env.py:212; ``agents_with_tasks``: the per-agent skip of wildfire.py:434 and
rideshare.py:276).  A stale flag does not fault, it silently steps a batch the reference would not step (or skips one it
would), so the flags are compared with the oracle's too, and every test keeps stepping after the state was set.
Integers, masks and dones are compared bit-exactly, float rewards within golden_util's tolerance.
"""
import importlib
import types

import numpy as np
import pytest
import torch

from free_range_zoo_b200 import presets
from tests import golden_util as G
from tests import philox_ref as P
from tests.engine_util import cpu, cyber_outputs, rideshare_outputs
from tests.test_philox_parity_gpu import WILDFIRE_GEOMETRIES, fast_wildfire_compare

pytestmark = pytest.mark.gpu

CYBER_PO = dict(show_bad_actions=False, partially_observable=True)


def make(domain, config, B, max_steps, **kwargs):
    module = importlib.import_module(f'free_range_zoo_b200.envs.{domain}_v0')
    return module.parallel_env(parallel_envs=B, max_steps=max_steps, configuration=config, device=torch.device('cuda'),
                               **kwargs).unwrapped


def wildfire_config(spec):
    return presets.wildfire_3x3() if spec == 'wildfire_3x3' else presets.wildfire_large(**spec)


class Given(types.SimpleNamespace):
    """An ``initial_state`` for ``reset(options=...)``: named tensors, batch-major."""

    def __len__(self):
        return next(iter(vars(self).values())).shape[0]


def given(**arrays):
    return Given(**{name: torch.as_tensor(value) for name, value in arrays.items()})


# ------------------------------------------------------------------------------------------------ state generators


def wildfire_state(oracle, rng, dead=(), all_lit=()):
    """Seeded valid wildfire states (invariants of oracle/wildfire.py:55-154): per cell one of lit (+type, intensity
    1..S-2, the burn-out branch S-2 included), burnable (-type, intensity 0, fuel -1..initial fuel), burnt out (-type,
    intensity S-1) or empty (0 / 0 / 0); per agent suppressant on a 0.5 grid from exactly 0, every possible capacity,
    every equipment state.  Environments in ``dead`` have nothing lit and no fuel (they terminate on the first step),
    those in ``all_lit`` have every cell with a fire type lit."""
    B, H, W, A, S = oracle.B, oracle.H, oracle.W, oracle.A, oracle.S
    types_ = np.broadcast_to(oracle.fire_types, (B, H, W))
    kind = rng.integers(0, 4, (B, H, W))
    kind[list(all_lit)] = 0
    kind[list(dead)] = rng.choice([2, 3], size=(len(dead), H, W))
    kind[types_ == 0] = 3
    fuel0 = oracle.initial_fuel
    fires = np.where(kind == 0, types_, np.where(kind == 3, 0, -types_)).astype(np.int32)
    intensity = np.select([kind == 0, kind == 2], [rng.integers(1, S - 1, (B, H, W)), np.full((B, H, W), S - 1)], 0)
    fuel = np.select([kind == 0, kind == 1, kind == 2], [rng.integers(0, fuel0 + 1, (B, H, W)),
                                                         rng.integers(-1, fuel0 + 1, (B, H, W)),
                                                         rng.integers(0, fuel0 + 1, (B, H, W))], 0)
    fuel[list(dead)] = 0
    capacity = rng.choice(oracle.capacities, size=(B, A)).astype(np.float32)
    supply = np.floor(rng.random((B, A)) * (2 * capacity + 1)).astype(np.float32) * np.float32(0.5)
    supply[rng.random((B, A)) < 0.2] = 0.0
    equipment = rng.integers(0, oracle.E, (B, A)).astype(np.int32)
    return dict(fires=fires, intensity=intensity.astype(np.int32), fuel=fuel.astype(np.int32), suppressants=supply,
                capacity=capacity, equipment=equipment)


def cyber_state(oracle, rng, absent=()):
    """Every network state, defenders at home (-1) and on every node, mixed presence; ``absent`` environments have
    no agent present."""
    B = oracle.B
    presence = rng.random((B, oracle.n_agents)) < 0.6
    presence[list(absent)] = False
    return dict(network_state=rng.integers(0, oracle.num_states, (B, oracle.N)).astype(np.int32),
                location=rng.integers(-1, oracle.N, (B, oracle.n_def)).astype(np.int32), presence=presence)


def rideshare_state(oracle, config, rng, steps):
    """Drivers anywhere, passenger tables from empty to as full as the table can be while the schedule keeps adding
    rows for ``steps`` steps; every passenger state, with a driver association iff accepted, riding passengers on their
    driver's cell (where the oracle's pick-up leaves them), drivers at their pool limit, waiting passengers on a
    driver's cell; entry times ascending in table order.  Returns (agents [B, A, 2], flat passengers [N, 11])."""
    B, A, K = oracle.B, oracle.A, oracle.K
    H, W = int(config.grid_height), int(config.grid_width)
    fares = oracle.schedule[:, 6]
    agents = np.stack([rng.integers(0, H, (B, A)), rng.integers(0, W, (B, A))], axis=2).astype(np.int32)
    rows = []
    for b in range(B):
        entering = sum(1 for row in oracle.schedule if row[0] <= steps + 1 and row[1] in (b, -1))
        room = max(K - entering, 0)
        count = room if b % 5 == 1 else int(rng.integers(0, room + 1))
        load = np.zeros(A, int)
        entered = np.sort(rng.integers(-6, 1, count))
        for i in range(count):
            state = int(rng.integers(0, 3))
            a = int(rng.integers(0, A))
            if state and load[a] >= oracle.pool_limit and b % 3 != 0:
                state = 0
            y, x = int(rng.integers(0, H)), int(rng.integers(0, W))
            if state == 2 or rng.random() < 0.3:
                y, x = int(agents[b, a, 0]), int(agents[b, a, 1])
            accepted = int(entered[i] + rng.integers(0, 1 - entered[i])) if state else -1
            picked = int(accepted + rng.integers(0, 1 - accepted)) if state == 2 else -1
            load[a] += state > 0
            rows.append([b, y, x, int(rng.integers(0, H)), int(rng.integers(0, W)), int(rng.choice(fares)), state,
                         a if state else -1, int(entered[i]), accepted, picked])
    return agents, np.asarray(rows, np.int32).reshape(-1, 11)


# ------------------------------------------------------------------------------------------------ comparisons


def assert_flags(raw, terminated, truncated, agent_task_count=None, context=''):
    """The control block's published flags == the oracle's batch-wide conditions."""
    block = raw.control_block()
    alive = (1 if not np.all(terminated) else 0) | (2 if not np.all(truncated) else 0)
    assert block['alive'] == alive, f"{context}: alive {block['alive']} != {alive}"
    if agent_task_count is not None:
        bits = sum(1 << a for a in np.nonzero(agent_task_count.sum(axis=0) > 0)[0])
        assert block['agents_with_tasks'] == bits, f"{context}: agents_with_tasks {block['agents_with_tasks']:#x} != {bits:#x}"


def check_wildfire(raw, oracle, context):
    fast_wildfire_compare(raw, oracle, context)
    assert_flags(raw, oracle.terminated, oracle.truncated, oracle.agent_task_count, context)


def check_cyber(raw, oracle, context):
    want = {key: value[None] for key, value in oracle.outputs(raw.agents).items()}
    G.compare(cyber_outputs(raw), want, 0, context=context)
    assert np.array_equal(cpu(raw.state().network_state), oracle.network_state), context
    assert_flags(raw, oracle.terminated, oracle.truncated, context=context)


def check_rideshare(raw, oracle, context):
    want = {key: value[None] for key, value in oracle.outputs().items()}
    G.compare(rideshare_outputs(raw, oracle.K), want, 0, context=context)
    assert np.array_equal(cpu(raw._cumulative), oracle.cumulative_rewards), context
    assert_flags(raw, oracle.terminated, oracle.truncated, oracle.agent_task_count, context)


def wildfire_actions(oracle, rng):
    counts = oracle.environment_task_count[:, None] + 0 * oracle.agent_task_count if oracle.show_bad_actions \
        else oracle.agent_task_count
    k = np.minimum((rng.random(counts.shape) * (counts + 1)).astype(np.int64), counts)
    return np.stack([k, np.where(k == counts, -1, 0)], axis=2).astype(np.int32)


def rideshare_actions(oracle, rng):
    acts = np.zeros((oracle.B, oracle.A, 2), np.int32)
    for b in range(oracle.B):
        for a in range(oracle.A):
            mine = oracle._task_list(b, a)
            k = min(int(rng.random() * (len(mine) + 1)), len(mine))
            acts[b, a] = (k, -1) if k == len(mine) else (k, oracle.tables[b][mine[k]][6])
    return acts


class Rollout:
    """One engine and its oracle stepped together: injected uniforms or (``philox``) the in-kernel Philox stream
    restated by tests/philox_ref.py for the engine's global environment indices."""

    def __init__(self, domain, raw, oracle, rng, philox=False, seed=0, offset=0):
        self.domain, self.raw, self.oracle, self.rng = domain, raw, oracle, rng
        self.philox, self.seed, self.envs = philox, seed, offset + np.arange(oracle.B)

    def check(self, context):
        {'wildfire': check_wildfire, 'cybersecurity': check_cyber, 'rideshare': check_rideshare}[self.domain](
            self.raw, self.oracle, context)

    def step(self, context, actions=None):
        """One step of both; returns whether the oracle stepped (False: the whole batch was finished)."""
        o, raw = self.oracle, self.raw
        step = raw.control_block()['step']
        if self.domain == 'wildfire':
            actions = wildfire_actions(o, self.rng) if actions is None else actions
            if self.philox:
                uniforms = P.wildfire_uniforms(self.seed, step, self.envs, o.H, o.W, o.A)
            else:
                uniforms = self.rng.random((3, o.B, o.H, o.W), dtype=np.float32), self.rng.random((5, o.B, o.A), dtype=np.float32)
        elif self.domain == 'cybersecurity':
            from tests.test_cyber_gpu import legal_actions
            actions = legal_actions(o, self.rng) if actions is None else actions
            if self.philox:
                uniforms = P.cyber_uniforms(self.seed, step, self.envs, o.N, o.n_agents)
            else:
                uniforms = (self.rng.random((1, o.B, o.N), dtype=np.float32),
                            self.rng.random((1, o.B, o.n_agents), dtype=np.float32))
        else:
            actions = rideshare_actions(o, self.rng) if actions is None else actions
            uniforms = ()
        stepped = o.step(actions, *uniforms)
        if uniforms and not self.philox:
            raw.inject_uniforms(*(torch.from_numpy(u) for u in uniforms))
        raw.step_all(torch.from_numpy(actions).cuda())
        self.check(context)
        assert raw.control_block()['step'] == step + int(stepped), f'{context}: the Philox step counter'
        return stepped

    def run(self, steps, context):
        for t in range(steps):
            self.step(f'{context} t={t}')
        assert not getattr(self.oracle, 'faults', None)
        self.raw.check_errors()


def setup(domain, config, B, max_steps, rng, kernel='auto', philox=False, offset=0, seed=7, kwargs=None, state=None,
          **generator):
    """Engine + oracle reset from a generated (or the given) state through ``reset(options={'initial_state': ...})``."""
    kwargs = dict(kwargs or {})
    if domain == 'wildfire':
        from oracle.wildfire import WildfireOracle
        oracle = WildfireOracle(config, B, max_steps, **kwargs)
        state = wildfire_state(oracle, rng, **generator) if state is None else state
        oracle.reset(initial_state=state)
        raw = make(domain, config, B, max_steps, step_kernel=kernel, env_offset=offset, **kwargs)
        raw.reset(seed=seed, options={'initial_state': given(**state)})
    elif domain == 'cybersecurity':
        from oracle.cybersecurity import CybersecurityOracle
        oracle = CybersecurityOracle(config, B, max_steps, **kwargs)
        state = cyber_state(oracle, rng, **generator) if state is None else state
        oracle.reset(initial_state=state)
        raw = make(domain, config, B, max_steps, env_offset=offset, **kwargs)
        raw.reset(seed=seed, options={'initial_state': given(**state)})
    else:
        from oracle.rideshare import RideshareOracle
        oracle = RideshareOracle(config, B, max_steps)
        agents, passengers = rideshare_state(oracle, config, rng, max_steps + 10) if state is None else state
        oracle.reset(initial_state=dict(agents=agents, passengers=passengers))
        raw = make(domain, config, B, max_steps, step_kernel=kernel)
        raw.reset(seed=seed, options={'initial_state': given(agents=agents, passengers=passengers)})
    return Rollout(domain, raw, oracle, rng, philox=philox, seed=seed, offset=offset)


# ------------------------------------------------------------------------------------------------ 1. initial_state reset

WILDFIRE_RESETS = [  # (spec, B, kernels)
    ('wildfire_large', 129, ['auto']),  # C4
    ('wildfire_3x3', 31, ['groups', 'tiles']),  # C1
    ('wildfire_3x3', 2049, ['groups', 'tiles']),
    (dict(height=4, width=5, num_agents=4, seed=32), 1, ['groups', 'tiles']),  # spare lanes feed the agents' words
    (dict(height=4, width=5, num_agents=4, seed=32), 129, ['groups', 'tiles']),
    (dict(height=16, width=16, num_agents=32, seed=12), 31, ['auto']),  # the engine's size limits
]


@pytest.mark.parametrize('mode', ['injected', 'philox'])
@pytest.mark.parametrize('spec,B,kernel', [(s, B, k) for s, B, ks in WILDFIRE_RESETS for k in ks],
                         ids=lambda v: str(v).replace(' ', ''))
def test_wildfire_initial_state_reset_matches_oracle(spec, B, kernel, mode):
    config = wildfire_config('wildfire_3x3' if spec == 'wildfire_3x3' else ({} if spec == 'wildfire_large' else spec))
    rng = np.random.default_rng(B)
    dead, lit = ([0], [B - 1]) if B > 1 else ((), ())
    run = setup('wildfire', config, B, 40, rng, kernel=kernel, philox=mode == 'philox', offset=5 * B + 3,
                seed=(0x5EED << 32) | B, kwargs=dict(show_bad_actions=B % 2 == 1 and B > 1), dead=dead, all_lit=lit)
    run.check('t=0')
    run.run(12, f'{spec} B={B}')


@pytest.mark.parametrize('preset,B,kernel', [
    ('rideshare_c2', 129, 'groups'), ('rideshare_c2', 129, 'tiles'), ('rideshare_c2', 1, 'tiles'),
    (('rideshare_synthetic', dict(drivers=20, rows=64)), 31, 'auto'),
])
def test_rideshare_initial_state_reset_matches_oracle(preset, B, kernel):
    config = getattr(presets, preset)() if isinstance(preset, str) else getattr(presets, preset[0])(**preset[1])
    run = setup('rideshare', config, B, 12, np.random.default_rng(B + 1), kernel=kernel)
    run.check('t=0')
    run.run(12, f'{preset} B={B}')


@pytest.mark.parametrize('mode', ['injected', 'philox'])
@pytest.mark.parametrize('preset,B,kwargs', [
    ('cyber_c3', 129, CYBER_PO),
    ('cyber_c3', 2049, dict(show_bad_actions=True, partially_observable=False)),
    (('cyber_synthetic', dict(nodes=32, attackers=16, defenders=16)), 31, dict(show_bad_actions=True)),  # direct kernel
])
def test_cyber_initial_state_reset_matches_oracle(preset, B, kwargs, mode):
    config = getattr(presets, preset)() if isinstance(preset, str) else getattr(presets, preset[0])(**preset[1])
    run = setup('cybersecurity', config, B, 30, np.random.default_rng(B + 2), philox=mode == 'philox',
                offset=7 * B + 1, seed=(0xC1 << 40) | B, kwargs=kwargs, absent=[0, B - 1])
    run.check('t=0')
    run.run(12, f'{preset} B={B}')


# ------------------------------------------------------------------------------------------------ 2. refresh


def edit_and_refresh(run, state, done):
    """Write ``state`` and the done flags into the engine and the oracle, refresh both."""
    raw, o = run.raw, run.oracle
    terminated, truncated = done
    for name, value in state.items():
        getattr(raw.state(), name).copy_(torch.as_tensor(value).to(getattr(raw.state(), name).dtype))
        setattr(o, name, np.array(value))
    raw._terminated.copy_(torch.from_numpy(terminated.astype(np.uint8)))
    raw._truncated.copy_(torch.from_numpy(truncated.astype(np.uint8)))
    o.terminated, o.truncated = terminated.copy(), truncated.copy()
    raw.update_actions()
    raw.update_observations()


DONE_PATTERNS = ['some', 'all_terminated', 'all_truncated']


def done_flags(pattern, B, rng):
    if pattern == 'all_terminated':
        return np.ones(B, bool), rng.random(B) < 0.5
    if pattern == 'all_truncated':
        return rng.random(B) < 0.5, np.ones(B, bool)
    if pattern == 'some':
        return rng.random(B) < 0.3, rng.random(B) < 0.3
    return np.zeros(B, bool), np.zeros(B, bool)


@pytest.mark.parametrize('pattern', DONE_PATTERNS)
@pytest.mark.parametrize('kernel', ['groups', 'tiles'])
@pytest.mark.parametrize('spec,B,geometry', WILDFIRE_GEOMETRIES, ids=lambda v: str(v).replace(' ', ''))
def test_wildfire_refresh_on_an_edited_state_matches_oracle(spec, B, geometry, kernel, pattern):
    if kernel == 'tiles' and geometry[0] != 8:
        pytest.skip('grid too large for the tiled kernel')
    config = wildfire_config(spec)
    rng = np.random.default_rng(B + len(pattern))
    run = setup('wildfire', config, B, 30, rng, kernel=kernel, kwargs=dict(show_bad_actions=True))
    edit_and_refresh(run, wildfire_state(run.oracle, rng, dead=[1], all_lit=[0]), done_flags(pattern, B, rng))
    run.oracle.update_observations()
    run.oracle.update_actions()
    run.check(f'{spec} refresh')
    for t in range(3):  # the next steps see the republished flags: the oracle steps, or returns early, alike
        run.step(f'{spec} {pattern} t={t}')


RIDESHARE_TILE_SHAPES = [  # the shapes test_rideshare_gpu.py runs through the tiled kernel
    ('rideshare_c2', {}, 97), ('rideshare_synthetic', dict(drivers=7, rows=24), 200),
    ('rideshare_synthetic', dict(drivers=8, rows=40), 130), ('rideshare_synthetic', dict(drivers=6, rows=16), 97),
    ('rideshare_synthetic', dict(drivers=2, rows=64), 70),
]


@pytest.mark.parametrize('pattern', ['none', 'all_truncated'])
@pytest.mark.parametrize('kernel', ['groups', 'tiles'])
@pytest.mark.parametrize('preset,preset_kwargs,B', RIDESHARE_TILE_SHAPES)
def test_rideshare_refresh_on_an_edited_state_matches_oracle(preset, preset_kwargs, B, kernel, pattern):
    config = getattr(presets, preset)(**preset_kwargs)
    rng = np.random.default_rng(B + 3)
    run = setup('rideshare', config, B, 20, rng, kernel=kernel)
    raw, o = run.raw, run.oracle
    agents, passengers = rideshare_state(o, config, rng, 20)  # a second generated state, written by hand
    counts = np.bincount(passengers[:, 0], minlength=B) if len(passengers) else np.zeros(B, int)
    table = np.zeros((B, o.K, 11), np.int32)
    for b in range(B):
        table[b, :counts[b]] = passengers[passengers[:, 0] == b]
    raw.state().agents.copy_(torch.from_numpy(agents))
    raw.state().passenger_table.copy_(torch.from_numpy(table))
    raw.environment_task_count.copy_(torch.from_numpy(counts.astype(np.int32)))
    o.agents, o.tables = agents.copy(), [[list(map(int, row)) for row in table[b, :counts[b]]] for b in range(B)]
    terminated, truncated = done_flags(pattern, B, rng)
    raw._truncated.copy_(torch.from_numpy(truncated.astype(np.uint8)))
    o.truncated = truncated
    raw.update_actions()
    raw.update_observations()
    o._publish()
    run.check(f'{preset} refresh')
    for t in range(3):
        run.step(f'{preset} {pattern} t={t}')


@pytest.mark.parametrize('pattern', ['none', 'all_truncated'])
@pytest.mark.parametrize('preset,B,kwargs', [
    ('cyber_c3', 129, CYBER_PO),
    ('cyber_quirks', 300, dict(show_bad_actions=True, observe_other_location=True)),
    (('cyber_synthetic', dict(nodes=10, attackers=5, defenders=4)), 200, dict(show_bad_actions=True)),
    (('cyber_synthetic', dict(nodes=17, attackers=1, defenders=1)), 200, dict(show_bad_actions=True)),
    (('cyber_synthetic', dict(nodes=20, attackers=9, defenders=9)), 100, dict(show_bad_actions=True)),
    (('cyber_synthetic', dict(nodes=32, attackers=16, defenders=16)), 100, dict(show_bad_actions=True)),
])
def test_cyber_refresh_on_an_edited_state_matches_oracle(preset, B, kwargs, pattern):
    config = getattr(presets, preset)() if isinstance(preset, str) else getattr(presets, preset[0])(**preset[1])
    rng = np.random.default_rng(B + 4)
    run = setup('cybersecurity', config, B, 20, rng, kwargs=kwargs)
    state = cyber_state(run.oracle, rng, absent=[1])
    engine_state = dict(state, presence=state['presence'].astype(np.uint8))
    edit_and_refresh(run, engine_state, done_flags(pattern, B, rng))
    run.oracle.presence = state['presence']
    run.oracle._publish()
    run.check(f'{preset} refresh')
    for t in range(3):
        run.step(f'{preset} {pattern} t={t}')


# ------------------------------------------------------------------------------------------------ 3. masked reset


def masks(B):
    index = np.arange(B)
    return dict(empty=index < 0, all=index >= 0, first=index == 0, last=index == B - 1, every_third=index % 3 == 0)


MASKED = [  # (domain, preset, B, kernel, kwargs)
    ('wildfire', 'wildfire_large', 129, 'auto', {}),
    ('wildfire', 'wildfire_3x3', 300, 'tiles', dict(show_bad_actions=True)),
    ('rideshare', 'rideshare_c2', 300, 'groups', {}),
    ('rideshare', 'rideshare_c2', 300, 'tiles', {}),
    ('cybersecurity', 'cyber_c3', 129, 'auto', CYBER_PO),
]


def domain_config(domain, preset):
    if domain == 'wildfire':
        return wildfire_config('wildfire_3x3' if preset == 'wildfire_3x3' else {})
    return getattr(presets, preset)()


def engine_reset(raw, mask):
    raw.reset_batches(np.nonzero(mask)[0].tolist())


@pytest.mark.parametrize('mask_name', ['empty', 'all', 'first', 'last', 'every_third'])
@pytest.mark.parametrize('domain,preset,B,kernel,kwargs', MASKED)
def test_masked_reset_matches_oracle(domain, preset, B, kernel, kwargs, mask_name):
    rng = np.random.default_rng(B + 5)
    run = setup(domain, domain_config(domain, preset), B, 40, rng, kernel=kernel, kwargs=kwargs)
    for t in range(4):
        run.step(f'before t={t}')
    mask = masks(B)[mask_name]
    run.oracle.reset_batches(mask)
    engine_reset(run.raw, mask)
    run.check(f'{mask_name} reset')
    run.run(6, f'after {mask_name} reset')


@pytest.mark.parametrize('domain,preset,B,kernel,kwargs', [
    ('rideshare', 'rideshare_c2', 2100, 'tiles', {}),  # the last tile of 32 environments is partial
    ('cybersecurity', 'cyber_c3', 129, 'auto', CYBER_PO),
])
def test_masked_reset_ending_inside_the_last_tile(domain, preset, B, kernel, kwargs):
    rng = np.random.default_rng(B + 6)
    run = setup(domain, domain_config(domain, preset), B, 40, rng, kernel=kernel, kwargs=kwargs)
    for t in range(2):
        run.step(f'before t={t}')
    mask = np.zeros(B, bool)
    mask[B - B % 32 - 3:B - 1] = True
    run.oracle.reset_batches(mask)
    engine_reset(run.raw, mask)
    run.check('tail reset')
    run.run(5, 'after tail reset')


FINISHED = [  # how the whole batch finishes: every wildfire environment burns out at once, or the horizon passes
    ('wildfire', 'wildfire_large', 129, 40, dict(dead=range(129))),
    ('wildfire', 'wildfire_3x3', 100, 3, {}),
    ('rideshare', 'rideshare_c2', 100, 3, {}),
    ('cybersecurity', 'cyber_c3', 129, 3, {}),
]


def finish(run, context):
    for t in range(6):
        if not run.step(f'{context} finishing t={t}'):
            break
    o = run.oracle
    assert o.terminated.all() or o.truncated.all()


@pytest.mark.parametrize('domain,preset,B,max_steps,generator', FINISHED)
def test_an_empty_reset_of_a_finished_batch_leaves_the_next_step_a_noop(domain, preset, B, max_steps, generator):
    rng = np.random.default_rng(B + 7)
    kwargs = CYBER_PO if domain == 'cybersecurity' else {}
    run = setup(domain, domain_config(domain, preset), B, max_steps, rng, kwargs=kwargs, **generator)
    finish(run, preset)
    raw = run.raw
    before = {name: tensor.clone() for name, tensor in raw._bound.items() if tensor is not None}
    step = raw.control_block()['step']
    run.oracle.reset_batches(np.zeros(B, bool))
    raw.reset_batches([])
    run.check('empty reset')
    assert not run.step('after the empty reset')
    assert raw.control_block()['step'] == step
    for name, tensor in before.items():
        if name not in ('actions', 'field_uniforms', 'agent_uniforms', 'network_uniforms', 'control'):
            assert torch.equal(raw._bound[name], tensor), f'{name} changed by a step of a finished batch'


@pytest.mark.parametrize('domain,preset,B,max_steps,generator', FINISHED)
def test_a_finished_batch_revived_in_part_steps_the_revived_environments(domain, preset, B, max_steps, generator):
    rng = np.random.default_rng(B + 8)
    kwargs = CYBER_PO if domain == 'cybersecurity' else {}
    run = setup(domain, domain_config(domain, preset), B, max_steps, rng, kwargs=kwargs, **generator)
    finish(run, preset)
    mask = np.arange(B) % 3 == 1
    if domain == 'wildfire' and generator:  # revive into burning states: the dead initial state would end at once
        fresh = wildfire_state(run.oracle, rng)
        run.oracle.reset_batches(mask, fresh)
        raw = run.raw
        for name, value in fresh.items():
            getattr(raw._initial, name).copy_(torch.from_numpy(value))
    else:
        run.oracle.reset_batches(mask)
    moves = cpu(run.raw.num_moves).copy()
    engine_reset(run.raw, mask)
    run.check('partial revival')
    assert run.step('after the revival')
    assert (cpu(run.raw.num_moves)[mask] == 1).all() and (cpu(run.raw.num_moves)[~mask] == moves[~mask] + 1).all()
    run.run(2, 'revived')


# ------------------------------------------------------------------------------------------------ 4. checkpoint restore


def checkpoint(raw):
    return {name: tensor.clone() for name, tensor in raw._bound.items()
            if tensor is not None and not name.startswith('init_') and name != 'control'}, raw.generator_state_dict()


def restore(raw, saved):
    arrays, generator = saved
    for name, tensor in arrays.items():
        raw._bound[name].copy_(tensor)
    raw.load_generator_state_dict(generator)


def test_a_restore_clears_faults_recorded_before_it():
    """A checkpoint taken right after a step with an invalid action (a recorded data fault): the restored run did
    not commit that fault, so check_errors() stays quiet after the restore."""
    raw = make('cybersecurity', presets.cyber_c3(), 64, 10, show_bad_actions=False)
    raw.reset(seed=2)
    actions = torch.zeros((64, 4, 2), dtype=torch.int32, device='cuda')
    actions[:, :, 1] = -1
    actions[3, 0] = torch.tensor([7, 0])  # attack a node that does not exist (reference: ValueError, :341)
    raw.step_all(actions)
    saved = checkpoint(raw)
    restore(raw, saved)
    raw.check_errors()
    actions[3, 0] = torch.tensor([1, -1])
    raw.step_all(actions)
    raw.check_errors()


def test_a_restore_into_another_env_offset_is_refused():
    config = presets.wildfire_large()
    raw = make('wildfire', config, 64, 10, env_offset=64)
    raw.reset(seed=1)
    saved = checkpoint(raw)
    other = make('wildfire', config, 64, 10, env_offset=0)
    other.reset(seed=1)
    with pytest.raises(ValueError, match='env_offset'):
        other.load_generator_state_dict(saved[1])
    raw.load_generator_state_dict(saved[1])  # the same offset is accepted


@pytest.mark.parametrize('domain,preset', [('wildfire', 'wildfire_large'), ('rideshare', 'rideshare_c2'),
                                           ('cybersecurity', 'cyber_c3')])
def test_a_restored_finished_batch_does_not_step(domain, preset):
    """A checkpoint of a batch in which every environment is truncated: after the restore into a fresh environment
    (whose flags say "alive"), the next step is a no-op, as the reference's would be (utils/env.py:212)."""
    config = getattr(presets, preset)()
    raw = make(domain, config, 300, 4)
    raw.reset(seed=3)
    for _ in range(4):
        raw.sample_actions(1)
        raw.step_all()
    assert bool(raw.truncated.all())
    saved = checkpoint(raw)
    other = make(domain, config, 300, 4)
    other.reset(seed=3)
    restore(other, saved)
    assert other.control_block()['alive'] & 2 == 0
    other.sample_actions(1)
    other.step_all()
    for name, tensor in saved[0].items():
        if name != 'actions':
            assert torch.equal(other._bound[name], tensor), name
    assert other.control_block()['step'] == saved[1]['step']


# ------------------------------------------------------------------------------------------------ 5. sharding


def shard_rollouts(domain, config, state, B, split, kwargs, steps, actions_of, seed=0xABC):
    """The whole batch and its two shards, each an engine + the oracle run on exactly its environments (Philox)."""
    rng = np.random.default_rng(0)
    pieces = {'whole': (0, B), 'shard0': (0, split), 'shard1': (split, B)}
    runs = {}
    for name, (lo, hi) in pieces.items():
        part = {key: value[lo:hi] for key, value in state.items()}
        runs[name] = setup(domain, config, hi - lo, steps, rng, philox=True, offset=lo, seed=seed, kwargs=kwargs,
                           state=part)
    for t in range(steps):
        whole = actions_of(runs['whole'].oracle, t)
        for name, (lo, hi) in pieces.items():
            runs[name].step(f'{name} t={t}', actions=np.ascontiguousarray(whole[lo:hi]))
    return runs


def wildfire_fixed_actions(oracle, t):
    """Every agent aims at env-local task min(t % 3, tasks - 1) -- with bad actions shown, whether it can reach it or
    not -- and refills only where nothing is lit."""
    count = oracle.environment_task_count[:, None] + np.zeros((1, oracle.A), np.int64)
    k = np.minimum(t % 3, np.maximum(count - 1, 0))
    return np.stack([k, np.where(count == 0, -1, 0)], axis=2).astype(np.int32)


@pytest.mark.parametrize('case', ['agree', 'shard0_terminates', 'agent_idle_in_shard0'])
def test_wildfire_shards_follow_the_oracle_of_their_own_environments(case):
    """Each shard evaluates the batch-wide conditions over its own environments: it equals its slice of the whole batch
    while they agree, and the oracle run on the shard alone when they do not."""
    from oracle.wildfire import WildfireOracle
    config, B, split, steps = presets.wildfire_large(), 96, 40, 5
    kwargs = dict(show_bad_actions=True)
    rng = np.random.default_rng(11)
    probe = WildfireOracle(config, B, steps, **kwargs)
    # every cell lit and every tank full: each agent has tasks in both shards throughout, unless the case says otherwise
    state = wildfire_state(probe, rng, dead=range(split) if case == 'shard0_terminates' else (), all_lit=range(split, B))
    if case != 'shard0_terminates':
        state = wildfire_state(probe, rng, all_lit=range(B))
        state['suppressants'] = state['capacity'].copy()
    if case == 'agent_idle_in_shard0':
        state['suppressants'][:split, 0] = 0.0  # agent 0 has tasks in shard 1 only
    runs = shard_rollouts('wildfire', config, state, B, split, kwargs, steps, wildfire_fixed_actions)
    whole, first, second = (runs[name].raw for name in ('whole', 'shard0', 'shard1'))
    same = all(torch.equal(getattr(whole.state(), name)[:split], getattr(first.state(), name)) and
               torch.equal(getattr(whole.state(), name)[split:], getattr(second.state(), name))
               for name in ('fires', 'intensity', 'fuel', 'suppressants', 'equipment'))
    same = same and torch.equal(whole._cumulative[:split], first._cumulative) and torch.equal(whole.num_moves[:split], first.num_moves)
    assert same == (case == 'agree'), 'the shards should differ from the whole batch exactly when the conditions differ'


def test_cyber_shards_follow_the_oracle_of_their_own_environments():
    """Cybersecurity's only batch-wide condition is truncation: shard 0 reset later than shard 1 (a masked reset)
    keeps stepping in the whole batch after shard 1 alone has stopped."""
    config, B, split, steps = presets.cyber_c3(), 80, 30, 4
    rng = np.random.default_rng(12)
    from oracle.cybersecurity import CybersecurityOracle
    state = cyber_state(CybersecurityOracle(config, B, steps, **CYBER_PO), rng)
    runs = {}
    pieces = {'whole': (0, B), 'shard0': (0, split), 'shard1': (split, B)}
    for name, (lo, hi) in pieces.items():
        part = {key: value[lo:hi] for key, value in state.items()}
        runs[name] = setup('cybersecurity', config, hi - lo, steps, rng, philox=True, offset=lo, seed=99, kwargs=CYBER_PO,
                           state=part)
    for t in range(steps + 3):
        if t == 2:  # shard 0 starts over
            for name, (lo, hi) in pieces.items():
                mask = (np.arange(lo, hi) < split)
                runs[name].oracle.reset_batches(mask)
                engine_reset(runs[name].raw, mask)
        for name in pieces:
            runs[name].step(f'{name} t={t}')
    # the whole batch stepped shard 1's truncated environments on; shard 1 alone stopped at its horizon
    assert runs['shard1'].raw.control_block()['step'] == steps
    assert runs['whole'].raw.control_block()['step'] > steps
    assert (cpu(runs['whole'].raw.num_moves)[split:] > steps).all()
