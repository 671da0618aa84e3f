"""Policy inputs on the device (include/frz_inputs.h) against an independent torch restatement built only from the public
observation views and the published bounds: f32 bit for bit, bf16 as the restatement's f32 rounded once.  States come
from the generators of tests/test_lifecycle_gpu.py and are stepped by sampled actions, so counts shrink and grow."""
import numpy as np
import pytest
import torch

from free_range_zoo_b200 import presets
from tests.test_lifecycle_gpu import CYBER_PO, cyber_state, given, make, rideshare_state, wildfire_config, wildfire_state
from tests.test_philox_parity_gpu import WILDFIRE_GEOMETRIES

pytestmark = pytest.mark.gpu

BATCHES = [1, 31, 129, 2049]
PAD = -100


def scales(bounds, none=()):
    """(scale, offset) f32 tensors of the columns: 1 / high, or 1 / (high + 1) with offset 1 for a "none" column; 1
    where the bound is missing or not positive."""
    scale, offset = [], []
    for c, high in enumerate(bounds):
        high = None if high is None else float(high) + (1.0 if c in none else 0.0)
        scale.append(1.0 if high is None or high <= 0 else 1.0 / high)
        offset.append(1.0 if c in none else 0.0)
    return (torch.tensor(scale, dtype=torch.float32, device='cuda'),
            torch.tensor(offset, dtype=torch.float32, device='cuda'))


def affine(values, columns, bounds, none=()):
    """float(v + offset) * scale of the selected columns (integers add the offset as integers)."""
    scale, offset = scales(bounds, none)
    if values.is_floating_point():
        return (values.float() + offset[columns]) * scale[columns]
    return (values.long() + offset[columns].long()).float() * scale[columns]


def restate(raw, final=False, views=None):
    """(agent [B, A, Fa], tasks [B, V, T, Ft]) in f32 from ``observations`` (or ``final_observations``, or ``views``)."""
    if views is None:
        views = raw.final_observations if final else {agent: raw.observe(agent) for agent in raw.agents}
    name = raw.metadata['name']
    B = raw.parallel_envs
    agent_rows, task_rows = [], []
    if name == 'wildfire_v0':
        observed = [0, 1] + ([2] if raw.observe_other_power else []) + ([3] if raw.observe_other_suppressant else [])
        for agent in raw.agents:
            v = views[agent]
            own = affine(v['self'], [0, 1, 2, 3], raw.agent_observation_bounds)
            others = affine(v['others'], observed, raw.agent_observation_bounds).reshape(B, -1)
            agent_rows.append(torch.cat([own, others], dim=1))
        v = views[raw.agents[0]]
        padded, count = v['tasks_padded'], v['task_count']
        live = torch.arange(padded.shape[1], device='cuda').unsqueeze(0) < count.unsqueeze(1)
        columns = affine(padded, [0, 1, 2, 3], raw.fire_observation_bounds)
        task_rows.append(torch.where(live.unsqueeze(2), torch.cat([torch.ones_like(columns[..., :1]), columns], 2), 0.0))
    elif name == 'rideshare_v0':
        for agent in raw.agents:
            v = views[agent]
            own = affine(v['self'], [0, 1, 2, 3], raw.agent_observation_bounds)
            others = affine(v['others'], [0, 1, 2, 3], raw.agent_observation_bounds).reshape(B, -1)
            agent_rows.append(torch.cat([own, others], dim=1))
        padded = views[raw.agents[0]]['tasks_padded']
        if final:  # rows past the count are padding
            live = padded[..., 0] != PAD
        else:
            live = torch.arange(padded.shape[1], device='cuda').unsqueeze(0) < raw.environment_task_count.unsqueeze(1)
        none = padded.clone()
        none[..., 4:6] = torch.where(none[..., 4:6] == PAD, -1, none[..., 4:6])
        columns = affine(none, list(range(8)), raw.passenger_observation_bounds, none=(4, 5))
        task_rows.append(torch.where(live.unsqueeze(2), torch.cat([torch.ones_like(columns[..., :1]), columns], 2), 0.0))
    else:
        config = raw.config
        p = raw.unwrapped._params
        criticality = max(abs(int(c)) for c in torch.as_tensor(config.network_config.adj_matrix).long().sum(1))
        network = (config.network_observation_bounds[0], criticality)
        for agent in raw.agents:
            v = views[agent]
            attacker = agent.startswith('attacker')
            bounds = config.attacker_observation_bounds if attacker else config.defender_observation_bounds
            none = () if attacker else (2, )
            flags = (raw.observe_other_power, raw.observe_other_presence) + (() if attacker else
                                                                            (raw.observe_other_location, ))
            observed = [c for c, on in enumerate(flags) if on]
            own = affine(v['self'], list(range(len(bounds))), bounds, none)
            others = affine(v['others'], observed, bounds, none).reshape(B, -1) if observed else own[:, :0]
            agent_rows.append(torch.cat([own, others], dim=1))
            tasks = v['tasks']  # -100 where the view hides the network
            seen = (tasks[..., 0] != PAD)
            columns = affine(tasks, [0, 1], network)
            task_rows.append(torch.where(seen.unsqueeze(2), torch.cat([torch.ones_like(columns[..., :1]), columns], 2),
                                         0.0))
        width = max(row.shape[1] for row in agent_rows)
        agent_rows = [torch.nn.functional.pad(row, (0, width - row.shape[1])) for row in agent_rows]
        assert int(p.num_nodes) == task_rows[0].shape[1]
    return torch.stack(agent_rows, dim=1), torch.stack(task_rows, dim=1)


def check(raw, context, final=False, where=None):
    want_agent, want_tasks = restate(raw, final)
    shapes = raw.policy_input_shapes
    B = raw.parallel_envs
    assert tuple(want_agent.shape) == (B, ) + shapes['agent'], context
    assert tuple(want_tasks.shape) == (B, ) + shapes['tasks'], context
    for dtype in (torch.float32, torch.bfloat16):
        agent, tasks = raw.policy_inputs(dtype, final=final)
        wa, wt = want_agent.to(dtype), want_tasks.to(dtype)
        if where is not None:
            agent, tasks, wa, wt = agent[where], tasks[where], wa[where], wt[where]
        assert torch.equal(agent, wa), f'{context} {dtype}: agent inputs'
        assert torch.equal(tasks, wt), f'{context} {dtype}: task inputs'
        # the flag is exactly 0 / 1 and a row with flag 0 is all zeros
        assert bool(((tasks[..., 0] == 0) | (tasks[..., 0] == 1)).all()), context
        assert bool((tasks[..., 1:][tasks[..., 0] == 0] == 0).all()), context


def roll(raw, steps, context, seed=2026):
    """check, then step with sampled actions, ``steps`` times"""
    for t in range(steps):
        check(raw, f'{context} t={t}')
        raw.sample_actions(seed + t)
        raw.step_all(None)
    check(raw, f'{context} t={steps}')
    raw.check_errors()


def wildfire_env(config, B, rng, kernel='auto', **kwargs):
    from oracle.wildfire import WildfireOracle
    oracle = WildfireOracle(config, B, 8)
    dead, lit = (range(0, B, 7), range(3, B, 11)) if B > 1 else ((), ())
    state = wildfire_state(oracle, rng, dead=dead, all_lit=lit)
    raw = make('wildfire', config, B, 8, step_kernel=kernel, **kwargs)
    raw.reset(seed=7, options={'initial_state': given(**state)})
    return raw


def rideshare_env(config, B, rng, kernel='auto'):
    from oracle.rideshare import RideshareOracle
    oracle = RideshareOracle(config, B, 8)
    agents, passengers = rideshare_state(oracle, config, rng, 18)
    raw = make('rideshare', config, B, 8, step_kernel=kernel)
    raw.reset(seed=7, options={'initial_state': given(agents=agents, passengers=passengers)})
    return raw


def cyber_env(config, B, rng, **kwargs):
    from oracle.cybersecurity import CybersecurityOracle
    oracle = CybersecurityOracle(config, B, 8)
    state = cyber_state(oracle, rng, absent=range(0, B, 5))
    raw = make('cybersecurity', config, B, 8, **kwargs)
    raw.reset(seed=7, options={'initial_state': given(**state)})
    return raw


OBSERVE = [dict(), dict(observe_other_power=True), dict(observe_other_power=True, observe_other_suppressant=True)]
WILDFIRE_CASES = [(spec, BATCHES[i % len(BATCHES)], kernel, OBSERVE[i % len(OBSERVE)])
                  for i, (spec, _, geometry) in enumerate(WILDFIRE_GEOMETRIES)
                  for kernel in (['groups', 'tiles'] if geometry[0] == 8 else ['auto'])]


@pytest.mark.parametrize('spec,B,kernel,observe', WILDFIRE_CASES, ids=lambda v: str(v).replace(' ', ''))
def test_wildfire_matches_the_restatement(spec, B, kernel, observe):
    rng = np.random.default_rng(B)
    raw = wildfire_env(wildfire_config(spec), B, rng, kernel, show_bad_actions=B % 2 == 1, **observe)
    roll(raw, 4, f'{spec} B={B}')


@pytest.mark.parametrize('B', BATCHES)
@pytest.mark.parametrize('observe', [0, 2])
def test_wildfire_c4_matches_the_restatement(B, observe):
    raw = wildfire_env(presets.wildfire_large(), B, np.random.default_rng(B), **OBSERVE[observe])
    roll(raw, 4, f'C4 B={B}')


@pytest.mark.parametrize('B', BATCHES)
@pytest.mark.parametrize('kernel', ['groups', 'tiles'])
def test_rideshare_matches_the_restatement(kernel, B):
    raw = rideshare_env(presets.rideshare_c2(), B, np.random.default_rng(B), kernel)
    roll(raw, 4, f'rideshare {kernel} B={B}')


def test_every_passenger_state_is_encoded():
    raw = rideshare_env(presets.rideshare_c2(), 129, np.random.default_rng(9))
    task_obs = raw._task_obs[:, :, 4:6]
    live = torch.arange(task_obs.shape[1], device='cuda').unsqueeze(0) < raw.environment_task_count.unsqueeze(1)
    assert bool(((task_obs[..., 0] == PAD) & live).any()) and bool(((task_obs[..., 1] != PAD) & live).any())
    assert bool(((task_obs[..., 0] != PAD) & (task_obs[..., 1] == PAD) & live).any())
    check(raw, 'passenger states')


CYBER_CASES = [
    ('cyber_c3', 1, CYBER_PO),
    ('cyber_c3', 129, dict(CYBER_PO, observe_other_presence=True, observe_other_location=True)),
    ('cyber_c3', 2049, dict(show_bad_actions=True, partially_observable=False, observe_other_power=False)),
    (('cyber_synthetic', dict(nodes=20, attackers=9, defenders=9)), 31, dict(show_bad_actions=True)),
    (('cyber_synthetic', dict(nodes=20, attackers=3, defenders=9)), 129, dict(CYBER_PO, observe_other_location=True)),
    (('cyber_synthetic', dict(nodes=32, attackers=16, defenders=16)), 31, CYBER_PO),
]


@pytest.mark.parametrize('preset,B,kwargs', CYBER_CASES, ids=lambda v: str(v).replace(' ', ''))
def test_cybersecurity_matches_the_restatement(preset, B, kwargs):
    config = getattr(presets, preset)() if isinstance(preset, str) else getattr(presets, preset[0])(**preset[1])
    raw = cyber_env(config, B, np.random.default_rng(B), **kwargs)
    location = raw.state().location
    assert B < 31 or (bool((location == -1).any()) and int(raw._presence.min()) == 0), 'home defenders / absent agents'
    if kwargs.get('partially_observable'):
        raw.sample_actions(5)  # some defenders monitor in the first step
        raw.step_all(None)
        monitored = raw._monitored
        assert B < 31 or (bool((monitored == 0).any()) and bool((monitored != 0).any()))
    roll(raw, 4, f'{preset} B={B}')


@pytest.mark.parametrize('domain,B', [('wildfire', 31), ('wildfire', 2049), ('rideshare', 31), ('rideshare', 2049)])
def test_one_agent(domain, B):
    rng = np.random.default_rng(B)
    if domain == 'wildfire':
        raw = wildfire_env(presets.wildfire_large(height=4, width=5, num_agents=1, seed=32), B, rng,
                           observe_other_power=True)
    else:
        raw = rideshare_env(presets.rideshare_synthetic(drivers=1, rows=16, horizon=10), B, rng)
    assert len(raw.agents) == 1 and raw.policy_input_shapes['agent'] == (1, 4)
    roll(raw, 4, f'{domain} one agent')


def test_wildfire_c4_at_65536():
    raw = make('wildfire', presets.wildfire_large(), 65536, 20)
    raw.reset(seed=3)
    roll(raw, 3, 'C4 65536')


# ------------------------------------------------------------------------------------------------ padding, slots


def poison(raw, rng):
    """Random values in every task row at or past the count (the rows the encoder must never read)."""
    task_obs = raw._task_obs
    rows = torch.arange(task_obs.shape[1], device='cuda').unsqueeze(0) >= raw.environment_task_count.unsqueeze(1)
    noise = torch.from_numpy(rng.integers(-2**31, 2**31 - 1, tuple(task_obs.shape), dtype=np.int64).astype(np.int32))
    task_obs.copy_(torch.where(rows.unsqueeze(2), noise.cuda(), task_obs))


@pytest.mark.parametrize('domain', ['wildfire', 'rideshare', 'cybersecurity'])
def test_padding_and_hidden_rows_are_never_read(domain):
    rng = np.random.default_rng(4)
    if domain == 'wildfire':
        raw = wildfire_env(presets.wildfire_large(), 129, rng)
    elif domain == 'rideshare':
        raw = rideshare_env(presets.rideshare_c2(), 129, rng)
    else:
        raw = cyber_env(presets.cyber_c3(), 129, rng, **CYBER_PO)
        raw.sample_actions(5)
        raw.step_all(None)
    for dtype in (torch.float32, torch.bfloat16):
        before = [t.clone() for t in raw.policy_inputs(dtype)]
        saved = raw._task_obs.clone()
        if domain == 'cybersecurity':
            # the hidden views' rows: change the network wherever no defender sees it and check those views stay zero
            hidden = raw._monitored == 0
            raw._task_obs.copy_(torch.from_numpy(rng.integers(0, 3, tuple(saved.shape)).astype(np.int32)).cuda())
            after = raw.policy_inputs(dtype)[1]
            A_att = raw._n_att
            assert bool((after[:, A_att:][hidden] == 0).all())
        else:
            poison(raw, rng)
            after = raw.policy_inputs(dtype)
            assert torch.equal(after[0], before[0]) and torch.equal(after[1], before[1]), dtype
        raw._task_obs.copy_(saved)


@pytest.mark.parametrize('domain,show_bad', [('wildfire', False), ('wildfire', True), ('rideshare', False)])
def test_every_legal_task_slot_is_a_flagged_row(domain, show_bad):
    rng = np.random.default_rng(12)
    raw = wildfire_env(presets.wildfire_large(), 257, rng, show_bad_actions=show_bad) if domain == 'wildfire' \
        else rideshare_env(presets.rideshare_c2(), 257, rng)
    for t in range(4):
        _, tasks = raw.policy_inputs()
        T = tasks.shape[2]
        legal = raw.legal_actions()[..., :T]
        flag = tasks[:, 0, :, 0] == 1
        assert bool((flag.unsqueeze(1) | ~legal).all()), t
        if show_bad:
            assert torch.equal(legal, flag.unsqueeze(1).expand_as(legal)), t
        raw.sample_actions(t)
        raw.step_all(None)


# ------------------------------------------------------------------------------------------------ final observations


@pytest.mark.parametrize('domain,config', [('wildfire', presets.wildfire_large), ('rideshare', presets.rideshare_c2),
                                           ('cybersecurity', presets.cyber_c3)])
def test_final_observations_are_encoded(domain, config):
    kwargs = dict(partially_observable=True) if domain == 'cybersecurity' else {}
    raw = make(domain, config(), 513, 3, autoreset=True, keep_final_observations=True, **kwargs)
    raw.reset(seed=8)
    finished = 0
    for t in range(7):
        raw.sample_actions(t)
        raw.step_all(None)
        done = raw.episode_statistics['done']
        finished += int(done.sum())
        if bool(done.any()):
            check(raw, f'{domain} final t={t}', final=True, where=done)
        check(raw, f'{domain} live t={t}')
    assert finished > 0
    plain = make(domain, config(), 8, 3, autoreset=True)
    plain.reset(seed=1)
    with pytest.raises(RuntimeError, match='keep_final_observations'):
        plain.policy_inputs(final=True)


# ------------------------------------------------------------------------------------------------ buffers, out=


def test_buffers_and_out():
    raw = make('wildfire', presets.wildfire_large(), 64, 10, observe_other_power=True)
    raw.reset(seed=2)
    shapes = raw.policy_input_shapes
    first = raw.policy_inputs()
    addresses = [t.data_ptr() for t in first]
    for dtype in (torch.float32, torch.bfloat16):
        agent, tasks = raw.policy_inputs(dtype)
        again = raw.policy_inputs(dtype)
        assert [t.data_ptr() for t in again] == [agent.data_ptr(), tasks.data_ptr()]
    assert [t.data_ptr() for t in raw.policy_inputs()] == addresses
    want = [t.clone() for t in raw.policy_inputs()]
    storage = (torch.zeros((5, 64) + shapes['agent'], device='cuda'), torch.zeros((5, 64) + shapes['tasks'], device='cuda'))
    got = raw.policy_inputs(out=(storage[0][3], storage[1][3]))
    assert got[0].data_ptr() == storage[0][3].data_ptr()
    assert torch.equal(storage[0][3], want[0]) and torch.equal(storage[1][3], want[1])
    assert not bool(storage[0][2].any()) and not bool(storage[1][4].any())
    # a bf16 slice at an odd element offset: scalar stores
    flat = torch.zeros(1 + 64 * int(np.prod(shapes['tasks'])), dtype=torch.bfloat16, device='cuda')
    odd = flat[1:].view((64, ) + shapes['tasks'])
    agent_bf16 = torch.zeros((64, ) + shapes['agent'], dtype=torch.bfloat16, device='cuda')
    raw.policy_inputs(torch.bfloat16, out=(agent_bf16, odd))
    assert torch.equal(odd, want[1].to(torch.bfloat16)) and torch.equal(agent_bf16, want[0].to(torch.bfloat16))
    assert float(flat[0]) == 0.0
    good = (torch.zeros((64, ) + shapes['agent'], device='cuda'), torch.zeros((64, ) + shapes['tasks'], device='cuda'))
    bad_outs = [
        (good[0][:, :-1], good[1]),  # shape
        (good[0].to(torch.bfloat16), good[1]),  # dtype
        (good[0].cpu(), good[1]),  # device
        (good[0], torch.zeros((64, ) + shapes['tasks'][:-1] + (2 * shapes['tasks'][-1], ), device='cuda')[..., ::2]),
        (good[0], ),
    ]
    for out in bad_outs:
        with pytest.raises(ValueError):
            raw.policy_inputs(out=out)
    with pytest.raises(ValueError):
        raw.policy_inputs(torch.float16)


def test_the_parallel_wrapper_forwards_policy_inputs():
    from free_range_zoo_b200.envs import cybersecurity_v0
    env = cybersecurity_v0.parallel_env(parallel_envs=64, max_steps=10, configuration=presets.cyber_c3(),
                                        device=torch.device('cuda'))
    env.reset(seed=3)
    assert env.policy_input_shapes == env.unwrapped.policy_input_shapes
    agent, tasks = env.policy_inputs()
    assert tuple(tasks.shape) == (64, ) + env.policy_input_shapes['tasks']
    check(env.unwrapped, 'parallel wrapper')


# ------------------------------------------------------------------------------------------------ graph capture


class Policy(torch.nn.Module):
    """A fixed two-layer MLP: agent rows -> hidden h, task rows -> g; slot t < T scores h . g[t], the rest h @ W."""

    def __init__(self, raw, hidden=32):
        super().__init__()
        gen = torch.Generator().manual_seed(0)
        Fa, (V, T, Ft) = raw.policy_input_shapes['agent'][1], raw.policy_input_shapes['tasks']
        self.agent = torch.nn.Sequential(torch.nn.Linear(Fa, hidden), torch.nn.ReLU(), torch.nn.Linear(hidden, hidden))
        self.task = torch.nn.Sequential(torch.nn.Linear(Ft, hidden), torch.nn.ReLU(), torch.nn.Linear(hidden, hidden))
        self.extra = torch.nn.Linear(hidden, raw.action_slots - T)
        for p in self.parameters():
            p.data.copy_(torch.randn(p.shape, generator=gen) * 0.3)
        self.cuda()

    @torch.no_grad()
    def forward(self, agent, tasks):
        h = self.agent(agent)  # [B, A, H]
        g = self.task(tasks)  # [B, V, T, H]
        if g.shape[1] == 1:
            scores = torch.einsum('bah,bth->bat', h, g[:, 0])
        else:
            scores = torch.einsum('bah,bath->bat', h, g)
        return torch.cat([scores, self.extra(h)], dim=2).contiguous()


@pytest.mark.parametrize('domain,config', [('wildfire', presets.wildfire_large), ('rideshare', presets.rideshare_c2),
                                           ('cybersecurity', presets.cyber_c3)])
def test_graph_capture_of_the_device_loop_replays_equal_to_eager(domain, config):
    B, K = 1000, 6
    eager = make(domain, config(), B, 4, autoreset=True)
    graphed = make(domain, config(), B, 4, autoreset=True)
    policy = Policy(eager)

    def loop(raw, record):
        for _ in range(K):
            agent, tasks = raw.policy_inputs()
            slots, log_prob = raw.sample_actions_from_logits(policy(agent, tasks), 2026)
            record.append((agent.clone(), tasks.clone(), slots.clone(), log_prob.clone()))
            raw.step_all(None)
            record.append(raw._rewards.clone())

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):  # warm-up: modules, cuBLAS, the first call's buffers
        graphed.reset(seed=5)
        loop(graphed, [])
    torch.cuda.current_stream().wait_stream(side)
    graphed.reset(seed=5)
    eager.reset(seed=5)
    torch.cuda.synchronize()
    captured = []
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        loop(graphed, captured)
    want = []
    for replay in range(2):
        graph.replay()
        loop(eager, want)
        torch.cuda.synchronize()
        for i, (got, expected) in enumerate(zip(captured, want[-len(captured):])):
            got = got if isinstance(got, tuple) else (got, )
            expected = expected if isinstance(expected, tuple) else (expected, )
            for a, b in zip(got, expected):
                assert torch.equal(a, b), f'replay {replay} record {i}'
    graphed.check_errors()
    eager.check_errors()
