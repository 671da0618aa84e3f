"""GAE advantages on the device (``utils.returns.advantages``, include/frz_returns.h): against a float64 restatement of
the recurrence, bit-for-bit independent of the batch, against the engine's own episode statistics, inside a captured
rollout, and with offsets past 2^31; and ``reward_table``."""
import importlib

import numpy as np
import pytest
import torch

from free_range_zoo_b200 import presets
from free_range_zoo_b200.utils.returns import advantages
from tests.engine_util import cpu
from tests.test_lifecycle_gpu import CYBER_PO, cyber_state, given, make, rideshare_state, wildfire_state
from tests.test_policy_inputs_gpu import Policy

pytestmark = pytest.mark.gpu

EPS = 2.0**-23


def restate(r, v, term, trunc, next_v, final_v, gamma, lam):
    """The recurrence of include/frz_returns.h in float64 on host arrays: (A, S) with S the same recurrence on |delta|
    (the scale of the rounding error)."""
    r, v, next_v = (np.asarray(x, np.float64) for x in (r, v, next_v))
    term, trunc = np.asarray(term).astype(bool)[..., None], np.asarray(trunc).astype(bool)[..., None]
    gamma, lam = float(np.float32(gamma)), float(np.float32(lam))
    following = np.concatenate([v[1:], next_v[None]], axis=0)
    final = 0.0 if final_v is None else np.asarray(final_v, np.float64)
    nv = np.where(term, 0.0, np.where(trunc, final, following))
    delta = (r + gamma * nv) - v
    c = gamma * lam * (1.0 - (term | trunc))
    A, S = np.zeros_like(r), np.zeros_like(r)
    a = s = 0.0
    for t in range(r.shape[0] - 1, -1, -1):
        a = delta[t] + c[t] * a
        s = np.abs(delta[t]) + c[t] * s
        A[t], S[t] = a, s
    return A, S


def assert_close(got, want, S, context):
    T = want.shape[0]
    bound = (T - np.arange(T) + 2).reshape((T, ) + (1, ) * (want.ndim - 1)) * EPS * (1.0 + S)
    err = np.abs(np.asarray(got, np.float64) - want)
    assert np.all(err <= bound), f'{context}: max excess {np.max(err - bound)} at {np.unravel_index(np.argmax(err - bound), err.shape)}'


def synthetic(T, B, A, density, dtype, final, seed):
    gen = torch.Generator(device='cuda').manual_seed(seed)
    uniform = lambda *shape: torch.rand(shape, generator=gen, device='cuda') * 2 - 1  # noqa: E731
    flags = lambda: torch.rand((T, B), generator=gen, device='cuda') < density  # noqa: E731
    term, trunc = flags(), flags().to(torch.uint8)
    return dict(rewards=uniform(T, B, A), values=uniform(T, B, A).to(dtype), terminated=term, truncated=trunc,
                next_values=uniform(B, A).to(dtype), final_values=uniform(T, B, A).to(dtype) if final else None)


def host(x):
    return None if x is None else cpu(x.float() if x.dtype == torch.bfloat16 else x)


def check_against_restatement(inputs, gamma, lam, with_returns, context):
    T, B, A = inputs['rewards'].shape
    out = (torch.full((T, B, A), np.nan, device='cuda'), torch.full((T, B, A), np.nan, device='cuda') if with_returns else None)
    got, returns = advantages(**inputs, gamma=gamma, lam=lam, out=out)
    assert got.data_ptr() == out[0].data_ptr()
    want, S = restate(*(host(inputs[k]) for k in ('rewards', 'values', 'terminated', 'truncated', 'next_values',
                                                  'final_values')), gamma, lam)
    assert_close(cpu(got), want, S, context)
    if with_returns:
        # R = A + v, one f32 add on top of A
        v = host(inputs['values']).astype(np.float64)
        assert_close(cpu(returns), want + v, S + np.abs(want + v), f'{context} returns')
    else:
        assert returns is None


# ------------------------------------------------------------------------------------------------ restatement sweep

DISCOUNTS = [(0.99, 0.95), (1.0, 1.0), (0.0, 0.0), (0.5, 1.0)]
SHAPES = [(1, 1), (31, 3), (129, 10), (2049, 1), (65536, 10)]
SWEEP = [(T, B, A) for T in (1, 2, 15, 16, 17, 128, 1000, 4096) for B, A in SHAPES if B * A < 65536 or T <= 128]


@pytest.mark.parametrize('T,B,A', SWEEP)
def test_matches_the_float64_restatement(T, B, A):
    case = 0
    for density in (0.0, 0.05, 0.5, 1.0):
        for dtype in (torch.float32, torch.bfloat16):
            final = case % 2 == 0
            gamma, lam = DISCOUNTS[(case // 2 + T) % len(DISCOUNTS)]
            with_returns = (case // 3) % 2 == 0
            inputs = synthetic(T, B, A, density, dtype, final, seed=T * 7919 + B * 31 + A + case)
            context = f'T={T} B={B} A={A} density={density} {dtype} final={final} gamma={gamma} lam={lam}'
            check_against_restatement(inputs, gamma, lam, with_returns, context)
            case += 1


def test_every_discount_value_type_and_final_option_at_one_shape():
    for gamma, lam in DISCOUNTS:
        for dtype in (torch.float32, torch.bfloat16):
            for final in (False, True):
                for with_returns in (False, True):
                    inputs = synthetic(40, 31, 3, 0.2, dtype, final, seed=5)
                    check_against_restatement(inputs, gamma, lam, with_returns, f'{gamma} {lam} {dtype} {final}')


def test_both_flags_on_one_step_bootstrap_from_zero():
    T, B, A = 3, 2, 2
    inputs = dict(rewards=torch.ones((T, B, A), device='cuda'), values=torch.zeros((T, B, A), device='cuda'),
                  terminated=torch.ones((T, B), dtype=torch.bool, device='cuda'),
                  truncated=torch.ones((T, B), dtype=torch.bool, device='cuda'),
                  next_values=torch.full((B, A), 100.0, device='cuda'),
                  final_values=torch.full((T, B, A), 100.0, device='cuda'))
    got, returns = advantages(**inputs, gamma=1.0, lam=1.0)
    assert torch.equal(got, torch.ones_like(got)) and torch.equal(returns, got)
    inputs['terminated'].zero_()  # truncation alone: bootstrap from the final values, without them from 0
    assert torch.equal(advantages(**inputs, gamma=0.5, lam=1.0)[0], torch.full_like(got, 51.0))
    inputs['final_values'] = None
    assert torch.equal(advantages(**inputs, gamma=0.5, lam=1.0)[0], torch.ones_like(got))


# ------------------------------------------------------------------------------------------------ invariance


def columnwise(x):
    """[T, B, A] -> [B, A, T], contiguous: the steps of a column adjacent."""
    return x.permute(1, 2, 0).contiguous()


@pytest.mark.parametrize('T,dtype', [(37, torch.float32), (600, torch.bfloat16)])
def test_a_column_alone_gives_the_same_bits_as_in_a_batch(T, dtype):
    B, A = 4099, 7
    inputs = synthetic(T, B, A, 0.05, dtype, True, seed=T)
    batch = advantages(**inputs, gamma=0.99, lam=0.95)
    again = advantages(**inputs, gamma=0.99, lam=0.95)
    assert torch.equal(batch[0], again[0]) and torch.equal(batch[1], again[1])
    r, v, fv = (columnwise(inputs[k]) for k in ('rewards', 'values', 'final_values'))
    term, trunc = inputs['terminated'].t().contiguous(), inputs['truncated'].t().contiguous()
    nv = inputs['next_values']
    alone = [torch.empty((B, A, T), device='cuda') for _ in range(2)]
    for b in range(B):
        for a in range(A):
            advantages(r[b, a].view(T, 1, 1), v[b, a].view(T, 1, 1), term[b].view(T, 1), trunc[b].view(T, 1),
                       nv[b, a].view(1, 1), fv[b, a].view(T, 1, 1), gamma=0.99, lam=0.95,
                       out=(alone[0][b, a].view(T, 1, 1), alone[1][b, a].view(T, 1, 1)))
    assert torch.equal(alone[0].permute(2, 0, 1), batch[0])
    assert torch.equal(alone[1].permute(2, 0, 1), batch[1])


# ------------------------------------------------------------------------------------------------ the engine


def engine(domain, B, max_steps, kernel='auto'):
    """An autoreset engine keeping final observations, reset into a generated state whose environments finish at
    different steps (wildfire: some with nothing lit, some fully lit; cybersecurity: some with nobody present)."""
    rng = np.random.default_rng(B + 3)
    kwargs = dict(autoreset=True, keep_final_observations=True)
    if domain == 'wildfire':
        from oracle.wildfire import WildfireOracle
        config = presets.wildfire_large()
        state = wildfire_state(WildfireOracle(config, B, max_steps), rng, dead=range(0, B, 7), all_lit=range(3, B, 11))
        raw = make(domain, config, B, max_steps, step_kernel=kernel, **kwargs)
    elif domain == 'rideshare':
        from oracle.rideshare import RideshareOracle
        config = presets.rideshare_c2()
        agents, passengers = rideshare_state(RideshareOracle(config, B, max_steps), config, rng, 3 * max_steps + 10)
        state = dict(agents=agents, passengers=passengers)
        raw = make(domain, config, B, max_steps, step_kernel=kernel, **kwargs)
    else:
        from oracle.cybersecurity import CybersecurityOracle
        config = presets.cyber_c3()
        state = cyber_state(CybersecurityOracle(config, B, max_steps, **CYBER_PO), rng, absent=range(0, B, 5))
        raw = make(domain, config, B, max_steps, **CYBER_PO, **kwargs)
    raw.reset(seed=11, options={'initial_state': given(**state)})
    return raw


def value_of(agent, tasks):
    """A fixed function of the policy inputs: f32 [B, A]."""
    task_sum = tasks.float().sum(dim=(2, 3))  # [B, V], V = 1 or A
    return (0.1 * agent.float().sum(dim=2) + 0.01 * task_sum).contiguous()


def record(raw, T, seed=100):
    """T steps of sampled actions with everything ``advantages`` reads, the episode statistics and the done flags."""
    B, A = raw.parallel_envs, len(raw.possible_agents)
    rec = dict(rewards=torch.zeros((T, B, A), device='cuda'), values=torch.zeros((T, B, A), device='cuda'),
               terminated=torch.zeros((T, B), dtype=torch.bool, device='cuda'),
               truncated=torch.zeros((T, B), dtype=torch.bool, device='cuda'),
               final_values=torch.zeros((T, B, A), device='cuda'))
    returns = torch.zeros((T, B, A), device='cuda')
    for t in range(T):
        rec['values'][t].copy_(value_of(*raw.policy_inputs()))
        raw.sample_actions(seed + t)
        raw.step_all(None)
        rec['rewards'][t].copy_(raw.reward_table)
        rec['terminated'][t].copy_(raw.terminated)
        rec['truncated'][t].copy_(raw.truncated)
        rec['final_values'][t].copy_(value_of(*raw.policy_inputs(final=True)))
        returns[t].copy_(raw.episode_statistics['return'])
    rec['next_values'] = value_of(*raw.policy_inputs())
    raw.check_errors()
    return rec, returns


def check_episode_returns(raw, T, from_reset, context):
    rec, episode_return = record(raw, T)
    zeros = torch.zeros_like(rec['values'])
    got, _ = advantages(rec['rewards'], zeros, rec['terminated'], rec['truncated'], torch.zeros_like(rec['next_values']),
                        zeros, gamma=1.0, lam=1.0)
    got, r, ret = cpu(got), cpu(rec['rewards']), cpu(episode_return)
    done = cpu(rec['terminated']) | cpu(rec['truncated'])
    B = done.shape[1]
    start = np.full(B, 0 if from_reset else -1)  # the step the current episode started at, -1 before the window
    checked = 0
    for t in range(T):
        for b in np.nonzero(done[t] & (start >= 0))[0]:
            s = start[b]
            scale = np.maximum(np.abs(ret[t, b]), np.abs(r[s:t + 1, b]).sum(axis=0))
            assert np.all(np.abs(got[s, b] - ret[t, b]) <= 1e-5 * scale), f'{context}: env {b} steps {s}..{t}'
            checked += 1
        start[done[t]] = t + 1
    assert checked > 0, context
    # values from the policy inputs, final values from the final observations: the kernel on the recorded tensors
    for dtype in (torch.float32, torch.bfloat16):
        inputs = dict(rec, values=rec['values'].to(dtype), next_values=rec['next_values'].to(dtype),
                      final_values=rec['final_values'].to(dtype))
        check_against_restatement(inputs, 0.99, 0.95, True, f'{context} {dtype}')
    return checked


@pytest.mark.parametrize('domain,kernel', [('wildfire', 'auto'), ('rideshare', 'groups'), ('rideshare', 'tiles'),
                                           ('cybersecurity', 'auto')])
def test_episode_returns_and_bootstraps_match_the_engine(domain, kernel):
    max_steps = 5
    T = 3 * max_steps + 2  # two segments
    raw = engine(domain, 67, max_steps, kernel)
    check_episode_returns(raw, T, True, f'{domain} {kernel} from reset')
    # staggered horizons: a third of the environments start over mid-episode, then a window that begins mid-episode
    raw = engine(domain, 67, max_steps, kernel)
    for t in range(3):
        if t == 1:
            raw.reset_batches(list(range(0, 67, 3)))
        raw.sample_actions(50 + t)
        raw.step_all(None)
    check_episode_returns(raw, T, False, f'{domain} {kernel} staggered')


# ------------------------------------------------------------------------------------------------ graph capture


@pytest.mark.parametrize('domain,config', [('wildfire', presets.wildfire_large), ('rideshare', presets.rideshare_c2),
                                           ('cybersecurity', presets.cyber_c3)])
def test_a_captured_rollout_with_advantages_replays_equal_to_eager(domain, config):
    B, T = 1000, 20
    kwargs = dict(autoreset=True, keep_final_observations=True)
    eager, graphed = make(domain, config(), B, 4, **kwargs), make(domain, config(), B, 4, **kwargs)
    policy = Policy(eager)
    shapes = eager.policy_input_shapes
    A = shapes['agent'][0]

    def storage():
        return dict(agent=torch.zeros((T, B) + shapes['agent'], device='cuda'),
                    tasks=torch.zeros((T, B) + shapes['tasks'], device='cuda'),
                    values=torch.zeros((T, B, A), device='cuda'), log_prob=torch.zeros((T, B, A), device='cuda'),
                    rewards=torch.zeros((T, B, A), device='cuda'),
                    terminated=torch.zeros((T, B), dtype=torch.bool, device='cuda'),
                    truncated=torch.zeros((T, B), dtype=torch.bool, device='cuda'),
                    final_values=torch.zeros((T, B, A), device='cuda'), next_values=torch.zeros((B, A), device='cuda'),
                    advantages=torch.zeros((T, B, A), device='cuda'), returns=torch.zeros((T, B, A), device='cuda'))

    def loop(raw, s):
        for t in range(T):
            agent, tasks = raw.policy_inputs(out=(s['agent'][t], s['tasks'][t]))
            s['values'][t].copy_(value_of(agent, tasks))
            _, log_prob = raw.sample_actions_from_logits(policy(agent, tasks), 2026)
            s['log_prob'][t].copy_(log_prob)
            raw.step_all(None)
            s['rewards'][t].copy_(raw.reward_table)
            s['terminated'][t].copy_(raw.terminated)
            s['truncated'][t].copy_(raw.truncated)
            s['final_values'][t].copy_(value_of(*raw.policy_inputs(final=True)))
        s['next_values'].copy_(value_of(*raw.policy_inputs()))
        advantages(s['rewards'], s['values'], s['terminated'], s['truncated'], s['next_values'], s['final_values'],
                   gamma=0.99, lam=0.95, out=(s['advantages'], s['returns']))

    captured, want = storage(), storage()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):  # warm-up: modules, cuBLAS, the first calls' buffers
        graphed.reset(seed=5)
        loop(graphed, storage())
    torch.cuda.current_stream().wait_stream(side)
    graphed.reset(seed=5)
    eager.reset(seed=5)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        loop(graphed, captured)
    finished = 0
    for replay in range(2):
        graph.replay()
        loop(eager, want)
        torch.cuda.synchronize()
        for name in want:
            assert torch.equal(captured[name], want[name]), f'replay {replay}: {name}'
        finished += int((want['terminated'] | want['truncated']).sum())
    assert finished > 0
    graphed.check_errors()
    eager.check_errors()


# ------------------------------------------------------------------------------------------------ 64-bit offsets


def test_offsets_past_two_to_the_31():
    T, B, A = 2048, 32769, 32
    assert T * B * A > 2**31
    inputs = synthetic(T, B, A, 0.01, torch.bfloat16, True, seed=64)
    got, _ = advantages(**inputs, gamma=0.99, lam=0.95, out=(torch.empty((T, B, A), device='cuda'), None))
    C = B * A
    first_high = 2**31 - (T - 1) * C  # the first column whose last step lies past 2^31 elements
    rng = np.random.default_rng(0)
    columns = np.unique(np.concatenate([rng.integers(first_high, C, 62), [first_high, C - 1]]))
    index = torch.as_tensor(columns, device='cuda')
    envs = torch.as_tensor(columns // A, device='cuda')
    # the picked columns restated as a batch of len(columns) one-agent environments: values [T, n, 1], flags [T, n]
    pick = lambda x: x.reshape(T, C)[:, index, None]  # noqa: E731
    want, S = restate(host(pick(inputs['rewards'])), host(pick(inputs['values'])), cpu(inputs['terminated'][:, envs]),
                      cpu(inputs['truncated'][:, envs]), host(inputs['next_values'].reshape(C)[index, None]),
                      host(pick(inputs['final_values'])), 0.99, 0.95)
    assert_close(cpu(pick(got)), want, S, 'offsets past 2^31')


# ------------------------------------------------------------------------------------------------ reward_table


@pytest.mark.parametrize('domain,preset,kwargs', [('wildfire', 'wildfire_large', {}), ('rideshare', 'rideshare_c2', {}),
                                                  ('cybersecurity', 'cyber_c3', CYBER_PO)])
def test_reward_table_is_the_stable_buffer_the_rewards_view(domain, preset, kwargs):
    module = importlib.import_module(f'free_range_zoo_b200.envs.{domain}_v0')
    env = module.parallel_env(parallel_envs=257, max_steps=6, configuration=getattr(presets, preset)(),
                              device=torch.device('cuda'), **kwargs)
    env.reset(seed=4)
    raw = env.unwrapped
    table = env.reward_table
    assert table is raw.reward_table and table.dtype == torch.float32 and tuple(table.shape) == (257, len(env.agents))
    nonzero = False
    for t in range(8):
        raw.sample_actions(t)
        _, rewards, _, _, _ = env.step(raw._actions.clone())
        assert env.reward_table.data_ptr() == table.data_ptr()
        assert torch.equal(env.reward_table, torch.stack([rewards[a] for a in env.agents], -1)), f'{domain} t={t}'
        nonzero |= bool(env.reward_table.any())
    assert nonzero, domain
