"""Policy actions on the device (include/frz_policy.h): legality and decoding against ``action_space``, the equal-logit
sampler against ``sample_actions`` bit for bit, the inverse-CDF draw against a float64 restatement on the host Philox
stream, bf16 and strided logits, faults, shards and CUDA-graph capture.  States come from the generators of
tests/test_lifecycle_gpu.py and are stepped by the sampled actions themselves."""
import numpy as np
import pytest
import torch

from free_range_zoo_b200 import presets
from tests import philox_ref as P
from tests.engine_util import cpu
from tests.test_lifecycle_gpu import CYBER_PO, make, setup, wildfire_config
from tests.test_philox_parity_gpu import WILDFIRE_GEOMETRIES

pytestmark = pytest.mark.gpu

BATCHES = [1, 31, 129, 2049]
SEED = 2026


def reference(raw):
    """(legal bool [B, A, C], k int64 [B, A, C], id int64 [B, A, C]) built on the host side of the API: the choices of
    ``action_space(agent)`` (``starts`` / ``counts``) placed on their slots in increasing slot order; k and id are
    defined where legal."""
    B, C = raw.parallel_envs, raw.action_slots
    dev = raw.device
    legal, starts_all = [], []
    for index, agent in enumerate(raw.agents):
        space = raw.action_space(agent)
        counts, starts = space.counts.long(), space.starts.long()
        if raw.metadata['name'] == 'cybersecurity_v0':
            choice = torch.arange(starts.shape[1], device=dev).unsqueeze(0).expand(B, -1)
            nodes = C - 3
            slot = torch.where(starts == 0, choice, nodes - 1 - starts)
            valid = choice < counts.unsqueeze(1)
            mask = torch.zeros((B, C + 1), dtype=torch.bool, device=dev)
            mask.scatter_(1, torch.where(valid, slot, C), True)
            mask = mask[:, :C]
            # the choices' slots increase with the choice index
            ordered = torch.where(valid, slot, C + choice)
            assert bool((ordered[:, 1:] > ordered[:, :-1]).all())
        else:
            if raw.metadata['name'] == 'wildfire_v0':
                cells = C - 1
                if raw.show_bad_actions:
                    tasks = torch.arange(cells, device=dev).unsqueeze(0) < raw.environment_task_count.unsqueeze(1)
                else:
                    tasks = raw.action_mask[:, index] != 0
            else:
                tasks = raw.task_mask[:, index]
            mask = torch.cat([tasks, torch.ones((B, 1), dtype=torch.bool, device=dev)], dim=1)
        assert torch.equal(mask.sum(1), counts), f'{agent}: legal slots != action_space choices'
        legal.append(mask)
        starts_all.append(starts)
    legal = torch.stack(legal, dim=1)
    k = (torch.cumsum(legal.long(), dim=2) - 1).clamp(min=0)
    width = max(s.shape[1] for s in starts_all)
    starts = torch.stack([torch.nn.functional.pad(s, (0, width - s.shape[1]), value=-99) for s in starts_all], dim=1)
    ident = starts.gather(2, k.clamp(max=width - 1))
    return legal, k, ident


def noop_slot(raw):
    return raw.action_slots - (3 if raw.metadata['name'] == 'cybersecurity_v0' else 1)


def check_decoding(raw, ref, rng, every_slot):
    legal, k, ident = ref
    assert torch.equal(raw.legal_actions(), legal)
    out = torch.zeros(legal.shape, dtype=torch.uint8, device=raw.device)
    assert torch.equal(raw.legal_actions(out=out), legal.to(torch.uint8))

    def decode(slots):
        actions = raw.actions_from_slots(slots).clone()
        want_k = k.gather(2, slots.long().unsqueeze(2)).squeeze(2)
        want_id = ident.gather(2, slots.long().unsqueeze(2)).squeeze(2)
        assert torch.equal(actions[..., 0].long(), want_k)
        assert torch.equal(actions[..., 1].long(), want_id)

    scores = torch.from_numpy(rng.random(legal.shape, dtype=np.float32)).to(raw.device)
    decode(scores.masked_fill(~legal, -1.0).argmax(2).to(torch.int32))  # random legal slots
    decode(torch.full(legal.shape[:2], noop_slot(raw), dtype=torch.int32, device=raw.device))
    if every_slot:
        noop = torch.full(legal.shape[:2], noop_slot(raw), dtype=torch.int32, device=raw.device)
        for s in range(raw.action_slots):
            decode(torch.where(legal[..., s], s, noop).to(torch.int32))
    raw.check_errors()


def host_uniforms(raw, step):
    """u [B, A] the uniform sampler draws (tests/philox_ref.py), for the engine's global environment indices."""
    envs = raw.env_offset + np.arange(raw.parallel_envs)
    A = len(raw.agents)
    words = P._calls(SEED, envs, step, np.uint32(0xC0000000) | np.arange(A, dtype=np.uint32))[:, :, 0]
    return P.u01(words).astype(np.float64)


def check_sampling(raw, ref, logits, slots, log_prob, step):
    """The chosen slot is legal and satisfies cum(< i) <= u * S < cum(<= i) in float64 (a neighbour is accepted within
    a 1e-5 relative band); log_prob is the masked log-softmax at the chosen slot."""
    legal = cpu(ref[0])
    x = cpu(logits.float()).astype(np.float64)
    s = cpu(slots).astype(np.int64)
    assert np.take_along_axis(legal, s[..., None], 2).all(), 'an illegal slot was chosen'
    x = np.where(legal, x, -np.inf)
    m = x.max(axis=2, keepdims=True)
    e = np.where(legal, np.exp(x - m), 0.0)
    cum = np.cumsum(e, axis=2)
    S = cum[..., -1]
    target = host_uniforms(raw, step) * S
    below = np.take_along_axis(cum - e, s[..., None], 2)[..., 0]
    upto = np.take_along_axis(cum, s[..., None], 2)[..., 0]
    band = 1e-5 * S
    assert np.all(below <= target + band) and np.all(target < upto + band), 'inverse CDF violated'
    want = (np.take_along_axis(x, s[..., None], 2)[..., 0] - m[..., 0]) - np.log(S)
    assert np.allclose(cpu(log_prob), want, rtol=0, atol=1e-5)
    masked = logits.float().masked_fill(~ref[0], float('-inf'))
    torch_lp = torch.log_softmax(masked, dim=2).gather(2, slots.long().unsqueeze(2)).squeeze(2)
    assert torch.allclose(log_prob, torch_lp, rtol=0, atol=1e-5)


def roll(raw, rng, steps, every_slot=False):
    """Each step: decoding, equal logits vs sample_actions, random logits (f32, bf16, strided, legal_out) checked, then
    the sampled actions step the batch."""
    A, C = len(raw.agents), raw.action_slots
    B = raw.parallel_envs
    legal_out = torch.zeros((B, A, C), dtype=torch.bool, device=raw.device)
    for t in range(steps):
        ref = reference(raw)
        step = raw.control_block()['step']
        check_decoding(raw, ref, rng, every_slot and t < 2)
        uniform = raw.sample_actions(SEED).clone()
        slots, log_prob = raw.sample_actions_from_logits(torch.zeros((B, A, C), device=raw.device), SEED)
        assert torch.equal(raw._actions, uniform), f't={t}: equal logits != sample_actions'
        assert torch.allclose(log_prob, -torch.log(ref[0].sum(2).float()), rtol=1e-6, atol=0)
        wide = torch.from_numpy(rng.normal(0.0, 3.0, (B, A, C + 5)).astype(np.float32)).to(raw.device)
        logits = wide[..., :C]
        bf16 = logits.to(torch.bfloat16)
        slots, log_prob = raw.sample_actions_from_logits(bf16, SEED)
        got = (slots.clone(), log_prob.clone(), raw._actions.clone())
        slots, log_prob = raw.sample_actions_from_logits(bf16.float(), SEED)
        assert torch.equal(slots, got[0]) and torch.equal(log_prob, got[1]) and torch.equal(raw._actions, got[2])
        check_sampling(raw, ref, bf16, got[0], got[1], step)
        slots, log_prob = raw.sample_actions_from_logits(logits, SEED, legal_out=legal_out)
        got = (slots.clone(), log_prob.clone(), raw._actions.clone())
        assert torch.equal(legal_out, ref[0])
        raw.sample_actions_from_logits(logits.contiguous(), SEED)
        assert torch.equal(slots, got[0]) and torch.equal(log_prob, got[1]) and torch.equal(raw._actions, got[2])
        check_sampling(raw, ref, logits, slots, log_prob, step)
        decoded = got[2]
        k, ident = ref[1].gather(2, slots.long().unsqueeze(2))[..., 0], ref[2].gather(2, slots.long().unsqueeze(2))[..., 0]
        assert torch.equal(decoded[..., 0].long(), k) and torch.equal(decoded[..., 1].long(), ident)
        raw.step_all(None)
    raw.check_errors()


# ------------------------------------------------------------------------------------------------ 1-4 over states

WILDFIRE_CASES = [(spec, BATCHES[i % len(BATCHES)], kernel)
                  for i, (spec, _, geometry) in enumerate(WILDFIRE_GEOMETRIES)
                  for kernel in (['groups', 'tiles'] if geometry[0] == 8 else ['auto'])]


@pytest.mark.parametrize('spec,B,kernel', WILDFIRE_CASES, ids=lambda v: str(v).replace(' ', ''))
def test_wildfire(spec, B, kernel):
    rng = np.random.default_rng(B)
    run = setup('wildfire', wildfire_config(spec), B, 6, rng, kernel=kernel,
                kwargs=dict(show_bad_actions=B % 2 == 1 and B > 1), dead=range(0, B, 7), all_lit=range(3, B, 11))
    roll(run.raw, rng, 4, every_slot=B <= 31)


@pytest.mark.parametrize('B', BATCHES)
@pytest.mark.parametrize('show_bad', [False, True])
def test_wildfire_c4(B, show_bad):
    rng = np.random.default_rng(B + show_bad)
    run = setup('wildfire', presets.wildfire_large(), B, 6, rng, kwargs=dict(show_bad_actions=show_bad))
    roll(run.raw, rng, 3, every_slot=B <= 31)


@pytest.mark.parametrize('B', BATCHES)
@pytest.mark.parametrize('kernel', ['groups', 'tiles'])
def test_rideshare(kernel, B):
    rng = np.random.default_rng(B)
    run = setup('rideshare', presets.rideshare_c2(), B, 8, rng, kernel=kernel)
    roll(run.raw, rng, 4, every_slot=B <= 31)


@pytest.mark.parametrize('preset,B,kwargs', [
    ('cyber_c3', 1, CYBER_PO),
    ('cyber_c3', 129, CYBER_PO),
    ('cyber_c3', 2049, dict(show_bad_actions=True, partially_observable=False)),
    (('cyber_synthetic', dict(nodes=20, attackers=9, defenders=9)), 31, dict(show_bad_actions=True)),
    (('cyber_synthetic', dict(nodes=20, attackers=9, defenders=9)), 129, CYBER_PO),
    (('cyber_synthetic', dict(nodes=32, attackers=16, defenders=16)), 31, CYBER_PO),
    (('cyber_synthetic', dict(nodes=32, attackers=16, defenders=16)), 1, dict(show_bad_actions=True)),
])
def test_cybersecurity(preset, B, kwargs):
    config = getattr(presets, preset)() if isinstance(preset, str) else getattr(presets, preset[0])(**preset[1])
    rng = np.random.default_rng(B)
    run = setup('cybersecurity', config, B, 6, rng, kwargs=kwargs, absent=range(0, B, 5))
    raw = run.raw
    location = cpu(raw.state().location)
    assert B < 31 or ((location == -1).any() and cpu(raw._presence).min() == 0), 'home defenders / absent agents'
    roll(raw, rng, 4, every_slot=B <= 31)


@pytest.mark.parametrize('domain,B', [('wildfire', 31), ('wildfire', 2049), ('rideshare', 31), ('rideshare', 2049)])
def test_one_agent(domain, B):
    rng = np.random.default_rng(B)
    if domain == 'wildfire':
        run = setup('wildfire', presets.wildfire_large(height=4, width=5, num_agents=1, seed=32), B, 6, rng)
    else:
        run = setup('rideshare', presets.rideshare_synthetic(drivers=1, rows=16, horizon=10), B, 8, rng)
    assert len(run.raw.agents) == 1
    roll(run.raw, rng, 4, every_slot=B <= 31)


def test_wildfire_c4_at_65536():
    raw = make('wildfire', presets.wildfire_large(), 65536, 20)
    raw.reset(seed=3)
    roll(raw, np.random.default_rng(5), 3)


def test_every_passenger_state_is_decoded():
    """The generated tables hold unaccepted, accepted and riding passengers in drivers' task lists."""
    rng = np.random.default_rng(9)
    raw = setup('rideshare', presets.rideshare_c2(), 129, 8, rng).raw
    ref = reference(raw)
    seen = set(cpu(ref[2][ref[0]]).tolist())
    assert {0, 1, 2, -1} <= seen, seen
    check_decoding(raw, ref, rng, True)


@pytest.mark.parametrize('domain,config,kwargs', [
    ('wildfire', presets.wildfire_large, dict(show_bad_actions=False)),
    ('wildfire', presets.wildfire_3x3, dict(show_bad_actions=True)),
    ('rideshare', presets.rideshare_c2, {}),
    ('cybersecurity', presets.cyber_c3, CYBER_PO),
    ('cybersecurity', presets.cyber_c3, dict(show_bad_actions=True))])
def test_equal_logits_stage_what_the_uniform_sampler_stages_over_12_steps(domain, config, kwargs):
    uniform = make(domain, config(), 129, 8, **kwargs)
    policy = make(domain, config(), 129, 8, **kwargs)
    uniform.reset(seed=11)
    policy.reset(seed=11)
    zeros = torch.zeros((129, len(policy.agents), policy.action_slots), device='cuda', dtype=torch.bfloat16)
    for t in range(12):
        uniform.sample_actions(SEED)
        _, log_prob = policy.sample_actions_from_logits(zeros, SEED)
        assert torch.equal(policy._actions, uniform._actions), t
        assert torch.allclose(log_prob, -torch.log(policy.legal_actions().sum(2).float()), rtol=1e-6, atol=0), t
        uniform.step_all(None)
        policy.step_all(None)
    assert torch.equal(policy._rewards, uniform._rewards)


# ------------------------------------------------------------------------------------------------ 3. distribution

def test_chi_square_of_fixed_logits():
    from scipy import stats
    B = 1 << 18  # x 4 agents = 2^20 draws
    raw = make('cybersecurity', presets.cyber_c3(), B, 10, show_bad_actions=True, partially_observable=False)
    raw.reset(seed=1)
    C = raw.action_slots
    row = torch.tensor([0.5, -1.0, 1.5, 0.0, -0.5, 2.0], device=raw.device)[:C]
    logits = row.expand(B, len(raw.agents), C).contiguous()
    legal = raw.legal_actions().clone()
    slots, _ = raw.sample_actions_from_logits(logits, SEED)
    slots, legal = cpu(slots), cpu(legal)
    for a in range(len(raw.agents)):
        mask = legal[0, a]
        assert (legal[:, a] == mask).all()
        p = np.where(mask, np.exp(cpu(row).astype(np.float64)), 0.0)
        p /= p.sum()
        counts = np.bincount(slots[:, a], minlength=C)
        assert counts[~mask].sum() == 0
        _, pvalue = stats.chisquare(counts[mask], p[mask] * B)
        assert pvalue > 1e-3, (a, counts, p * B, pvalue)


@pytest.mark.parametrize('value', [1e30, float('inf'), float('nan')])
def test_illegal_slots_are_never_chosen(value):
    rng = np.random.default_rng(1)
    raw = setup('wildfire', presets.wildfire_large(), 2049, 6, rng).raw
    legal = raw.legal_actions().clone()
    logits = torch.randn(legal.shape, device=raw.device).masked_fill(~legal, value)
    slots, log_prob = raw.sample_actions_from_logits(logits, SEED)
    assert bool(legal.gather(2, slots.long().unsqueeze(2)).all())
    assert bool(torch.isfinite(log_prob).all())
    raw.check_errors()


# ------------------------------------------------------------------------------------------------ 5. faults

@pytest.mark.parametrize('domain,config', [('wildfire', presets.wildfire_large), ('rideshare', presets.rideshare_c2),
                                           ('cybersecurity', presets.cyber_c3)])
def test_faults_stage_the_noop_and_are_raised(domain, config):
    rng = np.random.default_rng(2)
    kwargs = dict(kwargs=CYBER_PO) if domain == 'cybersecurity' else {}
    raw = setup(domain, config(), 129, 6, rng, **kwargs).raw
    legal, k, ident = reference(raw)
    noop = noop_slot(raw)
    noop_action = torch.stack([k[..., noop], ident[..., noop]], dim=2).to(torch.int32)
    B, A, C = legal.shape
    first_legal = legal.float().argmax(2)  # a legal slot of every row
    for name, poison in (('nan', float('nan')), ('inf', float('inf'))):
        logits = torch.zeros((B, A, C), device=raw.device)
        logits[5, 0, first_legal[5, 0]] = poison
        slots, log_prob = raw.sample_actions_from_logits(logits, SEED)
        assert int(slots[5, 0]) == noop and bool(torch.isnan(log_prob[5, 0])), name
        assert torch.equal(raw._actions[5, 0], noop_action[5, 0]), name
        assert raw.control_block()['error_word'] == 0x10, name
        with pytest.raises(ValueError, match='logits'):
            raw.check_errors()
    logits = torch.zeros((B, A, C), device=raw.device)
    logits[7, A - 1] = float('-inf')
    slots, _ = raw.sample_actions_from_logits(logits, SEED)
    assert int(slots[7, A - 1]) == noop and torch.equal(raw._actions[7, A - 1], noop_action[7, A - 1])
    with pytest.raises(ValueError, match='logits'):
        raw.check_errors()
    illegal = (~legal).float().argmax(2)  # an illegal slot where the row has one
    has_illegal = (~legal).any(2)
    b, a = [int(v) for v in torch.nonzero(has_illegal)[0]]
    for bad in (C, -1, int(illegal[b, a])):
        slots = torch.full((B, A), noop, dtype=torch.int32, device=raw.device)
        slots[b, a] = bad
        actions = raw.actions_from_slots(slots)
        assert torch.equal(actions, noop_action), bad
        assert raw.control_block()['error_word'] == 0x20, bad
        with pytest.raises(ValueError, match='slot'):
            raw.check_errors()


# ------------------------------------------------------------------------------------------------ 6. shards

def test_a_shard_samples_its_slice_of_the_whole_batch():
    B, half = 258, 129
    whole = make('wildfire', presets.wildfire_large(), B, 10)
    shard = make('wildfire', presets.wildfire_large(), half, 10, env_offset=half)
    whole.reset(seed=4)
    shard.reset(seed=4)
    rng = np.random.default_rng(4)
    for t in range(3):
        logits = torch.from_numpy(rng.normal(0, 2, (B, 10, whole.action_slots)).astype(np.float32)).cuda()
        s_whole, lp_whole = whole.sample_actions_from_logits(logits, SEED)
        s_shard, lp_shard = shard.sample_actions_from_logits(logits[half:].contiguous(), SEED)
        assert torch.equal(s_whole[half:], s_shard), t
        assert torch.equal(lp_whole[half:], lp_shard), t
        assert torch.equal(whole._actions[half:], shard._actions), t
        whole.step_all(None)
        shard.step_all(None)


# ------------------------------------------------------------------------------------------------ 7. graph capture

@pytest.mark.parametrize('autoreset', [False, True])
@pytest.mark.parametrize('domain,config', [('wildfire', presets.wildfire_large), ('rideshare', presets.rideshare_c2),
                                           ('cybersecurity', presets.cyber_c3)])
def test_graph_capture_replays_equal_to_eager(domain, config, autoreset):
    B, max_steps = 1000, 4
    eager = make(domain, config(), B, max_steps, autoreset=autoreset)
    graphed = make(domain, config(), B, max_steps, autoreset=autoreset)
    logits = torch.zeros((B, len(eager.agents), eager.action_slots), device='cuda')
    # warm-up outside capture (module loading, the first call's buffers), then start both from the same reset
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        graphed.reset(seed=5)
        graphed.sample_actions_from_logits(logits, SEED)
        graphed.step_all(None)
    torch.cuda.current_stream().wait_stream(side)
    graphed.reset(seed=5)
    eager.reset(seed=5)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        graphed.sample_actions_from_logits(logits, SEED)
        graphed.step_all(None)
    rng = np.random.default_rng(6)
    for t in range(10):
        logits.copy_(torch.from_numpy(rng.normal(0, 2, tuple(logits.shape)).astype(np.float32)))
        graph.replay()
        slots, log_prob = eager.sample_actions_from_logits(logits, SEED)
        eager.step_all(None)
        assert torch.equal(graphed._policy['slots'], slots), t
        assert torch.equal(graphed._policy['log_prob'], log_prob), t
        for name, tensor in eager._bound.items():
            if tensor is not None:
                assert torch.equal(graphed._bound[name], tensor), f't={t} {name}'
        if autoreset:
            assert torch.equal(graphed._autoreset_flags, eager._autoreset_flags), t
    graphed.check_errors()
    eager.check_errors()


def test_the_parallel_wrapper_forwards_policy_actions():
    from free_range_zoo_b200.envs import rideshare_v0
    env = rideshare_v0.parallel_env(parallel_envs=64, max_steps=10, configuration=presets.rideshare_c2(),
                                    device=torch.device('cuda'))
    twin = make('rideshare', presets.rideshare_c2(), 64, 10)
    env.reset(seed=3)
    twin.reset(seed=3)
    assert env.action_slots == twin.action_slots == 33
    rng = np.random.default_rng(3)
    for t in range(3):
        logits = torch.from_numpy(rng.normal(0, 2, (64, len(twin.agents), 33)).astype(np.float32)).cuda()
        assert torch.equal(env.legal_actions(), twin.legal_actions()), t
        slots, log_prob = env.sample_actions_from_logits(logits, SEED)
        twin_slots, twin_log_prob = twin.sample_actions_from_logits(logits, SEED)
        assert torch.equal(slots, twin_slots) and torch.equal(log_prob, twin_log_prob), t
        _, rewards, _, _, _ = env.step(None)
        twin.step_all(None)
        for index, agent in enumerate(twin.agents):
            assert torch.equal(rewards[agent], twin._rewards[:, index]), t
    slots, _ = env.sample_actions_from_logits(logits, SEED)  # legal in the current state
    host_slots = slots.cpu()  # a CPU policy's choices
    assert torch.equal(env.actions_from_slots(host_slots), twin.actions_from_slots(host_slots.cuda()))
    env.check_errors()
