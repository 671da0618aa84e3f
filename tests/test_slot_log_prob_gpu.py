"""Masked slot log-probabilities, entropies and their gradient on the device (include/frz_logprob.h): a float64
restatement of the contract over every row mapping, bit-for-bit agreement with the sampler in every domain, the packed
legal masks of include/frz_policy.h, per-row invariance, edge rows, CUDA-graph capture and offsets past 2^31."""
import math

import numpy as np
import pytest
import torch

from free_range_zoo_b200 import _lib, presets
from free_range_zoo_b200.utils.policy import legal_words, slot_log_prob, unpack_legal
from tests.test_lifecycle_gpu import CYBER_PO, setup, wildfire_config
from tests.test_philox_parity_gpu import WILDFIRE_GEOMETRIES
from tests.test_slot_log_prob import pack_legal

pytestmark = pytest.mark.gpu

SEED = 2026
U = 2.0 ** -24  # unit roundoff of f32
# every (G, PER) row mapping of frz_slots.cuh and its edges: (1, 16) C <= 16, (8, 4) <= 32, (16, 4) <= 64,
# (32, 4) <= 128, (32, 9) <= 288
SLOT_COUNTS = [2, 6, 10, 16, 17, 32, 33, 64, 65, 101, 128, 129, 257, 288]
DENSITIES = [0.0, 0.1, 0.5, 0.9, 1.0]  # 0: only the noop (the last slot) is legal; 1: every slot


def random_mask(lead, C, density, generator):
    mask = torch.rand(lead + (C, ), generator=generator, device='cuda') < density
    mask[..., -1] = True  # the noop
    return mask


def as_mask(mask, kind):
    return {'bool': mask, 'uint8': mask.to(torch.uint8), 'packed': pack_legal(mask)}[kind]


def reference(logits, slots, legal, g_lp, g_h):
    """The contract of include/frz_logprob.h in float64 (on the host), from the logits' own values."""
    x = logits.double().cpu().numpy()
    legal = legal.cpu().numpy()
    s = slots.long().cpu().numpy()
    C = x.shape[-1]
    with np.errstate(invalid='ignore', divide='ignore', over='ignore'):
        lx = np.where(legal, x, -np.inf)
        bad = (np.where(legal, np.isnan(x) | (x == np.inf), False)).any(-1)
        m = lx.max(-1, keepdims=True)
        bad |= m[..., 0] == -np.inf
        e = np.where(legal, np.exp(lx - m), 0.0)
        S = e.sum(-1, keepdims=True)
        log_S = np.log(S)
        d = np.where(e > 0, lx - m, 0.0)
        H = log_S[..., 0] - (e * d).sum(-1) / S[..., 0]
        in_range = (s >= 0) & (s < C)
        chosen_legal = in_range & np.take_along_axis(legal, np.clip(s, 0, C - 1)[..., None], -1)[..., 0]
        l_s = np.take_along_axis(lx, np.clip(s, 0, C - 1)[..., None], -1)[..., 0]
        lp = np.where(chosen_legal, (l_s - m[..., 0]) - log_S[..., 0], -np.inf)
        p = e / S
        ind = (np.arange(C) == s[..., None]) & chosen_legal[..., None]
        a = g_lp[..., None] * (ind - p)
        b = np.where(p > 0, g_h[..., None] * p * ((lx - m - log_S) + H[..., None]), 0.0)
        g = np.where(legal, a - b, 0.0)
        lp = np.where(bad, np.nan, lp)
        H = np.where(bad, np.nan, H)
        g = np.where(legal & bad[..., None], np.nan, g)
        n = legal.sum(-1)
        # error bounds from f32 rounding: n-term sums (relative n u), expf / logf / division (a few u each)
        tol_lp = 4 * U * (np.abs(np.where(chosen_legal, l_s - m[..., 0], 0)) + np.abs(log_S[..., 0]) + n + 4)
        spread = (e * np.abs(d)).sum(-1) / S[..., 0]
        tol_h = 8 * U * (n + 4) * (1 + np.abs(log_S[..., 0]) + spread)
        size = 1 + np.abs(d) + np.abs(log_S) + np.abs(H)[..., None]
        tol_g = 8 * U * (n[..., None] + 8) * (np.abs(g_lp)[..., None] * (ind + p) + np.abs(g_h)[..., None] * p * size)
        tol_g += 1e-37 * (np.abs(g_lp)[..., None] + np.abs(g_h)[..., None] * size)  # denormal exp terms
    return lp, H, g, tol_lp, tol_h, tol_g


def assert_within(got, want, tol, what):
    got = got.double().cpu().numpy() if isinstance(got, torch.Tensor) else got
    both_nan = np.isnan(got) & np.isnan(want)
    same_inf = np.isinf(want) & (got == want)
    with np.errstate(invalid='ignore'):
        close = np.abs(got - want) <= tol
    ok = both_nan | same_inf | close
    assert ok.all(), f'{what}: {int((~ok).sum())} of {ok.size} outside the bound, e.g. got ' \
                     f'{got[~ok][:4]} want {want[~ok][:4]} tol {np.broadcast_to(tol, want.shape)[~ok][:4]}'


def run(logits, slots, legal, g_lp, g_h, entropy=True):
    x = logits.detach().requires_grad_(True)
    lp, h = slot_log_prob(x, slots, legal, entropy=entropy)
    terms = []
    if g_lp is not None:
        terms.append((lp * g_lp).sum())
    if g_h is not None and entropy:
        terms.append((h * g_h).sum())
    grad = None
    if terms:
        sum(terms).backward()
        grad = x.grad
    return lp.detach(), None if h is None else h.detach(), grad


# ------------------------------------------------------------------------------------------------ 1. float64 reference

@pytest.mark.parametrize('C', SLOT_COUNTS)
@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16], ids=['f32', 'bf16'])
def test_against_a_float64_restatement(C, dtype):
    generator = torch.Generator(device='cuda').manual_seed(C)
    lead = (3, 7, 5)  # [T, B, A]
    for density in DENSITIES:
        legal = random_mask(lead, C, density, generator)
        wide = torch.randn(lead + (C + 3, ), generator=generator, device='cuda') * 3.0
        logits = wide.to(dtype)[..., :C]  # row_stride = C + 3
        choose = torch.rand(lead + (C, ), generator=generator, device='cuda').masked_fill(~legal, -1.0)
        slots = choose.argmax(-1).to(torch.int32)
        slots[0, 0] = C - 1
        slots[1, 1, :2] = torch.tensor([-1, C], dtype=torch.int32)  # outside [0, C)
        g_lp = torch.randn(lead, generator=generator, device='cuda')
        g_h = torch.randn(lead, generator=generator, device='cuda')
        for kind in ('bool', 'uint8', 'packed'):
            for glp, gh in ((g_lp, g_h), (g_lp, None), (None, g_h)):
                lp, h, grad = run(logits, slots, as_mask(legal, kind), glp, gh)
                zeros = np.zeros(lead)
                want = reference(logits, slots, legal, zeros if glp is None else glp.cpu().numpy(),
                                 zeros if gh is None else gh.cpu().numpy())
                what = f'C={C} {dtype} density={density} {kind} g_lp={glp is not None} g_H={gh is not None}'
                assert_within(lp, want[0], want[3], 'log_prob ' + what)
                assert_within(h, want[1], want[4], 'entropy ' + what)
                assert grad.dtype == dtype and grad.is_contiguous() and grad.shape == logits.shape
                tol = want[5] + (np.abs(want[2]) * 2.0 ** -8 if dtype == torch.bfloat16 else 0)  # bf16: one rounding
                assert_within(grad, want[2], tol, 'gradient ' + what)
                assert bool((grad.float()[~legal] == 0).all()), 'illegal slots get exactly 0'


def test_empty_leading_shapes_return_empty_outputs():
    logits = torch.zeros((0, 4, 33), device='cuda', requires_grad=True)
    lp, h = slot_log_prob(logits, torch.zeros((0, 4), dtype=torch.int32, device='cuda'),
                          torch.zeros((0, 4, 2), dtype=torch.int32, device='cuda'))
    assert lp.shape == h.shape == (0, 4)
    (lp.sum() + h.sum()).backward()
    assert logits.grad.shape == (0, 4, 33)


# ------------------------------------------------------------------------------------------------ 2-3. the sampler

def sampler_cases():
    cases = [('wildfire', wildfire_config(spec), 31, dict(show_bad_actions=i % 2 == 1))
             for i, (spec, _, _) in enumerate(WILDFIRE_GEOMETRIES)]
    cases += [('wildfire', presets.wildfire_large(), 129, dict(show_bad_actions=False)),
              ('wildfire', presets.wildfire_large(height=16, width=16, num_agents=32, seed=12), 31, {}),
              ('rideshare', presets.rideshare_c2(), 129, dict(kernel='groups')),
              ('rideshare', presets.rideshare_c2(), 129, dict(kernel='tiles')),
              ('rideshare', presets.rideshare_synthetic(drivers=1, rows=16, horizon=10), 31, {}),
              ('cybersecurity', presets.cyber_c3(), 129, CYBER_PO),
              ('cybersecurity', presets.cyber_c3(), 129, dict(show_bad_actions=True, partially_observable=False)),
              ('cybersecurity', presets.cyber_synthetic(nodes=20, attackers=9, defenders=9), 31, CYBER_PO),
              ('cybersecurity', presets.cyber_synthetic(nodes=32, attackers=16, defenders=16), 31,
               dict(show_bad_actions=True))]
    return cases


@pytest.mark.parametrize('case', range(len(sampler_cases())))
def test_the_sampler_log_prob_and_packed_masks_bit_for_bit(case):
    domain, config, B, kwargs = sampler_cases()[case]
    kwargs = dict(kwargs)
    kernel = kwargs.pop('kernel', 'auto')
    rng = np.random.default_rng(case)
    raw = setup(domain, config, B, 8, rng, kernel=kernel, kwargs=kwargs).raw
    twin = setup(domain, config, B, 8, np.random.default_rng(case), kernel=kernel, kwargs=kwargs).raw
    A, C = len(raw.agents), raw.action_slots
    W = legal_words(C)
    for t in range(3):
        legal = raw.legal_actions().clone()
        packed = raw.legal_actions(packed=True)
        assert packed.shape == (B, A, W) and packed.dtype == torch.int32
        assert torch.equal(packed, pack_legal(legal)), 'LEGAL'
        assert torch.equal(unpack_legal(packed, C), legal)
        out = torch.full((B, A, W), -1, dtype=torch.int32, device='cuda')
        assert raw.legal_actions(out=out) is out and torch.equal(out, packed)
        for dtype in (torch.float32, torch.bfloat16):
            wide = torch.from_numpy(rng.normal(0.0, 3.0, (B, A, C + 2)).astype(np.float32)).cuda().to(dtype)
            logits = wide[..., :C]
            byte_out = torch.zeros((B, A, C), dtype=torch.bool, device='cuda')
            slots, log_prob = raw.sample_actions_from_logits(logits, SEED, legal_out=byte_out)
            slots, log_prob, actions = slots.clone(), log_prob.clone(), raw._actions.clone()
            bits_out = torch.full((B, A, W), -1, dtype=torch.int32, device='cuda')
            slots2, log_prob2 = twin.sample_actions_from_logits(logits, SEED, legal_out=bits_out)
            # the flag changes nothing else the launch writes
            assert torch.equal(slots2, slots) and torch.equal(log_prob2, log_prob) and torch.equal(twin._actions, actions)
            assert torch.equal(byte_out, legal) and torch.equal(bits_out, pack_legal(legal)), 'SAMPLE'
            for mask in (byte_out, byte_out.to(torch.uint8), bits_out):
                lp, h = slot_log_prob(logits, slots, mask)
                assert torch.equal(lp, log_prob), f't={t} {dtype} {mask.dtype}: != the sampler'
                assert torch.equal(slot_log_prob(logits, slots, mask, entropy=False)[0], lp)
        # DECODE writes the same packed mask
        decode_out = torch.full((B, A, W), -1, dtype=torch.int32, device='cuda')
        raw._policy_launch(_lib.POLICY_DECODE, legal=decode_out)
        assert torch.equal(decode_out, packed), 'DECODE'
        # equal logits: -logf(n) and logf(n) exactly
        zeros = torch.zeros((B, A, C), device='cuda')
        slots, log_prob = raw.sample_actions_from_logits(zeros, SEED)
        lp, h = slot_log_prob(zeros, slots, packed)
        assert torch.equal(lp, log_prob) and torch.equal(h, -lp)
        n = legal.sum(-1).double()
        assert torch.allclose(h.double(), torch.log(n), rtol=2 * U, atol=0)
        twin.sample_actions_from_logits(zeros, SEED)
        raw.step_all(None)
        twin.step_all(None)
    raw.check_errors()
    twin.check_errors()


def test_the_parallel_wrapper_forwards_packed_masks():
    from free_range_zoo_b200.envs import rideshare_v0
    env = rideshare_v0.parallel_env(parallel_envs=64, max_steps=10, configuration=presets.rideshare_c2(),
                                    device=torch.device('cuda'))
    env.reset(seed=3)
    packed = env.legal_actions(packed=True)
    assert packed.shape == (64, len(env.agents), 2)
    assert env.unwrapped.legal_actions(packed=True) is packed  # env-owned, allocated once
    assert torch.equal(unpack_legal(packed, 33), env.legal_actions())
    out = torch.zeros_like(packed)
    env.sample_actions_from_logits(torch.zeros((64, len(env.agents), 33), device='cuda'), SEED, legal_out=out)
    assert torch.equal(out, packed)
    with pytest.raises(ValueError, match='W = ceil'):
        env.legal_actions(out=torch.zeros((64, len(env.agents), 3), dtype=torch.int32, device='cuda'))


# ------------------------------------------------------------------------------------------------ 4. invariance

@pytest.mark.parametrize('C', [6, 17, 33, 101, 257])
@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16], ids=['f32', 'bf16'])
def test_a_row_gives_the_same_bits_alone_in_a_batch_and_with_either_mask(C, dtype):
    generator = torch.Generator(device='cuda').manual_seed(C + 1)
    R = 4099
    legal = random_mask((R, ), C, 0.5, generator)
    logits = (torch.randn((R, C), generator=generator, device='cuda') * 4.0).to(dtype)
    slots = torch.randint(-1, C + 1, (R, ), generator=generator, device='cuda', dtype=torch.int32)
    g_lp = torch.randn((R, ), generator=generator, device='cuda')
    g_h = torch.randn((R, ), generator=generator, device='cuda')
    bits = as_mask(legal, 'packed')
    batch = run(logits, slots, legal, g_lp, g_h)
    assert all(torch.equal(a, b) for a, b in zip(batch, run(logits, slots, bits, g_lp, g_h)))
    lp_only = run(logits, slots, bits, g_lp, None, entropy=False)
    assert torch.equal(lp_only[0], batch[0]) and lp_only[1] is None
    assert torch.equal(lp_only[2], run(logits, slots, legal, g_lp, None)[2])
    for r in (0, 1, 31, 32, 33, 2048, R - 2, R - 1):
        alone = run(logits[r:r + 1].clone(), slots[r:r + 1].clone(), bits[r:r + 1].clone(), g_lp[r:r + 1].clone(),
                    g_h[r:r + 1].clone())
        for got, want in zip(alone, batch):
            assert torch.equal(got, want[r:r + 1]), r


# ------------------------------------------------------------------------------------------------ 5. edge rows

@pytest.mark.parametrize('C', [6, 33, 101])
def test_edge_rows(C):
    inf, nan = float('inf'), float('nan')
    legal = torch.zeros((8, C), dtype=torch.bool, device='cuda')
    legal[:, ::2] = True
    legal[:, -1] = True
    base = torch.randn((8, C), device='cuda', generator=torch.Generator(device='cuda').manual_seed(C))
    logits = base.clone()
    slots = torch.zeros((8, ), dtype=torch.int32, device='cuda')
    g = torch.ones((8, ), device='cuda')
    # rows 0-2: NaN, +inf, -inf in illegal slots change nothing
    for r, value in enumerate((nan, inf, -inf)):
        logits[r][~legal[r]] = value
    # row 3: partly -inf legal logits: finite entropy, no NaN
    logits[3, 2] = -inf
    # row 4: the chosen slot is illegal; row 5: out of range
    slots[4], slots[5] = 1, C + 7
    # rows 6, 7: a NaN / +inf legal logit
    logits[6, 0], logits[7, 2] = nan, inf
    for kind in ('bool', 'packed'):
        lp, h, grad = run(logits, slots, as_mask(legal, kind), g, g)
        clean = run(base, slots, as_mask(legal, kind), g, g)
        for r in range(3):
            assert torch.equal(lp[r], clean[0][r]) and torch.equal(h[r], clean[1][r])
            assert torch.equal(grad[r], clean[2][r]), r
        assert torch.isfinite(h[3]) and torch.isfinite(lp[3]) and not torch.isnan(grad[3]).any()
        assert grad[3, 2] == 0.0  # p = 0 and not chosen
        want = reference(logits[3:4], slots[3:4], legal[3:4], np.ones(1), np.ones(1))
        assert_within(h[3:4], want[1], want[4], 'partly -inf entropy')
        assert_within(grad[3:4], want[2], want[5], 'partly -inf gradient')
        for r in (4, 5):
            assert lp[r] == -inf and torch.isfinite(h[r])
            want = reference(logits[r:r + 1], slots[r:r + 1], legal[r:r + 1], np.ones(1), np.ones(1))
            assert_within(grad[r:r + 1], want[2], want[5], 'illegal chosen slot')
        for r in (6, 7):
            assert torch.isnan(lp[r]) and torch.isnan(h[r])
            assert torch.isnan(grad[r][legal[r]]).all() and (grad[r][~legal[r]] == 0).all()
    # no legal slot / every legal logit -inf
    none = torch.zeros((2, C), dtype=torch.bool, device='cuda')
    none[1, :3] = True
    x = torch.full((2, C), -inf, device='cuda')
    x[0] = 1.0
    lp, h, grad = run(x, torch.zeros((2, ), dtype=torch.int32, device='cuda'), none, g[:2], g[:2])
    assert torch.isnan(lp).all() and torch.isnan(h).all()
    assert (grad[0] == 0).all() and torch.isnan(grad[1, :3]).all() and (grad[1, 3:] == 0).all()
    # a -inf chosen legal slot with others finite: log_prob -inf, gradient g_lp there
    y = torch.zeros((1, C), device='cuda')
    y[0, 0] = -inf
    lp, h, grad = run(y, torch.zeros((1, ), dtype=torch.int32, device='cuda'), torch.ones((1, C), dtype=torch.bool,
                                                                                          device='cuda'), g[:1], None)
    assert lp[0] == -inf and grad[0, 0] == 1.0


# ------------------------------------------------------------------------------------------------ 6. CUDA graph

def test_a_captured_forward_backward_and_update_replays_equal_to_eager():
    torch.manual_seed(0)
    B, A, C, F = 257, 10, 101, 16
    generator = torch.Generator(device='cuda').manual_seed(1)
    features = torch.randn((4, B, A, F), generator=generator, device='cuda')
    legal = as_mask(random_mask((4, B, A), C, 0.3, generator), 'packed')
    slots = torch.randint(0, C, (4, B, A), generator=generator, device='cuda', dtype=torch.int32)
    old = torch.randn((4, B, A), generator=generator, device='cuda')

    class Policy(torch.nn.Module):  # reductions only (no GEMM): the same kernels eager and captured
        def __init__(self):
            super().__init__()
            self.weight = torch.nn.Parameter(torch.randn((F, C + 3), device='cuda') * 0.3)

        def forward(self, x):
            return (x.unsqueeze(-1) * self.weight).sum(-2)

    def model():
        return Policy()

    def step(net, optimizer):
        optimizer.zero_grad(set_to_none=False)
        logits = net(features)[..., :C]
        lp, h = slot_log_prob(logits, slots, legal)
        ratio = torch.exp(torch.nan_to_num(lp, neginf=-30.0) - old)
        loss = -(ratio.clamp(0.8, 1.2)).mean() - 0.01 * h.mean()
        loss.backward()
        optimizer.step()

    eager, captured = model(), model()
    captured.load_state_dict(eager.state_dict())
    opt_e = torch.optim.SGD(eager.parameters(), lr=0.1)
    opt_c = torch.optim.SGD(captured.parameters(), lr=0.1)
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream):
        step(captured, opt_c)  # warm-up (allocates the gradients)
    torch.cuda.current_stream().wait_stream(stream)
    step(eager, opt_e)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step(captured, opt_c)
    for _ in range(3):
        graph.replay()
        step(eager, opt_e)
    torch.cuda.synchronize()
    for a, b in zip(eager.parameters(), captured.parameters()):
        assert torch.equal(a, b)


# ------------------------------------------------------------------------------------------------ 7. past 2^31

def test_offsets_past_2_31_elements():
    R, C = 21_300_000, 101
    assert R * C > 2 ** 31
    generator = torch.Generator(device='cuda').manual_seed(31)
    logits = torch.randn((R, C), generator=generator, device='cuda', dtype=torch.bfloat16)
    W = legal_words(C)
    bits = torch.randint(-2 ** 31, 2 ** 31, (R, W), generator=generator, device='cuda', dtype=torch.int64)
    bits = bits.to(torch.int32)
    bits[:, -1] &= (1 << (C - 32 * (W - 1))) - 1  # no bits at or beyond C
    bits[:, -1] |= 1 << (C - 1 - 32 * (W - 1))  # the noop
    slots = torch.full((R, ), C - 1, dtype=torch.int32, device='cuda')
    g = torch.ones((R, ), device='cuda')
    lp, h, grad = run(logits, slots, bits, g, g)
    assert grad.dtype == torch.bfloat16 and grad.shape == (R, C)
    for r in (0, 2 ** 31 // C - 1, 2 ** 31 // C, 2 ** 31 // C + 1, R - 1):
        alone = run(logits[r:r + 1].clone(), slots[r:r + 1].clone(), bits[r:r + 1].clone(), g[:1], g[:1])
        assert torch.equal(alone[0], lp[r:r + 1]) and torch.equal(alone[1], h[r:r + 1]), r
        assert torch.equal(alone[2], grad[r:r + 1]), r
    tail = slice(R - 64, R)
    want = reference(logits[tail], slots[tail], unpack_legal(bits[tail], C), np.ones(64), np.ones(64))
    assert_within(lp[tail], want[0], want[3], 'log_prob past 2^31')
    assert_within(grad[tail], want[2], want[5] + np.abs(want[2]) * 2.0 ** -8, 'gradient past 2^31')
    assert not math.isnan(float(lp.sum()))
