"""CPU oracle for the wildfire step path -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Only ``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` may
import this module; the product path (``free_range_zoo_b200``) never does and fails loudly without its CUDA library.

This is a numpy restatement (batched over the leading ``parallel_envs`` axis, plain loops over agents) of the
reference's wildfire hot path; every function cites the reference lines it follows (paths relative to
``free_range_zoo/`` in /root/reference).  Parity pin: ``tests/test_oracle_golden.py`` replays the trajectories
recorded from the unmodified reference (``tests/golden/wildfire_*.npz``, made by ``tests/golden/gen_golden.py``) and
``tests/test_oracle_kat.py`` re-states the reference's own transition unit-test vectors
(tests/free_range_zoo/envs/wildfire/env/transitions/test_*.py).
"""
from __future__ import annotations

import numpy as np

PAD = -100
F32 = np.float32


def _f32(x):
    return np.asarray(x.detach().cpu().numpy() if hasattr(x, 'detach') else x, dtype=np.float32)


def _i32(x):
    return np.asarray(x.detach().cpu().numpy() if hasattr(x, 'detach') else x, dtype=np.int32)


def spread_lut(weights: np.ndarray) -> np.ndarray:
    """fp32 ignition probability for each of the 16 lit-neighbour patterns (bit0 N, bit1 W, bit2 E, bit3 S).

    The reference runs a 3x3 ``nn.Conv2d`` over the lit mask (envs/wildfire/env/transitions/fire_spreads.py:29,46) with
    the filter [[0,N,0],[W,0,E],[0,S,0]] (envs/wildfire/env/structures/configuration.py:347-363).  Its fp32
    accumulation order on CPU is ascending filter index -- N, W, E, S -- verified bit-for-bit against
    ``spread_lut`` in the golden fixtures (the reference's own conv2d output for the 16 patterns).
    """
    w = np.asarray(weights, dtype=np.float32).reshape(3, 3)
    taps = (w[0, 1], w[1, 0], w[1, 2], w[2, 1])
    lut = np.zeros(16, dtype=np.float32)
    for pattern in range(16):
        acc = F32(0.0)
        for bit, tap in enumerate(taps):
            if (pattern >> bit) & 1:
                acc = F32(acc + tap)
        lut[pattern] = acc
    return lut


# ---------------------------------------------------------------------------------------------------------------------
# The seven transitions as pure functions over numpy arrays (state arrays are updated in place where the reference
# mutates its state).  ``WildfireOracle.step`` chains them; tests/test_oracle_kat.py feeds them the inputs of the
# reference's own transition unit tests.


def suppressant_decrease(suppressants, users, u, stochastic, p):
    """transitions/suppressant_decrease.py:34-63."""
    decrease = users & (u < F32(p)) if stochastic else users
    return np.maximum(np.where(decrease, suppressants - F32(1), suppressants), F32(0)).astype(np.float32)


def equipment_transition(equipment, u, num_states, stochastic_repair, p_repair, stochastic_degrade, p_degrade,
                         critical_error, p_critical):
    """transitions/equipment.py:42-77 -- all masks from the pre-update equipment, one uniform for the three tests."""
    pristine = equipment == num_states - 1
    damaged = equipment == 0
    intermediate = ~pristine & ~damaged
    repairs = damaged & (u < F32(p_repair)) if stochastic_repair else damaged
    updated = equipment.copy()
    updated[repairs] = num_states - 1
    criticals = np.zeros_like(pristine)
    if critical_error:
        criticals = pristine & (u < F32(p_critical))
        updated[criticals] = 0
    degrades = (pristine | intermediate) & (u < F32(p_degrade)) if stochastic_degrade else (pristine | intermediate)
    degrades = degrades & ~criticals
    updated[degrades] -= 1
    return updated


def suppressant_refill(suppressants, capacity, equipment, refills, u, stochastic, p, capacity_bonuses):
    """transitions/suppressant_refill.py:43-74 (``equipment`` is the state AFTER the equipment transition)."""
    increase = refills & (u < F32(p)) if stochastic else refills.copy()
    bonus = np.asarray(capacity_bonuses, np.float32)[equipment]
    return np.where(increase, (capacity + bonus).astype(np.float32), suppressants).astype(np.float32), increase


def capacity_transition(suppressants, capacity, targets, u_size, u_switch, stochastic, p_switch, capacities, cumulative):
    """transitions/capacity.py:39-66 (bucketize right=False: first i with r <= cum[i])."""
    capacities = np.asarray(capacities, np.float32)
    size_index = np.searchsorted(np.asarray(cumulative, np.float32), u_size, side='left')
    new_max = capacities[np.minimum(size_index, len(capacities) - 1)]
    switch = targets & (u_switch < F32(p_switch)) if stochastic else targets
    extra = (suppressants - capacity).astype(np.float32)
    new_capacity = np.where(switch, new_max, capacity).astype(np.float32)
    new_suppressants = np.where(switch, (new_max + extra).astype(np.float32), suppressants).astype(np.float32)
    return new_suppressants, new_capacity


def fire_increase(fires, intensity, fuel, attack, u, num_states, stochastic_increase, p_increase, stochastic_burnouts,
                  p_burnout):
    """transitions/fire_increase.py:43-95; mutates fires / intensity / fuel, returns the just-burned-out mask."""
    required = np.where(fires >= 0, fires, 0).astype(np.float32)
    diff = required - attack
    burning = (fires > 0) & (intensity > 0)
    unmet = (diff > 0) & burning
    almost = unmet & (intensity == num_states - 2)
    prob = np.zeros(fires.shape, np.float32)
    prob[unmet & ~almost] = F32(p_increase) if stochastic_increase else F32(1.0)
    prob[almost] = F32(p_burnout) if stochastic_burnouts else F32(p_increase)
    prob = np.clip(prob, 0, 1)
    grow = u < prob
    intensity[grow] += 1
    burned = grow & (intensity >= num_states - 1)
    fires[burned] *= -1
    fuel[burned] = np.maximum(fuel[burned] - 1, 0)
    return burned


def fire_decrease(fires, intensity, fuel, attack, u, stochastic_decrease, p_decrease, bonus):
    """transitions/fire_decrease.py:36-80 (no FMA: multiply then add, each rounded to fp32); returns put-out mask."""
    required = np.where(fires >= 0, fires, 0).astype(np.float32)
    diff = required - attack
    burning = (fires > 0) & (intensity > 0)
    met = (diff <= 0) & burning
    prob = np.zeros(fires.shape, np.float32)
    if stochastic_decrease:
        prob[met] = (F32(p_decrease) + (F32(-1) * diff[met]).astype(np.float32) * F32(bonus)).astype(np.float32)
    else:
        prob[met] = 1.0
    prob = np.clip(prob, 0, 1)
    shrink = u < prob
    intensity[shrink] -= 1
    put_out = shrink & (intensity <= 0)
    fires[put_out] *= -1
    fuel[put_out] -= 1
    return put_out


def fire_spread(fires, intensity, fuel, u, lut, p_random, ignition_temp, use_fuel):
    """transitions/fire_spreads.py:33-59 on [B, H, W] arrays; mutates fires / intensity."""
    B, H, W = fires.shape
    burning = (fires > 0) & (intensity > 0)
    padded = np.pad(burning, ((0, 0), (1, 1), (1, 1)))
    pattern = (padded[:, 0:H, 1:W + 1].astype(np.int32) | (padded[:, 1:H + 1, 0:W].astype(np.int32) << 1) |
               (padded[:, 1:H + 1, 2:W + 2].astype(np.int32) << 2) | (padded[:, 2:H + 2, 1:W + 1].astype(np.int32) << 3))
    prob = np.asarray(lut, np.float32)[pattern]
    unlit = (fires < 0) & (intensity == 0)
    if use_fuel:
        unlit &= fuel > 0
    prob = np.where(unlit, (prob + F32(p_random)).astype(np.float32), F32(0))
    ignite = u < prob
    fires[ignite] *= -1
    intensity[ignite] = np.broadcast_to(np.asarray(ignition_temp), fires.shape)[ignite]
    return ignite


class WildfireOracle:
    """Reference semantics of ``wildfire_v0`` for one batch of environments, state held as numpy arrays.

    Attribute names follow the reference env (``num_moves``, ``num_burnouts``, ``environment_task_count`` ...).
    ``agent_task_count`` is stored [B, A] (the reference keeps [A, B], utils/env.py:160).
    """

    def __init__(self, configuration, parallel_envs: int, max_steps: int = 1, show_bad_actions: bool = False,
                 observe_other_suppressant: bool = False, observe_other_power: bool = False):
        c = configuration
        fc, ac, rc, sc = c.fire_config, c.agent_config, c.reward_config, c.stochastic_config
        self.B, self.H, self.W = parallel_envs, c.grid_height, c.grid_width
        self.A = ac.agents.shape[0]
        self.max_steps = max_steps
        self.show_bad_actions = show_bad_actions
        # envs/wildfire/env/wildfire.py:230-233 -- column mask applied to the other agents' observations
        self.other_columns = [0, 1] + ([2] if observe_other_power else []) + ([3] if observe_other_suppressant else [])

        self.fire_types = _i32(fc.fire_types)
        self.lit0 = np.asarray(fc.lit.cpu().numpy(), dtype=bool)
        self.ignition_temp = _i32(fc.ignition_temp)
        self.initial_fuel = int(fc.initial_fuel)
        self.S = int(fc.num_fire_states)
        self.p_increase = F32(fc.intensity_increase_probability)
        self.p_decrease = F32(fc.intensity_decrease_probability)
        self.decrease_bonus = F32(fc.extra_power_decrease_bonus)
        self.p_burnout = F32(fc.burnout_probability)
        self.spread_weights = _f32(c.fire_spread_weights)
        self.spread_lut = spread_lut(self.spread_weights)
        self.p_random = F32(c.fire_random_spread_weight)

        self.agent_pos = _i32(ac.agents)
        self.power = _f32(ac.fire_reduction_power)
        self.attack_range = _f32(ac.attack_range)
        self.equipment_states = _f32(ac.equipment_states)
        self.E = self.equipment_states.shape[0]
        self.p_supp_decrease = F32(ac.suppressant_decrease_probability)
        self.p_refill = F32(ac.suppressant_refill_probability)
        self.p_repair = F32(ac.repair_probability)
        self.p_degrade = F32(ac.degrade_probability)
        self.p_critical = F32(ac.critical_error_probability)
        self.p_tank_switch = F32(ac.tank_switch_probability)
        self.capacities = _f32(ac.possible_capacities)
        # transitions/capacity.py:28 -- cumulative probabilities are a torch fp32 cumsum (sequential)
        self.capacity_cum = np.cumsum(_f32(ac.capacity_probabilities), dtype=np.float32)
        self.initial = (F32(ac.initial_suppressant), F32(ac.initial_capacity), int(ac.initial_equipment_state))

        self.fire_rewards = _f32(rc.fire_rewards)
        self.bad_attack_penalty = F32(rc.bad_attack_penalty)
        self.burnout_penalty = F32(rc.burnout_penalty)
        self.burnout_penalty_scaled = bool(rc.burnout_penalty_scaled)
        self.termination_reward = F32(rc.termination_reward)
        self.termination_kappa = F32(rc.termination_kappa)
        self.localize_putouts = bool(rc.localize_putouts)
        self.sc = sc

    # ------------------------------------------------------------------ reset

    STATE_KEYS = ('fires', 'intensity', 'fuel', 'suppressants', 'capacity', 'equipment')

    def reset_batches(self, mask, initial_state: dict | None = None):
        """utils/env.py:163-189 + envs/wildfire/env/wildfire.py:376-397: the environments selected by ``mask`` (bool
        [B]) go back to the saved initial state (``initial_state`` replaces it first when given) with zeroed AEC fields
        and counters; then observations and actions are published for the whole batch."""
        mask = np.asarray(mask, bool)
        if initial_state is not None:
            self.initial_state = {key: np.array(initial_state[key]) for key in self.STATE_KEYS}
        for key in self.STATE_KEYS:
            getattr(self, key)[mask] = self.initial_state[key][mask]
        for key in ('rewards', 'cumulative_rewards', 'terminated', 'truncated', 'num_moves', 'num_burnouts', 'burnouts',
                    'putouts'):
            getattr(self, key)[mask] = 0
        self.update_observations()
        self.update_actions()

    def reset(self, initial_state: dict | None = None):
        """utils/env.py:95-160 + envs/wildfire/env/wildfire.py:291-373."""
        B, H, W, A = self.B, self.H, self.W, self.A
        if initial_state is not None:
            for key in self.STATE_KEYS:
                setattr(self, key, np.array(initial_state[key]))
        else:
            self.fires = np.zeros((B, H, W), np.int32)
            self.intensity = np.zeros((B, H, W), np.int32)
            self.fuel = np.zeros((B, H, W), np.int32)
            self.fires[:, self.lit0] = self.fire_types[self.lit0]  # wildfire.py:347
            self.fires[:, ~self.lit0] = -1 * self.fire_types[~self.lit0]  # :348
            self.intensity[:, self.lit0] = self.ignition_temp[self.lit0]  # :349
            self.fuel[self.fires != 0] = self.initial_fuel  # :350
            self.suppressants = np.full((B, A), self.initial[0], np.float32)  # :352-354
            self.capacity = np.full((B, A), self.initial[1], np.float32)
            self.equipment = np.full((B, A), self.initial[2], np.int32)
        # State.save_initial (utils/state.py:36-38): what reset_batches restores
        self.initial_state = {key: getattr(self, key).copy() for key in self.STATE_KEYS}
        self.rewards = np.zeros((B, A), np.float32)
        self.cumulative_rewards = np.zeros((B, A), np.float32)
        self.terminated = np.zeros(B, bool)
        self.truncated = np.zeros(B, bool)
        self.num_moves = np.zeros(B, np.int32)
        self.num_burnouts = np.zeros(B, np.int32)  # wildfire.py:360
        self.burnouts = np.zeros(B, np.int32)
        self.putouts = np.zeros(B, np.int32)
        self.update_observations()
        self.update_actions()

    # ------------------------------------------------------------------ derived views

    def _lit_rank(self):
        """Env-local task index of every lit cell = rank in row-major ``nonzero`` order (wildfire.py:420,595)."""
        lit = (self.fires > 0).reshape(self.B, -1)
        rank = np.cumsum(lit, axis=1) - 1
        return lit, rank

    def update_actions(self):
        """envs/wildfire/env/wildfire.py:587-666 with the range test of env/utils/in_range_check.py:5-23."""
        B, A, HW = self.B, self.A, self.H * self.W
        lit, rank = self._lit_rank()
        ys, xs = np.divmod(np.arange(HW), self.W)
        self.environment_task_count = lit.sum(axis=1).astype(np.int32)
        self.agent_task_count = np.zeros((B, A), np.int32)
        self.available = np.zeros((B, A, HW), bool)  # (agent can fight the fire of this cell)
        for a in range(A):
            cheb = np.maximum(np.abs(self.agent_pos[a, 0] - ys), np.abs(self.agent_pos[a, 1] - xs))  # [HW]
            true_range = self.attack_range[a] + self.equipment_states[self.equipment[:, a], 2]  # wildfire.py:606-609
            in_range = cheb[None, :] <= true_range[:, None]
            has_suppressant = self.suppressants[:, a] > 0  # :619
            self.available[:, a] = lit & in_range & has_suppressant[:, None]
            self.agent_task_count[:, a] = self.available[:, a].sum(axis=1)
        self._lit, self._rank = lit, rank

    def action_map(self, a: int, bad: bool = False):
        """Padded ``agent_action_mapping[a]`` / ``agent_bad_actions[a]`` (wildfire.py:642-662)."""
        B, HW = self.B, self.H * self.W
        out = np.full((B, HW), PAD, np.int32)
        if bad:
            member = self._lit & ~self.available[:, a]
        elif self.show_bad_actions:
            member = self._lit
        else:
            member = self.available[:, a]
        for b in range(B):
            tasks = self._rank[b, member[b]]
            out[b, :len(tasks)] = tasks
        return out

    def update_observations(self):
        """envs/wildfire/env/wildfire.py:669-717."""
        B, A, HW = self.B, self.A, self.H * self.W
        self.self_obs = np.zeros((B, A, 4), np.float32)
        self.self_obs[:, :, 0] = self.agent_pos[None, :, 0]
        self.self_obs[:, :, 1] = self.agent_pos[None, :, 1]
        self.self_obs[:, :, 2] = self.power[None, :]
        self.self_obs[:, :, 3] = self.suppressants
        lit = (self.fires > 0).reshape(B, HW)
        ys, xs = np.divmod(np.arange(HW), self.W)
        self.task_obs = np.full((B, HW, 4), PAD, np.int32)
        fires, intensity = self.fires.reshape(B, HW), self.intensity.reshape(B, HW)
        for b in range(B):
            cells = np.nonzero(lit[b])[0]
            self.task_obs[b, :len(cells)] = np.stack([ys[cells], xs[cells], fires[b, cells], intensity[b, cells]], axis=1)

    def others_obs(self, a: int):
        keep = [i for i in range(self.A) if i != a]
        return self.self_obs[:, keep][:, :, self.other_columns]

    # ------------------------------------------------------------------ step

    def step(self, actions: np.ndarray, u_field: np.ndarray, u_agent: np.ndarray):
        """One full AEC cycle: utils/env.py:203-242 around envs/wildfire/env/wildfire.py:400-584.

        actions: int32 [B, A, 2]; u_field: f32 [3, B, H, W]; u_agent: f32 [5, B, A] (event order of wildfire.py:409-410).
        A batch in which every env is already terminated (or truncated) is not stepped at all (utils/env.py:212).
        """
        if self.terminated.all() or self.truncated.all():
            return False
        B, H, W, A, HW = self.B, self.H, self.W, self.A, self.H * self.W
        sc = self.sc
        rewards = np.zeros((B, A), np.float32)
        lit, rank = self._lit, self._rank

        # ---- action decode, wildfire.py:412-486
        refills = actions[:, :, 1] == -1
        users = np.zeros((B, A), bool)
        attack = np.zeros((B, HW), np.float32)
        hit = np.zeros((B, A, HW), bool)
        for a in range(A):
            if self.agent_task_count[:, a].sum() == 0:  # :434
                continue
            choice_mask = lit if self.show_bad_actions else self.available[:, a]
            full_power = (self.power[a] + self.equipment_states[self.equipment[:, a], 1]).astype(np.float32)  # :455-457
            for b in range(B):
                if refills[b, a]:
                    continue
                cells = np.nonzero(choice_mask[b])[0]
                k = actions[b, a, 0]
                if k < 0 or k >= len(cells):
                    continue  # the reference would index padding here; never produced by a legal policy
                cell = cells[k]
                if self.show_bad_actions and not self.available[b, a, cell]:  # :464-468
                    rewards[b, a] = self.bad_attack_penalty  # :477 (assignment)
                    continue
                attack[b, cell] = F32(attack[b, cell] + full_power[b])  # :470, agents in order
                users[b, a] = True
                hit[b, a, cell] = True

        # ---- agent transitions, in the reference order (wildfire.py:488-514)
        self.suppressants = suppressant_decrease(self.suppressants, users, u_agent[0], sc.suppressant_decrease,
                                                 self.p_supp_decrease)
        self.equipment = equipment_transition(self.equipment, u_agent[1], self.E, sc.repair, self.p_repair, sc.degrade,
                                              self.p_degrade, sc.critical_error, self.p_critical)
        self.suppressants, increase = suppressant_refill(self.suppressants, self.capacity, self.equipment, refills,
                                                         u_agent[2], sc.suppressant_refill, self.p_refill,
                                                         self.equipment_states[:, 0])
        self.suppressants, self.capacity = capacity_transition(self.suppressants, self.capacity, increase, u_agent[3],
                                                               u_agent[4], sc.tank_switch, self.p_tank_switch,
                                                               self.capacities, self.capacity_cum)

        # ---- fire transitions, each on the state left by the previous one (wildfire.py:516-532)
        fires, intensity, fuel = self.fires, self.intensity, self.fuel
        attack3 = attack.reshape(B, H, W)
        burned = fire_increase(fires, intensity, fuel, attack3, u_field[0], self.S, sc.fire_increase, self.p_increase,
                               sc.special_burnout_probability, self.p_burnout)
        put_out = fire_decrease(fires, intensity, fuel, attack3, u_field[1], sc.fire_decrease, self.p_decrease,
                                self.decrease_bonus)
        fire_spread(fires, intensity, fuel, u_field[2], self.spread_lut, self.p_random, self.ignition_temp, sc.fire_fuel)
        fires, intensity, fuel = (x.reshape(B, HW) for x in (fires, intensity, fuel))
        burned, put_out = burned.reshape(B, HW), put_out.reshape(B, HW)

        # ---- rewards, wildfire.py:534-557
        cell_reward = np.broadcast_to(self.fire_rewards.reshape(1, HW), (B, HW))
        putout_reward = np.where(put_out, cell_reward, F32(0))
        if self.burnout_penalty_scaled:
            penalty = np.where(burned, -cell_reward, F32(0))
        else:
            penalty = np.where(burned, self.burnout_penalty, F32(0))
        penalty_total = penalty.sum(axis=1, dtype=np.float32)
        if self.localize_putouts:
            for a in range(A):
                rewards[:, a] += (putout_reward * hit[:, a]).sum(axis=1, dtype=np.float32) + penalty_total
        else:
            rewards += (putout_reward.sum(axis=1, dtype=np.float32) + penalty_total)[:, None]

        # ---- termination, wildfire.py:559-582
        dead = fires.max(axis=1) <= 0
        if sc.fire_fuel:
            dead &= fuel.sum(axis=1) <= 0
        fires[dead] = 0  # :570
        newly = ~self.terminated & dead
        term_reward = np.maximum(
            self.termination_reward - self.termination_kappa * np.log(self.num_burnouts.astype(np.float32) + F32(1.0)),
            F32(0)).astype(np.float32)
        rewards[newly] += term_reward[newly, None]
        self.terminated = self.terminated | dead
        self.burnouts = burned.sum(axis=1).astype(np.int32)
        self.putouts = put_out.sum(axis=1).astype(np.int32)
        self.num_burnouts = self.num_burnouts + self.burnouts

        self.fires, self.intensity, self.fuel = (x.reshape(B, H, W) for x in (fires, intensity, fuel))

        # ---- utils/env.py:223-237
        self.rewards = rewards
        self.num_moves = self.num_moves + 1
        if self.max_steps is not None:
            self.truncated = self.num_moves >= self.max_steps
        self.cumulative_rewards = self.cumulative_rewards + rewards
        self.update_observations()
        self.update_actions()
        return True

    # ------------------------------------------------------------------ golden-format dump

    def outputs(self) -> dict:
        """Same keys/layout as tests/golden/gen_golden.py::wildfire_outputs."""
        A = self.A
        out = dict(
            fires=self.fires, intensity=self.intensity, fuel=self.fuel, suppressants=self.suppressants,
            capacity=self.capacity, equipment=self.equipment, rewards=self.rewards,
            terminated=np.repeat(self.terminated[:, None], A, axis=1),
            truncated=np.repeat(self.truncated[:, None], A, axis=1),
            num_moves=self.num_moves, num_burnouts=self.num_burnouts, burnouts=self.burnouts, putouts=self.putouts,
            env_task_count=self.environment_task_count, agent_task_count=self.agent_task_count,
            self_obs=self.self_obs, others_obs=np.stack([self.others_obs(a) for a in range(A)], axis=0),
            task_obs=self.task_obs, action_map=np.stack([self.action_map(a) for a in range(A)], axis=0),
        )
        if self.show_bad_actions:
            out['bad_map'] = np.stack([self.action_map(a, bad=True) for a in range(A)], axis=0)
        return out
