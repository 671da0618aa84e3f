"""wildfire_v0 on the B200 engine.

Public surface of the reference module (free_range_zoo/envs/wildfire/env/wildfire.py:126-762): ``parallel_env``,
``env``, ``raw_env`` with the same constructor flags, ``reset / step / reset_batches / action_space /
observation_space`` and attributes.  The reference's Python step (seven ``nn.Module`` transitions, per-agent decode
loop, ``nonzero``/nested-tensor plumbing) is replaced by ``frz_wildfire_step`` -- one fused sm_100a launch.
"""
from __future__ import annotations

import ctypes
from typing import Any, Callable, Dict, List, Optional, Tuple

import numpy as np
import torch

from free_range_zoo_b200 import _lib
from free_range_zoo_b200.envs.wildfire.env.structures.state import WildfireState
from free_range_zoo_b200.utils.containers import (LazyDict, ObservationDict, jagged_from_padded,
                                                  jagged_indices_from_mask)
from free_range_zoo_b200.utils.conversions import batched_aec_to_batched_parallel
from free_range_zoo_b200.utils import compact
from free_range_zoo_b200.utils.env import AutoresetRows, BatchedAECEnv
from free_range_zoo_b200.utils.spaces import BatchedActionSpace, Space


def parallel_env(wrappers: List[Callable] = [], **kwargs):
    """Parallel-API wildfire environment (reference wildfire.py:126-142)."""
    env = raw_env(**kwargs)
    for wrapper in wrappers:
        env = wrapper(env)
    return batched_aec_to_batched_parallel(env)


def env(wrappers: List[Callable] = [], **kwargs):
    """AEC-API wildfire environment (reference wildfire.py:145-160)."""
    environment = raw_env(**kwargs)
    for wrapper in wrappers:
        environment = wrapper(environment)
    return environment


def _np(tensor, dtype):
    return np.ascontiguousarray(torch.as_tensor(tensor).detach().cpu().numpy().astype(dtype))


def spread_lut(weights) -> np.ndarray:
    """fp32 ignition probability for the 16 lit-neighbour patterns (bit0 N, bit1 W, bit2 E, bit3 S), accumulated in
    the order the reference's 3x3 conv2d accumulates on CPU: ascending filter index N, W, E, S
    (transitions/fire_spreads.py:29,46; structures/configuration.py:347-363)."""
    w = _np(weights, np.float32).reshape(3, 3)
    taps = (w[0, 1], w[1, 0], w[1, 2], w[2, 1])
    lut = np.zeros(16, dtype=np.float32)
    for pattern in range(16):
        acc = np.float32(0.0)
        for bit, tap in enumerate(taps):
            if pattern >> bit & 1:
                acc = np.float32(acc + tap)
        lut[pattern] = acc
    return lut


def flatten_configuration(config, max_steps, show_bad_actions: bool, env_offset: int = 0):
    """WildfireConfiguration -> (FrzWildfireParams, cell_reward, cell_ignition, range_mask) -- done once."""
    fc, ac, rc, sc = config.fire_config, config.agent_config, config.reward_config, config.stochastic_config
    H, W = int(config.grid_height), int(config.grid_width)
    A = int(ac.agents.shape[0])
    equipment_states = _np(ac.equipment_states, np.float32)
    E = equipment_states.shape[0]
    capacities = _np(ac.possible_capacities, np.float32)
    if H * W > _lib.MAX_CELLS or A > _lib.MAX_AGENTS or E > _lib.MAX_EQUIPMENT or len(capacities) > _lib.MAX_CAPACITIES:
        raise ValueError(f'wildfire configuration exceeds the engine limits: H*W={H * W} (<= {_lib.MAX_CELLS}), '
                         f'agents={A} (<= {_lib.MAX_AGENTS}), equipment states={E}, capacities={len(capacities)}')

    p = _lib.WildfireParams()
    p.height, p.width, p.num_agents = H, W, A
    p.num_fire_states = int(fc.num_fire_states)
    p.num_equipment_states = E
    p.num_capacities = len(capacities)
    p.max_steps = 2**31 - 1 if max_steps is None else int(max_steps)
    flags = 0
    for name, bit in _lib.WF_FLAGS.items():
        if getattr(sc, name):
            flags |= bit
    if rc.burnout_penalty_scaled:
        flags |= _lib.WF_BURNOUT_SCALED
    if rc.localize_putouts:
        flags |= _lib.WF_LOCALIZE_PUTOUTS
    if show_bad_actions:
        flags |= _lib.WF_SHOW_BAD_ACTIONS
    p.flags = flags
    p.env_offset = env_offset
    p.p_increase = fc.intensity_increase_probability
    p.p_burnout = fc.burnout_probability
    p.p_decrease = fc.intensity_decrease_probability
    p.decrease_bonus = fc.extra_power_decrease_bonus
    p.p_random_ignition = config.fire_random_spread_weight
    p.spread_lut[:] = spread_lut(config.fire_spread_weights).tolist()
    p.p_suppressant_decrease = ac.suppressant_decrease_probability
    p.p_refill = ac.suppressant_refill_probability
    p.p_repair = ac.repair_probability
    p.p_degrade = ac.degrade_probability
    p.p_critical = ac.critical_error_probability
    p.p_tank_switch = ac.tank_switch_probability
    cumulative = np.cumsum(_np(ac.capacity_probabilities, np.float32), dtype=np.float32)  # capacity.py:28
    for i in range(len(capacities)):
        p.capacity_cum[i] = cumulative[i]
        p.capacity_value[i] = capacities[i]
    for e in range(E):
        p.equipment_capacity_bonus[e] = equipment_states[e, 0]
        p.equipment_power_bonus[e] = equipment_states[e, 1]
    p.bad_attack_penalty = rc.bad_attack_penalty
    p.burnout_penalty = rc.burnout_penalty
    p.termination_reward = rc.termination_reward
    p.termination_kappa = rc.termination_kappa
    positions = _np(ac.agents, np.int32)
    power = _np(ac.fire_reduction_power, np.float32)
    for a in range(A):
        p.agent_y[a], p.agent_x[a], p.agent_power[a] = int(positions[a, 0]), int(positions[a, 1]), float(power[a])

    # Chebyshev range test of update_actions (wildfire.py:606-616, utils/in_range_check.py:5-23), tabulated per
    # (agent, equipment state): agents never move, so the in-range set only depends on the equipment state.
    words = (H * W + 31) // 32
    ys, xs = np.divmod(np.arange(H * W), W)
    attack_range = _np(ac.attack_range, np.float32)
    range_mask = np.zeros((A, E, words), dtype=np.uint32)
    for a in range(A):
        chebyshev = np.maximum(np.abs(positions[a, 0] - ys), np.abs(positions[a, 1] - xs)).astype(np.float32)
        for e in range(E):
            reach = np.float32(attack_range[a] + equipment_states[e, 2])
            for c in np.nonzero(chebyshev <= reach)[0]:
                range_mask[a, e, c >> 5] |= np.uint32(1 << (c & 31))
    return p, _np(rc.fire_rewards, np.float32).reshape(-1), _np(fc.ignition_temp, np.int32).reshape(-1), range_mask


def compact_bounds(config) -> Dict[str, int]:
    """Largest |value| of the integer observations, from the configuration (utils/compact.py picks the types)."""
    H, W, fc = int(config.grid_height), int(config.grid_width), config.fire_config
    max_fire_type = max(int(fc.max_fire_type), int(torch.as_tensor(fc.fire_types).abs().max()))
    return dict(task_obs=max(H - 1, W - 1, max_fire_type, int(fc.num_fire_states) - 1),  # (y, x, fire type, intensity)
                agent_task_count=H * W)


def transpose_range_mask(range_mask: np.ndarray, cells: int) -> np.ndarray:
    """[A, E, words] (bit c of agent a's row) -> [E, cells] (bit a of cell c's word): who reaches a cell."""
    agents, states, _ = range_mask.shape
    cell_agents = np.zeros((states, cells), dtype=np.uint32)
    for a in range(agents):
        for e in range(states):
            for c in range(cells):
                if int(range_mask[a, e, c >> 5]) >> (c & 31) & 1:
                    cell_agents[e, c] |= np.uint32(1 << a)
    return cell_agents


class raw_env(BatchedAECEnv):
    """Wildfire environment whose step is one fused CUDA kernel."""

    metadata = {"render.modes": ["human", "rgb_array"], "name": "wildfire_v0", "is_parallelizable": True,
                "render_fps": 2}

    @torch.no_grad()
    def __init__(self, *args, observe_other_suppressant: bool = False, observe_other_power: bool = False,
                 show_bad_actions: bool = False, step_kernel: str = 'auto', **kwargs) -> None:
        """``step_kernel`` ('auto' | 'tiles' | 'groups'): grids of at most 32 cells with at most 8 agents have two step
        kernels (one thread per environment for large batches, eight lanes per environment otherwise) with identical
        results and random streams; 'auto' picks by batch size, the other two force one (tests, kernel timing --
        include/frz.h FRZ_WF_KERNEL_*).  Larger grids ignore it."""
        super().__init__(*args, **kwargs)
        if step_kernel not in ('auto', 'tiles', 'groups'):
            raise ValueError(f"step_kernel must be 'auto', 'tiles' or 'groups', not {step_kernel!r}")
        self._step_kernel = step_kernel
        self.observe_other_suppressant = observe_other_suppressant
        self.observe_other_power = observe_other_power
        self.show_bad_actions = show_bad_actions

        A = int(self.agent_config.agents.shape[0])
        self.possible_agents = tuple(f"firefighter_{i}" for i in range(1, A + 1))
        self.agents = self.possible_agents
        self.agent_name_mapping = dict(zip(self.possible_agents, range(A)))
        self.max_x, self.max_y = int(self.config.grid_width), int(self.config.grid_height)
        self.ignition_temp = self.fire_config.ignition_temp
        self.agent_observation_bounds = (self.max_y, self.max_x, self.agent_config.max_fire_reduction_power,
                                         self.agent_config.suppressant_states)
        self.fire_observation_bounds = (self.max_y, self.max_x, self.fire_config.max_fire_type,
                                        self.fire_config.num_fire_states)
        other_columns = [0, 1] + ([2] if observe_other_power else []) + ([3] if observe_other_suppressant else [])
        self._other_columns = torch.tensor(other_columns, device=self.device)
        self._other_agents = {
            agent: torch.tensor([i for i in range(A) if i != index], dtype=torch.int64, device=self.device)
            for agent, index in self.agent_name_mapping.items()
        }

        self._params, cell_reward, cell_ignition, range_mask = flatten_configuration(
            self.config, self.max_steps, show_bad_actions, self.env_offset)
        self._params.flags |= {'auto': 0, 'tiles': _lib.WF_KERNEL_TILES, 'groups': _lib.WF_KERNEL_GROUPS}[step_kernel]
        B, HW, dev = self.parallel_envs, self.max_y * self.max_x, self.device
        self._allocate_runtime(A)
        self._mask_stride = (HW + 3) // 4 * 4
        i32, f32 = torch.int32, torch.float32
        self._state = WildfireState(
            fires=torch.zeros((B, self.max_y, self.max_x), dtype=i32, device=dev),
            intensity=torch.zeros((B, self.max_y, self.max_x), dtype=i32, device=dev),
            fuel=torch.zeros((B, self.max_y, self.max_x), dtype=i32, device=dev),
            agents=torch.as_tensor(self.agent_config.agents, dtype=i32).to(dev),
            suppressants=torch.ones((B, A), dtype=f32, device=dev),
            capacity=torch.ones((B, A), dtype=f32, device=dev),
            equipment=torch.ones((B, A), dtype=i32, device=dev),
        )
        self._initial = self._state.clone()
        self.num_burnouts = torch.zeros(B, dtype=i32, device=dev)
        self._burnouts = torch.zeros(B, dtype=i32, device=dev)
        self._putouts = torch.zeros(B, dtype=i32, device=dev)
        self._action_mask = torch.zeros((B, A, self._mask_stride), dtype=torch.uint8, device=dev)
        self._self_obs = torch.zeros((B, A, 4), dtype=f32, device=dev)
        self._task_obs = torch.full((B, HW, 4), _lib.PAD, dtype=i32, device=dev)
        self._cell_reward = torch.from_numpy(cell_reward).to(dev)
        self._cell_ignition = torch.from_numpy(cell_ignition).to(dev)
        self._range_mask = torch.from_numpy(range_mask.view(np.int32)).to(dev)
        self._cell_agents = torch.from_numpy(transpose_range_mask(range_mask, HW).view(np.int32)).to(dev)
        self._uniforms = (None, None)
        self._io = self._bind_buffers()

    def _bind_buffers(self) -> _lib.WildfireBuffers:
        s, init = self._state, self._initial
        io = _lib.WildfireBuffers()
        tensors = dict(
            fires=s.fires, intensity=s.intensity, fuel=s.fuel, suppressants=s.suppressants, capacity=s.capacity,
            equipment=s.equipment, init_fires=init.fires, init_intensity=init.intensity, init_fuel=init.fuel,
            init_suppressants=init.suppressants, init_capacity=init.capacity, init_equipment=init.equipment,
            actions=self._actions, rewards=self._rewards, cumulative_rewards=self._cumulative,
            terminated=self._terminated, truncated=self._truncated, num_moves=self.num_moves,
            num_burnouts=self.num_burnouts, burnouts=self._burnouts, putouts=self._putouts,
            env_task_count=self.environment_task_count, agent_task_count=self._agent_task_count,
            action_mask=self._action_mask, self_obs=self._self_obs, task_obs=self._task_obs,
            cell_reward=self._cell_reward, cell_ignition=self._cell_ignition, range_mask=self._range_mask,
            cell_agents=self._cell_agents,
            control=self._control, field_uniforms=self._uniforms[0], agent_uniforms=self._uniforms[1])
        for name, tensor in tensors.items():
            if tensor is not None:
                assert tensor.is_contiguous() and tensor.device == self.device, name
            setattr(io, name, _lib.pointer(tensor))
        io.mask_stride = self._mask_stride
        io.mask_words = self._range_mask.shape[-1]
        self._bound = tensors  # keeps every tensor alive for as long as the pointers are in use
        return io

    # ------------------------------------------------------------------------------------------ reset

    @torch.no_grad()
    def reset(self, seed=None, options: Dict[str, Any] = None) -> None:
        """Reference wildfire.py:291-373: build (or take) the initial state, save it, publish observations/actions."""
        super().reset(seed=seed, options=options)
        self._params.max_steps = self._horizon()
        fc, ac, dev = self.fire_config, self.agent_config, self.device
        init = self._initial
        if options is not None and options.get('initial_state') is not None:
            given = options['initial_state']
            if len(given) != self.parallel_envs:
                raise ValueError("Initial state must have the same number of environments as the parallel environments")
            for name in ('fires', 'intensity', 'fuel', 'suppressants', 'capacity', 'equipment'):
                getattr(init, name).copy_(getattr(given, name).to(dev))
        else:
            lit = torch.as_tensor(fc.lit, dtype=torch.bool).to(dev)
            fire_types = torch.as_tensor(fc.fire_types, dtype=torch.int32).to(dev)
            ignition = torch.as_tensor(fc.ignition_temp, dtype=torch.int32).to(dev)
            fires = torch.where(lit, fire_types, -fire_types)  # wildfire.py:347-348
            init.fires.copy_(fires.unsqueeze(0).expand_as(init.fires))
            init.intensity.copy_(torch.where(lit, ignition, torch.zeros_like(ignition)).unsqueeze(0).expand_as(init.fires))
            init.fuel.copy_(torch.where(fires != 0, int(fc.initial_fuel), 0).unsqueeze(0).expand_as(init.fires))
            init.suppressants.fill_(float(ac.initial_suppressant))
            init.capacity.fill_(float(ac.initial_capacity))
            init.equipment.fill_(int(ac.initial_equipment_state))
        self._state.initial_state = init
        self.fire_reduction_power = ac.fire_reduction_power
        self.suppressant_states = ac.suppressant_states
        self._reset_masked(None)
        self._snapshot_reset()
        self.infos = dict({agent: {} for agent in self.agents}, burnouts=self._burnouts, putouts=self._putouts)
        self._rebind_outputs()
        if self.log_directory is not None:
            self._log_environment(reset=True)

    def _reset_masked(self, mask: Optional[torch.Tensor]) -> None:
        """frz_wildfire_reset: restore initial rows, zero AEC fields (+ num_burnouts, wildfire.py:393), refresh."""
        _lib.check(self._lib.frz_wildfire_reset(ctypes.byref(self._params), ctypes.byref(self._io), self.parallel_envs,
                                                _lib.pointer(mask), self._stream()), 'frz_wildfire_reset')

    @classmethod
    def _autoreset_rows(cls) -> AutoresetRows:
        """A restart as wildfire_restore_kernel + refresh: state from init_*, the refresh's outputs from the snapshot,
        AEC fields and the burn-out total zeroed; rewards and the per-step burn-out / put-out counts are written for
        every environment by every step."""
        state = ('fires', 'intensity', 'fuel', 'suppressants', 'capacity', 'equipment')
        return AutoresetRows(
            init={name: f'init_{name}' for name in state},
            snapshot=('action_mask', 'self_obs', 'task_obs', 'env_task_count', 'agent_task_count'),
            zero=('cumulative_rewards', 'terminated', 'truncated', 'num_moves', 'num_burnouts'),
            overwritten=('rewards', 'burnouts', 'putouts'),
            static=tuple(f'init_{name}' for name in state) + (
                'actions', 'cell_reward', 'cell_ignition', 'range_mask', 'cell_agents', 'control', 'field_uniforms',
                'agent_uniforms'),
            agents_with_tasks=True,
            final=('self_obs', 'task_obs', 'action_mask', 'env_task_count', 'agent_task_count'))

    # ------------------------------------------------------------------------------------------ step

    def step_environment(self) -> Tuple[Dict[str, torch.Tensor], Dict[str, torch.Tensor], Dict[str, Dict]]:
        _lib.check(self._lib.frz_wildfire_step(ctypes.byref(self._params), ctypes.byref(self._io), self.parallel_envs,
                                               self._stream()), 'frz_wildfire_step')
        return self._reward_views, self.terminations, self.infos

    def _host_entry(self):
        return self._lib.frz_wildfire_step_host

    def _refresh(self) -> None:
        _lib.check(self._lib.frz_wildfire_refresh(ctypes.byref(self._params), ctypes.byref(self._io),
                                                  self.parallel_envs, self._stream()), 'frz_wildfire_refresh')

    def _observation_download(self, buffers=None):
        """Host-side observation download (``gather_observations``): self observations and per-agent task counts whole,
        the live rows of the task observations and of every agent's action-mask row packed."""
        b = self._observation_buffers() if buffers is None else buffers
        dense = dict(self_obs=b['self_obs'], agent_task_count=b['agent_task_count'])
        ragged = dict(task_obs=(b['task_obs'], 1), action_mask=(b['action_mask'], len(self.possible_agents)))
        return dense, ragged

    def _compact_schema(self, buffers=None):
        """Compact download (utils/compact.py): live task rows and the action mask as bits; of ``self_obs`` only the
        suppressant -- y, x and power are the configuration's and are restored by ``unpack()``."""
        b = self._observation_buffers() if buffers is None else buffers
        A, p = len(self.possible_agents), self._params
        bounds = compact_bounds(self.config)
        fill = torch.tensor([[float(p.agent_y[a]), float(p.agent_x[a]), p.agent_power[a], 0.0] for a in range(A)],
                            dtype=torch.float32)
        return compact.Schema(capacity=self.max_y * self.max_x, mask_groups=A, arrays=[
            compact.rows('task_obs', b['task_obs'], bound=bounds['task_obs']),
            compact.mask('action_mask', b['action_mask'], groups=A),
            compact.dense('self_obs', b['self_obs'], columns=(3, 1), fill=fill),
            compact.dense('agent_task_count', b['agent_task_count'], bound=bounds['agent_task_count']),
        ])

    def update_actions(self) -> None:
        """Recompute task counts / masks from the current state (wildfire.py:587-666). The fused step already does
        this; call it only after editing ``env.state()`` by hand."""
        self._refresh()

    def update_observations(self) -> None:
        """Recompute observations from the current state (wildfire.py:669-717); see ``update_actions``."""
        self._refresh()
        self.update_observation_views()

    def inject_uniforms(self, field: Optional[torch.Tensor], agent: Optional[torch.Tensor]) -> None:
        """Parity mode: use caller-supplied uniforms, shaped like the reference's ``generator.generate`` output
        (field f32 [3, B, H, W], agent f32 [5, B, A]; wildfire.py:409-410), instead of in-kernel Philox."""
        self._uniforms = (None if field is None else field.to(self.device, torch.float32).contiguous(),
                          None if agent is None else agent.to(self.device, torch.float32).contiguous())
        self._io = self._bind_buffers()

    def sample_actions(self, sampler_seed: int = 2026) -> torch.Tensor:
        _lib.check(self._lib.frz_wildfire_sample_actions(ctypes.byref(self._params), ctypes.byref(self._io),
                                                         self.parallel_envs, ctypes.c_uint64(sampler_seed),
                                                         self._stream()), 'frz_wildfire_sample_actions')
        return self._actions

    @property
    def action_slots(self) -> int:
        """H*W + 1: slot t < H*W acts on env-local task t (row t of ``tasks_padded``), slot H*W is the noop."""
        return int(self._params.height) * int(self._params.width) + 1

    def _policy_entry(self):
        return self._lib.frz_wildfire_policy_actions

    # ------------------------------------------------------------------------------------------ logging tap

    def _log_snapshot(self) -> Dict[str, torch.Tensor]:
        s = self._state
        return dict(super()._log_snapshot(), fires=s.fires, intensity=s.intensity, fuel=s.fuel,
                    suppressants=s.suppressants, capacity=s.capacity, equipment=s.equipment,
                    action_mask=self._action_mask, burnouts=self._burnouts, putouts=self._putouts)

    def _log_state_columns(self, host) -> Dict[str, Any]:
        """WildfireState.to_dataframe (utils/state.py:180-191): per-env cells, the shared agent positions last."""
        from free_range_zoo_b200.utils.logging_tap import nested
        B = self.parallel_envs
        columns = {name: [nested(host[name][b]) for b in range(B)]
                   for name in ('fires', 'intensity', 'fuel', 'suppressants', 'capacity', 'equipment')}
        columns['agents'] = [str(torch.as_tensor(self.agent_config.agents).tolist())] * B
        return columns

    def _log_mappings(self, host, agent_index: int):
        """(action map, observation map) cells: env-local task indices the agent may act on / observes."""
        from free_range_zoo_b200.utils.logging_tap import index_list
        counts = host['env_task_count']
        slots = np.arange(host['action_mask'].shape[2])[None, :] < counts[:, None]
        allowed = slots if self.show_bad_actions else (host['action_mask'][:, agent_index] != 0) & slots
        return [index_list(row) for row in allowed], [index_list(row) for row in slots]

    def _log_extra_columns(self, host, reset: bool) -> Dict[str, Any]:
        """wildfire.py:755-762: the per-step burn-out / put-out counters (absent from infos right after a reset)."""
        B = self.parallel_envs
        return {'burnouts': [None] * B if reset else host['burnouts'].tolist(),
                'putouts': [None] * B if reset else host['putouts'].tolist()}

    # ------------------------------------------------------------------------------------------ views

    @property
    def action_mask(self) -> torch.Tensor:
        """uint8 [B, A, H*W]: 1 iff the agent may fight env-local task t (in range and has suppressant)."""
        return self._action_mask[:, :, :self.max_y * self.max_x]

    @property
    def task_store(self) -> torch.Tensor:
        """Jagged int64 [B, #lit, 4] = (y, x, fires, intensity) like the reference (wildfire.py:699)."""
        return jagged_from_padded(self._task_obs, self.environment_task_count, torch.int64)

    def _observation_views(self, buffers) -> Dict[str, ObservationDict]:
        B = self.parallel_envs
        self_obs, task_obs, counts = buffers['self_obs'], buffers['task_obs'], buffers['env_task_count']
        action_mask = buffers['action_mask'][:, :, :self.max_y * self.max_x]
        tasks = LazyDict({'tasks': lambda: jagged_from_padded(task_obs, counts, torch.int64)})
        views = {}
        for agent, index in self.agent_name_mapping.items():
            others, columns = self._other_agents[agent], self._other_columns
            views[agent] = ObservationDict(
                {
                    'self': self_obs[:, index],
                    'others': (lambda o=others, c=columns: self_obs[:, o][:, :, c]),
                    'tasks': (lambda: tasks['tasks']),
                    'tasks_padded': task_obs,
                    'task_count': counts,
                    'action_mask': action_mask[:, index],
                },
                batch_size=[B],
                device=self.device,
            )
        return views

    def update_observation_views(self) -> None:
        self.observations = self._observation_views(self._observation_buffers())
        good = {a: (lambda i=i: jagged_indices_from_mask(self.action_mask[:, i] != 0))
                for a, i in self.agent_name_mapping.items()}
        every = LazyDict({'all': lambda: jagged_indices_from_mask(
            torch.arange(self.max_y * self.max_x, device=self.device).unsqueeze(0) < self.environment_task_count.unsqueeze(1))})
        lit_steps = lambda: torch.arange(self.max_y * self.max_x, device=self.device).unsqueeze(0) < \
            self.environment_task_count.unsqueeze(1)
        if self.show_bad_actions:  # wildfire.py:658-662
            self.agent_action_mapping = LazyDict({a: (lambda: every['all']) for a in self.agents})
            self.agent_bad_actions = LazyDict({
                a: (lambda i=i: jagged_indices_from_mask((self.action_mask[:, i] == 0) & lit_steps()))
                for a, i in self.agent_name_mapping.items()
            })
        else:
            self.agent_action_mapping = LazyDict(good)
            self.agent_bad_actions = {a: None for a in self.agents}
        self.agent_observation_mapping = LazyDict({a: (lambda: every['all']) for a in self.agents})

    # ------------------------------------------------------------------------------------------ spaces

    @torch.no_grad()
    def action_space(self, agent: str) -> BatchedActionSpace:
        """Per environment ``OneOf([Discrete(1, start=0)] * n + [Discrete(1, start=-1)])`` with n the number of tasks
        the agent may act on (reference wildfire.py:720-734, spaces/actions.py:10-41)."""
        if self.show_bad_actions:
            counts = self.environment_task_count
        else:
            counts = self._agent_task_count[:, self.agent_name_mapping[agent]]
        slots = torch.arange(self.max_y * self.max_x + 1, device=self.device, dtype=torch.int32).unsqueeze(0)
        starts = torch.where(slots == counts.unsqueeze(1), -1, 0).to(torch.int32)
        return BatchedActionSpace(starts, counts + 1)

    @torch.no_grad()
    def observation_space(self, agent: str) -> List[Space]:
        """Reference wildfire.py:736-753 + spaces/observations.py:11-101 (one ``Space.Dict`` per environment)."""
        agent_high, fire_high = self.agent_observation_bounds, self.fire_observation_bounds
        other_high = tuple(agent_high[i] for i in self._other_columns.tolist())
        A = len(self.agents)

        def single(num_tasks: int) -> Space:
            return Space.Dict({
                'self': Space.Box(low=[0] * 4, high=agent_high),
                'others': Space.Tuple([Space.Box(low=[0] * len(other_high), high=other_high) for _ in range(A - 1)]),
                'tasks': Space.Tuple([Space.Box(low=[0] * 4, high=fire_high) for _ in range(num_tasks)]),
            })

        cache: Dict[int, Space] = {}
        return [cache.setdefault(n, single(n)) for n in self.environment_task_count.tolist()]
