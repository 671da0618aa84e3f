"""rideshare_v0 on the B200 engine.

Public surface of the reference module (free_range_zoo/envs/rideshare/env/rideshare.py:98-504): ``parallel_env``,
``env``, ``raw_env``.  The reference's step (decode through padded nested mappings, ``unique`` loop for accept
conflicts, boolean-mask compaction, ``cat`` + stable ``argsort`` for entries, a dozen ``bincount`` calls) is replaced
by ``frz_rideshare_step`` -- one fused sm_100a launch over per-environment passenger tables.
"""
from __future__ import annotations

import ctypes
from typing import Any, Callable, Dict, List, Optional, Tuple

import numpy as np
import torch

from free_range_zoo_b200 import _lib
from free_range_zoo_b200.envs.rideshare.env.structures.state import RideshareState
from free_range_zoo_b200.utils.containers import (LazyDict, ObservationDict, jagged_indices_from_mask,
                                                  jagged_rows_from_mask)
from free_range_zoo_b200.utils.conversions import batched_aec_to_batched_parallel
from free_range_zoo_b200.utils import compact
from free_range_zoo_b200.utils.env import (AutoresetRows, BatchedAECEnv, InputKind, PolicyInputLayout,
                                           PolicyInputSchema, input_column)
from free_range_zoo_b200.utils.spaces import BatchedActionSpace, Space


def parallel_env(wrappers: List[Callable] = [], **kwargs):
    """Parallel-API rideshare environment (reference rideshare.py:98-114)."""
    env = raw_env(**kwargs)
    for wrapper in wrappers:
        env = wrapper(env)
    return batched_aec_to_batched_parallel(env)


def env(wrappers: List[Callable] = [], **kwargs):
    """AEC-API rideshare environment (reference rideshare.py:117-132)."""
    environment = raw_env(**kwargs)
    for wrapper in wrappers:
        environment = wrapper(environment)
    return environment


def _np(tensor, dtype):
    return np.ascontiguousarray(torch.as_tensor(tensor).detach().cpu().numpy().astype(dtype))


def flatten_configuration(config, max_steps, parallel_envs: int, env_offset: int = 0):
    """RideshareConfiguration -> (FrzRideshareParams, time-sorted schedule int32 [S, 7])."""
    ac, rc = config.agent_config, config.reward_config
    schedule = _np(config.passenger_config.schedule, np.int32).reshape(-1, 7)
    # stable sort by entry time: rows entering in the same step keep schedule order (passenger_entry.py:52,69-70)
    schedule = schedule[np.argsort(schedule[:, 0], kind='stable')]
    A = int(ac.start_positions.shape[0])
    if A > _lib.MAX_AGENTS:
        raise ValueError(f'rideshare configuration exceeds the engine limit of {_lib.MAX_AGENTS} agents')
    # rows an environment can ever hold: wildcard rows + rows addressed to it
    wildcard = int((schedule[:, 1] == -1).sum())
    local = schedule[(schedule[:, 1] >= env_offset) & (schedule[:, 1] < env_offset + parallel_envs), 1]
    addressed = int(np.bincount(local - env_offset).max()) if len(local) else 0
    capacity = max(1, min(wildcard + addressed, _lib.MAX_PASSENGERS))
    p = _lib.RideshareParams()
    p.num_agents, p.capacity, p.schedule_rows, p.pool_limit = A, capacity, len(schedule), int(ac.pool_limit)
    p.schedule_horizon = int(schedule[:, 0].max()) if len(schedule) else -1
    p.max_steps = 2**31 - 1 if max_steps is None else int(max_steps)
    p.flags = ((_lib.RS_FAST_TRAVEL if ac.use_fast_travel else 0) | (_lib.RS_DIAGONAL_TRAVEL if ac.use_diagonal_travel else 0) |
               (_lib.RS_VARIABLE_MOVE_COST if rc.use_variable_move_cost else 0) |
               (_lib.RS_WAITING_COSTS if rc.use_waiting_costs else 0))
    p.env_offset = env_offset
    for i, limit in enumerate(_np(rc.wait_limit, np.int64)):
        p.wait_limit[i] = int(limit)
    p.long_wait_time = int(rc.long_wait_time)
    for name in ('move_cost', 'drop_cost', 'noop_cost', 'accept_cost', 'pool_limit_cost', 'general_wait_cost',
                 'long_wait_cost'):
        setattr(p, name, float(getattr(rc, name)))
    return p, schedule


def compact_bounds(config, params, max_steps) -> Dict[str, int]:
    """Largest |value| of the integer observations, from the configuration (utils/compact.py picks the types): task
    rows (y, x, dest_y, dest_x, accepted_by, riding_by, fare, entered) hold grid positions, driver indices or the
    padding value, the schedule's fares and entry steps (at most the horizon); self observations (y, x, #accepted,
    #riding) grid positions and passenger counts."""
    H, W, A, K = int(config.grid_height), int(config.grid_width), int(params.num_agents), int(params.capacity)
    schedule = torch.as_tensor(config.passenger_config.schedule).reshape(-1, 7)
    max_fare = int(schedule[:, 6].abs().max()) if schedule.numel() else 0
    horizon = 2**31 - 1 if max_steps is None else max(int(max_steps), int(params.schedule_horizon))
    return dict(task_obs=max(H - 1, W - 1, A - 1, -_lib.PAD, max_fare, horizon), self_obs=max(H - 1, W - 1, K),
                agent_task_count=K)


def schedule_index(schedule: np.ndarray, horizon: int) -> np.ndarray:
    """index[t] = first row of the time-sorted schedule whose entry step is >= t, for t in [0, horizon + 1]."""
    return np.searchsorted(schedule[:, 0], np.arange(horizon + 2), side='left').astype(np.int32)


class raw_env(BatchedAECEnv):
    """Rideshare environment whose step is one fused CUDA kernel."""

    metadata = {"render.modes": ["human", "rgb_array"], "name": "rideshare_v0", "is_parallelizable": True,
                "render_fps": 2}

    @torch.no_grad()
    def __init__(self, *args, step_kernel: str = 'auto', **kwargs):
        """``step_kernel`` ('auto' | 'tiles' | 'groups') picks the step kernel: by batch size, or one of the two
        whatever the batch size (identical results; for tests and kernel timing -- include/frz.h FRZ_RS_KERNEL_*)."""
        super().__init__(*args, **kwargs)
        if step_kernel not in ('auto', 'tiles', 'groups'):
            raise ValueError(f"step_kernel must be 'auto', 'tiles' or 'groups', not {step_kernel!r}")
        A = int(self.agent_config.start_positions.shape[0])
        self.possible_agents = tuple(f'driver_{i}' for i in range(1, A + 1))
        self.agents = self.possible_agents
        self.agent_name_mapping = {agent: index for index, agent in enumerate(self.possible_agents)}
        self.max_x, self.max_y = int(self.config.grid_width), int(self.config.grid_height)
        self.agent_observation_bounds = (self.max_y, self.max_x, self.agent_config.pool_limit,
                                         self.agent_config.pool_limit)
        self.passenger_observation_bounds = (self.max_y, self.max_x, self.max_y, self.max_x, A, A, self.config.max_fare,
                                             self.max_steps)
        self._params, schedule = flatten_configuration(self.config, self.max_steps, self.parallel_envs, self.env_offset)
        self._params.flags |= {'auto': 0, 'tiles': _lib.RS_KERNEL_TILES, 'groups': _lib.RS_KERNEL_GROUPS}[step_kernel]
        B, K, dev = self.parallel_envs, self._params.capacity, self.device
        self._capacity = K
        self._allocate_runtime(A)
        i32 = torch.int32
        self._state = RideshareState(agents=torch.zeros((B, A, 2), dtype=i32, device=dev),
                                     passenger_table=torch.zeros((B, K, 11), dtype=i32, device=dev),
                                     passenger_count=self.environment_task_count)
        self._init_agents = torch.zeros((B, A, 2), dtype=i32, device=dev)
        self._init_passengers = torch.zeros((B, K, 11), dtype=i32, device=dev)
        self._init_count = torch.zeros(B, dtype=i32, device=dev)
        self._schedule = torch.from_numpy(schedule).to(dev) if len(schedule) else torch.zeros((1, 7), dtype=i32, device=dev)
        index = schedule_index(schedule, self._params.schedule_horizon) if len(schedule) else np.zeros(1, np.int32)
        self._schedule_index = torch.from_numpy(index).to(dev)
        self._task_mask = torch.zeros((B, A, K), dtype=torch.uint8, device=dev)
        self._self_obs = torch.zeros((B, A, 4), dtype=i32, device=dev)
        self._task_obs = torch.full((B, K, 8), _lib.PAD, dtype=i32, device=dev)
        self._other_agents = {
            agent: torch.tensor([i for i in range(A) if i != index], dtype=torch.int64, device=dev)
            for agent, index in self.agent_name_mapping.items()
        }
        self._io = self._bind_buffers()

    def _bind_buffers(self) -> _lib.RideshareBuffers:
        io = _lib.RideshareBuffers()
        tensors = dict(agents=self._state.agents, passengers=self._state.passenger_table, init_agents=self._init_agents,
                       init_passengers=self._init_passengers, init_count=self._init_count, schedule=self._schedule,
                       schedule_index=self._schedule_index,
                       actions=self._actions, rewards=self._rewards, cumulative_rewards=self._cumulative,
                       terminated=self._terminated, truncated=self._truncated, num_moves=self.num_moves,
                       env_task_count=self.environment_task_count, agent_task_count=self._agent_task_count,
                       task_mask=self._task_mask, self_obs=self._self_obs, task_obs=self._task_obs,
                       control=self._control)
        for name, tensor in tensors.items():
            assert tensor.is_contiguous() and tensor.device == self.device, name
            setattr(io, name, _lib.pointer(tensor))
        self._bound = tensors
        return io

    # ------------------------------------------------------------------------------------------ reset

    @torch.no_grad()
    def reset(self, seed=None, options: Optional[Dict[str, Any]] = None):
        """Reference rideshare.py:188-229: place the drivers, admit the t = 0 passengers, publish."""
        super().reset(seed=seed, options=options)
        self._params.max_steps = self._horizon()
        dev = self.device
        self._init_passengers.zero_()
        self._init_count.zero_()
        if options is not None and options.get('initial_state') is not None:
            given = options['initial_state']
            if len(given) != self.parallel_envs:
                raise ValueError("Initial state must have the same number of environments as the parallel environments")
            self._init_agents.copy_(given.agents.to(dev))
            flat = getattr(given, 'passengers', None)
            if flat is not None and flat.numel():
                flat = flat.to(dev).to(torch.int32)
                flat = flat[torch.argsort(flat[:, 0], stable=True)]
                batch = flat[:, 0].long()
                counts = torch.bincount(batch, minlength=self.parallel_envs)
                if int(counts.max()) > self._capacity:
                    raise ValueError(f'initial_state holds more than {self._capacity} passengers in one environment')
                starts = torch.cumsum(counts, 0) - counts
                slot = torch.arange(flat.shape[0], device=dev) - starts[batch]
                self._init_passengers[batch, slot] = flat
                self._init_count.copy_(counts.to(torch.int32))
        else:
            starts = torch.as_tensor(self.agent_config.start_positions, dtype=torch.int32).to(dev)
            self._init_agents.copy_(starts.unsqueeze(0).expand_as(self._init_agents))
        self._reset_masked(None)
        self._snapshot_reset()
        self._rebind_outputs()
        if self.log_directory is not None:
            self._log_environment(reset=True)

    def _reset_masked(self, mask: Optional[torch.Tensor]) -> None:
        _lib.check(self._lib.frz_rideshare_reset(ctypes.byref(self._params), ctypes.byref(self._io), self.parallel_envs,
                                                 _lib.pointer(mask), self._stream()), 'frz_rideshare_reset')

    @classmethod
    def _autoreset_rows(cls) -> AutoresetRows:
        """A restart as rideshare_restore_kernel + the t = 0 entry: drivers from init_agents; the passenger table and its
        count after the entry, like the observations, masks and counts, from the snapshot (the t = 0 entry depends on
        the schedule and the environment's index only); AEC fields zeroed; rewards written by every step."""
        return AutoresetRows(
            init={'agents': 'init_agents'},
            snapshot=('passengers', 'env_task_count', 'agent_task_count', 'task_mask', 'self_obs', 'task_obs'),
            zero=('cumulative_rewards', 'terminated', 'truncated', 'num_moves'),
            overwritten=('rewards', ),
            static=('init_agents', 'init_passengers', 'init_count', 'schedule', 'schedule_index', 'actions', 'control'),
            agents_with_tasks=True,
            final=('self_obs', 'task_obs', 'task_mask', 'env_task_count', 'agent_task_count'))

    # ------------------------------------------------------------------------------------------ step

    def step_environment(self) -> Tuple[Dict[str, torch.Tensor], Dict[str, torch.Tensor], Dict[str, Dict]]:
        _lib.check(self._lib.frz_rideshare_step(ctypes.byref(self._params), ctypes.byref(self._io), self.parallel_envs,
                                                self._stream()), 'frz_rideshare_step')
        return self._reward_views, self.terminations, self.infos

    def _host_entry(self):
        return self._lib.frz_rideshare_step_host

    def _refresh(self) -> None:
        _lib.check(self._lib.frz_rideshare_refresh(ctypes.byref(self._params), ctypes.byref(self._io),
                                                   self.parallel_envs, self._stream()), 'frz_rideshare_refresh')

    def _observation_download(self, buffers=None):
        """Host-side observation download (``gather_observations``): self observations and per-driver task counts whole,
        the live rows of the task observations and of every driver's task-mask row packed."""
        b = self._observation_buffers() if buffers is None else buffers
        dense = dict(self_obs=b['self_obs'], agent_task_count=b['agent_task_count'])
        ragged = dict(task_obs=(b['task_obs'], 1), task_mask=(b['task_mask'], len(self.possible_agents)))
        return dense, ragged

    def _compact_schema(self, buffers=None):
        """Compact download (utils/compact.py): live task rows, the task mask as bits, self observations and counts."""
        b = self._observation_buffers() if buffers is None else buffers
        A = len(self.possible_agents)
        bounds = compact_bounds(self.config, self._params, self.max_steps)
        return compact.Schema(capacity=self._capacity, mask_groups=A, arrays=[
            compact.rows('task_obs', b['task_obs'], bound=bounds['task_obs']),
            compact.mask('task_mask', b['task_mask'], groups=A),
            compact.dense('self_obs', b['self_obs'], bound=bounds['self_obs']),
            compact.dense('agent_task_count', b['agent_task_count'], bound=bounds['agent_task_count']),
        ])

    def update_actions(self) -> None:
        """Recompute task lists from the current table (rideshare.py:368-395); only needed after manual edits."""
        self._refresh()

    def update_observations(self) -> None:
        """Recompute observations from the current table (rideshare.py:398-467); only needed after manual edits."""
        self._refresh()
        self.update_observation_views()

    def sample_actions(self, sampler_seed: int = 2026) -> torch.Tensor:
        _lib.check(self._lib.frz_rideshare_sample_actions(ctypes.byref(self._params), ctypes.byref(self._io),
                                                          self.parallel_envs, ctypes.c_uint64(sampler_seed),
                                                          self._stream()), 'frz_rideshare_sample_actions')
        return self._actions

    @property
    def action_slots(self) -> int:
        """K + 1: slot t < K acts on passenger-table row t with the id its state requires, slot K is the noop."""
        return int(self._params.capacity) + 1

    def _policy_entry(self):
        return self._lib.frz_rideshare_policy_actions

    # the task columns accepted_by / riding_by hold a driver index or FRZ_PAD for nobody
    _NONE_TASK_COLUMNS = (False, ) * 4 + (True, True) + (False, ) * 2

    def _policy_input_layout(self) -> PolicyInputLayout:
        """Self (y, x, #accepted, #riding), the same four of every other driver; every passenger row, one view."""
        p = self._params
        return PolicyInputLayout(kinds=(InputKind(int(p.num_agents), 4, (0, 1, 2, 3)), ), task_rows=int(p.capacity),
                                 views=1, task_columns=self._NONE_TASK_COLUMNS)

    def _policy_input_schema(self) -> PolicyInputSchema:
        """``1 / high`` of ``agent_observation_bounds`` and ``passenger_observation_bounds``; accepted_by / riding_by
        map nobody to 0 and driver i to (i + 1) / (A + 1)."""
        return PolicyInputSchema(self._policy_input_layout(),
                                 self_columns=(tuple(input_column(h) for h in self.agent_observation_bounds), ),
                                 task_columns=tuple(input_column(h, none) for h, none in
                                                    zip(self.passenger_observation_bounds, self._NONE_TASK_COLUMNS)))

    def _inputs_entry(self):
        return self._lib.frz_rideshare_policy_inputs

    # ------------------------------------------------------------------------------------------ logging tap

    def _log_snapshot(self) -> Dict[str, torch.Tensor]:
        return dict(super()._log_snapshot(), agents=self._state.agents, passengers=self._state.passenger_table,
                    task_mask=self._task_mask)

    def _log_state_columns(self, host) -> Dict[str, Any]:
        """RideshareState.to_dataframe (envs/rideshare/env/structures/state.py:50-66): driver positions, then the rows of
        the passenger table that belong to the environment (with their batch column)."""
        from free_range_zoo_b200.utils.logging_tap import nested
        B = self.parallel_envs
        counts = host['env_task_count']
        return {'agents': [nested(host['agents'][b]) for b in range(B)],
                'passengers': [nested(host['passengers'][b, :counts[b]]) for b in range(B)]}

    def _log_mappings(self, host, agent_index: int):
        from free_range_zoo_b200.utils.logging_tap import index_list
        cells = [index_list(row) for row in host['task_mask'][:, agent_index] != 0]
        return cells, cells  # rideshare.py:394-395: the observation mapping is the action mapping

    # ------------------------------------------------------------------------------------------ views

    @property
    def task_mask(self) -> torch.Tensor:
        """bool [B, A, K]: table row p is in the agent's task list (unaccepted, or associated with the agent)."""
        return self._task_mask.view(torch.bool)

    @property
    def task_store(self) -> torch.Tensor:
        """Jagged int32 [B, #passengers, 8] like the reference (rideshare.py:418-422)."""
        rows = torch.arange(self._capacity, device=self.device).unsqueeze(0) < self.environment_task_count.unsqueeze(1)
        return jagged_rows_from_mask(self._task_obs, rows)

    def _observation_views(self, buffers) -> Dict[str, ObservationDict]:
        B = self.parallel_envs
        self_obs, task_obs, task_mask = buffers['self_obs'], buffers['task_obs'], buffers['task_mask'].view(torch.bool)
        views = {}
        for agent, index in self.agent_name_mapping.items():
            others = self._other_agents[agent]
            views[agent] = ObservationDict(
                {
                    'self': self_obs[:, index],
                    'others': (lambda o=others: self_obs[:, o]),
                    'tasks': (lambda i=index: jagged_rows_from_mask(task_obs, task_mask[:, i])),
                    'tasks_padded': task_obs,
                    'task_mask': task_mask[:, index],
                },
                batch_size=[B],
                device=self.device,
            )
        return views

    def update_observation_views(self) -> None:
        self.observations = self._observation_views(self._observation_buffers())
        mapping = {a: (lambda i=i: jagged_indices_from_mask(self.task_mask[:, i])) for a, i in self.agent_name_mapping.items()}
        self.agent_action_mapping = LazyDict(dict(mapping))
        self.agent_observation_mapping = LazyDict(dict(mapping))
        self.agent_bad_actions = {a: None for a in self.agents}

    # ------------------------------------------------------------------------------------------ spaces

    def _task_states(self) -> torch.Tensor:
        """Passenger state (0 unaccepted, 1 accepted, 2 riding) of every table row, from the observation columns."""
        accepted_by, riding_by = self._task_obs[:, :, 4], self._task_obs[:, :, 5]
        return torch.where(riding_by != _lib.PAD, 2, torch.where(accepted_by != _lib.PAD, 1, 0)).to(torch.int32)

    @torch.no_grad()
    def action_space(self, agent: str) -> BatchedActionSpace:
        """Per environment ``OneOf([Discrete(1, start=state_i) for the agent's tasks] + [Discrete(1, start=-1)])``
        (reference rideshare.py:470-487, spaces/actions.py:10-50)."""
        index = self.agent_name_mapping[agent]
        K = self._capacity
        mask = self.task_mask[:, index]
        position = torch.cumsum(mask, dim=1) - 1
        position = torch.where(mask, position, K + 1)  # rows outside the list land in a scratch column
        starts = torch.full((self.parallel_envs, K + 2), -1, dtype=torch.int32, device=self.device)
        starts.scatter_(1, position, self._task_states())
        return BatchedActionSpace(starts[:, :K + 1].contiguous(), self._agent_task_count[:, index] + 1)

    @torch.no_grad()
    def observation_space(self, agent: str) -> List[Space]:
        """Reference rideshare.py:489-504 + spaces/observations.py:5-88 (one ``Space.Dict`` per environment)."""
        agent_high, passenger_high = self.agent_observation_bounds, self.passenger_observation_bounds
        A = len(self.agents)

        def single(num_tasks: int) -> Space:
            return Space.Dict({
                'self': Space.Box(low=[0] * 4, high=agent_high),
                'others': Space.Tuple([Space.Box(low=[0] * 4, high=agent_high) for _ in range(A - 1)]),
                'tasks': Space.Tuple([Space.Box(low=[0] * 8, high=passenger_high) for _ in range(num_tasks)]),
            })

        cache: Dict[int, Space] = {}
        counts = self._agent_task_count[:, self.agent_name_mapping[agent]].tolist()
        return [cache.setdefault(n, single(n)) for n in counts]
