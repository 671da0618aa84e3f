"""cybersecurity_v0 on the B200 engine.

Public surface of the reference module (free_range_zoo/envs/cybersecurity/env/cybersecurity.py:112-584):
``parallel_env``, ``env``, ``raw_env`` with the same constructor flags.  The Python step (per-agent decode loop with
host-synchronising ValueError guards, three ``nn.Module`` transitions, per-agent clones of the task store) is replaced
by ``frz_cyber_step`` -- one fused sm_100a launch; the ValueError conditions become device-side fault bits that
``env.check_errors()`` reports.
"""
from __future__ import annotations

import ctypes
from typing import Any, Callable, Dict, List, Optional, Tuple

import numpy as np
import torch

from free_range_zoo_b200 import _lib
from free_range_zoo_b200.envs.cybersecurity.env.structures.state import CybersecurityState
from free_range_zoo_b200.utils.containers import LazyDict, ObservationDict, jagged_indices_from_mask
from free_range_zoo_b200.utils.conversions import batched_aec_to_batched_parallel
from free_range_zoo_b200.utils import compact
from free_range_zoo_b200.utils.env import AutoresetRows, BatchedAECEnv
from free_range_zoo_b200.utils.spaces import BatchedActionSpace, Space


def parallel_env(wrappers: List[Callable] = [], **kwargs):
    """Parallel-API cybersecurity environment (reference cybersecurity.py:112-128)."""
    env = raw_env(**kwargs)
    for wrapper in wrappers:
        env = wrapper(env)
    return batched_aec_to_batched_parallel(env)


def env(wrappers: List[Callable] = [], **kwargs):
    """AEC-API cybersecurity environment (reference cybersecurity.py:131-146)."""
    environment = raw_env(**kwargs)
    for wrapper in wrappers:
        environment = wrapper(environment)
    return environment


def _np(tensor, dtype):
    return np.ascontiguousarray(torch.as_tensor(tensor).detach().cpu().numpy().astype(dtype))


def danger_score_table(threat: np.ndarray, mitigation: np.ndarray, temperature: float) -> torch.Tensor:
    """tanh((patches - attacks) / T) for every set of agents that can act on one node (index bit a = agent a,
    attackers first).  Sums run in agent order like the reference's decode loop (cybersecurity.py:350,375) and the
    tanh is torch's CPU tanh -- the routine the reference itself calls (transitions/subnetwork.py:53-54)."""
    n_att, n_def = len(threat), len(mitigation)
    size = 1 << (n_att + n_def)
    attacks = np.zeros(size, dtype=np.float32)
    patches = np.zeros(size, dtype=np.float32)
    for index in range(size):
        for a in range(n_att):
            if index >> a & 1:
                attacks[index] = np.float32(attacks[index] + threat[a])
        for d in range(n_def):
            if index >> (n_att + d) & 1:
                patches[index] = np.float32(patches[index] + mitigation[d])
    difference = torch.from_numpy(patches - attacks)
    return torch.tanh(difference / torch.tensor(temperature, dtype=torch.float32))


def flatten_configuration(config, max_steps, show_bad_actions: bool, env_offset: int = 0):
    """CybersecurityConfiguration -> (FrzCyberParams, score LUT or None)."""
    ac, dc, nc, rc = config.attacker_config, config.defender_config, config.network_config, config.reward_config
    threat, mitigation = _np(ac.threat, np.float32), _np(dc.mitigation, np.float32)
    n_att, n_def = len(threat), len(mitigation)
    N = int(nc.adj_matrix.shape[0])
    num_states = int(nc.patched_states + nc.vulnerable_states + nc.exploited_states)
    if N > _lib.MAX_NODES or n_att + n_def > _lib.MAX_AGENTS or num_states > _lib.MAX_NET_STATES:
        raise ValueError(f'cybersecurity configuration exceeds the engine limits: nodes={N} (<= {_lib.MAX_NODES}), '
                         f'agents={n_att + n_def} (<= {_lib.MAX_AGENTS}), states={num_states}')
    p = _lib.CyberParams()
    p.num_nodes, p.num_attackers, p.num_defenders, p.num_states = N, n_att, n_def, num_states
    p.max_steps = 2**31 - 1 if max_steps is None else int(max_steps)
    p.flags = (_lib.CY_STOCHASTIC_STATE if config.stochastic_config.network_state else 0) | \
        (_lib.CY_SHOW_BAD_ACTIONS if show_bad_actions else 0)
    p.env_offset = env_offset
    p.temperature = float(nc.temperature)
    p.patch_reward = float(rc.patch_reward)
    p.bad_action_penalty = float(rc.bad_action_penalty)
    persist = np.concatenate([_np(ac.persist_probs, np.float32), _np(dc.persist_probs, np.float32)])
    returns = np.concatenate([_np(ac.return_probs, np.float32), _np(dc.return_probs, np.float32)])
    power = np.concatenate([threat, mitigation])
    for a in range(n_att + n_def):
        p.power[a], p.persist[a], p.returns[a] = float(power[a]), float(persist[a]), float(returns[a])
    for s, value in enumerate(_np(rc.network_state_rewards, np.float32)):
        p.state_rewards[s] = float(value)
    criticality = _np(nc.adj_matrix, np.int64).sum(axis=1)
    for n in range(N):
        p.criticality[n] = float(criticality[n])
    lut = None
    if n_att + n_def <= _lib.CY_MAX_LUT_BITS:
        lut = danger_score_table(threat, mitigation, float(nc.temperature))
        p.lut_bits = n_att + n_def
    return p, lut


def compact_bounds(params) -> Dict[str, int]:
    """Largest |value| of the integer observations, from the configuration (utils/compact.py picks the types): task
    rows hold (state, criticality), task counts at most every subnetwork."""
    N = int(params.num_nodes)
    criticality = max(abs(int(params.criticality[n])) for n in range(N))
    return dict(task_obs=max(int(params.num_states) - 1, criticality), agent_task_count=N)


class raw_env(BatchedAECEnv):
    """Cybersecurity environment whose step is one fused CUDA kernel."""

    metadata = {"render.modes": ["human", "rgb_array"], "name": "cybersecurity_v0", "is_parallelizable": True,
                "render_fps": 2, "null_value": -100}

    @torch.no_grad()
    def __init__(self, *args, observe_other_location: bool = False, observe_other_presence: bool = False,
                 observe_other_power: bool = True, partially_observable: bool = True, show_bad_actions: bool = True,
                 **kwargs) -> None:
        super().__init__(*args, **kwargs)
        self.observe_other_power = observe_other_power
        self.observe_other_location = observe_other_location
        self.observe_other_presence = observe_other_presence
        self.partially_obserable = partially_observable  # (sic) attribute name of the reference, cybersecurity.py:191
        self.partially_observable = partially_observable
        self.show_bad_actions = show_bad_actions

        n_att = int(self.attacker_config.threat.shape[0])
        n_def = int(self.defender_config.mitigation.shape[0])
        self._n_att, self._n_def, self._n_nodes = n_att, n_def, int(self.network_config.adj_matrix.shape[0])
        attackers = tuple(f"attacker_{i}" for i in range(1, n_att + 1))
        defenders = tuple(f"defender_{i}" for i in range(1, n_def + 1))
        self.possible_agents = attackers + defenders
        self.agents = self.possible_agents
        self.attacker_name_mapping = dict(zip(attackers, range(n_att)))
        self.defender_name_mapping = dict(zip(defenders, range(n_def)))
        self.agent_name_mapping = {**self.attacker_name_mapping, **self.defender_name_mapping}
        self.offset_agent_name_mapping = dict(zip(self.possible_agents, range(n_att + n_def)))
        dev = self.device
        columns = lambda flags: torch.tensor([i for i, on in enumerate(flags) if on], dtype=torch.int64, device=dev)
        self._attacker_columns = columns((observe_other_power, observe_other_presence))  # env/utils/masking.py:7-28
        self._defender_columns = columns((observe_other_power, observe_other_presence, observe_other_location))

        self._params, lut = flatten_configuration(self.config, self.max_steps, show_bad_actions, self.env_offset)
        B, N, n = self.parallel_envs, self._n_nodes, n_att + n_def
        self._allocate_runtime(n)
        i32, f32, u8 = torch.int32, torch.float32, torch.uint8
        self._presence = torch.zeros((B, n), dtype=u8, device=dev)
        self._state = CybersecurityState(network_state=torch.zeros((B, N), dtype=i32, device=dev),
                                         location=torch.zeros((B, n_def), dtype=i32, device=dev),
                                         presence=self._presence.view(torch.bool))
        self._init_network = torch.zeros((B, N), dtype=i32, device=dev)
        self._init_location = torch.zeros((B, n_def), dtype=i32, device=dev)
        self._init_presence = torch.zeros((B, n), dtype=u8, device=dev)
        self._attacker_self = torch.zeros((B, n_att, 2), dtype=f32, device=dev)
        self._defender_self = torch.zeros((B, n_def, 3), dtype=f32, device=dev)
        self._task_obs = torch.zeros((B, N, 2), dtype=i32, device=dev)
        self._monitored = torch.zeros((B, n_def), dtype=u8, device=dev)
        self._score_lut = None if lut is None else lut.to(dev).contiguous()
        self._uniforms = (None, None)
        self._io = self._bind_buffers()

    def _bind_buffers(self) -> _lib.CyberBuffers:
        s = self._state
        io = _lib.CyberBuffers()
        tensors = dict(network_state=s.network_state, location=s.location, presence=self._presence,
                       init_network_state=self._init_network, init_location=self._init_location,
                       init_presence=self._init_presence, actions=self._actions, rewards=self._rewards,
                       cumulative_rewards=self._cumulative, terminated=self._terminated, truncated=self._truncated,
                       num_moves=self.num_moves, env_task_count=self.environment_task_count,
                       agent_task_count=self._agent_task_count, attacker_self=self._attacker_self,
                       defender_self=self._defender_self, task_obs=self._task_obs, monitored=self._monitored,
                       score_lut=self._score_lut, control=self._control, network_uniforms=self._uniforms[0],
                       agent_uniforms=self._uniforms[1])
        for name, tensor in tensors.items():
            if tensor is not None:
                assert tensor.is_contiguous() and tensor.device == self.device, name
            setattr(io, name, _lib.pointer(tensor))
        self._bound = tensors
        return io

    # ------------------------------------------------------------------------------------------ reset

    @torch.no_grad()
    def reset(self, seed=None, options: Dict[str, Any] = None) -> None:
        """Reference cybersecurity.py:222-271."""
        super().reset(seed=seed, options=options)
        self._params.max_steps = self._horizon()
        dev = self.device
        if options is not None and options.get('initial_state') is not None:
            given = options['initial_state']
            if len(given) != self.parallel_envs:
                raise ValueError("Initial state must have the same number of environments as the parallel environments")
            self._init_network.copy_(given.network_state.to(dev))
            self._init_location.copy_(given.location.to(dev))
            self._init_presence.copy_(given.presence.to(dev).to(torch.uint8))
        else:
            self._init_network.copy_(torch.as_tensor(self.network_config.initial_state, dtype=torch.int32).to(dev)
                                     .unsqueeze(0).expand_as(self._init_network))
            self._init_location.copy_(torch.as_tensor(self.defender_config.initial_location, dtype=torch.int32).to(dev)
                                      .unsqueeze(0).expand_as(self._init_location))
            self._init_presence.copy_(torch.as_tensor(self.config.initial_presence).to(dev).to(torch.uint8)
                                      .unsqueeze(0).expand_as(self._init_presence))
        self._actions.fill_(-2)  # cybersecurity.py:233-236
        self._reset_masked(None)
        self._snapshot_reset()
        self._rebind_outputs()
        if self.log_directory is not None:
            self._log_environment(reset=True)

    def _reset_masked(self, mask: Optional[torch.Tensor]) -> None:
        _lib.check(self._lib.frz_cyber_reset(ctypes.byref(self._params), ctypes.byref(self._io), self.parallel_envs,
                                             _lib.pointer(mask), self._stream()), 'frz_cyber_reset')

    # ------------------------------------------------------------------------------------------ logging tap

    def _log_snapshot(self) -> Dict[str, torch.Tensor]:
        s = self._state
        return dict(super()._log_snapshot(), network_state=s.network_state, location=s.location, presence=self._presence)

    def _log_state_columns(self, host) -> Dict[str, Any]:
        """CybersecurityState.to_dataframe (utils/state.py:180-191): network state, defender locations, presence."""
        from free_range_zoo_b200.utils.logging_tap import nested
        B = self.parallel_envs
        return {'network_state': [nested(host['network_state'][b]) for b in range(B)],
                'location': [nested(host['location'][b]) for b in range(B)],
                'presence': [nested(host['presence'][b] != 0) for b in range(B)]}

    def _log_mappings(self, host, agent_index: int):
        """cybersecurity.py:428-457: a present agent may act on every node, an absent one on none; the observation
        mapping is the full node range wrapped in one more list (it is a [1, N] slice of a nested tensor)."""
        nodes = list(range(self._n_nodes))
        present = host['agent_task_count'][:, agent_index] > 0
        return [str(nodes if here else []) for here in present], [str([nodes])] * self.parallel_envs

    def _log_extra_columns(self, host, reset: bool) -> Dict[str, Any]:
        """cybersecurity.py:580-584: the adjacency matrix on every row."""
        adjacency = str(torch.as_tensor(self.network_config.adj_matrix).int().tolist())
        return {'adj_matrix': [adjacency] * self.parallel_envs}

    @classmethod
    def _autoreset_rows(cls) -> AutoresetRows:
        """A restart as cyber_restore_kernel + refresh: state from init_*, the refresh's outputs from the snapshot,
        AEC fields and ``monitored`` (the last actions are -2 again) zeroed; rewards written by every step.  The domain
        has no per-agent skip: agents_with_tasks stays 0."""
        return AutoresetRows(
            init={'network_state': 'init_network_state', 'location': 'init_location', 'presence': 'init_presence'},
            snapshot=('env_task_count', 'agent_task_count', 'attacker_self', 'defender_self', 'task_obs'),
            zero=('monitored', 'cumulative_rewards', 'terminated', 'truncated', 'num_moves'),
            overwritten=('rewards', ),
            static=('init_network_state', 'init_location', 'init_presence', 'actions', 'score_lut', 'control',
                    'network_uniforms', 'agent_uniforms'),
            agents_with_tasks=False,
            final=('attacker_self', 'defender_self', 'task_obs', 'monitored', 'env_task_count', 'agent_task_count'))

    # ------------------------------------------------------------------------------------------ step

    def step_environment(self) -> Tuple[Dict[str, torch.Tensor], Dict[str, torch.Tensor], Dict[str, Dict]]:
        _lib.check(self._lib.frz_cyber_step(ctypes.byref(self._params), ctypes.byref(self._io), self.parallel_envs,
                                            self._stream()), 'frz_cyber_step')
        return self._reward_views, self.terminations, self.infos

    def _host_entry(self):
        return self._lib.frz_cyber_step_host

    def _refresh(self) -> None:
        _lib.check(self._lib.frz_cyber_refresh(ctypes.byref(self._params), ctypes.byref(self._io), self.parallel_envs,
                                               self._stream()), 'frz_cyber_refresh')

    def _observation_download(self, buffers=None):
        """Host-side observation download (``gather_observations``): every environment always has all N subnetworks as
        tasks, so everything is dense."""
        b = self._observation_buffers() if buffers is None else buffers
        dense = dict(attacker_self=b['attacker_self'], defender_self=b['defender_self'], task_obs=b['task_obs'],
                     monitored=b['monitored'], agent_task_count=b['agent_task_count'])
        return dense, {}

    def _compact_schema(self, buffers=None):
        """Compact download (utils/compact.py): task rows and counts narrowed; the float arrays and ``monitored`` as
        they are.  Every environment has all subnetworks as tasks, so everything is dense."""
        b = self._observation_buffers() if buffers is None else buffers
        bounds = compact_bounds(self._params)
        return compact.Schema(capacity=int(self._params.num_nodes), arrays=[
            compact.dense('attacker_self', b['attacker_self']),
            compact.dense('defender_self', b['defender_self']),
            compact.dense('task_obs', b['task_obs'], bound=bounds['task_obs']),
            compact.dense('monitored', b['monitored']),
            compact.dense('agent_task_count', b['agent_task_count'], bound=bounds['agent_task_count']),
        ])

    def update_actions(self) -> None:
        """Recompute task counts from the current state (cybersecurity.py:414-457); only needed after manual edits."""
        self._refresh()

    def update_observations(self) -> None:
        """Recompute observations from the current state (cybersecurity.py:460-526); only needed after manual edits."""
        self._refresh()
        self.update_observation_views()

    def inject_uniforms(self, network: Optional[torch.Tensor], agent: Optional[torch.Tensor]) -> None:
        """Parity mode: caller-supplied uniforms shaped like ``generator.generate`` output (network f32 [1, B, N],
        agent f32 [1, B, Att+D]; cybersecurity.py:304-315) instead of in-kernel Philox."""
        self._uniforms = (None if network is None else network.to(self.device, torch.float32).contiguous(),
                          None if agent is None else agent.to(self.device, torch.float32).contiguous())
        self._io = self._bind_buffers()

    def sample_actions(self, sampler_seed: int = 2026) -> torch.Tensor:
        _lib.check(self._lib.frz_cyber_sample_actions(ctypes.byref(self._params), ctypes.byref(self._io),
                                                      self.parallel_envs, ctypes.c_uint64(sampler_seed), self._stream()),
                   'frz_cyber_sample_actions')
        return self._actions

    @property
    def action_slots(self) -> int:
        """N + 3 for every agent: slot t < N attacks / moves to node t, then noop, patch and monitor (the last two are
        never legal for attackers)."""
        return int(self._params.num_nodes) + 3

    def _policy_entry(self):
        return self._lib.frz_cyber_policy_actions

    # ------------------------------------------------------------------------------------------ views

    @property
    def task_store(self) -> torch.Tensor:
        """int64 [B, N, 2] = (state, criticality), like the reference (cybersecurity.py:488)."""
        return self._task_obs.to(torch.int64)

    def _tasks_for(self, agent: str, buffers):
        """A defender under partial observability sees -100 unless its last action was monitor (:497,510-511)."""
        task_obs, monitored = buffers['task_obs'], buffers['monitored']
        if agent in self.defender_name_mapping and self.partially_observable:
            d = self.defender_name_mapping[agent]
            return lambda: torch.where(monitored[:, d].view(-1, 1, 1) != 0, task_obs, -100).to(torch.int64)
        return lambda: task_obs.to(torch.int64)

    def _other_indices(self, count: int, index: int) -> torch.Tensor:
        """Indices of the other agents of the same kind (device tensors built once: this runs every step)."""
        cache = self.__dict__.setdefault('_other_index_cache', {})
        if (count, index) not in cache:
            cache[(count, index)] = torch.tensor([i for i in range(count) if i != index], dtype=torch.int64,
                                                 device=self.device)
        return cache[(count, index)]

    def _node_indices(self) -> torch.Tensor:
        if getattr(self, '_node_index_cache', None) is None:
            self._node_index_cache = torch.arange(self._n_nodes, device=self.device).unsqueeze(0)
        return self._node_index_cache

    def _observation_views(self, buffers) -> Dict[str, ObservationDict]:
        B = self.parallel_envs
        views = {}
        for agent in self.agents:
            if agent in self.attacker_name_mapping:
                index, table, columns, count = (self.attacker_name_mapping[agent], buffers['attacker_self'],
                                                self._attacker_columns, self._n_att)
            else:
                index, table, columns, count = (self.defender_name_mapping[agent], buffers['defender_self'],
                                                self._defender_columns, self._n_def)
            others = self._other_indices(count, index)
            views[agent] = ObservationDict(
                {
                    'self': table[:, index],
                    'others': (lambda t=table, o=others, c=columns: t[:, o][:, :, c]),
                    'tasks': self._tasks_for(agent, buffers),
                },
                batch_size=[B],
                device=self.device,
            )
        return views

    def update_observation_views(self) -> None:
        B = self.parallel_envs
        self.observations = self._observation_views(self._observation_buffers())
        nodes = self._node_indices()
        self.agent_action_mapping = LazyDict({
            a: (lambda i=i: jagged_indices_from_mask(nodes < self._agent_task_count[:, i].unsqueeze(1)))
            for a, i in self.offset_agent_name_mapping.items()
        })
        self.agent_observation_mapping = LazyDict({
            a: (lambda: jagged_indices_from_mask(nodes.expand(B, -1) >= 0)) for a in self.agents
        })
        self.agent_bad_actions = {a: None for a in self.agents}

    # ------------------------------------------------------------------------------------------ spaces

    @torch.no_grad()
    def action_space(self, agent: str) -> BatchedActionSpace:
        """Reference cybersecurity.py:529-551 + spaces/actions.py:11-99: attackers [attack x n, noop]; defenders
        [move x n, noop, patch, monitor] (patch hidden at the home node unless show_bad_actions)."""
        slot = self.offset_agent_name_mapping[agent]
        counts = self.environment_task_count if self.show_bad_actions else self._agent_task_count[:, slot]
        N = self._n_nodes
        slots = torch.arange(N + 3, device=self.device, dtype=torch.int32).unsqueeze(0)
        offset = slots - counts.unsqueeze(1)  # 0 -> noop, 1 / 2 -> patch / monitor
        if agent in self.attacker_name_mapping:
            starts = torch.where(offset == 0, -1, 0)
            return BatchedActionSpace(starts.to(torch.int32), counts + 1)
        location = self._state.location[:, self.defender_name_mapping[agent]]
        can_patch = torch.ones_like(location, dtype=torch.bool) if self.show_bad_actions else location != -1
        second = torch.where(can_patch, -2, -3).unsqueeze(1)
        starts = torch.where(offset <= 0, torch.where(offset == 0, -1, 0), torch.where(offset == 1, second, -3))
        present = counts > 0
        choices = torch.where(present, counts + 2 + can_patch.to(torch.int32), 1)
        return BatchedActionSpace(starts.to(torch.int32), choices.to(torch.int32))

    @torch.no_grad()
    def observation_space(self, agent: str) -> List[Space]:
        """Reference cybersecurity.py:553-576 + spaces/observations.py:7-165 (identical for every environment)."""
        config = self.config
        is_attacker = agent in self.attacker_name_mapping
        own_high = config.attacker_observation_bounds if is_attacker else config.defender_observation_bounds
        columns = (self._attacker_columns if is_attacker else self._defender_columns).tolist()
        other_high = tuple(own_high[i] for i in columns)
        others = (self._n_att if is_attacker else self._n_def) - 1
        network_high = config.network_observation_bounds
        space = Space.Dict({
            'self': Space.Box(low=[0] * len(own_high), high=own_high),
            'others': Space.Tuple([Space.Box(low=[0] * len(other_high), high=other_high) for _ in range(others)]),
            'tasks': Space.Tuple([Space.Box(low=[0] * len(network_high), high=network_high)
                                  for _ in range(self._n_nodes)]),
        })
        return [space] * self.parallel_envs
