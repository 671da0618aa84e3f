"""CPU oracle for the cybersecurity step path -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Only ``tests/``, ``__graft_entry__.smoke()`` and the CPU-baseline legs of ``bench.py`` may import this module.

numpy restatement of the reference's cybersecurity hot path (paths relative to ``free_range_zoo/`` in
/root/reference): envs/cybersecurity/env/cybersecurity.py:296-526 and env/transitions/{movement,presence,subnetwork}.py.
The single transcendental on the path, ``tanh`` (subnetwork.py:54), is evaluated with ``torch.tanh`` on CPU -- the
very routine the reference calls -- so the threshold compare ``|score| <= r`` sees identical bits.
Parity pin: tests/test_oracle_golden.py replays tests/golden/cyber_*.npz (recorded from the unmodified reference);
tests/test_oracle_kat.py re-states the reference's transition unit-test vectors.
"""
from __future__ import annotations

import numpy as np
import torch

PAD = -100
F32 = np.float32


def _np(x, dtype):
    return np.asarray(x.detach().cpu().numpy() if hasattr(x, 'detach') else x, dtype=dtype)


def danger_score(patches: np.ndarray, attacks: np.ndarray, temperature) -> np.ndarray:
    """tanh((patches - attacks) / T) in fp32 with torch's CPU tanh (subnetwork.py:53-54)."""
    diff = torch.from_numpy(np.ascontiguousarray(patches - attacks, dtype=np.float32))
    return torch.tanh(diff / torch.tensor(float(temperature), dtype=torch.float32)).numpy()


# ---------------------------------------------------------------------------------------------------------------------
# The three transitions as pure functions (tests/test_oracle_kat.py feeds them the reference's unit-test inputs).


def movement(location, targets, mask):
    """transitions/movement.py:17-32."""
    return np.where(mask, targets, location).astype(np.int32)


def presence_transition(presence, location, u, persist, returns, num_attackers):
    """transitions/presence.py:35-60; returns (presence, location)."""
    returning = ~presence & (u < returns)
    leaving = presence & (u >= persist)
    new_presence = (presence | returning) & ~leaving
    new_location = np.where(returning[:, num_attackers:], -1, location).astype(np.int32)
    return new_presence, new_location


def subnetwork(network_state, patches, attacks, u, temperature, stochastic, num_states):
    """transitions/subnetwork.py:40-72."""
    score = danger_score(patches, attacks, temperature)
    if stochastic:
        magnitude = np.abs(score)
        better = (score > 0) & (magnitude <= u)
        worse = (score < 0) & (magnitude <= u)
    else:
        better, worse = score > 0, score < 0
    state = network_state - better.astype(np.int32) + worse.astype(np.int32)
    return np.clip(state, 0, num_states - 1).astype(np.int32)


class CybersecurityOracle:
    """Reference semantics of ``cybersecurity_v0`` for one batch; agents are ordered attackers then defenders."""

    def __init__(self, configuration, parallel_envs: int, max_steps: int = 1, observe_other_location: bool = False,
                 observe_other_presence: bool = False, observe_other_power: bool = True,
                 partially_observable: bool = True, show_bad_actions: bool = True):
        c = configuration
        ac, dc, nc, rc = c.attacker_config, c.defender_config, c.network_config, c.reward_config
        self.B = parallel_envs
        self.max_steps = max_steps
        self.n_att, self.n_def = ac.threat.shape[0], dc.mitigation.shape[0]
        self.n_agents = self.n_att + self.n_def
        self.N = nc.adj_matrix.shape[0]
        self.num_states = nc.patched_states + nc.vulnerable_states + nc.exploited_states
        self.temperature = F32(nc.temperature)
        self.stochastic = bool(c.stochastic_config.network_state)
        self.threat = _np(ac.threat, np.float32)
        self.mitigation = _np(dc.mitigation, np.float32)
        self.persist = np.concatenate([_np(ac.persist_probs, np.float32), _np(dc.persist_probs, np.float32)])
        self.returns = np.concatenate([_np(ac.return_probs, np.float32), _np(dc.return_probs, np.float32)])
        self.initial_presence = np.concatenate([_np(ac.initial_presence, bool), _np(dc.initial_presence, bool)])
        self.initial_location = _np(dc.initial_location, np.int32)
        self.initial_network = _np(nc.initial_state, np.int32)
        self.criticality = _np(nc.adj_matrix, np.int64).sum(axis=1)  # configuration.py:215-217
        self.state_rewards = _np(rc.network_state_rewards, np.float32)
        self.patch_reward = F32(rc.patch_reward)
        self.bad_action_penalty = F32(rc.bad_action_penalty)
        self.partially_observable = partially_observable
        self.show_bad_actions = show_bad_actions
        # env/utils/masking.py:7-28
        self.attacker_columns = [i for i, on in enumerate((observe_other_power, observe_other_presence)) if on]
        self.defender_columns = [
            i for i, on in enumerate((observe_other_power, observe_other_presence, observe_other_location)) if on
        ]
        self.faults = []

    STATE_KEYS = ('network_state', 'location', 'presence')

    def reset(self, initial_state: dict | None = None):
        """cybersecurity.py:222-271 (``initial_state``: network_state [B, N], location [B, D], presence [B, n] instead
        of the configuration's): actions are pre-filled with -2, so no defender has 'monitored' yet."""
        B = self.B
        if initial_state is not None:
            self.network_state = np.array(initial_state['network_state'], np.int32)
            self.location = np.array(initial_state['location'], np.int32)
            self.presence = np.array(initial_state['presence'], bool)
        else:
            self.network_state = np.tile(self.initial_network, (B, 1))
            self.location = np.tile(self.initial_location, (B, 1))
            self.presence = np.tile(self.initial_presence, (B, 1))
        self.initial_state = {key: getattr(self, key).copy() for key in self.STATE_KEYS}  # utils/state.py:36-38
        self.last_action_id = np.full((B, self.n_agents), -2, np.int32)
        self.rewards = np.zeros((B, self.n_agents), np.float32)
        self.cumulative_rewards = np.zeros((B, self.n_agents), np.float32)
        self.terminated = np.zeros(B, bool)
        self.truncated = np.zeros(B, bool)
        self.num_moves = np.zeros(B, np.int32)
        self._publish()

    def reset_batches(self, mask, initial_state: dict | None = None):
        """utils/env.py:163-189 + cybersecurity.py:274-293: the environments selected by ``mask`` (bool [B]) go back to
        the saved initial state (``initial_state`` replaces it first when given), their AEC fields are zeroed and their
        last actions are -2 again (not monitored); then everything is published."""
        mask = np.asarray(mask, bool)
        if initial_state is not None:
            self.initial_state = {key: np.array(initial_state[key], getattr(self, key).dtype) for key in self.STATE_KEYS}
        for key in self.STATE_KEYS:
            getattr(self, key)[mask] = self.initial_state[key][mask]
        self.last_action_id[mask] = -2
        for key in ('rewards', 'cumulative_rewards', 'terminated', 'truncated', 'num_moves'):
            getattr(self, key)[mask] = 0
        self._publish()

    def _publish(self):
        """update_observations + update_actions (cybersecurity.py:414-526)."""
        B, N = self.B, self.N
        self.environment_task_count = np.full(B, N, np.int32)
        self.agent_task_count = np.where(self.presence, N, 0).astype(np.int32)
        self.attacker_self = np.stack(
            [np.broadcast_to(self.threat, (B, self.n_att)), self.presence[:, :self.n_att].astype(np.float32)], axis=2)
        self.defender_self = np.stack([
            np.broadcast_to(self.mitigation, (B, self.n_def)), self.presence[:, self.n_att:].astype(np.float32),
            self.location.astype(np.float32)
        ], axis=2)
        self.task_store = np.stack([self.network_state, np.broadcast_to(self.criticality, (B, N))],
                                   axis=2).astype(np.int32)

    def task_obs(self, agent: int) -> np.ndarray:
        tasks = self.task_store.copy()
        if agent >= self.n_att and self.partially_observable:
            not_monitor = self.last_action_id[:, agent] != -3  # cybersecurity.py:497,510-511
            tasks[not_monitor] = PAD
        return tasks

    def others_obs(self, agent: int) -> np.ndarray:
        if agent < self.n_att:
            keep = [i for i in range(self.n_att) if i != agent]
            return self.attacker_self[:, keep][:, :, self.attacker_columns]
        keep = [i for i in range(self.n_def) if i != agent - self.n_att]
        return self.defender_self[:, keep][:, :, self.defender_columns]

    def action_map(self, agent: int) -> np.ndarray:
        out = np.full((self.B, self.N), PAD, np.int32)
        out[self.presence[:, agent]] = np.arange(self.N)
        return out

    def step(self, actions: np.ndarray, u_network: np.ndarray, u_agent: np.ndarray):
        """One AEC round (utils/env.py:203-242 around cybersecurity.py:296-411).

        actions int32 [B, n_agents, 2]; u_network f32 [1, B, N]; u_agent f32 [1, B, n_agents].
        """
        if self.terminated.all() or self.truncated.all():
            return False
        B, N = self.B, self.N
        rewards = np.zeros((B, self.n_agents), np.float32)
        patches = np.zeros((B, N), np.float32)
        attacks = np.zeros((B, N), np.float32)
        rows = np.arange(B)
        target, ident = actions[:, :, 0], actions[:, :, 1]
        move_mask = np.zeros((B, self.n_def), bool)
        move_target = np.zeros((B, self.n_def), np.int32)
        for agent in range(self.n_agents):
            present = self.presence[:, agent]
            if not self.show_bad_actions and np.any(ident[:, agent][~present] != -1):
                self.faults.append('Invalid action for non-present agent')  # cybersecurity.py:345,362
            if agent < self.n_att:
                attack = ident[:, agent] == 0
                nodes = target[attack, agent]
                if not ((nodes >= 0) & (nodes < N)).all():
                    self.faults.append('Invalid attack target')  # :341
                ok = attack & (target[:, agent] >= 0) & (target[:, agent] < N)
                attacks[rows[ok], target[ok, agent]] += self.threat[agent]  # :350, agents in order
            else:
                d = agent - self.n_att
                move = ident[:, agent] == 0
                patch = (ident[:, agent] == -2) & (self.location[:, d] != -1)  # :354
                nodes = target[move, agent]
                if not ((nodes >= 0) & (nodes < N)).all():
                    self.faults.append('Invalid movement target')  # :357
                move_mask[:, d] = move
                move_target[:, d] = target[:, agent]
                patches[rows[patch], self.location[patch, d]] += self.mitigation[d]  # :375, pre-move location
                rewards[patch, agent] += self.patch_reward  # :376
                # :379-381 -- patch already requires location != -1, so the bad-action penalty never fires

        self.location = movement(self.location, move_target, move_mask)
        self.presence, self.location = presence_transition(self.presence, self.location, u_agent[0], self.persist,
                                                           self.returns, self.n_att)
        self.network_state = subnetwork(self.network_state, patches, attacks, u_network[0], self.temperature,
                                        self.stochastic, self.num_states)
        # rewards, cybersecurity.py:395-409: matmul([B,N] f32, criticality f32 [N]) accumulated in node order
        node_rewards = self.state_rewards[self.network_state]
        network = np.zeros(B, np.float32)
        for n in range(N):
            network = (network + node_rewards[:, n] * F32(self.criticality[n])).astype(np.float32)
        rewards[:, :self.n_att] += -network[:, None]
        rewards[:, self.n_att:] += network[:, None]

        self.last_action_id = ident.astype(np.int32).copy()
        self.rewards = rewards
        self.num_moves = self.num_moves + 1
        if self.max_steps is not None:
            self.truncated = self.num_moves >= self.max_steps
        self.cumulative_rewards = self.cumulative_rewards + rewards
        self._publish()
        return True

    def outputs(self, agent_names) -> dict:
        """Same keys/layout as tests/golden/gen_golden.py::cyber_outputs."""
        n = self.n_agents
        out = dict(
            network_state=self.network_state, location=self.location, presence=self.presence, rewards=self.rewards,
            terminated=np.repeat(self.terminated[:, None], n, axis=1),
            truncated=np.repeat(self.truncated[:, None], n, axis=1), num_moves=self.num_moves,
            env_task_count=self.environment_task_count, agent_task_count=self.agent_task_count,
            attacker_self=self.attacker_self, defender_self=self.defender_self,
            task_obs=np.stack([self.task_obs(a) for a in range(n)], axis=0), task_store=self.task_store,
        )
        for a, name in enumerate(agent_names):
            out[f'others__{name}'] = self.others_obs(a).astype(np.float32)
            out[f'action_map__{name}'] = self.action_map(a)
        return out
