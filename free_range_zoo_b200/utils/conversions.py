"""AEC -> Parallel adapter with the reference's Parallel API (free_range_zoo/utils/conversions.py:13-118).

``step(actions)`` takes ``{agent: IntTensor[B, 2]}`` and returns ``(observations, rewards, terminations, truncations,
infos)``.  The reference loops ``aec_env.step(actions[agent])`` over the agents (conversions.py:87-90); here the A
action tensors are stacked straight into the device action table (one launch) and the environment advances with one
fused launch.  A pre-stacked int32 ``[B, A, 2]`` tensor is accepted too.
"""
from __future__ import annotations

from typing import Any, Dict, List, Tuple, Union

import torch

from free_range_zoo_b200.utils.env import BatchedAECEnv


def batched_aec_to_batched_parallel(aec_env: BatchedAECEnv) -> 'batched_aec_to_batched_parallel_wrapper':
    """Wrap an AEC environment in the Parallel API (idempotent for an already wrapped environment)."""
    if isinstance(aec_env, batched_aec_to_batched_parallel_wrapper):
        return aec_env
    return batched_aec_to_batched_parallel_wrapper(aec_env)


class batched_aec_to_batched_parallel_wrapper:
    """Parallel view of a ``BatchedAECEnv``; unknown attributes are forwarded to the wrapped environment."""

    def __init__(self, aec_env: BatchedAECEnv):
        self.aec_env = aec_env
        self.metadata = getattr(aec_env, 'metadata', {})
        self.possible_agents = aec_env.possible_agents
        self.agents = list(getattr(aec_env, 'agents', aec_env.possible_agents))

    def __getattr__(self, name: str):
        if name == 'aec_env':
            raise AttributeError(name)
        return getattr(self.aec_env, name)

    @property
    def unwrapped(self) -> BatchedAECEnv:
        return self.aec_env.unwrapped

    def observation_space(self, agent: str):
        return self.aec_env.observation_space(agent)

    def action_space(self, agent: str):
        return self.aec_env.action_space(agent)

    def state(self):
        return self.aec_env.state()

    def reset_batches(self, *args, **kwargs) -> None:
        self.aec_env.reset_batches(*args, **kwargs)

    def reset(self, seed: Union[int, List[int]] = None,
              options: Dict[str, Any] = None) -> Tuple[Dict[str, Any], Dict[str, Any]]:
        self.aec_env.reset(seed=seed, options=options)
        self.agents = self.aec_env.agents
        return self.observe(), self.aec_env.infos

    def step(self, actions) -> Tuple[Dict, Dict, Dict, Dict, Dict]:
        env = self.aec_env.unwrapped
        if isinstance(actions, dict):
            torch.stack([actions[agent] for agent in env.agents], dim=1, out=env._actions)
            env.step_all(None)
        else:
            env.step_all(actions)
        self.agents = env.agents
        return self.observe(), env.rewards, env.terminations, env.truncations, env.infos

    def step_host(self, host_actions: torch.Tensor, chunks=None, observations: bool = False):
        """Parallel step with HOST buffers: page-locked int32 ``[B, A, 2]`` actions in, page-locked ``(rewards [B, A],
        terminated [B], truncated [B])`` out; upload, step and download are pipelined over slices of the batch
        (``BatchedAECEnv.step_host``).  Observations stay on the device (``observe()``) unless ``observations=True``:
        then a fourth element carries them in host memory, packed (``BatchedAECEnv.gather_observations``)."""
        env = self.aec_env.unwrapped
        results = env.step_host(host_actions, chunks, observations)
        self.agents = env.agents
        return results

    def observe(self) -> Dict[str, Any]:
        return {agent: self.aec_env.observe(agent) for agent in self.aec_env.agents}

    @property
    def finished(self) -> torch.Tensor:
        return self.aec_env.finished

    @property
    def final_observations(self) -> Dict[str, Any]:
        """``BatchedAECEnv.final_observations``: the observations the episodes of the last step ended with."""
        return self.aec_env.final_observations
