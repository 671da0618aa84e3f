"""AEC runtime shell of the B200 engine.

``BatchedAECEnv`` keeps the surface of the reference base class (free_range_zoo/utils/env.py:18-359): the same
constructor keywords, ``reset / reset_batches / step / observe / state / action_space / observation_space``, the
five domain hooks (``step_environment``, ``update_actions``, ``update_observations``, ``action_space``,
``observation_space``) and the public attributes (``agents``, ``rewards``, ``terminations``, ``truncations``,
``infos``, ``num_moves``, ``environment_task_count``, ``agent_task_count``, ``finished`` ...).

What changed underneath: the whole cycle the reference runs on the last agent of an AEC round --
``step_environment -> num_moves += 1 -> truncation -> accumulate rewards -> update_observations -> update_actions``
(utils/env.py:220-237) -- is ONE fused CUDA launch through the C ABI of ``include/frz.h``.  All per-step outputs
live in persistent device buffers that the kernel updates in place; the dictionaries handed to the caller are views
of those buffers, so there is no host round trip, no ``.tolist()``, no allocation on the step path.  The reference's
host-side "is every environment done?" test (utils/env.py:212, a device synchronisation per agent call) is evaluated
on the device from flags the previous launch published.

NOTE on aliasing: because buffers are updated in place, tensors returned by ``step`` are overwritten by the next
``step``.  Pass ``detach_outputs=True`` to get fresh copies (the reference's behaviour) at the cost of one copy each.
"""
from __future__ import annotations

import ctypes
import math
from abc import ABC, abstractmethod
from typing import Any, Dict, List, NamedTuple, Optional, Tuple

import torch

from free_range_zoo_b200 import _lib
from free_range_zoo_b200.utils import compact
from free_range_zoo_b200.utils.configuration import Configuration
from free_range_zoo_b200.utils.containers import ObservationDict
from free_range_zoo_b200.utils.selector import AgentSelector


# most slices ``step_host`` cuts a batch into by default (measured on B200, profiles/README.md)
HOST_STEP_MAX_DEFAULT_CHUNKS = 5


class AutoresetRows(NamedTuple):
    """What a restart does with each per-environment buffer a domain binds (``_bound`` keys).  Every key is in exactly
    one of the five groups, so a buffer added later needs a decision (tests/test_autoreset.py)."""
    init: Dict[str, str]  # state restored from its initial copy: {buffer: its init_* buffer}
    snapshot: Tuple[str, ...]  # outputs of the reset's refresh, restored from the snapshot taken at reset()
    zero: Tuple[str, ...]  # AEC fields the next step reads, zeroed as the domain's reset kernel zeroes them
    overwritten: Tuple[str, ...]  # written for every environment by every step: kept as the finishing step wrote them
    static: Tuple[str, ...]  # not changed by a restart: init_* copies, inputs, configuration tables, the control block
    agents_with_tasks: bool  # whether the domain publishes FrzControl.agents_with_tasks (a refresh publishes 0 otherwise)
    # the arrays the observations are built from (views and host downloads), all restored by a restart: what
    # keep_final_observations copies aside before the restart overwrites them
    final: Tuple[str, ...]


class InputKind(NamedTuple):
    """Agents of one kind in the policy inputs: ``count`` agents (consecutive in the action table) whose self table
    has ``columns`` columns, of which ``observed`` appear for every other agent of the kind in its ``others`` view."""
    count: int
    columns: int
    observed: Tuple[int, ...]

    @property
    def width(self) -> int:
        return self.columns + (self.count - 1) * len(self.observed)


class PolicyInputLayout(NamedTuple):
    """The structure of the policy inputs (include/frz_inputs.h)."""
    kinds: Tuple[InputKind, ...]  # one, or cybersecurity's attackers and defenders
    task_rows: int  # T
    views: int  # V
    task_columns: Tuple[bool, ...]  # one per task_obs column: True for a "none" column whose FRZ_PAD means nobody
    flags: int = 0  # _lib.INPUTS_*


class PolicyInputSchema(NamedTuple):
    """A layout and the ``(scale, offset)`` of every source column (self columns per kind, then task columns)."""
    layout: PolicyInputLayout
    self_columns: Tuple[Tuple[Tuple[float, int], ...], ...]
    task_columns: Tuple[Tuple[float, int], ...]


def input_column(high, none: bool = False) -> Tuple[float, int]:
    """``(scale, offset)`` of a column bounded by ``high``: ``(1 / high, 0)``, or ``(1 / (high + 1), 1)`` for a "none"
    column (its "none" value -1 then maps to 0); scale 1 where the bound is missing or not positive."""
    high = None if high is None else float(high) + (1.0 if none else 0.0)
    return (1.0 if high is None or not high > 0 else 1.0 / high), (1 if none else 0)


class _DeviceBound:
    """libfrz entry points bound to one CUDA device: every call of the C ABI works on the CURRENT device
    (include/frz.h), so calls made while another device is current switch to the environment's device for their
    duration.  When it already is current (the normal case) the call goes straight through."""

    def __init__(self, library, device: torch.device):
        self._library, self._index = library, device.index

    def __getattr__(self, name):
        entry, index = getattr(self._library, name), self._index

        def call(*args):
            if torch.cuda.current_device() == index:
                return entry(*args)
            with torch.cuda.device(index):
                return entry(*args)

        self.__dict__[name] = call
        return call


def _seed_to_u64(seed) -> int:
    """Fold whatever ``reset(seed=...)`` received (None / int / list / tensor) into one 64-bit Philox key."""
    if seed is None:
        return int(torch.randint(0, 2**62, (1, )).item())
    if isinstance(seed, torch.Tensor):
        seed = seed.flatten().tolist()
    if isinstance(seed, (list, tuple)):
        folded = 0x9E3779B97F4A7C15
        for value in seed:
            folded = ((folded ^ (int(value) & 0xFFFFFFFFFFFFFFFF)) * 0x100000001B3) & 0xFFFFFFFFFFFFFFFF
        return folded
    return int(seed) & 0xFFFFFFFFFFFFFFFF


class BatchedAECEnv(ABC):
    """Batched agent-environment-cycle environment whose step runs as one CUDA kernel."""

    metadata: Dict[str, Any] = {}

    def __init__(
        self,
        *args,
        configuration: Configuration = None,
        max_steps: int = 1,
        parallel_envs: int = 1,
        device: torch.device = torch.device('cuda'),
        render_mode: str | None = None,
        log_directory: str = None,
        single_seeding: bool = False,
        buffer_size: int = 0,
        override_initialization_check: bool = False,
        env_offset: int = 0,
        detach_outputs: bool = False,
        autoreset: bool = False,
        keep_final_observations: bool = False,
        **kwargs,
    ):
        """
        Args (same meaning as the reference, utils/env.py:21-48):
            configuration: the domain's configuration structure
            max_steps: truncation horizon
            parallel_envs: number of environments stepped together
            device: must be a CUDA device -- there is no CPU path
            render_mode: accepted; rendering is a host-side subsystem outside this engine
            log_directory / override_initialization_check: a directory turns on the asynchronous logging tap
                (utils/logging_tap.py; same files as the reference's CSVLogger), a ``sqlite://`` URL its SQL form
                (utils/sql_tap.py; the reference's SQLLogger tables); other connection strings are refused
            single_seeding / buffer_size: accepted and ignored -- randomness is counter-based Philox generated inside
                the step kernel, keyed by (seed, global env index, step), so there are no generator states to juggle
            env_offset: global index of this shard's first environment.  Random streams are keyed by the global index,
                so a shard draws what its environments draw in the whole batch.  The two batch-wide conditions of the
                reference -- every environment terminated / truncated (utils/env.py:212), an agent without a task in
                any environment (wildfire.py:434, rideshare.py:276) -- are evaluated over this shard's environments
                only: a shard equals its slice of the whole batch while those conditions agree, and otherwise equals
                the reference run on the shard alone
            detach_outputs: return copies instead of views of the in-place updated device buffers
            autoreset: restart every environment that is terminated or truncated at the end of the step that finished
                it ("same-step" autoreset), on the device and in the same stream / CUDA graph as the step: ``step``,
                ``step_all``, the Parallel ``step``, ``step_host`` and every step of a ``capture_graph(steps=K)`` replay.
                Afterwards state, observations, masks, counts and the batch-wide flags are what ``reset_batches`` of the
                finished environments leaves.  What the step returns (rewards, terminations, truncations, infos) is what
                the finishing step produced; ``terminated`` / ``truncated`` / ``finished`` / ``terminations`` /
                ``truncations`` read copies of the step's done flags ("the episode ended at the last step") and
                ``episode_statistics`` gives each finished episode's return and length.  Restarted environments keep
                drawing random numbers with the global step counter, as after ``reset_batches``.  The observations
                after the step are the restarted environment's; ``keep_final_observations`` keeps the ones the finished
                episode ended with.  Every full ``reset()`` snapshots the per-environment outputs of its refresh
                (observations, masks, counts, rideshare's passenger table), which a restart copies back: about 2.8 KB
                per environment at wildfire C4 (184 MB at 65 536 environments).  Not available with a
                ``log_directory``.
            keep_final_observations: with ``autoreset`` only (``ValueError`` otherwise): before a restart overwrites
                them, the restart copies the finished environments' observation arrays to a set of final-observation
                buffers, in the same launch.  ``final_observations`` reads them on the device and
                ``gather_observations(final=True)`` downloads them, e.g. to bootstrap a truncated episode from the value
                of its last observation.  Costs one more copy of the observation arrays in device memory (as much again
                as the snapshot at wildfire C4) and, on a step that finishes environments, one more pass over their
                observation rows; nothing on a step where none finished.
        """
        device = torch.device(device)
        if device.type != 'cuda':
            raise RuntimeError(f'free_range_zoo_b200 runs on CUDA devices only (got device={device}); '
                               'there is no CPU fallback -- use the reference implementation on CPU.')
        if device.index is None:
            device = torch.device('cuda', torch.cuda.current_device())
        if log_directory is not None and str(log_directory).startswith(('postgres', 'mysql')):
            raise NotImplementedError('the asynchronous logging tap writes CSV files or sqlite:// databases; '
                                      f'no driver for {log_directory!r} is available')
        self.parallel_envs = int(parallel_envs)
        self.max_steps = max_steps
        self.device = device
        self.render_mode = render_mode
        self.log_directory = log_directory
        self.override_initialization_check = override_initialization_check
        self.single_seeding = single_seeding
        self.log_description = None
        self.logger = None
        self.env_offset = int(env_offset)
        self.detach_outputs = detach_outputs
        self.autoreset = bool(autoreset)
        if self.autoreset and log_directory is not None:
            raise ValueError('autoreset restarts environments on the device inside the step, which the logging tap does not '
                             'record; autoreset=True needs log_directory=None')
        self.keep_final_observations = bool(keep_final_observations)
        if self.keep_final_observations and not self.autoreset:
            raise ValueError('keep_final_observations keeps what the autoreset overwrites: it needs autoreset=True '
                             '(without it the observations of a finished environment stay until reset_batches)')

        if configuration is not None:
            self.config = configuration
            # hoist the sub-configurations as attributes, like the reference (utils/env.py:58-63)
            for key, value in vars(configuration).items():
                if hasattr(value, 'validate') and not isinstance(value, torch.Tensor):
                    setattr(self, key, value)

        self._lib = _DeviceBound(_lib.library(), self.device)
        self._tap = None  # asynchronous CSV logging (utils/logging_tap.py), created by the first reset
        self._control = torch.zeros(8, dtype=torch.int64, device=self.device)  # FrzControl, 64 bytes
        self._seed_value = None
        self._graph = None

    def __del__(self):
        handle = getattr(self, '_host_events', None)
        if handle is not None:
            try:
                self._lib.frz_host_pipeline_destroy(handle)
            except Exception:
                pass
            self._host_events = None

    # ------------------------------------------------------------------------------------------ random stream

    def generator_state_dict(self) -> Dict[str, int]:
        """The whole random state of the engine (reference: ``RandomGenerator.state_dict``, one pickled
        ``torch.Generator`` state per environment, utils/random_generator.py:148-162): every draw is
        Philox(seed; global environment index, step, event), so ``seed`` and the step counter say it all.
        Synchronises (reads the device control block)."""
        block = self.control_block()
        return {'seed': block['seed'], 'step': block['step'], 'env_offset': self.env_offset}

    def load_generator_state_dict(self, state: Dict[str, int]) -> None:
        """Continue the random stream of a checkpoint (reference: ``RandomGenerator.load_state_dict``,
        utils/random_generator.py:164-176).  Restore the state tensors FIRST (``env.state().load(...)`` /
        ``reset(options={'initial_state': ...})``, the AEC buffers included), then call this: it sets (seed, step),
        clears recorded faults and re-publishes observations, masks and the batch-wide flags from the restored state.

        The checkpoint must come from an environment with the same ``env_offset``: the random streams are keyed by the
        global environment index, so another offset would continue on other streams (``ValueError``)."""
        if int(state['env_offset']) != self.env_offset:
            raise ValueError(f"the checkpoint was taken with env_offset={int(state['env_offset'])}, this environment has "
                             f'env_offset={self.env_offset}: its environments would continue on other random streams')
        self._seed_value = int(state['seed'])
        _lib.check(self._lib.frz_control_restore(self._control.data_ptr(), ctypes.c_uint64(int(state['seed'])),
                                                 ctypes.c_uint64(int(state['step'])), self._stream()),
                   'frz_control_restore')
        self._refresh()
        self._mid_cycle = False
        self._rebind_outputs()

    # ------------------------------------------------------------------------------------------ properties

    @property
    def num_agents(self) -> int:
        return len(self.agents)

    @property
    def max_num_agents(self) -> int:
        return len(self.possible_agents)

    @property
    def unwrapped(self) -> 'BatchedAECEnv':
        return self

    @property
    def terminated(self) -> torch.Tensor:
        """bool [B]; every agent of an environment terminates together (reference utils/env.py:341-349).  With
        ``autoreset`` a copy of what the last step produced (the live flags of a restarted environment are clear)."""
        if self.autoreset:
            return self._autoreset_flags[1].view(torch.bool)
        return self._terminated.view(torch.bool)

    @property
    def truncated(self) -> torch.Tensor:
        if self.autoreset:
            return self._autoreset_flags[2].view(torch.bool)
        return self._truncated.view(torch.bool)

    @property
    def episode_statistics(self) -> Dict[str, torch.Tensor]:
        """The episodes the last step finished (``autoreset=True`` only), device tensors overwritten by the next step:
        ``done`` / ``terminated`` / ``truncated`` bool [B], ``return`` f32 [B, A] (the cumulative reward of the episode)
        and ``length`` int32 [B] (its number of steps).  ``return`` and ``length`` are defined only where ``done`` is
        set; elsewhere they hold an earlier episode's values or zeros, so select with ``done`` before reducing (e.g.
        ``distributed.episode_statistics(s['return'][s['done']], ...)``)."""
        if not self.autoreset:
            raise RuntimeError('episode_statistics is recorded by the autoreset: construct the environment with autoreset=True')
        flags = self._autoreset_flags.view(torch.bool)
        return {'done': flags[0], 'terminated': flags[1], 'truncated': flags[2], 'return': self._episode_return,
                'length': self._episode_length}

    @property
    def final_observations(self) -> Dict[str, ObservationDict]:
        """The observations the episodes of the last step ended with (``keep_final_observations=True`` only):
        ``{agent: ObservationDict}`` with the keys, shapes and dtypes of ``observations[agent]``, built over device
        buffers that the next step overwrites where it finishes an environment.  Environment b's entry is the
        observation its episode ended with wherever ``episode_statistics['done'][b]`` is set; elsewhere it holds an
        earlier episode's or the last full ``reset()``'s observation, so select with ``done`` (e.g.
        ``final_observations[agent]['self'][done]``).  ``reset_batches`` leaves them alone."""
        if not self.keep_final_observations:
            raise RuntimeError('final_observations are kept by the autoreset: construct the environment with '
                               'autoreset=True, keep_final_observations=True')
        return self._observation_views(self._final_buffers)

    @property
    def finished(self) -> torch.Tensor:
        return torch.logical_or(self.terminated, self.truncated)

    @property
    def agent_task_count(self) -> torch.Tensor:
        """int32 [A, B] like the reference (utils/env.py:160); a transposed view of the kernel's [B, A] buffer."""
        return self._agent_task_count.t()

    @property
    def rewards(self) -> Dict[str, torch.Tensor]:
        """Per-agent rewards of the last environment step.  In the middle of an AEC round the reference has cleared
        them to zero (utils/env.py:215,251-254); that is mirrored without touching device memory."""
        if self._mid_cycle:
            return {agent: self._zero_rewards for agent in self.agents}
        return self._reward_views

    @property
    def reward_table(self) -> torch.Tensor:
        """f32 [B, A] on the device: the rewards of the last environment step, agents in the order of ``possible_agents``.
        It is the buffer ``rewards[agent]`` views column by column and keeps its address on every step, so a rollout
        stores a step with one ``storage[t].copy_(env.reward_table)`` (capturable).  The next step overwrites it; unlike
        ``rewards`` it is not zeroed in the middle of an AEC round, and ``detach_outputs`` does not copy it."""
        return self._rewards

    # ------------------------------------------------------------------------------------------ allocation

    def _allocate_runtime(self, num_agents: int) -> None:
        """Persistent AEC buffers (what the reference re-creates in reset, utils/env.py:129-160)."""
        B, A, dev = self.parallel_envs, num_agents, self.device
        self._actions = torch.zeros((B, A, 2), dtype=torch.int32, device=dev)
        self._rewards = torch.zeros((B, A), dtype=torch.float32, device=dev)
        self._cumulative = torch.zeros((B, A), dtype=torch.float32, device=dev)
        self._terminated = torch.zeros(B, dtype=torch.uint8, device=dev)
        self._truncated = torch.zeros(B, dtype=torch.uint8, device=dev)
        self.num_moves = torch.zeros(B, dtype=torch.int32, device=dev)
        self.environment_task_count = torch.zeros(B, dtype=torch.int32, device=dev)
        self._agent_task_count = torch.zeros((B, A), dtype=torch.int32, device=dev)
        self._zero_rewards = torch.zeros(B, dtype=torch.float32, device=dev)
        if self.autoreset:
            self._autoreset_flags = torch.zeros((3, B), dtype=torch.uint8, device=dev)  # done, terminated, truncated
            self._episode_return = torch.zeros((B, A), dtype=torch.float32, device=dev)
            self._episode_length = torch.zeros(B, dtype=torch.int32, device=dev)
            self._autoreset_list = torch.zeros(B, dtype=torch.int32, device=dev)
            self._autoreset_count = torch.zeros(1, dtype=torch.int32, device=dev)
            self._autoreset_scratch = torch.zeros(2, dtype=torch.int32, device=dev)  # left zero by every launch

    def _stream(self) -> ctypes.c_void_p:
        return _lib.stream_handle(self.device)

    def _horizon(self) -> int:
        return 2**31 - 1 if self.max_steps is None else int(self.max_steps)

    # ------------------------------------------------------------------------------------------ reset

    @torch.no_grad()
    def reset(self, seed=None, options: Optional[Dict[str, Any]] = None) -> None:
        """Reset every environment (reference utils/env.py:95-160). Subclasses extend this with their state."""
        options = options or {}
        if options.get('max_steps') is not None:
            self.max_steps = options['max_steps']
        self._log_label = options.get('log_label')
        self.log_description = options.get('log_description')

        if options.get('skip_seeding'):
            if self._seed_value is None:
                raise ValueError("Seed must be set before skipping seeding is possible")
        else:
            self._seed_value = _seed_to_u64(seed)
        self.seeds = torch.full((self.parallel_envs, ), self._seed_value & 0x7FFFFFFF, dtype=torch.int32,
                                device=self.device)
        _lib.check(self._lib.frz_control_init(self._control.data_ptr(), ctypes.c_uint64(self._seed_value), self._stream()),
                   'frz_control_init')

        self.agents = self.possible_agents
        self.infos = {agent: {} for agent in self.agents}
        self._reward_views = {a: self._rewards[:, i] for i, a in enumerate(self.agents)}
        self._cumulative_rewards = {a: self._cumulative[:, i] for i, a in enumerate(self.agents)}
        terminated, truncated = self.terminated, self.truncated
        self.terminations = {a: terminated for a in self.agents}
        self.truncations = {a: truncated for a in self.agents}
        self.actions = {a: self._actions[:, i] for i, a in enumerate(self.agents)}
        self._agent_slot = {a: i for i, a in enumerate(self.agents)}
        self._mid_cycle = False

        self.agent_selector = AgentSelector(self.agents)
        self.agent_selection = self.agent_selector.reset()

    @torch.no_grad()
    def reset_batches(self, batch_indices, seed=None, options: Optional[Dict[str, Any]] = None) -> None:
        """Reset only the environments ``batch_indices`` (reference utils/env.py:163-189; index list or tensor)."""
        mask = torch.zeros(self.parallel_envs, dtype=torch.uint8, device=self.device)
        mask[torch.as_tensor(batch_indices, device=self.device, dtype=torch.int64)] = 1
        self._reset_masked(mask)
        if self.autoreset:  # a restarted environment's episode did not end at the last step
            self._autoreset_flags.masked_fill_(mask.bool(), 0)
        # the observation dictionaries hold gathered copies (other agents' rows, per-agent task views): rebuild them
        # from the refreshed buffers, as a step does
        self._mid_cycle = False
        self._rebind_outputs()

    @abstractmethod
    def _reset_masked(self, mask: Optional[torch.Tensor]) -> None:
        """Launch the domain's reset kernel for the environments selected by ``mask`` (uint8 [B]; None = all)."""

    # ------------------------------------------------------------------------------------------ autoreset

    @classmethod
    def _autoreset_rows(cls) -> AutoresetRows:
        """How a restart treats each buffer of ``_bound``.  Domain hook."""
        raise NotImplementedError

    def _snapshot_reset(self) -> None:
        """After a full reset: with ``autoreset``, keep the outputs of the reset's refresh, which are what a restart
        restores, and describe the rows of ``frz_autoreset`` (include/frz_autoreset.h)."""
        if not self.autoreset:
            return
        B, rows, bound = self.parallel_envs, self._autoreset_rows(), self._bound
        if getattr(self, '_reset_snapshot', None) is None:
            self._reset_snapshot = {name: torch.empty_like(bound[name]) for name in rows.snapshot}
        for name, tensor in self._reset_snapshot.items():
            tensor.copy_(bound[name])
        if self.keep_final_observations:  # (kept apart from _bound, which mirrors the domain's C buffer struct)
            if getattr(self, '_final_buffers', None) is None:
                self._final_buffers = {name: torch.empty_like(bound[name]) for name in rows.final}
                self._final_counts = torch.zeros(B, dtype=torch.int32, device=self.device)
            for name, tensor in self._final_buffers.items():  # well-formed before any episode has finished
                tensor.copy_(bound[name])
        keep = self._final_buffers if self.keep_final_observations else {}
        self._autoreset_flags.zero_()
        pairs = ([(name, bound[src]) for name, src in rows.init.items()] +
                 [(name, self._reset_snapshot[name]) for name in rows.snapshot] +
                 [(name, None) for name in rows.zero])
        table = (_lib.AutoresetRow * len(pairs))()
        for at, (name, src) in enumerate(pairs):
            dst = bound[name]
            assert dst.shape[0] == B and dst.is_contiguous() and (src is None or src.shape == dst.shape)
            table[at].dst, table[at].src, table[at].keep = dst.data_ptr(), _lib.pointer(src), _lib.pointer(keep.get(name))
            table[at].bytes = dst.numel() * dst.element_size() // B
        block = _lib.Autoreset()
        block.terminated, block.truncated = self._terminated.data_ptr(), self._truncated.data_ptr()
        block.done, block.step_terminated, block.step_truncated = (row.data_ptr() for row in self._autoreset_flags)
        block.cumulative_rewards, block.episode_return = self._cumulative.data_ptr(), self._episode_return.data_ptr()
        block.num_moves, block.episode_length = self.num_moves.data_ptr(), self._episode_length.data_ptr()
        if rows.agents_with_tasks:
            block.agent_task_count = self._agent_task_count.data_ptr()
            block.reset_agent_task_count = self._reset_snapshot['agent_task_count'].data_ptr()
        block.control = self._control.data_ptr()
        block.finished, block.finished_count = self._autoreset_list.data_ptr(), self._autoreset_count.data_ptr()
        block.scratch = self._autoreset_scratch.data_ptr()
        block.rows, block.row_count = table, len(pairs)
        block.num_agents = self._cumulative.shape[1]
        self._autoreset_block = (block, table)  # (the table must outlive the block that points at it)

    def _autoreset_launch(self) -> None:
        """Restart the environments the step just finished (two launches on the current stream; no host read)."""
        if self.autoreset:
            _lib.check(self._lib.frz_autoreset(ctypes.byref(self._autoreset_block[0]), self.parallel_envs, self._stream()),
                       'frz_autoreset')

    # ------------------------------------------------------------------------------------------ step

    @abstractmethod
    def step_environment(self) -> Tuple[Dict[str, torch.Tensor], Dict[str, torch.Tensor], Dict[str, Dict]]:
        """Launch the domain's fused step kernel; returns (rewards, terminations, infos) views."""

    @abstractmethod
    def update_actions(self) -> None:
        """Refresh task counts / action masks from the current state (already done inside the fused step)."""

    @abstractmethod
    def update_observations(self) -> None:
        """Refresh observations from the current state (already done inside the fused step)."""

    @abstractmethod
    def action_space(self, agent: str):
        """Per-environment action spaces of ``agent`` (a lazily materialised ``Space.Vector``)."""

    @abstractmethod
    def observation_space(self, agent: str):
        """Per-environment observation spaces of ``agent``."""

    @torch.no_grad()
    def step(self, actions: torch.Tensor) -> None:
        """AEC step of the currently selected agent (reference utils/env.py:203-242).

        The agent's ``[B, 2]`` actions are staged into the device action table; when the last agent of the round has
        acted, one fused launch advances every environment.
        """
        self._actions[:, self._agent_slot[self.agent_selection]].copy_(actions, non_blocking=True)
        self._mid_cycle = True
        if self.agent_selector.is_last():
            self._advance()
        self.agent_selection = self.agent_selector.next()

    @torch.no_grad()
    def step_all(self, actions: Optional[torch.Tensor] = None) -> None:
        """One environment step for all agents at once: ``actions`` int32 [B, A, 2] (None = already staged in
        ``env._actions``, e.g. by ``sample_actions``).  Equivalent to A consecutive ``step`` calls."""
        if actions is not None and actions.data_ptr() != self._actions.data_ptr():
            self._actions.copy_(actions, non_blocking=True)
        self._advance()

    # ------------------------------------------------------------------------------------------ host-buffer step

    def _host_entry(self):
        """The domain's ``frz_<domain>_step_host`` entry point."""
        raise NotImplementedError

    def _host_pipeline(self, chunks: Optional[int]):
        """Page-locked result buffers, per-slice control blocks and streams of ``step_host`` (built once per slicing)."""
        B, A = self.parallel_envs, len(self.possible_agents)
        if chunks is None:  # slices of >= 12 288 environments: below that the copies are too short to be worth hiding
            chunks = max(1, min(HOST_STEP_MAX_DEFAULT_CHUNKS, B // 12288))
        chunks = max(1, min(int(chunks), _lib.MAX_CHUNKS))
        cached = getattr(self, '_host_state', None)
        if cached is not None and cached['chunks'] == chunks:
            return cached
        state = dict(
            chunks=chunks,
            # (initialised from the device: a step that is skipped because every environment is done writes nothing)
            rewards=self._rewards.cpu().pin_memory(),
            done=torch.stack([self._terminated, self._truncated]).cpu().pin_memory(),
            controls=torch.zeros((chunks, 8), dtype=torch.int64, device=self.device),
            streams=[torch.cuda.Stream(self.device) for _ in range(chunks)],
            # the stream the pipeline is issued on: a capturable one (the legacy default stream is not), so that the
            # library can replay the whole pipeline as one CUDA graph from the second call on
            main=torch.cuda.Stream(self.device),
            packed=torch.zeros((B, A, 2), dtype=torch.int16, device=self.device),  # staging of int16 action uploads
        )
        if getattr(self, '_host_events', None) is None:  # this environment's own events (never shared, include/frz.h)
            handle = ctypes.c_void_p()
            _lib.check(self._lib.frz_host_pipeline_create(ctypes.byref(handle)), 'frz_host_pipeline_create')
            self._host_events = handle
        handles = (ctypes.c_void_p * chunks)(*[stream.cuda_stream for stream in state['streams']])
        block = _lib.HostStep()
        block.rewards = state['rewards'].data_ptr()
        block.terminated = state['done'][0].data_ptr()
        block.truncated = state['done'][1].data_ptr()
        block.chunk_controls = state['controls'].data_ptr()
        block.streams = ctypes.cast(handles, ctypes.POINTER(ctypes.c_void_p))
        block.chunks = chunks
        block.packed_actions = state['packed'].data_ptr()
        block.pipeline = self._host_events
        done = state['done'].view(torch.bool)
        state.update(handles=handles, block=block, terminated=done[0], truncated=done[1])
        self._host_state = state
        return state

    # ------------------------------------------------------------------------------------------ observations on the host

    def _observation_buffers(self) -> Dict[str, torch.Tensor]:
        """The live arrays the observations are built from, by ``_bound`` name (``_autoreset_rows().final``); the
        final-observation buffers have the same names."""
        buffers = self.__dict__.get('_live_observation_buffers')
        if buffers is None:  # (the tensors live as long as the environment; rebinding keeps them)
            buffers = self._live_observation_buffers = {name: self._bound[name] for name in self._autoreset_rows().final}
        return buffers

    def _observation_views(self, buffers: Dict[str, torch.Tensor]) -> Dict[str, ObservationDict]:
        """``{agent: ObservationDict}`` as views of ``buffers`` (live or final, see ``_observation_buffers``).  Domain
        hook."""
        raise NotImplementedError

    def _observation_download(self, buffers: Optional[Dict[str, torch.Tensor]] = None
                              ) -> Tuple[Dict[str, torch.Tensor], Dict[str, Tuple[torch.Tensor, int]]]:
        """What a policy on the host reads after a step, from ``buffers`` (None = the live ones): ``(dense, ragged)``.
        ``dense`` arrays leave the device whole; ``ragged`` maps a name to ``(padded array [B, groups, capacity, ...] or
        [B, capacity, ...], groups)`` of which only the first ``counts[b]`` rows per environment (and row block) are
        live.  Domain hook."""
        raise NotImplementedError

    def _download_counts(self, final: bool) -> torch.Tensor:
        """Live rows per environment of a download: the task counts, or for the final observations the final counts
        of the environments the last step finished and 0 elsewhere (computed on the current stream)."""
        if not final:
            return self.environment_task_count
        done = self._autoreset_flags[0]  # uint8 0 / 1
        torch.mul(self._final_buffers['env_task_count'], done, out=self._final_counts)
        return self._final_counts

    def _download_buffers(self, final: bool) -> Dict[str, torch.Tensor]:
        if final and not self.keep_final_observations:
            raise RuntimeError('final observations are kept by the autoreset: construct the environment with '
                               'autoreset=True, keep_final_observations=True')
        return self._final_buffers if final else self._observation_buffers()

    def _gather_state(self, final: bool = False):
        attribute = '_gather_final' if final else '_gather'
        state = getattr(self, attribute, None)
        if state is not None:
            return state
        B, dev = self.parallel_envs, self.device
        dense, ragged = self._observation_download(self._download_buffers(final))
        arrays = (_lib.GatherArray * max(1, len(ragged)))()
        packed, layout = {}, {}
        for at, (name, (tensor, groups)) in enumerate(ragged.items()):
            capacity = tensor.shape[2] if tensor.dim() >= 3 and groups > 1 else tensor.shape[1]
            row_shape = tuple(tensor.shape[3:] if groups > 1 else tensor.shape[2:])
            row_bytes = tensor.element_size() * math.prod(row_shape)
            packed[name] = torch.empty(tensor.numel(), dtype=tensor.dtype, device=dev)
            arrays[at].src, arrays[at].dst = tensor.data_ptr(), packed[name].data_ptr()
            arrays[at].row_bytes, arrays[at].capacity, arrays[at].groups = row_bytes, capacity, groups
            layout[name] = (groups, row_shape, row_bytes // tensor.element_size())
        state = dict(
            final=final, dense=dense, ragged=ragged, arrays=arrays, packed=packed, layout=layout,
            offsets=torch.zeros(B + 1, dtype=torch.int32, device=dev),
            scratch=torch.zeros((B + 1023) // 1024 + 1, dtype=torch.int32, device=dev),
            host_counts=torch.zeros(B, dtype=torch.int32).pin_memory(),
            host_offsets=torch.zeros(B + 1, dtype=torch.int32).pin_memory(),
            host_dense={name: torch.empty(tensor.shape, dtype=tensor.dtype).pin_memory() for name, tensor in dense.items()},
            host_packed={name: torch.empty(tensor.numel(), dtype=tensor.dtype).pin_memory() for name, tensor in packed.items()},
        )
        setattr(self, attribute, state)
        return state

    def _enqueue_gather(self, state) -> None:
        """Compaction kernels + the downloads whose size is known up front (counts, offsets, dense arrays), on the
        current stream of the device."""
        counts = self._download_counts(state['final'])
        _lib.check(self._lib.frz_gather_live_rows(counts.data_ptr(), self.parallel_envs,
                                                  state['offsets'].data_ptr(), state['scratch'].data_ptr(), state['arrays'],
                                                  len(state['ragged']), self._stream()), 'frz_gather_live_rows')
        state['host_counts'].copy_(counts, non_blocking=True)
        state['host_offsets'].copy_(state['offsets'], non_blocking=True)
        for name, tensor in state['dense'].items():
            state['host_dense'][name].copy_(tensor, non_blocking=True)

    def _finish_gather(self, state) -> Dict[str, Any]:
        """Second half, after the stream has been synchronised once: the packed rows, exactly as many bytes as are live
        (one copy per array), then the host views."""
        B = self.parallel_envs
        total = int(state['host_offsets'][B])
        moved = state['host_counts'].numel() * 4 + state['host_offsets'].numel() * 4
        moved += sum(t.numel() * t.element_size() for t in state['host_dense'].values())
        out: Dict[str, Any] = {'counts': state['host_counts'], 'offsets': state['host_offsets'], 'total': total}
        out.update(state['host_dense'])
        for name, device_rows in state['packed'].items():
            groups, row_shape, row_elements = state['layout'][name]
            live = total * groups * row_elements
            host_rows = state['host_packed'][name][:live]
            if live:
                host_rows.copy_(device_rows[:live], non_blocking=True)
            moved += live * device_rows.element_size()
            # environment b's block g = rows [offsets[b] * groups + g * counts[b], ... + counts[b])
            out[name] = host_rows.view((total * groups, ) + row_shape) if row_shape else host_rows
        torch.cuda.current_stream(self.device).synchronize()
        out['bytes'] = moved
        return out

    def _compact_schema(self, buffers: Optional[Dict[str, torch.Tensor]] = None) -> compact.Schema:
        """The domain's compact observation format (utils/compact.py) over ``buffers`` (None = the live ones): which
        array is narrowed to which type, from bounds the configuration guarantees.  Domain hook."""
        raise NotImplementedError

    def _compact_download(self, final: bool = False) -> compact.CompactDownload:
        attribute = '_compact_final' if final else '_compact'
        download = getattr(self, attribute, None)
        if download is None or download.key != self.max_steps:  # (rideshare bounds depend on the horizon)
            schema = self._compact_schema(self._download_buffers(final))
            counts = self._final_counts if final else self.environment_task_count
            download = compact.CompactDownload(schema, counts, key=self.max_steps)
            setattr(self, attribute, download)
        return download

    def _enqueue_compact(self, final: bool = False) -> compact.CompactDownload:
        """The compact download of the current state (frz_observe_compact), on the current stream of the device."""
        download = self._compact_download(final)
        self._download_counts(final)
        _lib.check(self._lib.frz_observe_compact(ctypes.byref(download.block), self.parallel_envs, self._stream()),
                   'frz_observe_compact')
        return download

    @torch.no_grad()
    def gather_observations(self, compact: bool = False, final: bool = False) -> Dict[str, Any]:
        """The observations of the current state in page-locked HOST memory, packed like the reference's jagged nested
        tensors (a value buffer + offsets; wildfire.py:669-717, rideshare.py:398-467): ``counts`` int32 [B] live tasks
        per environment, ``offsets`` int32 [B + 1] their exclusive prefix sum, the dense arrays (``self_obs``,
        ``agent_task_count``, ...) whole, and for every padded array its live rows only -- environment b's row block
        g of array ``name`` is ``out[name][offsets[b] * groups + g * counts[b] :][:counts[b]]`` (groups = 1 for task
        observations, = agents for the action / task masks).  The live rows are compacted on the device
        (``frz_gather_live_rows``) so that each array crosses PCIe in one copy of exactly its live bytes.  The
        returned tensors are overwritten by the next call.  ``out['bytes']`` = bytes copied device -> host.

        ``compact=True`` returns the same observations in the compact format instead (a ``CompactObservations``,
        utils/compact.py: narrow integers, bit masks, no configuration constants; ``.unpack()`` gives this dict), encoded
        on the device and stored straight into page-locked host buffers: one synchronisation, fewer bytes.

        ``final=True`` (``keep_final_observations=True`` only) downloads ``final_observations`` instead, in either
        format: ``counts`` is environment b's final task count where ``episode_statistics['done'][b]`` is set and 0
        elsewhere, so only the finished environments' rows cross the link; the dense arrays come whole and are defined
        where ``done`` is set.  Its host buffers are separate from those of the live download."""
        with torch.cuda.device(self.device):
            if compact:
                download = self._enqueue_compact(final)
                torch.cuda.current_stream(self.device).synchronize()
                return download.result()
            state = self._gather_state(final)
            self._enqueue_gather(state)
            torch.cuda.current_stream(self.device).synchronize()
            return self._finish_gather(state)

    @torch.no_grad()
    def step_host(self, host_actions: torch.Tensor, chunks: Optional[int] = None, observations: bool | str = False
                  ) -> Tuple[torch.Tensor, ...]:
        """One environment step for callers that live on the host: ``host_actions`` is a page-locked int32 -- or int16 /
        int8 (at most 127 tasks per environment), which halve / quarter the upload and are widened on the device --
        ``[B, A, 2]`` CPU tensor (agent order = ``env.agents``);
        returns page-locked CPU tensors ``(rewards f32 [B, A],
        terminated bool [B], truncated bool [B])`` that are valid when the call returns and are overwritten by the next
        ``step_host``.  Equivalent to copying the actions to the device, ``step_all`` and copying the results back,
        but the batch is cut into ``chunks`` slices whose uploads, step kernels and downloads overlap
        (``frz_<domain>_step_host``, include/frz.h); the results are bit-identical.  Observations, masks and counts stay
        on the device as usual -- unless ``observations=True``: then the call also returns, as a fourth element, what
        ``gather_observations()`` returns (the next observations in host memory, packed), which is what a policy that
        runs on the CPU needs for its next decision.  ``observations='compact'`` returns them as
        ``gather_observations(compact=True)`` does: encoded on the device after the step and stored into page-locked
        host buffers, with one stream synchronisation for the whole call."""
        if not (isinstance(observations, bool) or (isinstance(observations, str) and observations == 'compact')):
            raise ValueError(f"observations must be False, True or 'compact', not {observations!r}")
        B, A = self.parallel_envs, len(self.possible_agents)
        if (host_actions.device.type != 'cpu' or host_actions.dtype not in (torch.int32, torch.int16, torch.int8)
                or not host_actions.is_contiguous() or tuple(host_actions.shape) != (B, A, 2)
                or not host_actions.is_pinned()):
            raise ValueError(f'step_host expects a page-locked contiguous int32 / int16 / int8 CPU tensor of shape {(B, A, 2)} '
                             '(torch.empty(..., dtype=torch.int32).pin_memory())')
        state = self._host_pipeline(chunks)
        state['block'].actions = host_actions.data_ptr()
        state['block'].action_format = {torch.int32: _lib.HOST_ACTIONS_I32, torch.int16: _lib.HOST_ACTIONS_I16,
                                        torch.int8: _lib.HOST_ACTIONS_I8}[host_actions.dtype]
        current, main = torch.cuda.current_stream(self.device), state['main']
        main.wait_stream(current)
        _lib.check(self._host_entry()(ctypes.byref(self._params), ctypes.byref(self._io), B,
                                      ctypes.byref(state['block']), ctypes.c_void_p(main.cuda_stream)), 'step_host')
        # (every slice's reward download and the done-flag download are on `main` before this point, so the host
        # results are the finishing step's)
        with torch.cuda.stream(main):
            self._autoreset_launch()
        current.wait_stream(main)  # later work on the caller's stream sees the stepped state
        # host-side bookkeeping while the device works; the views do not depend on the data
        self._mid_cycle = False
        self._rebind_outputs()
        if self.log_directory is not None:
            self._log_environment()
        if not observations:
            main.synchronize()
            return state['rewards'], state['terminated'], state['truncated']
        if observations == 'compact':
            with torch.cuda.stream(main):
                download = self._enqueue_compact()
            main.synchronize()
            return state['rewards'], state['terminated'], state['truncated'], download.result()
        with torch.cuda.stream(main):  # compaction + fixed-size downloads ride on the same synchronisation
            gather = self._gather_state()
            self._enqueue_gather(gather)
            main.synchronize()
            packed = self._finish_gather(gather)
        return state['rewards'], state['terminated'], state['truncated'], packed

    def _advance(self) -> None:
        _, _, infos = self.step_environment()
        self._autoreset_launch()
        self.infos = infos
        self._mid_cycle = False
        self._rebind_outputs()
        if self.log_directory is not None:
            self._log_environment()

    # ------------------------------------------------------------------------------------------ logging tap

    def _log_environment(self, reset: bool = False) -> None:
        """Queue one CSV row per environment (reference utils/env.py:256-271 -> CSVLogger); nothing here waits for the
        device: see utils/logging_tap.py."""
        if self._tap is None:
            from free_range_zoo_b200.utils.logging_tap import LoggingTap
            if str(self.log_directory).startswith('sqlite://'):  # reference utils/env.py:65-86
                from free_range_zoo_b200.utils.sql_tap import SqliteSink
                sink = SqliteSink(self.log_directory, self.metadata['name'], self.parallel_envs)
                self._tap = LoggingTap(self.log_directory, self.parallel_envs, self.device, self._log_snapshot,
                                       self._log_records, sink=sink, agents=self.possible_agents)
            else:
                self._tap = LoggingTap(self.log_directory, self.parallel_envs, self.device, self._log_snapshot,
                                       self._log_columns,
                                       override_initialization_check=self.override_initialization_check)
        self._tap.capture(reset, self.log_description, getattr(self, '_log_label', None))

    def flush_logs(self) -> None:
        """Wait until every queued log row is on disk."""
        if self._tap is not None:
            self._tap.flush()

    def _log_snapshot(self) -> Dict[str, torch.Tensor]:
        """Live device tensors the log rows are built from (domain tensors are added by the subclasses)."""
        return dict(actions=self._actions, rewards=self._rewards, num_moves=self.num_moves, terminated=self._terminated,
                    truncated=self._truncated, env_task_count=self.environment_task_count,
                    agent_task_count=self._agent_task_count)

    def _log_columns(self, host: Dict[str, Any], reset: bool) -> Dict[str, Any]:
        """Ordered CSV columns from the host copy of a snapshot: state columns, the per-agent action / reward columns,
        step, complete, the per-agent mappings, then the domain's extra columns (logging_handlers.py:77-100)."""
        from free_range_zoo_b200.utils.logging_tap import nested
        B = self.parallel_envs
        columns = dict(self._log_state_columns(host))
        finished = (host['terminated'] != 0) | (host['truncated'] != 0)
        for index, agent in enumerate(self.possible_agents):
            columns[f'{agent}_action'] = [None] * B if reset else [nested(host['actions'][b, index]) for b in range(B)]
            columns[f'{agent}_rewards'] = [None] * B if reset else host['rewards'][:, index].astype(float).tolist()
        columns['step'] = [-1] * B if reset else host['num_moves'].tolist()
        columns['complete'] = [None] * B if reset else finished.tolist()
        for index, agent in enumerate(self.possible_agents):
            action_map, observation_map = self._log_mappings(host, index)
            columns[f'{agent}_action_map'] = action_map
            columns[f'{agent}_observation_map'] = observation_map
        columns.update(self._log_extra_columns(host, reset))
        return columns

    def _log_records(self, host: Dict[str, Any], reset: bool) -> Dict[str, Any]:
        """The SQL sink's record of one snapshot (utils/sql_tap.py::SqliteSink.write): the same state / mapping cells as
        the CSV columns, raw action and reward values per agent (logging_handlers.py:160-241)."""
        state = dict(self._log_state_columns(host))
        state.update({name: cells for name, cells in self._log_extra_columns(host, reset).items()
                      if name not in ('burnouts', 'putouts')})
        agents = {}
        for index, agent in enumerate(self.possible_agents):
            action_map, observation_map = self._log_mappings(host, index)
            agents[agent] = dict(reward=host['rewards'][:, index], action_field=host['actions'][:, index, 1],
                                 task_field=host['actions'][:, index, 0], action_map=action_map,
                                 observation_map=observation_map)
        return dict(timestep=host['num_moves'], state=state, agents=agents)

    def _log_state_columns(self, host) -> Dict[str, Any]:
        raise NotImplementedError

    def _log_mappings(self, host, agent_index: int):
        raise NotImplementedError

    def _log_extra_columns(self, host, reset: bool) -> Dict[str, Any]:
        return {}

    def _rebind_outputs(self) -> None:
        """Re-create the lazily evaluated observation views after the device buffers changed."""
        self.update_observation_views()
        if self.detach_outputs:
            self._reward_views = {a: self._rewards[:, i].clone() for i, a in enumerate(self.agents)}
            terminated, truncated = self.terminated.clone(), self.truncated.clone()
            self.terminations = {a: terminated for a in self.agents}
            self.truncations = {a: truncated for a in self.agents}

    @abstractmethod
    def update_observation_views(self) -> None:
        """Build ``self.observations`` (dict agent -> ObservationDict) as views of the device buffers."""

    @torch.no_grad()
    def observe(self, agent: str) -> ObservationDict:
        return self.observations[agent]

    @torch.no_grad()
    def state(self):
        return self._state

    def last(self, observe: bool = True):
        """pettingzoo AEC convenience: (observation, reward, termination, truncation, info) of the selected agent."""
        agent = self.agent_selection
        observation = self.observe(agent) if observe else None
        return (observation, self._cumulative_rewards[agent], self.terminations[agent], self.truncations[agent],
                self.infos[agent])

    # ------------------------------------------------------------------------------------------ diagnostics

    def control_block(self) -> Dict[str, int]:
        """Host copy of the device control block (synchronises; diagnostics / tests only)."""
        raw = self._control.cpu().numpy().tobytes()
        block = _lib.Control.from_buffer_copy(raw)
        return {name: getattr(block, name) for name, _ in _lib.Control._fields_ if name != 'reserved'}

    def check_errors(self) -> None:
        """Raise ``ValueError`` for data-dependent faults the kernels recorded (the reference raises these eagerly,
        at the price of a host sync per step: cybersecurity.py:341-363).  Synchronises; call it off the hot path."""
        word = self.control_block()['error_word']
        if word:
            self._control.view(torch.int32)[7] = 0
            reasons = [text for bit, text in _lib.FAULT_NAMES.items() if word & bit]
            raise ValueError('invalid actions were submitted: ' + '; '.join(reasons))

    # ------------------------------------------------------------------------------------------ CUDA graph

    def capture_graph(self, sample: bool = False, sampler_seed: int = 2026, steps: int = 1) -> None:
        """Capture ``steps`` x ``[sample_actions ->] step [-> autoreset]`` in a CUDA graph; ``replay()`` then costs one graph launch
        per ``steps`` environment steps (small batches are bound by launch latency: several steps per launch keep the
        kernels back to back).  Kernel arguments are pointer-stable and the step counter lives on the device, so the
        graph needs no updates.  Capturing leaves the environment where it was (the warm-up launch is undone).  Replays
        do not feed the logging tap, so a ``log_directory`` is refused."""
        if self.log_directory is not None:
            raise RuntimeError('graph replays bypass the logging tap; capture_graph needs log_directory=None')
        torch.cuda.synchronize(self.device)
        # the warm-up launch outside capture (lazy module load, occupancy query) steps for real: every tensor the
        # kernels write -- state, outputs, the control block with the Philox step counter -- is put back afterwards,
        # so capturing does not advance the environment
        saved = {name: tensor.clone() for name, tensor in self._bound.items()
                 if tensor is not None and not name.startswith('init_')}
        autoreset = [self._autoreset_flags, self._episode_return, self._episode_length] if self.autoreset else []
        if self.keep_final_observations:
            autoreset += list(self._final_buffers.values())
        saved_autoreset = [tensor.clone() for tensor in autoreset]
        side = torch.cuda.Stream(self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):
            if sample:
                self.sample_actions(sampler_seed)
            self.step_environment()
            self._autoreset_launch()
        torch.cuda.current_stream(self.device).wait_stream(side)
        torch.cuda.synchronize(self.device)
        for name, tensor in saved.items():
            self._bound[name].copy_(tensor)
        for tensor, copy in zip(autoreset, saved_autoreset):
            tensor.copy_(copy)
        del saved
        torch.cuda.synchronize(self.device)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for _ in range(max(1, int(steps))):
                if sample:
                    self.sample_actions(sampler_seed)
                self.step_environment()
                self._autoreset_launch()
        self._graph = graph

    def replay(self) -> None:
        """Launch the captured graph (``steps`` environment steps); outputs are re-bound like after ``step``."""
        self._graph.replay()
        self._mid_cycle = False
        if self.detach_outputs:
            self._rebind_outputs()

    def sample_actions(self, sampler_seed: int = 2026) -> torch.Tensor:
        """Uniform random legal actions for every agent, generated on the device into the staged action table
        (the caller side of the path: replaces ``action_space(agent).sample_nested()`` per agent per step)."""
        raise NotImplementedError

    # ------------------------------------------------------------------------------------------ policy actions

    @property
    def action_slots(self) -> int:
        """C: the fixed number of action slots per agent a policy scores (include/frz_policy.h) -- wildfire H*W + 1
        (slot t acts on env-local task t, the last is the noop), rideshare K + 1 (table row t, then the noop),
        cybersecurity N + 3 (node t, then noop, patch, monitor).  The legal slots of (environment, agent) are, in slot
        order, the choices of ``action_space(agent)`` for that environment.  Domain hook."""
        raise NotImplementedError

    def _policy_entry(self):
        """The domain's ``frz_<domain>_policy_actions`` entry point."""
        raise NotImplementedError

    def _policy_buffers(self) -> Dict[str, torch.Tensor]:
        """Env-owned outputs of the policy launches, allocated by the first call (later calls allocate nothing)."""
        buffers = self.__dict__.get('_policy')
        if buffers is None:
            B, A, dev = self.parallel_envs, len(self.possible_agents), self.device
            buffers = self._policy = dict(slots=torch.zeros((B, A), dtype=torch.int32, device=dev),
                                          log_prob=torch.zeros((B, A), dtype=torch.float32, device=dev),
                                          legal=torch.zeros((B, A, self.action_slots), dtype=torch.bool, device=dev))
        return buffers

    def _legal_kind(self, tensor: torch.Tensor, what: str) -> bool:
        """Check a legal-mask output: bool / uint8 [B, A, C], or int32 [B, A, W] (W = ceil(C / 32)) for the packed mask
        (include/frz_policy.h), contiguous.  Returns whether it is packed."""
        B, A, C = self.parallel_envs, len(self.possible_agents), self.action_slots
        packed = isinstance(tensor, torch.Tensor) and tensor.dtype == torch.int32
        if not packed:
            self._check_policy_tensor(tensor, what, (torch.bool, torch.uint8))
        elif tensor.device != self.device or tuple(tensor.shape) != (B, A, (C + 31) // 32):
            raise ValueError(f'{what} (packed) must be an int32 tensor of shape {(B, A, (C + 31) // 32)} on '
                             f'{self.device} (W = ceil({C} / 32) words per row)')
        if not tensor.is_contiguous():
            raise ValueError(f'{what} must be contiguous')
        return packed

    def _check_policy_tensor(self, tensor: torch.Tensor, what: str, dtypes, slots: bool = True) -> None:
        B, A = self.parallel_envs, len(self.possible_agents)
        shape = (B, A, self.action_slots) if slots else (B, A)
        if not isinstance(tensor, torch.Tensor) or tensor.device != self.device or tensor.dtype not in dtypes \
                or tuple(tensor.shape) != shape:
            raise ValueError(f'{what} must be a {" / ".join(str(d) for d in dtypes)} tensor of shape {shape} on '
                             f'{self.device}')

    def _policy_launch(self, mode: int, logits: Optional[torch.Tensor] = None, legal: Optional[torch.Tensor] = None,
                       sampler_seed: int = 0) -> None:
        buffers = self._policy_buffers()
        block = _lib.PolicyActions()
        if legal is not None and legal.dtype == torch.int32:
            mode |= _lib.POLICY_PACKED_LEGAL
        block.mode, block.slots = mode, self.action_slots
        block.slot, block.log_prob = buffers['slots'].data_ptr(), buffers['log_prob'].data_ptr()
        block.legal = _lib.pointer(legal)
        block.sampler_seed = int(sampler_seed) & 0xFFFFFFFFFFFFFFFF
        if logits is not None:
            block.logits, block.row_stride = logits.data_ptr(), logits.stride(1)
            block.logits_type = _lib.LOGITS_BF16 if logits.dtype == torch.bfloat16 else _lib.LOGITS_F32
        _lib.check(self._policy_entry()(ctypes.byref(self._params), ctypes.byref(self._io), self.parallel_envs,
                                        ctypes.byref(block), self._stream()), 'policy_actions')

    def legal_actions(self, out: Optional[torch.Tensor] = None, packed: bool = False) -> torch.Tensor:
        """bool [B, A, C] on the device: slot t of (environment, agent) is legal (``action_slots``).  Written into
        ``out`` (bool or uint8, contiguous) when given, else into an env-owned buffer the next call overwrites.

        ``packed=True`` returns the mask bit-packed instead, int32 [B, A, W] with W = ceil(C / 32): bit t % 32 of word
        t / 32 is slot t, bits at or beyond C are 0 (``utils.policy.unpack_legal`` unpacks it).  An int32 ``out`` of
        that shape receives the packed mask too."""
        if out is None:
            buffers = self._policy_buffers()
            if packed and 'legal_packed' not in buffers:
                B, A, C = self.parallel_envs, len(self.possible_agents), self.action_slots
                buffers['legal_packed'] = torch.zeros((B, A, (C + 31) // 32), dtype=torch.int32, device=self.device)
            out = buffers['legal_packed' if packed else 'legal']
        else:
            self._legal_kind(out, 'out')
        self._policy_launch(_lib.POLICY_LEGAL, legal=out)
        return out

    def sample_actions_from_logits(self, logits: torch.Tensor, sampler_seed: int = 2026,
                                   legal_out: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
        """Sample every agent's action from ``logits`` (f32 or bf16 [B, A, C] on the device, C = ``action_slots``; rows
        may be a view with a larger stride, e.g. ``wide[..., :C]``) restricted to the legal slots, and stage it for
        ``step_all(None)`` / the Parallel ``step``.  One launch, no host read: capturable in a CUDA graph.

        Returns ``(slots, log_prob)``: int32 [B, A] chosen slots and f32 [B, A] their log-probability under the masked
        softmax, env-owned buffers overwritten by the next call.  ``legal_out`` (bool / uint8 [B, A, C], or int32
        [B, A, ceil(C / 32)] for the packed mask of ``legal_actions(packed=True)``; contiguous) receives the legal mask
        in the same launch, e.g. for a learner that recomputes log-probabilities with gradients
        (``utils.policy.slot_log_prob``).
        The random draw of (environment, agent) is the one ``sample_actions(sampler_seed)`` makes, so equal logits
        stage exactly what ``sample_actions`` stages.  NaN / +inf in a legal slot, or -inf in all of them, records a
        fault (``check_errors``) and stages the noop."""
        self._check_policy_tensor(logits, 'logits', (torch.float32, torch.bfloat16))
        if logits.stride(2) != 1 or logits.stride(0) != logits.stride(1) * logits.shape[1]:
            raise ValueError('logits rows must be evenly spaced with unit stride along the slots '
                             '(a contiguous tensor, or a [..., :C] view of one)')
        if legal_out is not None:
            self._legal_kind(legal_out, 'legal_out')
        self._policy_launch(_lib.POLICY_SAMPLE, logits=logits, legal=legal_out, sampler_seed=sampler_seed)
        buffers = self._policy_buffers()
        return buffers['slots'], buffers['log_prob']

    def actions_from_slots(self, slots: torch.Tensor) -> torch.Tensor:
        """Stage the actions of chosen slots (int [B, A], on the device or the host), e.g. a greedy
        ``logits.masked_fill(~legal, -inf).argmax(-1)`` or a CPU policy's choices.  An out-of-range or illegal slot
        records a fault (``check_errors``) and stages the noop.  Returns the staged [B, A, 2] action table."""
        shape = (self.parallel_envs, len(self.possible_agents))
        if not isinstance(slots, torch.Tensor) or tuple(slots.shape) != shape or slots.is_floating_point() \
                or slots.is_complex() or slots.dtype == torch.bool:
            raise ValueError(f'slots must be an integer tensor of shape {shape}')
        buffers = self._policy_buffers()
        if slots.data_ptr() != buffers['slots'].data_ptr():
            buffers['slots'].copy_(slots, non_blocking=True)
        self._policy_launch(_lib.POLICY_DECODE)
        return self._actions

    # ------------------------------------------------------------------------------------------ policy inputs

    def _policy_input_layout(self) -> PolicyInputLayout:
        """The structure of the policy inputs (include/frz_inputs.h), from ``_params`` and the observe flags only (no
        device, no configuration).  Domain hook."""
        raise NotImplementedError

    def _policy_input_schema(self) -> PolicyInputSchema:
        """The layout and every column's ``(scale, offset)``, from the bounds of ``observation_space``.  Domain hook."""
        raise NotImplementedError

    def _inputs_entry(self):
        """The domain's ``frz_<domain>_policy_inputs`` entry point."""
        raise NotImplementedError

    @property
    def policy_input_shapes(self) -> Dict[str, Tuple[int, ...]]:
        """``{'agent': (A, Fa), 'tasks': (V, T, Ft)}``: the per-environment shapes of ``policy_inputs``.  Row t < T of
        a view's task block is padded task row t, which action slot t acts on (``action_slots``): wildfire env-local
        task t, rideshare table row t, cybersecurity node t."""
        layout = self._policy_input_layout()
        A = sum(kind.count for kind in layout.kinds)
        Fa = max(kind.width for kind in layout.kinds if kind.count > 0)
        return {'agent': (A, Fa), 'tasks': (layout.views, layout.task_rows, len(layout.task_columns) + 1)}

    def _policy_inputs_block(self) -> _lib.PolicyInputs:
        """The launch block with the schema's column tables (built once; the call fills in outputs and type)."""
        block = self.__dict__.get('_inputs_block')
        if block is None:
            schema = self._policy_input_schema()
            layout = schema.layout
            block = _lib.PolicyInputs()
            shapes = self.policy_input_shapes
            block.agent_width = shapes['agent'][1]
            block.views, block.task_rows, block.task_width = shapes['tasks']
            block.flags = layout.flags
            for index, (kind, columns) in enumerate(zip(layout.kinds, schema.self_columns)):
                target = block.self_columns[index]
                target.columns = kind.columns
                target.observed = sum(1 << c for c in kind.observed)
                for c, (scale, offset) in enumerate(columns):
                    target.scale[c], target.offset[c] = scale, offset
            target = block.task_columns
            target.columns = len(layout.task_columns)
            target.pad_is_none = sum(1 << c for c, none in enumerate(layout.task_columns) if none)
            for c, (scale, offset) in enumerate(schema.task_columns):
                target.scale[c], target.offset[c] = scale, offset
            self._inputs_block = block
        return block

    def _inputs_io(self, final: bool):
        """The domain's buffer struct, with the observation arrays of ``final_observations`` when ``final``."""
        if not final:
            return self._io
        if not self.keep_final_observations:
            raise RuntimeError('final_observations are kept by the autoreset: construct the environment with '
                               'autoreset=True, keep_final_observations=True')
        io = type(self._io).from_buffer_copy(self._io)
        for name, tensor in self._final_buffers.items():
            setattr(io, name, tensor.data_ptr())
        return io

    def policy_inputs(self, dtype: torch.dtype = torch.float32, final: bool = False,
                      out: Optional[Tuple[torch.Tensor, torch.Tensor]] = None) -> Tuple[torch.Tensor, torch.Tensor]:
        """The observations of every environment and agent as fixed-width policy inputs (include/frz_inputs.h), in one
        launch with no host read (capturable in a CUDA graph).  Returns ``(agent, tasks)`` of ``dtype`` (f32 or bf16):

        - ``agent`` [B, A, Fa]: the agent's ``self`` columns, then the observed columns of each agent of its ``others``
          view, in the view's order (cybersecurity: the shorter kind zero-padded);
        - ``tasks`` [B, V, T, Ft]: row t is padded task row t, i.e. action slot t.  Column 0 is 1 iff the row is a live
          task the view may see, then the row's columns; other rows are all zeros.  V = 1 when every agent sees the same
          tasks (wildfire, rideshare), V = A when views differ (cybersecurity: an unmonitored defender under partial
          observability sees none).

        Every column is ``float(v + offset) * scale`` in f32 (bf16: rounded once, to nearest even), with scale
        ``1 / high`` of the column's bound in ``observation_space`` (1 where a bound is missing or not positive) and
        offset 0; "none" columns (rideshare accepted_by / riding_by, the cybersecurity defender location) use offset 1
        and scale ``1 / (high + 1)``, so that "none" is exactly 0.  No clamping.

        ``final=True`` encodes ``final_observations`` (``keep_final_observations=True`` only).  The result buffers
        belong to the environment, one pair per ``(dtype, final)``, allocated by the first call and overwritten by the
        next; ``out=(agent, tasks)`` writes into contiguous caller tensors of the right shape, dtype and device instead
        (e.g. ``storage[t]`` of a ``[T_rollout, B, ...]`` rollout buffer)."""
        if dtype not in (torch.float32, torch.bfloat16):
            raise ValueError(f'dtype must be torch.float32 or torch.bfloat16, not {dtype}')
        io = self._inputs_io(final)
        shapes = self.policy_input_shapes
        B = self.parallel_envs
        wanted = ((B, ) + shapes['agent'], (B, ) + shapes['tasks'])
        if out is None:
            buffers = self.__dict__.setdefault('_inputs', {})
            out = buffers.get((dtype, final))
            if out is None:
                out = buffers[(dtype, final)] = tuple(torch.zeros(shape, dtype=dtype, device=self.device)
                                                      for shape in wanted)
        else:
            if not isinstance(out, (tuple, list)) or len(out) != 2:
                raise ValueError('out must be a pair (agent, tasks)')
            for name, tensor, shape in zip(('agent', 'tasks'), out, wanted):
                if not isinstance(tensor, torch.Tensor) or tuple(tensor.shape) != shape or tensor.dtype != dtype \
                        or tensor.device != self.device or not tensor.is_contiguous():
                    raise ValueError(f'out {name} must be a contiguous {dtype} tensor of shape {shape} on {self.device}')
            out = tuple(out)
        block = _lib.PolicyInputs.from_buffer_copy(self._policy_inputs_block())
        block.agent, block.tasks = out[0].data_ptr(), out[1].data_ptr()
        block.output_type = _lib.INPUTS_BF16 if dtype == torch.bfloat16 else _lib.INPUTS_F32
        _lib.check(self._inputs_entry()(ctypes.byref(self._params), ctypes.byref(io), B, ctypes.byref(block),
                                        self._stream()), 'policy_inputs')
        return out
