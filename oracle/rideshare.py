"""CPU oracle for the rideshare step path -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Only ``tests/``, ``__graft_entry__.smoke()`` and the CPU-baseline legs of ``bench.py`` may import this module.

Scalar (per environment, per passenger) restatement of the reference's rideshare hot path (paths relative to
``free_range_zoo/`` in /root/reference): envs/rideshare/env/rideshare.py:249-467 and
env/transitions/{movement,passenger_state,passenger_exit,passenger_entry}.py.  The reference keeps ONE flat passenger
table ``[N_total, 11]`` sorted by environment; here every environment owns its slice of that table (same row order),
which is also how the CUDA engine stores it.
Parity pin: tests/test_oracle_golden.py replays tests/golden/rideshare_*.npz (recorded from the unmodified reference,
including illegal-but-accepted action ids in ``rideshare_wild``); tests/test_oracle_kat.py re-states the reference's
transition unit-test vectors.
"""
from __future__ import annotations

import numpy as np

PAD = -100
F32 = np.float32
# passenger columns (envs/rideshare/env/structures/state.py:11-22)
BATCH, Y, X, DEST_Y, DEST_X, FARE, STATE, ASSOC, ENTERED, ACCEPTED, PICKED = range(11)

CARDINAL = [(0, 0), (-1, 0), (0, 1), (1, 0), (0, -1)]  # stay, N, E, S, W (transitions/movement.py:27-36)
DIAGONAL = [(-1, -1), (-1, 1), (1, 1), (1, -1)]  # NW, NE, SE, SW (:37-45)


def _np(x, dtype):
    return np.asarray(x.detach().cpu().numpy() if hasattr(x, 'detach') else x, dtype=dtype)


def _norm(dy, dx) -> np.float32:
    return np.sqrt(F32(F32(dy) * F32(dy) + F32(dx) * F32(dx)))


class RideshareOracle:

    def __init__(self, configuration, parallel_envs: int, max_steps: int = 1):
        c = configuration
        ac, rc = c.agent_config, c.reward_config
        self.B = parallel_envs
        self.max_steps = max_steps
        self.starts = _np(ac.start_positions, np.int32)
        self.A = self.starts.shape[0]
        self.pool_limit = int(ac.pool_limit)
        self.fast = bool(ac.use_fast_travel)
        self.directions = CARDINAL + (DIAGONAL if ac.use_diagonal_travel else [])
        self.schedule = _np(c.passenger_config.schedule, np.int32)
        self.K = self.schedule.shape[0]
        self.rc = rc
        self.wait_limit = [int(v) for v in _np(rc.wait_limit, np.int64)]

    # ------------------------------------------------------------------ reset

    def reset(self, initial_state: dict | None = None):
        """rideshare.py:188-229: agents at their start positions (or ``initial_state['agents']`` [B, A, 2]), the
        passenger table empty (or the rows of ``initial_state['passengers']`` [N, 11] whose column 0 is the
        environment, in their order), then the passengers scheduled for t = 0 enter."""
        B, A = self.B, self.A
        if initial_state is not None:
            agents = np.array(initial_state['agents'], np.int32)
            rows = np.asarray(initial_state.get('passengers', np.zeros((0, 11))), np.int64)
            tables = [[[int(v) for v in row] for row in rows if row[0] == b] for b in range(B)]
        else:
            agents, tables = np.tile(self.starts[None], (B, 1, 1)).astype(np.int32), [[] for _ in range(B)]
        self.initial_state = dict(agents=agents, tables=tables)  # utils/state.py:36-38
        self.agents = agents.copy()
        self.tables = [[list(row) for row in table] for table in tables]  # per env: list of 11-int rows in table order
        self.num_moves = np.zeros(B, np.int32)
        self.rewards = np.zeros((B, A), np.float32)
        self.cumulative_rewards = np.zeros((B, A), np.float32)
        self.terminated = np.zeros(B, bool)
        self.truncated = np.zeros(B, bool)
        self._entry(self.num_moves)
        self._publish()

    def reset_batches(self, mask):
        """utils/env.py:163-189 for the environments selected by ``mask`` (bool [B]): drivers and passenger table back
        to the saved initial state, AEC fields zeroed, the t = 0 passengers enter again; then everything is published.
        The reference raises NotImplementedError for a partial rideshare reset (rideshare.py:231-246); this follows
        the engine's documented intent (include/frz.h, frz_rideshare_reset)."""
        mask = np.asarray(mask, bool)
        for b in np.nonzero(mask)[0]:
            self.agents[b] = self.initial_state['agents'][b]
            self.tables[b] = [list(row) for row in self.initial_state['tables'][b]]
        for key in ('rewards', 'cumulative_rewards', 'terminated', 'truncated', 'num_moves'):
            getattr(self, key)[mask] = 0
        self._entry(self.num_moves, mask)
        self._publish()

    def _entry(self, timesteps, mask=None):
        """transitions/passenger_entry.py:25-72: rows whose start time equals the env's timestep (and whose batch
        is the env or -1) are appended in schedule order (only in the environments selected by ``mask``)."""
        for b in range(self.B):
            if mask is not None and not mask[b]:
                continue
            for row in self.schedule:
                if row[0] == timesteps[b] and (row[1] == b or row[1] == -1):
                    self.tables[b].append(
                        [b, row[2], row[3], row[4], row[5], row[6], 0, -1, int(timesteps[b]), -1, -1])

    def _task_list(self, b: int, a: int):
        """Rows an agent may act on: unaccepted, or associated with it (rideshare.py:374-386)."""
        return [i for i, p in enumerate(self.tables[b]) if p[STATE] == 0 or p[ASSOC] == a]

    def _publish(self):
        """update_actions + update_observations (rideshare.py:368-467)."""
        B, A, K = self.B, self.A, self.K
        self.environment_task_count = np.array([len(t) for t in self.tables], np.int32)
        self.agent_task_count = np.zeros((B, A), np.int32)
        self.self_obs = np.zeros((B, A, 4), np.int32)
        self.self_obs[:, :, :2] = self.agents
        self.task_store = np.full((B, K, 8), PAD, np.int32)
        self.task_obs = np.full((A, B, K, 8), PAD, np.int32)
        self.action_map = np.full((A, B, K), PAD, np.int32)
        for b in range(B):
            rows = []
            for p in self.tables[b]:
                rows.append([p[Y], p[X], p[DEST_Y], p[DEST_X], p[ASSOC] if p[STATE] == 1 else PAD,
                             p[ASSOC] if p[STATE] == 2 else PAD, p[FARE], p[ENTERED]])
            if rows:
                self.task_store[b, :len(rows)] = rows
            for a in range(A):
                mine = self._task_list(b, a)
                self.agent_task_count[b, a] = len(mine)
                self.action_map[a, b, :len(mine)] = mine
                if mine:
                    self.task_obs[a, b, :len(mine)] = [rows[i] for i in mine]
                self.self_obs[b, a, 2] = sum(1 for p in self.tables[b] if p[STATE] == 1 and p[ASSOC] == a)
                self.self_obs[b, a, 3] = sum(1 for p in self.tables[b] if p[STATE] == 2 and p[ASSOC] == a)

    def others_obs(self, a: int):
        return self.self_obs[:, [i for i in range(self.A) if i != a]]

    def passengers_padded(self):
        table = np.full((self.B, self.K, 11), PAD, np.int32)
        for b, rows in enumerate(self.tables):
            if rows:
                table[b, :len(rows)] = rows
        return table

    # ------------------------------------------------------------------ transitions (one environment at a time)

    def movement(self, b: int, vector):
        """transitions/movement.py:94-116: move every agent one step towards its goal; riding passengers follow their
        driver.  Returns the distance cost of each agent."""
        cost = np.zeros(self.A, np.float32)
        moves = []
        for a in range(self.A):
            move, cost[a] = self._move(vector[a][:2], vector[a][2:])
            moves.append(move)
            self.agents[b, a, 0] += move[0]
            self.agents[b, a, 1] += move[1]
        for p in self.tables[b]:
            if p[STATE] == 2:
                move = moves[p[ASSOC]]  # ASSOC == -1 wraps to the last agent, exactly like the tensor index does
                p[Y] += move[0]
                p[X] += move[1]
        return cost

    def passenger_state(self, b: int, accept, pick, target, vector, t_now: int):
        """transitions/passenger_state.py:24-100; distances come from the PRE-move vectors.  Returns them."""
        A, table = self.A, self.tables[b]
        dist = [np.inf if v[0] == PAD else _norm(v[0] - v[2], v[1] - v[3]) for v in vector]
        claims = [target[a] if accept[a] else PAD for a in range(A)]
        duplicated = [claims[a] != PAD and claims.count(claims[a]) > 1 for a in range(A)]
        if any(duplicated):  # among ALL duplicated claims of the env only the closest claimant (first on ties) survives
            contest = [dist[a] if duplicated[a] else np.inf for a in range(A)]
            keep = int(np.argmin(np.array(contest, dtype=np.float32)))
            for a in range(A):
                if duplicated[a] and a != keep:
                    claims[a] = PAD
        for a in range(A):
            if claims[a] != PAD:
                p = table[claims[a]]
                p[STATE], p[ACCEPTED], p[ASSOC] = 1, t_now, a
        for a in range(A):
            if pick[a] and target[a] != PAD and dist[a] < 1e-6:
                p = table[target[a]]
                p[STATE], p[PICKED] = 2, t_now
        return dist

    def passenger_exit(self, b: int, drop, target, dist):
        """transitions/passenger_exit.py:23-56: a drop succeeds iff the driver stood on the destination."""
        table = self.tables[b]
        fares = np.zeros(self.A, np.int32)
        finished = set()
        for a in range(self.A):
            if drop[a] and target[a] != PAD and dist[a] == 0:
                fares[a] = table[target[a]][FARE]
                finished.add(target[a])
        self.tables[b] = [p for i, p in enumerate(table) if i not in finished]
        return fares

    # ------------------------------------------------------------------ step

    def _move(self, start, goal):
        """transitions/movement.py:57-116: first argmin of the L2 distance of each candidate to the goal."""
        if start[0] == PAD:
            return (0, 0), F32(0)
        if self.fast:
            move = (int(goal[0] - start[0]), int(goal[1] - start[1]))
        else:
            best, move = None, (0, 0)
            for dy, dx in self.directions:
                d = _norm(start[0] + dy - goal[0], start[1] + dx - goal[1])
                if best is None or d < best:
                    best, move = d, (dy, dx)
        if len(self.directions) == 9:
            cost = _norm(move[0], move[1])
        else:
            cost = F32(abs(move[0]) + abs(move[1]))
        return move, cost

    def step(self, actions: np.ndarray):
        """One AEC round (utils/env.py:203-242 around rideshare.py:249-365). actions int32 [B, A, 2]."""
        if self.terminated.all() or self.truncated.all():
            return False
        B, A, rc = self.B, self.A, self.rc
        rewards = np.zeros((B, A), np.float32)
        agent_active = self.agent_task_count.sum(axis=0) > 0  # rideshare.py:276 (a batch-wide test)
        for b in range(B):
            table = self.tables[b]
            t_now = int(self.num_moves[b])
            ident = actions[b, :, 1]
            noop, accept, pick, drop = ident == -1, ident == 0, ident == 1, ident == 2
            # ---- decode (rideshare.py:255-300)
            target = [PAD] * A
            vector = [(PAD, PAD, PAD, PAD)] * A
            for a in range(A):
                if agent_active[a] and not noop[a]:
                    mine = self._task_list(b, a)
                    k = int(actions[b, a, 0])
                    if 0 <= k < len(mine):
                        target[a] = mine[k]
                if target[a] == PAD:
                    continue
                p = table[target[a]]
                if accept[a] or pick[a]:
                    vector[a] = (self.agents[b, a, 0], self.agents[b, a, 1], p[Y], p[X])
                elif drop[a]:
                    vector[a] = (self.agents[b, a, 0], self.agents[b, a, 1], p[DEST_Y], p[DEST_X])
            cost = self.movement(b, vector)
            dist = self.passenger_state(b, accept, pick, target, vector, t_now)
            fares = self.passenger_exit(b, drop, target, dist)
            table = self.tables[b]
            # ---- entry at num_moves + 1 (rideshare.py:307)
            for row in self.schedule:
                if row[0] == t_now + 1 and (row[1] == b or row[1] == -1):
                    table.append([b, row[2], row[3], row[4], row[5], row[6], 0, -1, t_now + 1, -1, -1])
            # ---- rewards (rideshare.py:309-363)
            shared = F32(0)
            if rc.use_waiting_costs:
                stamp = (ENTERED, ACCEPTED, PICKED)
                for state in range(3):  # one statement per class; duplicate indices => the LAST row of the class lands
                    rows = [p for p in table if p[STATE] == state]
                    if rows:
                        elapsed = t_now - rows[-1][stamp[state]]
                        shared = F32(shared + F32(elapsed >= self.wait_limit[state]) * F32(rc.general_wait_cost))
                rows = [p for p in table if p[STATE] == 0]
                if rows:
                    elapsed = t_now - rows[-1][ENTERED]
                    shared = F32(shared + F32(elapsed >= rc.long_wait_time) * F32(rc.long_wait_cost))
                free = A * self.pool_limit - len(table)
                unaccepted = sum(1 for p in table if p[STATE] == 0)
                shared = F32(shared + F32(F32(unaccepted >= free) * F32(-0.5)) * F32(free))
            for a in range(A):
                accepted = sum(1 for p in table if p[ASSOC] == a)
                r = F32(0)
                r = F32(r + (F32(rc.pool_limit_cost) if accepted > self.pool_limit else F32(0)))
                r = F32(r + F32(noop[a]) * F32(rc.noop_cost))
                r = F32(r + F32(accept[a]) * F32(rc.accept_cost))
                r = F32(r + (F32(fares[a]) - F32(rc.drop_cost) if fares[a] > 0 else F32(0)))
                move_reward = F32(cost[a] * F32(rc.move_cost))
                if rc.use_variable_move_cost:
                    move_reward = F32(move_reward / F32(accepted + 1))
                r = F32(r + move_reward)
                rewards[b, a] = F32(r + shared)

        self.rewards = rewards
        self.num_moves = self.num_moves + 1
        if self.max_steps is not None:
            self.truncated = self.num_moves >= self.max_steps
        self.cumulative_rewards = self.cumulative_rewards + rewards
        self._publish()
        return True

    def outputs(self) -> dict:
        """Same keys/layout as tests/golden/gen_golden.py::rideshare_outputs."""
        A = self.A
        return dict(
            agents=self.agents, passengers=self.passengers_padded(), passenger_count=self.environment_task_count,
            rewards=self.rewards, terminated=np.repeat(self.terminated[:, None], A, axis=1),
            truncated=np.repeat(self.truncated[:, None], A, axis=1), num_moves=self.num_moves,
            env_task_count=self.environment_task_count, agent_task_count=self.agent_task_count,
            self_obs=self.self_obs, others_obs=np.stack([self.others_obs(a) for a in range(A)], axis=0),
            task_store=self.task_store, task_obs=self.task_obs, action_map=self.action_map,
        )
