"""VecMapfEnv -- B independent copies of one MapfEnv spec, stepped and expanded in bulk on one GPU.

This is the batched surface the reference lacks (SURVEY.md 8b): the same transition model as `MapfEnv.step` /
`MapfEnv.P` (reference mapf_env.py:237-266, 448-479), over device-resident tensors.

State tensors are `int64[B]` when L**n < 2**63, else `int64[B, 2]` (low word, high word).  Actions are `int32[B]`
base-5 joint actions.  Rewards / probabilities are float64, dones / collisions are bool.
"""
import collections

import numpy as np

Transitions = collections.namedtuple("Transitions", "row_ptr next_state prob reward flags")
Rollout = collections.namedtuple("Rollout", "next_state reward prob done collision")
# per episode: return f64, length i32 (steps taken), outcome u8 (0 timeout, 1 collision, 2 goal, 3 the start was terminal)
Evaluation = collections.namedtuple("Evaluation", "returns lengths outcomes")
# find_conflicts: the Evaluation, the attributed pair per episode (u8[E], i | j << 4 or NO_CONFLICT) and counts[i, j]
# (int64[n, n], i < j): the number of episodes attributed to the pair (i, j)
Conflicts = collections.namedtuple("Conflicts", "evaluation pairs counts")


def _int_root(x, k):
    r = int(round(x ** (1.0 / k)))
    while r > 0 and r ** k > x:
        r -= 1
    while (r + 1) ** k <= x:
        r += 1
    return r


class GroupPolicy(collections.namedtuple("GroupPolicy", "groups tables")):
    """A product of group policies: the agents are split into groups, and each group acts jointly by its own table.

    `groups`: a tuple of agent tuples that partitions agents 0..n-1, each ascending, in canonical order (by lowest
    agent).  `tables[g]`: int32[L**|g|] on the device, the group's joint action (base 5, agent g[k]'s digit at 5**k)
    indexed by the group's local state sum_k cell[g[k]] * L**k -- exactly the policy `value_iteration` returns on
    `get_local_view(env, g)`, and what `VecMapfEnv.project(states, g)` computes.  The constructor puts the groups (with
    their tables) in canonical order and rejects anything else it cannot use: agents out of order inside a group, a set
    of groups that does not partition 0..n-1, tables of the wrong dtype, length, device, or with entries outside
    [0, 5**|g|)."""
    __slots__ = ()

    def __new__(cls, groups, tables):
        import torch
        groups = [tuple(int(a) for a in g) for g in groups]
        tables = list(tables)
        if not groups or len(tables) != len(groups):
            raise ValueError("a GroupPolicy needs one table per group (got %d groups, %d tables)"
                             % (len(groups), len(tables)))
        for g in groups:
            if not g or any(a >= b for a, b in zip(g, g[1:])):
                raise ValueError("the agents of a group must be distinct and ascending (got %s)" % (g,))
        agents = sorted(a for g in groups for a in g)
        if agents != list(range(len(agents))):
            raise ValueError("the groups must partition the agents 0..n-1 (got %s)" % (groups,))
        order = sorted(range(len(groups)), key=lambda k: groups[k][0])
        groups, tables = tuple(groups[k] for k in order), [tables[k] for k in order]
        L, device = None, None
        for g, t in zip(groups, tables):
            if not isinstance(t, torch.Tensor) or t.dtype is not torch.int32 or t.dim() != 1 or t.numel() == 0:
                raise ValueError("the table of group %s must be a non-empty int32[L**%d] tensor" % (g, len(g)))
            r = _int_root(t.numel(), len(g))
            if r ** len(g) != t.numel() or (L is not None and r != L):
                raise ValueError("the table of group %s has %d entries, not L**%d%s"
                                 % (g, t.numel(), len(g), "" if L is None else " = %d" % L ** len(g)))
            if device is not None and t.device != device:
                raise ValueError("all tables must be on one device (got %s and %s)" % (device, t.device))
            L, device = r, t.device
            lo, hi = (int(v) for v in torch.aminmax(t))
            if lo < 0 or hi >= 5 ** len(g):
                raise ValueError("the entries of group %s's table must lie in [0, %d) (got [%d, %d])"
                                 % (g, 5 ** len(g), lo, hi))
        return super().__new__(cls, groups, tables)

    @property
    def n_agents(self):
        return sum(len(g) for g in self.groups)

    @property
    def n_cells(self):
        """L, the number of free cells the tables are indexed over."""
        return _int_root(self.tables[0].numel(), len(self.groups[0]))

    def group_of(self):
        """The group id of every agent (a list of n_agents ints)."""
        out = [0] * self.n_agents
        for gid, g in enumerate(self.groups):
            for a in g:
                out[a] = gid
        return out


def _canonical_groups(groups):
    """The groups as ascending agent tuples, and the order that sorts them by lowest agent; raises unless they
    partition the agents 0..n-1."""
    groups = [tuple(int(a) for a in g) for g in groups]
    for g in groups:
        if not g or any(a >= b for a, b in zip(g, g[1:])):
            raise ValueError("the agents of a group must be distinct and ascending (got %s)" % (g,))
    agents = sorted(a for g in groups for a in g)
    if not groups or agents != list(range(len(agents))):
        raise ValueError("the groups must partition the agents 0..n-1 (got %s)" % (groups,))
    return groups, sorted(range(len(groups)), key=lambda k: groups[k][0])


class GroupValues(collections.namedtuple("GroupValues", "groups values policy")):
    """Values of agent groups planned apart, the additive heuristic of `VecMapfEnv.rtdp`.

    `groups` partitions the agents as in GroupPolicy; `values[g]` is a float64[L**|g|] device tensor indexed by group g's
    local state (the V `value_iteration` returns on `get_local_view(env, g)`); `policy` is the GroupPolicy of the same
    groups (the fallback of the RTDP policy).  The heuristic of a joint state s is 0.0 when s is terminal, else
    ((0.0 + values[0][l_0(s)]) + values[1][l_1(s)]) + ... in group order.  The constructor puts groups and values in
    canonical order and rejects groups that do not partition the agents, values of the wrong dtype, shape or device,
    and a policy over other groups."""
    __slots__ = ()

    def __new__(cls, groups, values, policy):
        import torch
        values = list(values)
        if len(values) != len(groups):
            raise ValueError("GroupValues needs one value table per group (got %d groups, %d tables)"
                             % (len(groups), len(values)))
        groups, order = _canonical_groups(groups)
        groups, values = tuple(groups[k] for k in order), [values[k] for k in order]
        L, device = None, None
        for g, v in zip(groups, values):
            if not isinstance(v, torch.Tensor) or v.dtype is not torch.float64 or v.dim() != 1 or v.numel() == 0:
                raise ValueError("the values of group %s must be a non-empty float64[L**%d] tensor" % (g, len(g)))
            r = _int_root(v.numel(), len(g))
            if r ** len(g) != v.numel() or (L is not None and r != L):
                raise ValueError("the values of group %s have %d entries, not L**%d%s"
                                 % (g, v.numel(), len(g), "" if L is None else " = %d" % L ** len(g)))
            if device is not None and v.device != device:
                raise ValueError("all value tables must be on one device (got %s and %s)" % (device, v.device))
            L, device = r, v.device
        if not isinstance(policy, GroupPolicy) or policy.groups != groups or policy.n_cells != L or \
                policy.tables[0].device != device:
            raise ValueError("the policy must be a GroupPolicy of the groups %s on %d cells on %s" % (groups, L, device))
        return super().__new__(cls, groups, values, policy)


class ValueTable:
    """A device-resident value table for RTDP (C ABI `mapf_vtable`): `capacity` slots (a power of two, >= 64) of
    (key = one-word joint state, float64 value, int32 greedy joint action), open addressing with linear probing, at
    most capacity / 2 of them occupied.  Owns the five device tensors; the keys start as VTABLE_EMPTY."""

    def __init__(self, engine, capacity):
        capacity = int(capacity)
        if capacity < 64 or capacity & (capacity - 1):
            raise ValueError("capacity must be a power of two >= 64 (got %d)" % capacity)
        if engine.words != 1:
            raise ValueError("a value table is keyed by one-word states; this env's states take two words")
        import torch
        dev = engine.torch_device
        self.engine, self.capacity = engine, capacity
        self.keys = torch.full((capacity,), -1, dtype=torch.int64, device=dev)  # VTABLE_EMPTY as int64
        self.values = torch.zeros(capacity, dtype=torch.float64, device=dev)
        self.actions = torch.zeros(capacity, dtype=torch.int32, device=dev)
        self.count = torch.zeros(1, dtype=torch.int64, device=dev)

    def c_struct(self):
        from .. import _native
        return _native.MapfVtable(self.keys.data_ptr(), self.values.data_ptr(), self.actions.data_ptr(), self.capacity,
                                  self.count.data_ptr())

    def _count(self):
        return int(self.count.item()) & ((1 << 64) - 1)

    def __len__(self):
        """Occupied slots (synchronises with the device)."""
        return self._count() & ~(1 << 63)

    def overflowed(self):
        """True once a store was dropped because capacity / 2 slots were taken (synchronises with the device)."""
        return bool(self._count() >> 63)

    def lookup(self, states, heuristic):
        """(values f64[B], actions i32[B]): the stored value of each state, or `heuristic`'s (GroupValues) when it is not
        a key, and the stored action, or -1."""
        return self.engine.vtable_lookup(states, heuristic, self)

    def store(self, states, values, actions):
        """Stores (states[b], values[b], actions[b]); the states must be distinct."""
        self.engine.vtable_store(states, values, actions, self)

    def items(self):
        """(keys int64[K], values, actions) of the occupied slots, sorted by key (for inspection)."""
        occ = self.keys != -1
        keys, order = self.keys[occ].sort()
        return keys, self.values[occ][order], self.actions[occ][order]


class TablePolicy(collections.namedtuple("TablePolicy", "table fallback")):
    """The policy of a value table: in a state that is a key of `table` (ValueTable) take the action stored with it,
    anywhere else the action of `fallback` (GroupPolicy)."""
    __slots__ = ()

    def __new__(cls, table, fallback):
        if not isinstance(table, ValueTable):
            raise ValueError("table must be a ValueTable (got %s)" % type(table).__name__)
        if not isinstance(fallback, GroupPolicy):
            raise ValueError("fallback must be a GroupPolicy (got %s)" % type(fallback).__name__)
        return super().__new__(cls, table, fallback)


# rtdp: the value table, its TablePolicy (fallback: the heuristic's GroupPolicy) and one log record per iteration
Rtdp = collections.namedtuple("Rtdp", "table policy log")


def evaluation_summary(ev):
    """dict of the usual policy statistics of an Evaluation: mean / (population) standard deviation of the return, the
    shares of episodes that reached the goal, collided or ran out of steps, and the mean episode length."""
    from .. import _native
    n = ev.returns.numel()
    if n == 0:
        raise ValueError("an empty Evaluation has no statistics")
    rate = lambda code: float((ev.outcomes == code).sum().item()) / n  # noqa: E731
    return dict(mean_return=float(ev.returns.mean().item()), std_return=float(ev.returns.std(correction=0).item()),
                success_rate=rate(_native.EPISODE_GOAL), collision_rate=rate(_native.EPISODE_COLLISION),
                timeout_rate=rate(_native.EPISODE_TIMEOUT), mean_length=float(ev.lengths.double().mean().item()))


class VecMapfEnv:
    def __init__(self, env, num_envs, device=None, seed=0, auto_reset=True, reuse_outputs=False):
        """`env`: a MapfEnv (its spec and device context are shared).  `seed` keys the Philox sampling stream;
        `auto_reset`: an env whose step returns done restarts from the start state (its returned next state is then
        the start state, as in gym's vector envs).  `reuse_outputs`: `step()` alternates between two preallocated
        sets of result tensors instead of allocating five new ones per call (the tensors returned by a step are
        overwritten two steps later); with it a `step()` costs ~9 us of host time instead of ~20."""
        import torch
        self.env = env
        if device is not None and env._engine_obj is None:
            env.device = device
        self.engine = env.engine
        self.device = self.engine.torch_device
        self.num_envs = int(num_envs)
        self.seed = int(seed)
        self.auto_reset = bool(auto_reset)
        self.env_offset = 0      # index of this shard's first env in a sharded global batch
        self.step_count = 0
        self.n_agents, self.nS, self.nA = env.n_agents, env.nS, env.nA
        self.states = self.engine.new_states(self.num_envs)
        self._torch = torch
        self._ring = None
        if reuse_outputs:
            B, dev = self.num_envs, self.device
            self._ring = [(self.engine.new_states(B), torch.empty(B, dtype=torch.float64, device=dev),
                           torch.empty(B, dtype=torch.float64, device=dev), torch.empty(B, dtype=torch.bool, device=dev),
                           torch.empty(B, dtype=torch.bool, device=dev)) for _ in range(2)]
            self.states = self._ring[1][0]
        self.reset()

    # ---- encodings ---------------------------------------------------------------------------------------------
    def state_to_cells(self, states):
        """int32[B, n] per-agent cell ids (bulk `state_to_locations`, reference mapf_env.py:358-362)."""
        return self.engine.decode(states)

    def cells_to_state(self, cells):
        """Bulk `locations_to_state` (reference mapf_env.py:364-371) from int32[B, n] cell ids."""
        return self.engine.encode(cells.to(self._torch.int32).contiguous())

    def states_from_ints(self, values):
        return self.engine.states_from_ints(values)

    def states_to_ints(self, states):
        return self.engine.states_to_ints(states)

    # ---- episode control ---------------------------------------------------------------------------------------
    def reset(self):
        """Every env back on the start state (reference mapf_env.py:290-293).  Returns the state tensor."""
        s0 = self.engine.states_from_ints([self.engine.s0])
        self.states.copy_(s0.expand_as(self.states) if self.engine.words == 1 else s0.expand(self.num_envs, 2))
        return self.states

    def set_states(self, states):
        self.states.copy_(states)

    # ---- sampled transitions -----------------------------------------------------------------------------------
    def step(self, actions, uniforms=None):
        """One joint step of every env.  Returns (next_states, rewards, dones, info) with
        info = {"prob": f64[B], "collision": bool[B]}.  `uniforms` (f64[B, n]) replays given draws bit-exactly;
        without it the device-side Philox stream keyed by (seed, env, step) is used."""
        out = None if self._ring is None else self._ring[self.step_count & 1]
        if out is not None and out[0].data_ptr() == self.states.data_ptr():  # after an odd number of step_host() calls
            out = self._ring[(self.step_count + 1) & 1]
        ns, reward, prob, done, coll = self.engine.step(
            self.states, actions, uniforms=uniforms, seed=self.seed, step_index=self.step_count,
            env_offset=self.env_offset, auto_reset=self.auto_reset, out=out)
        self.states = ns
        self._states_shared = True  # the caller holds this tensor: step_host() must not advance it in place
        self.step_count += 1
        return ns, reward, done, {"prob": prob, "collision": coll}

    def rollout(self, T, actions=None, uniforms=None):
        """T steps in one launch.  `actions`: int32[T, B] or None for a uniformly random policy.  Returns a Rollout
        of step-major [T, B] tensors; the env states advance by T steps."""
        out = self.engine.rollout(self.states, actions, T, uniforms=uniforms, seed=self.seed,
                                  step_index=self.step_count, env_offset=self.env_offset, auto_reset=self.auto_reset)
        self.step_count += T
        return Rollout(*out)

    def step_host(self, actions, out=None, uniforms=None):
        """End-to-end host path, the batched `MapfEnv.step(action)` (reference mapf_env.py:237-266): `actions` is a CPU
        int32 array/tensor; the env states stay on the device, where `step` / `rollout` / `reset` / `set_states` keep
        them too (the reference keeps `self.s` in the env), so device-side and host-side steps can be mixed freely; the
        five results land in host memory (pinned tensors, or `out`)."""
        B = self.num_envs
        if out is None:
            out = (self._torch.empty(self.states.shape, dtype=self._torch.int64).pin_memory(),
                   self._torch.empty(B, dtype=self._torch.float64).pin_memory(),
                   self._torch.empty(B, dtype=self._torch.float64).pin_memory(),
                   self._torch.empty(B, dtype=self._torch.bool).pin_memory(),
                   self._torch.empty(B, dtype=self._torch.bool).pin_memory())
        if getattr(self, "_states_shared", False):
            self.states = self.states.clone()
            self._states_shared = False
        self.engine.step_host_resident(self.states, actions, out, uniforms=uniforms, seed=self.seed,
                                       step_index=self.step_count, env_offset=self.env_offset,
                                       auto_reset=self.auto_reset)
        self.step_count += 1
        return tuple(out)

    def evaluate(self, policy, n_episodes, max_steps, gamma=1.0, seed=None):
        """Runs `policy` for `n_episodes` episodes from the start state, in one launch: episode e is env e of this
        batch stepped from a reset with `actions = policy(states)` and no auto-reset, cut at its first done or after
        `max_steps` steps.  It draws from the Philox stream of `self.seed` (or `seed`) at `self.env_offset + e`, from
        step `self.step_count` on.  `policy`: None (uniformly random joint actions), int32[nS] joint actions by joint
        state (`value_iteration`'s policy), an integer [n_agents, L] table of per-agent actions by cell
        (`independent_policy`), a GroupPolicy (`group_policy`) or a TablePolicy (`rtdp`).  Returns an Evaluation; `self.states` and
        `step_count` are left as they are."""
        out = self.engine.evaluate(policy, n_episodes, max_steps, gamma=gamma, seed=self.seed if seed is None else seed,
                                   step_index=self.step_count, episode_offset=self.env_offset)
        return Evaluation(*out)

    def find_conflicts(self, policy, n_episodes, max_steps, gamma=1.0, seed=None):
        """`evaluate` of a GroupPolicy or TablePolicy that also names, for every episode that ends in a collision, the pair of agents
        (i < j) that clashed on its last step: the lexicographically smallest pair of agents in different groups, else
        the smallest pair inside one group.  This is sampled: it sees the collisions of these episodes, not every
        reachable one.  Returns Conflicts(evaluation, pairs u8[E] (i | j << 4, or NO_CONFLICT), counts int64[n, n])."""
        from .. import _native
        torch = self._torch
        if not isinstance(policy, (GroupPolicy, TablePolicy)):
            raise ValueError("find_conflicts needs a GroupPolicy or a TablePolicy (got %s)" % type(policy).__name__)
        E, n = int(n_episodes), self.n_agents
        pairs = torch.empty(max(E, 0), dtype=torch.uint8, device=self.device)
        run = self.engine.evaluate_table if isinstance(policy, TablePolicy) else self.engine.evaluate_groups
        out = run(policy, E, max_steps, gamma=gamma, seed=self.seed if seed is None else seed,
                  step_index=self.step_count, episode_offset=self.env_offset, conflicts=pairs)
        p = pairs[pairs != _native.NO_CONFLICT].long()
        counts = torch.bincount((p & 15) * n + (p >> 4), minlength=n * n).view(n, n)
        return Conflicts(Evaluation(*out), pairs, counts)

    # ---- transition table --------------------------------------------------------------------------------------
    def transitions(self, states, actions):
        """P[s][a] for B pairs as CSR: records row_ptr[b] .. row_ptr[b+1] are the row of pair b, in the
        reference's order.  flags bit 0 = done, bit 1 = collision."""
        return Transitions(*self.engine.transitions(states, actions))

    def build_table(self, s_begin, n_states):
        """The table slab [s_begin, s_begin + n_states) x [0, nA): row index = (s - s_begin) * nA + a."""
        return Transitions(*self.engine.table_range(int(s_begin), int(n_states)))

    def checksum(self, tr, index_base=0):
        """dict of mod-2**64 checksums of a Transitions (see include/mapf_b200.h: mapf_checksum)."""
        out = self.engine.checksum(tr.next_state, tr.prob, tr.reward, tr.flags, index_base=index_base)
        v = out.cpu().numpy().view(np.uint64)
        keys = ["count", "n_collision", "n_done", "sum_next_lo", "sum_next_hi", "sum_prob_bits", "sum_reward_bits",
                "ordered"]
        return dict(zip(keys, (int(x) for x in v)))

    # ---- consumers of the table (SURVEY.md 8f) -----------------------------------------------------------------
    def backup(self, V, gamma, states=None, actions=None, s_begin=0, n_states=None):
        """Bellman backup without materialising the table: for explicit (states, actions) pairs a float64[B], else
        Q[n_states, nA] of the slab [s_begin, s_begin + n_states) (default: every state).  Each entry is
        `q = 0; for ((p, c), s2, r, done) in P[s][a]: q += p * (r + gamma * V[s2])`, bit for bit."""
        if states is not None:
            return self.engine.backup(states, actions, V, gamma)
        if n_states is None:
            n_states = self.nS - int(s_begin)
        return self.engine.backup_range(int(s_begin), int(n_states), V, gamma)

    def greedy(self, Q):
        """(V, policy) = (max_a Q[s, a], first argmax) -- `max(q_sa)` / `np.argmax(q_sa)` of the classic planner loop."""
        return self.engine.greedy(Q)

    def value_iteration(self, gamma=1.0, eps=1e-2, max_iter=1000, slab=None):
        """Synchronous value iteration over the whole state space on the device (only for envs whose nS values fit
        in memory).  Stops when sum |V_new - V| <= eps (the classic gym loop).  Returns (V, policy, iterations)."""
        torch = self._torch
        nS = int(self.nS)
        V = torch.zeros(nS, dtype=torch.float64, device=self.device)
        slab = nS if slab is None else int(slab)
        it = 0
        for it in range(1, max_iter + 1):
            V_new = torch.empty_like(V)
            pi = torch.empty(nS, dtype=torch.int32, device=self.device)
            for s0 in range(0, nS, slab):
                n = min(slab, nS - s0)
                v, p = self.engine.greedy(self.engine.backup_range(s0, n, V, gamma))
                V_new[s0:s0 + n] = v
                pi[s0:s0 + n] = p
            delta = float((V_new - V).abs().sum().item())
            V = V_new
            if delta <= eps:
                break
        return V, pi, it

    def rtdp(self, heuristic, n_trials, max_depth, max_iterations, gamma=1.0, eps=1e-6, capacity=1 << 24, seed=None):
        """Real-time dynamic programming from the start state over a device-resident ValueTable, for joint spaces whose
        values do not fit in memory (one-word states).  `heuristic` (GroupValues) values every state the table does not
        hold.  The run is exactly
            every trial t in [0, n_trials) starts at s0
            for it in range(max_iterations):
                residual = 0
                for d in range(max_depth):
                    S = the distinct states of the live trials, sorted
                    v, a = rtdp_backup(S); old = lookup(S).values      (both read the table before the store)
                    residual = max(residual, max |v - old|); store(S, v, a)
                    every live trial steps with the a of its state (Philox stream `seed` (default self.seed), step
                        index it * max_depth + d, env index t, no auto-reset); one whose next state is terminal
                        (two agents on one cell, or every agent on its goal) stops for this iteration
                log one record; raise if the table overflowed
                if residual <= eps: stop
        A trial runs on through a done that is not terminal (a swap clash ends on distinct cells): in the MDP that
        `value_iteration` solves such a state keeps its future value.
        The value of s0 converges to the optimum V*(s0) only when the heuristic is optimistic, h >= V* at every state;
        under SoC with `reward_of_clash` below any path cost, the sum of the single-agent values (`group_values` of
        singleton groups) is such a heuristic.
        Returns Rtdp(table, policy = TablePolicy(table, heuristic.policy), log), one log record per iteration:
        {"residual", "v_s0", "table_size", "backups" (states backed up), "seconds"}."""
        import time
        torch = self._torch
        eng = self.engine
        if not isinstance(heuristic, GroupValues):
            raise ValueError("the heuristic must be a GroupValues (got %s)" % type(heuristic).__name__)
        n_trials, max_depth, max_iterations = int(n_trials), int(max_depth), int(max_iterations)
        if n_trials < 1 or max_depth < 1 or max_iterations < 1:
            raise ValueError("n_trials, max_depth and max_iterations must be >= 1")
        seed = self.seed if seed is None else int(seed)
        table = ValueTable(eng, capacity)
        s0 = eng.states_from_ints([eng.s0])
        goal = int(eng.goal_state)
        log = []
        for it in range(max_iterations):
            t_start = time.perf_counter()
            states = s0.repeat(n_trials)
            live = torch.ones(n_trials, dtype=torch.bool, device=self.device)
            residual = torch.zeros((), dtype=torch.float64, device=self.device)
            backups = 0
            for d in range(max_depth):
                idx = live.nonzero().squeeze(1)
                if idx.numel() == 0:
                    break
                S, inv = torch.unique(states[idx], sorted=True, return_inverse=True)
                v, a = eng.rtdp_backup(S, heuristic, table, gamma)
                old, _ = eng.vtable_lookup(S, heuristic, table)
                residual = torch.maximum(residual, (v - old).abs().max())
                eng.vtable_store(S, v, a, table)
                backups += S.numel()
                actions = torch.zeros(n_trials, dtype=torch.int32, device=self.device)
                actions[idx] = a[inv]
                ns = eng.step(states, actions, seed=seed, step_index=it * max_depth + d, env_offset=0)[0]
                states = torch.where(live, ns, states)
                cells = eng.decode(ns).sort(dim=1).values
                terminal = (ns == goal) | (cells[:, 1:] == cells[:, :-1]).any(dim=1)
                live = live & ~terminal
            res = float(residual.item())
            v_s0 = float(eng.vtable_lookup(s0, heuristic, table)[0].item())
            if table.overflowed():
                raise RuntimeError("rtdp: the value table of capacity %d is full (more than %d states); pass a larger "
                                   "capacity" % (table.capacity, table.capacity // 2))
            log.append(dict(residual=res, v_s0=v_s0, table_size=len(table), backups=backups,
                            seconds=time.perf_counter() - t_start))
            if res <= eps:
                break
        return Rtdp(table, TablePolicy(table, heuristic.policy), log)

    def predecessors(self, states):
        """(row_ptr, pred_states): the CSR of `MapfEnv.predecessors` (reference mapf_env.py:373-376) per state."""
        return self.engine.predecessors(states)

    def project(self, states, agent_indexes):
        """The joint states as `get_local_view(env, agent_indexes)` numbers them (reference utils.py:138-157)."""
        return self.engine.project(states, agent_indexes)


class MultiMapVecEnv:
    """A heterogeneous batch: counts[i] copies of envs[i] -- different grids, scenarios, rewards or criteria per
    segment -- stepped together (SURVEY.md 8f row 4).  Env b of the concatenated batch belongs to the spec whose
    segment [offsets[i], offsets[i + 1]) holds b.

    Specs that agree in agent count and state width (and whose move tables fit shared memory) are stepped by ONE
    launch of the grouped kernel (`mapf_group_step`); a batch that mixes agent counts or state widths is split into
    one group per (agent count, width) class, each over its own contiguous slice, so every class must be contiguous
    in `envs`.  Per-env semantics are those of `VecMapfEnv.step` / `MapfEnv.step` (reference mapf_env.py:237-266).
    State tensors are int64[B] (or int64[B, 2] when every spec needs two words)."""

    def __init__(self, envs, counts, seed=0, auto_reset=True, env_offset=0):
        """`env_offset`: index of this batch's first env in a larger (sharded) batch -- it keys the Philox streams, see
        `sharding.segment_shard`."""
        import torch
        from .. import _native
        if len(envs) != len(counts) or not envs:
            raise ValueError("one env count per env")
        self._torch = torch
        self.envs = list(envs)
        self.counts = [int(c) for c in counts]
        self.offsets = [0]
        for c in self.counts:
            self.offsets.append(self.offsets[-1] + c)
        self.num_envs = self.offsets[-1]
        self.seed, self.auto_reset, self.step_count = int(seed), bool(auto_reset), 0
        self.env_offset = int(env_offset)
        engines = [e.engine for e in self.envs]
        self.device = engines[0].torch_device
        words = {e.words for e in engines}
        if len(words) != 1:
            raise ValueError("all specs of a MultiMapVecEnv must have the same state width (1 or 2 words)")
        self.words = words.pop()
        # contiguous runs of compatible specs -> one mapf_group each; a spec whose table is not staged steps alone
        self._parts = []  # (first env, last env, Group or Engine)
        i = 0
        while i < len(engines):
            if not engines[i].moves_in_smem:
                self._parts.append((self.offsets[i], self.offsets[i + 1], engines[i]))
                i += 1
                continue
            j = i
            while j < len(engines) and engines[j].moves_in_smem and engines[j].n == engines[i].n:
                j += 1
            self._parts.append((self.offsets[i], self.offsets[j], _native.Group(engines[i:j], self.counts[i:j])))
            i = j
        shape = (self.num_envs,) if self.words == 1 else (self.num_envs, 2)
        self.states = torch.empty(shape, dtype=torch.int64, device=self.device)
        self.reset()

    def spec_of(self, b):
        """Index into `envs` of the spec env b belongs to."""
        import bisect
        return bisect.bisect_right(self.offsets, int(b)) - 1

    def reset(self):
        for i, env in enumerate(self.envs):
            lo, hi = self.offsets[i], self.offsets[i + 1]
            if hi > lo:
                self.states[lo:hi] = env.engine.states_from_ints([env.engine.s0])
        return self.states

    def set_states(self, states):
        self.states.copy_(states)

    def step(self, actions, uniforms=None):
        """One joint step of every env: (next_states, rewards, dones, {"prob", "collision"}).  `actions` is int32[B];
        `uniforms` (float64[B, n], groups of one agent count only) replays given draws bit-exactly."""
        torch = self._torch
        B, dev = self.num_envs, self.device
        ns = torch.empty_like(self.states)
        reward = torch.empty(B, dtype=torch.float64, device=dev)
        prob = torch.empty(B, dtype=torch.float64, device=dev)
        done = torch.empty(B, dtype=torch.bool, device=dev)
        coll = torch.empty(B, dtype=torch.bool, device=dev)
        if uniforms is not None and len(self._parts) != 1:
            raise ValueError("uniforms can only be replayed when every spec has the same agent count")
        for lo, hi, part in self._parts:
            if hi == lo:
                continue
            out = (ns[lo:hi], reward[lo:hi], prob[lo:hi], done[lo:hi], coll[lo:hi])
            part.step(self.states[lo:hi], actions[lo:hi], uniforms=uniforms, seed=self.seed, step_index=self.step_count,
                      env_offset=self.env_offset + lo, auto_reset=self.auto_reset, out=out)
        self.states = ns
        self._states_shared = True  # the caller holds this tensor: step_host() must not advance it in place
        self.step_count += 1
        return ns, reward, done, {"prob": prob, "collision": coll}
