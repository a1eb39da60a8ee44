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
        (`independent_policy`), or a GroupPolicy (`group_policy`).  Returns an Evaluation; `self.states` and
        `step_count` are left as they are."""
        out = self.engine.evaluate(policy, n_episodes, max_steps, gamma=gamma, seed=self.seed if seed is None else seed,
                                   step_index=self.step_count, episode_offset=self.env_offset)
        return Evaluation(*out)

    def find_conflicts(self, policy, n_episodes, max_steps, gamma=1.0, seed=None):
        """`evaluate` of a GroupPolicy that also names, for every episode that ends in a collision, the pair of agents
        (i < j) that clashed on its last step: the lexicographically smallest pair of agents in different groups, else
        the smallest pair inside one group.  This is sampled: it sees the collisions of these episodes, not every
        reachable one.  Returns Conflicts(evaluation, pairs u8[E] (i | j << 4, or NO_CONFLICT), counts int64[n, n])."""
        from .. import _native
        torch = self._torch
        if not isinstance(policy, GroupPolicy):
            raise ValueError("find_conflicts needs a GroupPolicy (got %s)" % type(policy).__name__)
        E, n = int(n_episodes), self.n_agents
        pairs = torch.empty(max(E, 0), dtype=torch.uint8, device=self.device)
        out = self.engine.evaluate_groups(policy, E, max_steps, gamma=gamma, seed=self.seed if seed is None else seed,
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
