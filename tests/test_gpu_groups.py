"""Products of group policies (mapf_evaluate_groups / GroupPolicy / group_policy), conflict attribution
(VecMapfEnv.find_conflicts) and independence detection, against the AGENTS and JOINT kinds, against a host loop over
`step` and `project`, and against the C oracle fed the host-side Philox draws.  Returns are compared as fp64 bit
patterns."""
import ctypes as C

import numpy as np
import pytest

import golden_util as G
from engine_util import make_engine, make_oracle, u64
from test_gpu_evaluate import Episodes, assert_same, c1_env, env_of, kinds, philox_words, vi_policy
from test_gpu_guard_bands import SIZES, Guarded

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


def random_groups(eng, groups, seed):
    """A GroupPolicy with uniformly random entries in [0, 5**|g|)."""
    import torch
    from gym_mapf_b200.envs.vec_env import GroupPolicy
    rng = np.random.default_rng(seed)
    return GroupPolicy(groups, [torch.from_numpy(rng.integers(0, 5 ** len(g), eng.L ** len(g)).astype(np.int32))
                                .to(eng.torch_device) for g in groups])


def groups_fn(eng, policy):
    """The joint action of a GroupPolicy, from `project`, table gathers and a digit scatter on the host side."""
    import torch

    def f(states):
        a = torch.zeros(states.shape[0], dtype=torch.int64, device=eng.torch_device)
        for g, table in zip(policy.groups, policy.tables):
            entry = table.to(torch.int64)[eng.project(states, list(g))]
            for k, agent in enumerate(g):
                a += (entry // 5 ** k) % 5 * 5 ** agent
        return a.to(torch.int32)
    return f


def host_pair(prev, nxt, group_of):
    """The attributed pair of a clash step, smallest cross-group pair first, else the smallest pair."""
    n = len(prev)
    pairs = [(i, j) for i in range(n) for j in range(i + 1, n)
             if nxt[i] == nxt[j] or (nxt[i] == prev[j] and nxt[j] == prev[i])]
    cross = [p for p in pairs if group_of[p[0]] != group_of[p[1]]]
    i, j = (cross or pairs)[0]
    return i | j << 4


def step_loop_pairs(eng, policy, E, T, gamma, seed=0, step_index=0, env_offset=0):
    """Episodes of `policy` stepped on the host side, and the conflict byte of each episode."""
    from gym_mapf_b200._native import NO_CONFLICT
    fn, gid = groups_fn(eng, policy), policy.group_of()
    states = eng.states_from_ints([eng.s0] * E)
    ep = Episodes(E, gamma)
    pair = np.full(E, NO_CONFLICT, np.uint8)
    for t in range(T):
        ns, r, prob, done, coll = eng.step(states, fn(states), seed=seed, step_index=step_index + t, env_offset=env_offset)
        d, c, p = done.cpu().numpy(), coll.cpu().numpy(), prob.cpu().numpy()
        hit = np.flatnonzero(ep.active & d & c)
        if len(hit):
            prev, nxt = eng.decode(states).cpu().numpy()[hit], eng.decode(ns).cpu().numpy()[hit]
            for k, e in enumerate(hit):
                pair[e] = host_pair(prev[k], nxt[k], gid)
        if not ep.add(t, r.cpu().numpy(), d, kinds(d, c, p)):
            break
        states = ns
    return ep, pair


# ---- 1. singleton groups == AGENTS --------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["rows_c2", "rows_c4", "rows_berlin"])
def test_singletons_equal_agents(name, torch):
    from gym_mapf_b200.envs.utils import group_policy, independent_policy
    from gym_mapf_b200.envs.vec_env import GroupPolicy
    env = env_of(G.load(name)[0])
    eng = env.engine
    table = independent_policy(env)
    gp = GroupPolicy([(i,) for i in range(eng.n)], list(table))
    if name == "rows_c2":  # group_policy of singletons plans exactly what independent_policy plans
        planned = group_policy(env, [(i,) for i in range(eng.n)])
        assert all(torch.equal(a, b) for a, b in zip(planned.tables, table))
    for gamma in (1.0, 0.95):
        want = eng.evaluate(table, 50000, 400, gamma=gamma, seed=13, step_index=3, episode_offset=77)
        got = eng.evaluate(gp, 50000, 400, gamma=gamma, seed=13, step_index=3, episode_offset=77)
        assert all(torch.equal(a, b) for a, b in zip(got, want))


# ---- 2. one group of every agent == JOINT -------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["c1", "room2"])
def test_one_group_equals_joint(case, torch):
    from gym_mapf_b200.envs.mapf_env import OptimizationCriteria
    from gym_mapf_b200.envs.utils import create_mapf_env
    from gym_mapf_b200.envs.vec_env import GroupPolicy
    env = c1_env(soc=True) if case == "c1" else \
        create_mapf_env("room-32-32-4", 1, 2, 0.2, -1000.0, 100.0, -1.0, OptimizationCriteria.SoC, device=0)
    eng = env.engine
    pi = vi_policy(eng, max_iter=300)
    gp = GroupPolicy([tuple(range(eng.n))], [pi])
    for gamma in (1.0, 0.95):
        want = eng.evaluate(pi, 100003, 300, gamma=gamma, seed=2, step_index=5)
        got = eng.evaluate(gp, 100003, 300, gamma=gamma, seed=2, step_index=5)
        assert all(torch.equal(a, b) for a, b in zip(got, want))


# ---- 3 + 5. mixed partitions == a host step loop, conflict bytes == the host's pair ------------------------------------
PARTITIONS = {"rows_c2": [(0, 2), (1,), (3,)], "rows_c4": [(0, 1), (2, 3), (4, 5), (6, 7)]}


@pytest.fixture(scope="module")
def mixed(torch):
    out = {}
    for name, groups in PARTITIONS.items():
        eng = make_engine(G.load(name)[0])
        out[name] = (eng, random_groups(eng, groups, 11))
    return out


@pytest.mark.parametrize("name", sorted(PARTITIONS))
@pytest.mark.parametrize("E", [1, 31, 33, 4097, 100003])
def test_mixed_groups_equal_step_loop(name, E, mixed, torch):
    eng, gp = mixed[name]
    T = 40
    want, want_pair = step_loop_pairs(eng, gp, E, T, 0.95, seed=9, step_index=4, env_offset=E)
    pairs = torch.empty(E, dtype=torch.uint8, device=eng.torch_device)
    got = eng.evaluate_groups(gp, E, T, gamma=0.95, seed=9, step_index=4, episode_offset=E, conflicts=pairs)
    assert_same(got, want)
    assert np.array_equal(pairs.cpu().numpy(), want_pair)
    plain = eng.evaluate_groups(gp, E, T, gamma=0.95, seed=9, step_index=4, episode_offset=E)
    assert all(torch.equal(a, b) for a, b in zip(got, plain))  # conflicts=None changes nothing else
    if E == 100003:
        assert (want.outcome == 1).any() and (want_pair != 0xFF).any()


def test_cross_group_pair_comes_first(torch):
    """A vertex clash of three agents: (0, 1) inside a group loses to (0, 2) across groups."""
    from gym_mapf_b200.envs.vec_env import GroupPolicy
    spec = dict(rows=["...", "...", "..."], n_agents=3, starts=[[1, 0], [1, 2], [0, 1]], goals=[[2, 0], [2, 2], [2, 1]],
                fail_prob=0.0, r_clash=-1000.0, r_goal=100.0, r_living=-1.0, soc=True)
    eng = make_engine(spec)
    L = eng.L
    dev = eng.torch_device
    # every agent steps onto the centre: agent 0 RIGHT, agent 1 LEFT, agent 2 DOWN (ACTIONS = STAY UP RIGHT DOWN LEFT)
    pair_table = torch.full((L * L,), 2 + 5 * 4, dtype=torch.int32, device=dev)
    one = torch.full((L,), 3, dtype=torch.int32, device=dev)
    for groups, tables, want in ([[(0, 1), (2,)], [pair_table, one], 0 | 2 << 4],
                                 [[(0,), (1,), (2,)], [torch.full((L,), 2, dtype=torch.int32, device=dev),
                                                       torch.full((L,), 4, dtype=torch.int32, device=dev), one], 0 | 1 << 4],
                                 [[(0, 1, 2)], [torch.full((L ** 3,), 2 + 5 * 4 + 25 * 3, dtype=torch.int32, device=dev)],
                                  0 | 1 << 4]):
        pairs = torch.empty(5, dtype=torch.uint8, device=dev)
        ret, length, outcome = eng.evaluate_groups(GroupPolicy(groups, tables), 5, 10, conflicts=pairs)
        assert bool((outcome == 1).all()) and bool((length == 1).all())
        assert bool((pairs == want).all()), (groups, pairs)


def test_attribution_at_13_agents(torch):
    """Thirteen agents on an open 3 x 13 grid (39**13 >= 2**63: two-word states, staged moves).  Agents 0-9 stand on
    row 0 and STAY.  Agent 10 on (1, 10) goes RIGHT, 11 on (0, 11) DOWN and 12 on (2, 11) UP: a 3-way vertex clash on
    (1, 11); or 10 STAYs and only 11 and 12 clash; optionally 4 and 5 swap.  The expected bytes are written out: the
    high nibble holds agents 10-12."""
    from gym_mapf_b200.envs.vec_env import GroupPolicy
    starts = [[0, c] for c in range(10)] + [[1, 10], [0, 11], [2, 11]]
    goals = [[2, c] for c in range(10)] + [[1, 0], [1, 1], [1, 2]]
    spec = dict(rows=["." * 13] * 3, n_agents=13, starts=starts, goals=goals, fail_prob=0.0, r_clash=-1000.0,
                r_goal=100.0, r_living=-1.0, soc=True)
    eng = make_engine(spec)
    assert (eng.L, eng.words, eng.moves_in_smem) == (39, 2, True)
    dev = eng.torch_device
    STAY, UP, RIGHT, DOWN, LEFT = range(5)
    three, two = {10: RIGHT, 11: DOWN, 12: UP}, {11: DOWN, 12: UP}
    swap = {4: RIGHT, 5: LEFT}
    single = [(i,) for i in range(10)]
    rest = [(i,) for i in range(10) if i not in (4, 5)]
    cases = [(three, single + [(10,), (11,), (12,)], 0xBA),
             (two, single + [(10,), (11,), (12,)], 0xCB),
             ({**three, **swap}, single + [(10,), (11,), (12,)], 0x54),
             (three, single + [(10, 11), (12,)], 0xCA),
             (two, single + [(10, 11, 12)], 0xCB),
             ({**three, **swap}, rest + [(4, 5), (10,), (11, 12)], 0xBA),
             ({**three, **swap}, rest + [(4, 5), (10, 11, 12)], 0x54)]
    for moves, groups, want in cases:
        tables = [torch.full((eng.L ** len(g),), sum(moves.get(a, STAY) * 5 ** k for k, a in enumerate(g)),
                             dtype=torch.int32, device=dev) for g in groups]
        pairs = torch.empty(64, dtype=torch.uint8, device=dev)
        ret, length, outcome = eng.evaluate_groups(GroupPolicy(groups, tables), 64, 10, conflicts=pairs)
        assert bool((outcome == 1).all()) and bool((length == 1).all()), (moves, groups)
        assert bool((pairs == want).all()), (moves, groups, pairs)


# ---- 4. the same episodes from the C oracle and the host Philox stream ------------------------------------------------
def test_groups_replayed_through_the_oracle(torch):
    spec, _ = G.load("rows_c2")
    eng, ora = make_engine(spec), make_oracle(spec)
    E, T, gamma, seed, step0, off = 6000, 120, 0.95, 0x5eed, 40, 12345
    gp = random_groups(eng, [(0, 3), (1, 2)], 5)
    got = eng.evaluate(gp, E, T, gamma=gamma, seed=seed, step_index=step0, episode_offset=off)
    sub = np.arange(0, E, 23)
    env = sub.astype(np.uint64) + np.uint64(off)
    tabs = [t.cpu().numpy().astype(np.int64) for t in gp.tables]
    lo = np.full(len(sub), eng.s0, np.uint64)
    hi = np.zeros_like(lo)
    ep = Episodes(len(sub), gamma)
    for t in range(T):
        cells = ora.decode(lo, hi).astype(np.int64)
        actions = np.zeros(len(sub), np.int64)
        for g, tab in zip(gp.groups, tabs):
            entry = tab[sum(cells[:, a] * eng.L ** k for k, a in enumerate(g))]
            for k, a in enumerate(g):
                actions += (entry // 5 ** k) % 5 * 5 ** a
        u = np.zeros((len(sub), eng.n))
        for b in range((eng.n + 3) // 4):
            words = philox_words(seed, env, step0 + t, b)
            for q in range(4):
                if 4 * b + q < eng.n:
                    u[:, 4 * b + q] = words[q].astype(np.float64) * 2.0 ** -32
        w = ora.step(lo, hi, actions, u)
        done = w["done"].astype(bool)
        k = np.where(w["collision"] == 1, 1, np.where(w["terminal"] == 1, 3, 2)).astype(np.uint8)
        if not ep.add(t, w["reward"], done, k):
            break
        lo, hi = w["next_lo"], w["next_hi"]
    assert np.array_equal(u64(got[0])[sub], ep.G.view(np.uint64))
    assert np.array_equal(got[1].cpu().numpy()[sub], ep.length)
    assert np.array_equal(got[2].cpu().numpy()[sub], ep.outcome)


# ---- 6. sharding -------------------------------------------------------------------------------------------------------
def test_sharded_calls_concatenate(mixed, torch):
    from gym_mapf_b200 import sharding
    eng, gp = mixed["rows_c2"]
    E, T, off = 100003, 150, 1000
    pairs = torch.empty(E, dtype=torch.uint8, device=eng.torch_device)
    whole = eng.evaluate_groups(gp, E, T, gamma=0.95, seed=8, step_index=1, episode_offset=off, conflicts=pairs)
    parts = []
    for rank in range(3):
        sh = sharding.split_range(E, 3, rank, begin=off)
        p = torch.empty(sh.count, dtype=torch.uint8, device=eng.torch_device)
        parts.append(eng.evaluate_groups(gp, sh.count, T, gamma=0.95, seed=8, step_index=1, episode_offset=sh.begin,
                                         conflicts=p) + (p,))
    for k in range(3):
        assert torch.equal(torch.cat([p[k] for p in parts]), whole[k])
    assert torch.equal(torch.cat([p[3] for p in parts]), pairs)


# ---- 7. rejected arguments -----------------------------------------------------------------------------------------
def test_evaluate_groups_errors(mixed, torch):
    from gym_mapf_b200 import _native
    from gym_mapf_b200._native import MAPF_ERR_INVALID, _ptr, lib
    from gym_mapf_b200.envs.vec_env import GroupPolicy
    eng, gp = mixed["rows_c2"]
    eng4, _ = mixed["rows_c4"]
    dev = eng.torch_device
    E, L = 10, eng.L
    tables = torch.cat(gp.tables)
    n_tab = tables.numel()
    assert n_tab == 2 * L + L * L
    ret, length, outcome = (torch.empty(E, dtype=torch.float64, device=dev), torch.empty(E, dtype=torch.int32, device=dev),
                            torch.empty(E, dtype=torch.uint8, device=dev))
    conflict = torch.empty(E, dtype=torch.uint8, device=dev)
    scratch = torch.empty(2, dtype=torch.int64, device=dev)

    def call(e=E, gof=(0, 1, 0, 2), tab=tables, tlen=n_tab, T=5, sc=scratch, r=ret, ln=length, oc=outcome, cf=conflict,
             h=None, e_ng=eng):
        g = None if gof is None else (C.c_int32 * len(gof))(*gof)
        return lib().mapf_evaluate_groups(e_ng._h if h is None else h, g, _ptr(tab), tlen, e, T, 1.0, 0, 0, 0, _ptr(sc),
                                          _ptr(r), _ptr(ln), _ptr(oc), _ptr(cf), e_ng._stream())

    assert call() == 0 and call(cf=None) == 0 and call(0, sc=None, r=None, ln=None, oc=None, cf=None) == 0
    invalid = [dict(h=C.c_void_p(0)), dict(gof=None), dict(tab=None), dict(sc=None), dict(r=None), dict(ln=None),
               dict(oc=None), dict(T=0), dict(T=-1), dict(T=1 << 31), dict(e=-1), dict(e=(1 << 30) + 1),
               dict(tlen=n_tab - 1), dict(tlen=n_tab + 1), dict(tlen=-1),
               dict(gof=(1, 0, 1, 2)), dict(gof=(0, 2, 1, 1)), dict(gof=(0, 1, -1, 2)), dict(gof=(0, 1, 0, 4)),
               dict(gof=(0, 0, 0, 0)),  # a valid partition, but its table would have L**4 entries
               dict(gof=(0,) * 8, e_ng=eng4, tlen=1 << 62)]  # L**8 > 2**63: the size overflows
    for kw in invalid:
        assert call(**kw) == MAPF_ERR_INVALID, kw
    # the Python layer
    with pytest.raises(ValueError):  # a policy for another agent count
        eng4.evaluate(gp, E, 5)
    other = GroupPolicy([(0, 1, 2, 3)], [torch.zeros(3 ** 4, dtype=torch.int32, device=dev)])
    with pytest.raises(ValueError):  # a policy for another map
        eng.evaluate(other, E, 5)
    with pytest.raises(ValueError):
        eng.evaluate_groups(gp, E, 5, conflicts=torch.empty(E + 1, dtype=torch.uint8, device=dev))
    with pytest.raises(ValueError):
        eng.evaluate_groups(gp, -1, 5)
    with pytest.raises(_native.NativeError) as ei:
        eng.evaluate(gp, E, 0)
    assert ei.value.code == MAPF_ERR_INVALID


# ---- 8. writes stay inside the outputs ---------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(PARTITIONS))
def test_evaluate_groups_writes_only_its_outputs(name, mixed, torch):
    from gym_mapf_b200._native import _ptr, check, lib
    eng, gp = mixed[name]
    g = Guarded(torch)
    tables = torch.cat(gp.tables)
    keep = tables.clone()
    gof = (C.c_int32 * eng.n)(*gp.group_of())
    sb = int(lib().mapf_evaluate_scratch_bytes())
    for E in SIZES:
        scratch = g.new((sb + 7) // 8, torch.int64)
        ret, length, outcome, conflict = g.new(E, torch.float64), g.new(E, torch.int32), g.new(E, torch.uint8), \
            g.new(E, torch.uint8)
        check(lib().mapf_evaluate_groups(eng._h, gof, _ptr(tables), tables.numel(), E, 64, 0.95, 3, 0, 0, _ptr(scratch),
                                         _ptr(ret), _ptr(length), _ptr(outcome), _ptr(conflict), eng._stream()))
        g.check("evaluate_groups E=%d" % E)
        assert torch.equal(keep, tables)
        assert bool(((length >= 1) & (length <= 64)).all()) and bool((outcome <= 3).all())
        coll = outcome == 1
        assert bool((conflict[~coll] == 0xFF).all()) and bool((conflict[coll] != 0xFF).all())


# ---- 9. independence detection -----------------------------------------------------------------------------------------
# Agents 0 and 1 swap the ends of a one-cell-wide corridor that has one passing bay (row 0); agent 2 walks in a room
# of its own.
CORRIDOR_MAP = "type octile\nheight 4\nwidth 7\nmap\n@@@.@@@\n.......\n@@@@@@@\n.......\n"
CORRIDOR_SCEN = "version 1\n" + "".join("0\tcorridor.map\t7\t4\t%d\t%d\t%d\t%d\t6\n" % rc for rc in
                                        [(1, 0, 1, 6), (1, 6, 1, 0), (3, 0, 3, 6)])


def corridor_env(fail_prob):
    from gym_mapf_b200.envs.mapf_env import OptimizationCriteria
    from gym_mapf_b200.envs.utils import create_mapf_env_from_text
    return create_mapf_env_from_text(CORRIDOR_MAP, CORRIDOR_SCEN, 3, fail_prob, -1000.0, 100.0, -1.0,
                                     OptimizationCriteria.SoC, device=0)


def test_independence_detection_merges_the_corridor_pair(torch):
    from gym_mapf_b200.envs.utils import independence_detection
    env = corridor_env(0.0)
    res = independence_detection(env, n_episodes=4096, max_steps=64, seed=3)
    first, last = res.log[0], res.log[-1]
    assert first["groups"] == ((0,), (1,), (2,))
    assert first["summary"]["collision_rate"] == 1.0
    counts = first["counts"]
    assert int(counts[0, 1]) == 4096 and int(counts.sum()) == 4096
    assert res.resolved and res.policy.groups == ((0, 1), (2,)) and len(res.log) == 2
    assert last["groups"] == ((0, 1), (2,))
    assert last["summary"]["collision_rate"] == 0.0 and last["summary"]["success_rate"] == 1.0
    again = independence_detection(env, n_episodes=4096, max_steps=64, seed=3)
    assert again.policy.groups == res.policy.groups
    assert all(torch.equal(a, b) for a, b in zip(again.policy.tables, res.policy.tables))
    assert [r["summary"] for r in again.log] == [r["summary"] for r in res.log]


def test_independence_detection_with_slips_lowers_the_collision_rate(torch):
    from gym_mapf_b200.envs.utils import independence_detection
    res = independence_detection(corridor_env(0.2), n_episodes=1 << 14, max_steps=64, seed=5)
    assert len(res.log) >= 2
    assert res.log[-1]["summary"]["collision_rate"] < res.log[0]["summary"]["collision_rate"]


def test_independence_detection_stops_at_the_group_size_limit(torch):
    from gym_mapf_b200.envs.utils import independence_detection
    res = independence_detection(corridor_env(0.0), n_episodes=1024, max_steps=64, seed=3, max_group_size=1)
    assert not res.resolved and res.policy.groups == ((0,), (1,), (2,)) and len(res.log) == 1


def test_find_conflicts_counts(mixed, torch):
    from gym_mapf_b200._native import NO_CONFLICT
    from gym_mapf_b200.envs.vec_env import VecMapfEnv
    env = env_of(G.load("rows_c2")[0])
    _, gp = mixed["rows_c2"]
    vec = VecMapfEnv(env, 1, seed=4)
    found = vec.find_conflicts(gp, 20000, 100)
    p = found.pairs.cpu().numpy()
    o = found.evaluation.outcomes.cpu().numpy()
    assert np.array_equal(p != NO_CONFLICT, o == 1)
    want = np.zeros((4, 4), np.int64)
    for x in p[p != NO_CONFLICT]:
        want[x & 15, x >> 4] += 1
    assert np.array_equal(found.counts.cpu().numpy(), want) and want.sum() > 0
    ev = vec.evaluate(gp, 20000, 100)
    assert all(torch.equal(a, b) for a, b in zip(ev, found.evaluation))


# ---- 10. out-of-range entries through the C ABI are clamped ------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(PARTITIONS))
def test_out_of_range_entries_are_clamped(name, mixed, torch):
    """Entries >= 5**|g| or negative (as u32, above 5**|g| - 1) act as 5**|g| - 1.  GroupPolicy rejects such tables,
    so only C callers reach the clamp."""
    from gym_mapf_b200._native import POLICY_GROUPS
    from test_gpu_evaluate import assert_clamped
    eng, gp = mixed[name]
    table = torch.cat(gp.tables).cpu().numpy()
    size = np.concatenate([np.full(t.numel(), 5 ** len(g), np.int64) for g, t in zip(gp.groups, gp.tables)])
    assert_clamped(torch, eng, lambda t: (POLICY_GROUPS, t, gp.group_of()), table, [size, -1, -(1 << 31)], size - 1,
                   np.random.default_rng(5))


# ---- 11. 2**30 episodes in one call: the env index crosses 2**32 -------------------------------------------------------
@pytest.mark.timeout(300)
def test_largest_call_crosses_2_32(mixed, torch):
    """n_episodes = 2**30, the most one call takes, from episode_offset 2**32 - 2**29: episode 2**29 is env 2**32.
    Every record is written, and episodes on both sides of the crossing and the last one are the oracle's."""
    from test_gpu_evaluate import SENTINEL_RET
    from test_gpu_kernel_matrix import SEED, assert_episodes, replay_episodes
    free, _ = torch.cuda.mem_get_info()
    if free < 24 << 30:
        pytest.skip("needs 24 GB of free device memory for 15 GB of outputs, %.1f GB free: the device is shared"
                    % (free / 2 ** 30))
    eng, gp = mixed["rows_c2"]
    E, T, gamma, step0, off = 1 << 30, 2, 0.95, (1 << 32) - 1, (1 << 32) - (1 << 29)
    dev = eng.torch_device
    ret = torch.full((E,), SENTINEL_RET, dtype=torch.int64, device=dev).view(torch.float64)
    length = torch.full((E,), -1, dtype=torch.int32, device=dev)
    outcome = torch.full((E,), 0xEE, dtype=torch.uint8, device=dev)
    pairs = torch.full((E,), 0xEE, dtype=torch.uint8, device=dev)
    eng.evaluate_groups(gp, E, T, gamma=gamma, seed=SEED, step_index=step0, episode_offset=off,
                        out=(ret, length, outcome), conflicts=pairs)
    assert bool((ret.view(torch.int64) != SENTINEL_RET).all())
    assert bool(((length >= 1) & (length <= T)).all()) and bool((outcome <= 3).all())
    assert bool(((pairs != 0xFF) == (outcome == 1)).all()) and bool((pairs != 0xEE).all())
    sub = np.concatenate([np.arange(0, 300), np.arange((1 << 29) - 300, (1 << 29) + 300), np.arange(E - 300, E)])
    ep = replay_episodes(eng, make_oracle(G.load("rows_c2")[0]), (gp.groups, [t.cpu().numpy() for t in gp.tables]),
                         "groups", T, gamma, step0, off, sub)
    got = tuple(x[torch.from_numpy(sub).to(dev)] for x in (ret, length, outcome, pairs))
    every = np.arange(len(sub))
    assert_episodes(got, ep, every, "E = 2**30")
    assert np.array_equal(got[3].cpu().numpy(), ep.pair) and (ep.length == T).any()
