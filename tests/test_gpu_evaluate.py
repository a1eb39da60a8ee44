"""Closed-loop policy evaluation (mapf_evaluate / Engine.evaluate / VecMapfEnv.evaluate) against what a user's loop
over `step` or `rollout` computes, against the C oracle fed the host-side Philox draws, and against the exact value of
the policy.  Returns are compared as fp64 bit patterns."""
import ctypes as C

import numpy as np
import pytest

import golden_util as G
from engine_util import make_engine, make_oracle, u64
from test_gpu_guard_bands import SIZES, Guarded
from test_gpu_parity import philox4x32_10

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


def env_of(spec, **over):
    from gym_mapf_b200.envs.grid import MapfGrid
    from gym_mapf_b200.envs.mapf_env import MapfEnv, OptimizationCriteria
    s = dict(spec, **over)
    crit = OptimizationCriteria.SoC if s["soc"] else OptimizationCriteria.Makespan
    return MapfEnv(MapfGrid(s["rows"]), s["n_agents"], tuple(map(tuple, s["starts"])), tuple(map(tuple, s["goals"])),
                   s["fail_prob"], s["r_clash"], s["r_goal"], s["r_living"], crit, device=0)


def c1_env(soc=False, fail_prob=0.2):
    from gym_mapf_b200.envs.mapf_env import OptimizationCriteria
    from gym_mapf_b200.envs.utils import create_mapf_env
    crit = OptimizationCriteria.SoC if soc else OptimizationCriteria.Makespan
    return create_mapf_env("empty-8-8", 1, 2, fail_prob, -1000.0, 100.0, -1.0, crit, device=0)


def vi_policy(eng, gamma=1.0, eps=1e-6, max_iter=1000):
    import torch
    V = torch.zeros(int(eng.nS), dtype=torch.float64, device=eng.torch_device)
    for _ in range(max_iter):
        V_new, pi = eng.greedy(eng.backup_range(0, int(eng.nS), V, gamma))
        delta = float((V_new - V).abs().sum())
        V = V_new
        if delta <= eps:
            break
    return pi


class Episodes:
    """Host accumulation of episode records from per-step results, each env masked at its FIRST done (without
    auto-reset a swap-clashed env keeps stepping with non-zero rewards)."""

    def __init__(self, E, gamma):
        self.G, self.disc = np.zeros(E), np.ones(E)
        self.length, self.outcome = np.zeros(E, np.int32), np.zeros(E, np.uint8)
        self.active, self.gamma = np.ones(E, bool), gamma

    def add(self, t, reward, done, kind):
        a = self.active
        self.G[a] = self.G[a] + self.disc[a] * reward[a]  # two binary64 operations, as the kernel does
        self.disc[a] = self.disc[a] * self.gamma
        self.length[a] = t + 1
        d = a & done
        self.outcome[d] = kind[d]
        self.active = a & ~done
        return bool(self.active.any())


def kinds(done, coll, prob):
    """EnvOut.kind of a step result: 1 clash, 3 step from a terminal state (prob 0), 2 goal, 0 not done."""
    return np.where(~done, 0, np.where(coll, 1, np.where(prob == 0.0, 3, 2))).astype(np.uint8)


def step_loop(eng, policy_fn, E, T, gamma, seed=0, step_index=0, env_offset=0):
    states = eng.states_from_ints([eng.s0] * E)
    ep = Episodes(E, gamma)
    for t in range(T):
        ns, r, prob, done, coll = eng.step(states, policy_fn(states), seed=seed, step_index=step_index + t,
                                           env_offset=env_offset)
        d, c, p = done.cpu().numpy(), coll.cpu().numpy(), prob.cpu().numpy()
        if not ep.add(t, r.cpu().numpy(), d, kinds(d, c, p)):
            break
        states = ns
    return ep


def joint_fn(pi):
    return lambda s: pi.index_select(0, s)


def agents_fn(eng, table):
    import torch
    pw = torch.tensor([5 ** i for i in range(eng.n)], dtype=torch.int64, device=eng.torch_device)
    tl = table.to(torch.int64)

    def f(states):
        cells = eng.decode(states).to(torch.int64)
        return (tl.gather(1, cells.t().contiguous()).t() * pw).sum(1).to(torch.int32)
    return f


def assert_same(got, want):
    ret, length, outcome = got
    assert np.array_equal(u64(ret), want.G.view(np.uint64))
    assert np.array_equal(length.cpu().numpy(), want.length)
    assert np.array_equal(outcome.cpu().numpy(), want.outcome)


def random_table(eng, seed):
    import torch
    rng = np.random.default_rng(seed)
    return torch.from_numpy(rng.integers(0, 5, (eng.n, eng.L)).astype(np.int32)).to(eng.torch_device)


# ---- 1. RANDOM == rollout(actions=None, auto_reset=False), cut at the first done --------------------------------------
@pytest.mark.parametrize("name,E,T", [("rows_c2", 20000, 40), ("rows_c4", 3000, 24)])
@pytest.mark.parametrize("gamma", [1.0, 0.95])
def test_random_policy_equals_rollout(name, E, T, gamma, torch):
    from gym_mapf_b200.envs.vec_env import VecMapfEnv
    spec, _ = G.load(name)
    vec = VecMapfEnv(env_of(spec), E, seed=0xfeed, auto_reset=False)
    vec.env_offset = 1 << 33
    vec.step(torch.zeros(E, dtype=torch.int32, device=vec.device))  # the stream starts at step_count
    vec.reset()
    before = vec.states.clone()
    ev = vec.evaluate(None, E, T, gamma=gamma)
    assert torch.equal(vec.states, before) and vec.step_count == 1
    ro = vec.rollout(T)
    d, c, p, r = (x.cpu().numpy() for x in (ro.done, ro.collision, ro.prob, ro.reward))
    want = Episodes(E, gamma)
    for t in range(T):
        want.add(t, r[t], d[t], kinds(d[t], c[t], p[t]))
    assert_same(ev, want)
    assert (want.outcome == 0).any() and (want.length < T).any()


# ---- 2. JOINT == a step loop over pi[states] --------------------------------------------------------------------------
JOINT_SPECS = ("c1_makespan", "c1_soc", "rows_obst4_n2_v0_soc")


@pytest.fixture(scope="module")
def joint_cases(torch):
    out = {}
    for key in JOINT_SPECS:
        eng = c1_env(soc=key == "c1_soc").engine if key.startswith("c1") else make_engine(G.load(key)[0])
        out[key] = (eng, vi_policy(eng))
    return out


@pytest.mark.parametrize("key", JOINT_SPECS)
@pytest.mark.parametrize("E", [1, 31, 33, 4097, 100003])
def test_joint_policy_equals_step_loop(key, E, joint_cases, torch):
    eng, pi = joint_cases[key]
    for T in (1, 7, 200):
        for gamma in (1.0, 0.95):
            got = eng.evaluate(pi, E, T, gamma=gamma, seed=5, step_index=9, episode_offset=E)
            assert_same(got, step_loop(eng, joint_fn(pi), E, T, gamma, seed=5, step_index=9, env_offset=E))


# ---- 3. AGENTS == a step loop over the per-agent table ----------------------------------------------------------------
@pytest.fixture(scope="module")
def agent_envs(torch):
    return {name: env_of(G.load(name)[0]) for name in ("rows_c2", "rows_c4", "rows_berlin")}


@pytest.mark.parametrize("name,E,T", [("rows_c2", 30000, 300), ("rows_c4", 4000, 400), ("rows_berlin", 3000, 600)])
@pytest.mark.parametrize("table_kind", ["random", "independent"])
def test_agents_policy_equals_step_loop(name, E, T, table_kind, agent_envs, torch):
    from gym_mapf_b200.envs.utils import independent_policy
    env = agent_envs[name]
    eng = env.engine
    table = random_table(eng, 3) if table_kind == "random" else independent_policy(env)
    assert table.dtype == torch.int32 and tuple(table.shape) == (eng.n, eng.L)
    for gamma in (1.0, 0.95):
        got = eng.evaluate(table, E, T, gamma=gamma, seed=21, step_index=2, episode_offset=100)
        want = step_loop(eng, agents_fn(eng, table), E, T, gamma, seed=21, step_index=2, env_offset=100)
        assert_same(got, want)


def test_local_view_numbers_cells_like_the_joint_env(agent_envs):
    from gym_mapf_b200.envs.utils import get_local_view
    for env in agent_envs.values():
        k, dest, prob, rc = env.engine.moves()
        for i in range(env.n_agents):
            sub = get_local_view(env, [i]).engine
            assert sub.L == env.engine.L and np.array_equal(sub.moves()[3], rc)
            assert sub.s0 == env.engine.decode(env.engine.states_from_ints([env.engine.s0]))[0, i].item()


def test_agents_equals_joint_table_on_c1(torch):
    eng = c1_env(soc=True).engine
    table = random_table(eng, 8)
    cells = eng.decode(torch.arange(int(eng.nS), dtype=torch.int64, device=eng.torch_device)).to(torch.int64)
    joint = (table.to(torch.int64)[0][cells[:, 0]] + 5 * table.to(torch.int64)[1][cells[:, 1]]).to(torch.int32)
    for gamma in (1.0, 0.95):
        a = eng.evaluate(table, 50000, 300, gamma=gamma, seed=4)
        b = eng.evaluate(joint, 50000, 300, gamma=gamma, seed=4)
        for x, y in zip(a, b):
            assert torch.equal(x, y)


# ---- 4. the same episodes from the C oracle and the host Philox stream ------------------------------------------------
def philox_words(seed, env, step, block):
    return philox4x32_10([env & np.uint64(0xFFFFFFFF), env >> np.uint64(32), np.full(len(env), step & 0xFFFFFFFF, np.uint64),
                          np.full(len(env), ((step >> 32) << 8) | block, np.uint64)], [seed & 0xFFFFFFFF, seed >> 32])


@pytest.mark.parametrize("kind", ["agents", "random"])
def test_episodes_replayed_through_the_oracle(kind, torch):
    spec, _ = G.load("rows_c2")
    eng, ora = make_engine(spec), make_oracle(spec)
    E, T, gamma, seed, step0, off = 6000, 120, 0.95, 0x5eed, 40, 12345
    table = random_table(eng, 2)
    got = eng.evaluate(table if kind == "agents" else None, E, T, gamma=gamma, seed=seed, step_index=step0,
                       episode_offset=off)
    sub = np.arange(0, E, 23)
    env = sub.astype(np.uint64) + np.uint64(off)
    tab = table.cpu().numpy().astype(np.int64)
    lo = np.full(len(sub), eng.s0, np.uint64)
    hi = np.zeros_like(lo)
    ep = Episodes(len(sub), gamma)
    for t in range(T):
        if kind == "agents":
            cells = ora.decode(lo, hi).astype(np.int64)
            actions = sum(tab[i][cells[:, i]] * 5 ** i for i in range(eng.n))
        else:  # k_rollout's random action: Philox block 15, words 0 and 1 as a 64-bit fraction of nA
            w = philox_words(seed, env, step0 + t, 15)
            nA = np.uint64(eng.nA)
            actions = ((w[0] * nA + ((w[1] * nA) >> np.uint64(32))) >> np.uint64(32)).astype(np.int64)
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


# ---- 5. statistics: the mean return estimates V_pi(s0) --------------------------------------------------------------
def policy_value(ora, pi, nS, gamma, iters=700):
    """V_pi by iterating V = sum over P[s][pi(s)] of p * (r + gamma * V[s2]), with no continuation after a done record."""
    s = np.arange(nS, dtype=np.uint64)
    w = ora.rows(s, np.zeros_like(s), pi.astype(np.int64))
    rows = np.repeat(np.arange(nS), np.diff(w["row_ptr"]))
    cont = gamma * (1 - w["done"].astype(np.float64))
    s2 = w["next_lo"].astype(np.int64)
    V = np.zeros(nS)
    for _ in range(iters):
        V = np.bincount(rows, weights=w["prob"] * (w["reward"] + cont * V[s2]), minlength=nS)
    return V


def test_mean_return_matches_policy_value(torch):
    from gym_mapf_b200.envs.vec_env import VecMapfEnv, evaluation_summary
    env = c1_env(soc=False)
    eng = env.engine
    gamma, E = 0.9, 1 << 20
    _, pi, _ = VecMapfEnv(env, 1).value_iteration(gamma=gamma, eps=1e-10)
    spec = dict(rows=["".join("@" if v else "." for v in r) for r in env.grid.obstacles], n_agents=2,
                goals=[list(g) for g in env.agents_goals], fail_prob=0.2, r_clash=-1000.0, r_goal=100.0, r_living=-1.0,
                soc=False)
    V = policy_value(make_oracle(spec), pi.cpu().numpy(), int(eng.nS), gamma)
    ev = VecMapfEnv(env, E, seed=77).evaluate(pi, E, 400, gamma=gamma)
    st = evaluation_summary(ev)
    se = st["std_return"] / np.sqrt(E)
    assert se > 0 and abs(st["mean_return"] - V[eng.s0]) < 5 * se, (st, V[eng.s0])
    # the summary is what torch computes from the records
    r, o = ev.returns.cpu().numpy(), ev.outcomes.cpu().numpy()
    assert st["mean_length"] == pytest.approx(ev.lengths.cpu().numpy().mean())
    assert st["success_rate"] + st["collision_rate"] + st["timeout_rate"] == pytest.approx(1.0)
    assert st["success_rate"] == pytest.approx((o == 2).mean()) and st["std_return"] == pytest.approx(r.std())


def test_deterministic_env_gives_the_oracle_trajectory(torch):
    from gym_mapf_b200.envs.vec_env import VecMapfEnv
    env = c1_env(soc=True, fail_prob=0.0)
    eng = env.engine
    gamma = 0.9
    _, pi, _ = VecMapfEnv(env, 1).value_iteration(gamma=gamma, eps=1e-10)
    ret, length, outcome = eng.evaluate(pi, 70001, 400, gamma=gamma, seed=3)
    spec = dict(rows=["".join("@" if v else "." for v in r) for r in env.grid.obstacles], n_agents=2,
                goals=[list(g) for g in env.agents_goals], fail_prob=0.0, r_clash=-1000.0, r_goal=100.0, r_living=-1.0,
                soc=True)
    ora, p = make_oracle(spec), pi.cpu().numpy()
    lo, ep = np.array([eng.s0], np.uint64), Episodes(1, gamma)
    for t in range(400):
        w = ora.step(lo, np.zeros_like(lo), np.array([p[int(lo[0])]], np.int64), np.full((1, 2), 0.5))
        k = np.where(w["collision"] == 1, 1, np.where(w["terminal"] == 1, 3, 2)).astype(np.uint8)
        if not ep.add(t, w["reward"], w["done"].astype(bool), k):
            break
        lo = w["next_lo"]
    assert ep.outcome[0] == 2 and ep.length[0] > 1
    assert np.all(u64(ret) == ep.G.view(np.uint64)[0])
    assert np.all(length.cpu().numpy() == ep.length[0]) and np.all(outcome.cpu().numpy() == ep.outcome[0])


# ---- 6. sharding: episode ranges split over calls concatenate to one call ---------------------------------------------
def test_sharded_calls_concatenate(torch):
    from gym_mapf_b200 import sharding
    spec, _ = G.load("rows_c2")
    eng = make_engine(spec)
    table = random_table(eng, 6)
    E, T, off = 100003, 150, 1000
    whole = eng.evaluate(table, E, T, gamma=0.95, seed=8, step_index=1, episode_offset=off)
    parts = []
    for rank in range(3):
        sh = sharding.split_range(E, 3, rank, begin=off)
        parts.append(eng.evaluate(table, sh.count, T, gamma=0.95, seed=8, step_index=1, episode_offset=sh.begin))
    for k in range(3):
        assert torch.equal(torch.cat([p[k] for p in parts]), whole[k])


# ---- 7. a start state that is already terminal ------------------------------------------------------------------------
def test_terminal_start(torch):
    from gym_mapf_b200.envs.vec_env import evaluation_summary
    base = c1_env()
    spec = dict(rows=["".join("@" if v else "." for v in r) for r in base.grid.obstacles], n_agents=2,
                starts=[list(g) for g in base.agents_goals], goals=[list(g) for g in base.agents_goals], fail_prob=0.2,
                r_clash=-1000.0, r_goal=100.0, r_living=-1.0, soc=True)
    eng = env_of(spec).engine
    zeros_joint = torch.zeros(int(eng.nS), dtype=torch.int32, device=eng.torch_device)
    for policy in (None, zeros_joint, random_table(eng, 1)):
        ev = eng.evaluate(policy, 1000, 50, gamma=0.95)
        assert np.all(u64(ev[0]) == 0) and bool((ev[1] == 1).all()) and bool((ev[2] == 3).all())
    from gym_mapf_b200.envs.vec_env import Evaluation
    st = evaluation_summary(Evaluation(*ev))
    assert st["success_rate"] == st["collision_rate"] == st["timeout_rate"] == 0.0 and st["mean_length"] == 1.0


# ---- 8. writes stay inside the outputs -------------------------------------------------------------------------------
@pytest.mark.parametrize("map_name,n", [("room-32-32-4", 4), ("room-64-64-8", 8), ("empty-8-8", 2)])
def test_evaluate_writes_only_its_outputs(map_name, n, torch):
    from gym_mapf_b200._native import POLICY_AGENTS, POLICY_JOINT, POLICY_RANDOM, _ptr, check, lib
    from gym_mapf_b200.envs.mapf_env import OptimizationCriteria
    from gym_mapf_b200.envs.utils import create_mapf_env
    eng = create_mapf_env(map_name, 1, n, 0.2, -1000.0, 100.0, -1.0, OptimizationCriteria.SoC, device=0).engine
    g = Guarded(torch)
    policies = [(POLICY_RANDOM, None, 0), (POLICY_AGENTS, random_table(eng, 4).to(torch.uint8), eng.n * eng.L)]
    if eng.words == 1 and eng.nS < (1 << 24):
        policies.append((POLICY_JOINT, torch.randint(0, int(eng.nA), (int(eng.nS),), dtype=torch.int32,
                                                       device=eng.torch_device), int(eng.nS)))
    sb = int(lib().mapf_evaluate_scratch_bytes())
    for E in SIZES:
        for kind, table, n_entries in policies:
            keep = None if table is None else table.clone()
            scratch = g.new((sb + 7) // 8, torch.int64)
            ret, length, outcome = g.new(E, torch.float64), g.new(E, torch.int32), g.new(E, torch.uint8)
            check(lib().mapf_evaluate(eng._h, kind, _ptr(table), n_entries, E, 64, 0.95, 3, 0, 0, _ptr(scratch),
                                      _ptr(ret), _ptr(length), _ptr(outcome), eng._stream()))
            g.check("evaluate kind=%d E=%d" % (kind, E))
            assert keep is None or torch.equal(keep, table)
            assert bool(((length >= 1) & (length <= 64)).all()) and bool((outcome <= 3).all())


# ---- 9. rejected arguments -----------------------------------------------------------------------------------------
def test_evaluate_errors(torch):
    from gym_mapf_b200 import _native
    from gym_mapf_b200._native import (MAPF_ERR_INVALID, MAPF_ERR_UNSUPPORTED, POLICY_AGENTS, POLICY_JOINT,
                                       POLICY_RANDOM, _ptr, lib)
    spec, _ = G.load("rows_obst4_n2_v0_soc")
    eng = make_engine(spec)
    eng4 = make_engine(G.load("rows_c4")[0])
    dev = eng.torch_device
    E = 10
    buf = lambda e: (torch.empty(e, dtype=torch.float64, device=dev), torch.empty(e, dtype=torch.int32, device=dev),  # noqa: E731
                     torch.empty(e, dtype=torch.uint8, device=dev))
    ret, length, outcome = buf(E)
    scratch = torch.empty(2, dtype=torch.int64, device=dev)
    joint = torch.zeros(int(eng.nS), dtype=torch.int32, device=dev)
    agents = torch.zeros(eng.n * eng.L, dtype=torch.uint8, device=dev)

    def call(e, kind=POLICY_RANDOM, pol=None, plen=0, T=5, sc=scratch, r=ret, ln=length, oc=outcome, h=None):
        return lib().mapf_evaluate(eng._h if h is None else h, kind, _ptr(pol), plen, e, T, 1.0, 0, 0, 0, _ptr(sc),
                                   _ptr(r), _ptr(ln), _ptr(oc), eng._stream())

    assert call(E) == 0 and call(0, sc=None, r=None, ln=None, oc=None) == 0
    assert call(E, POLICY_JOINT, joint, int(eng.nS)) == 0 and call(E, POLICY_AGENTS, agents, eng.n * eng.L) == 0
    invalid = [dict(h=C.c_void_p(0)), dict(sc=None), dict(r=None), dict(ln=None), dict(oc=None),
               dict(kind=3), dict(kind=-1), dict(kind=POLICY_JOINT, plen=int(eng.nS)),
               dict(kind=POLICY_AGENTS, plen=eng.n * eng.L), dict(T=0), dict(T=-1), dict(T=1 << 31),
               dict(kind=POLICY_JOINT, pol=joint, plen=int(eng.nS) - 1),
               dict(kind=POLICY_AGENTS, pol=agents, plen=eng.n * eng.L - 1),
               dict(kind=POLICY_AGENTS, pol=agents, plen=eng.n * eng.L + 1)]
    for kw in invalid:
        assert call(E, **kw) == MAPF_ERR_INVALID, kw
    assert call(-1) == MAPF_ERR_INVALID and call((1 << 30) + 1) == MAPF_ERR_INVALID
    j4 = torch.zeros(16, dtype=torch.int32, device=dev)
    assert lib().mapf_evaluate(eng4._h, POLICY_JOINT, _ptr(j4), 1 << 62, E, 5, 1.0, 0, 0, 0, _ptr(scratch), _ptr(ret),
                               _ptr(length), _ptr(outcome), eng4._stream()) == MAPF_ERR_UNSUPPORTED
    # the Python layer: shapes, dtypes and ranges
    bad = [joint.to(torch.int64), joint.double(), joint[:-1], torch.zeros((2, 2, 2), dtype=torch.int32, device=dev),
           joint.clone().fill_(-1), joint.clone().fill_(int(eng.nA)),
           torch.zeros((eng.n, eng.L), dtype=torch.float32, device=dev), torch.zeros((eng.n, eng.L - 1), dtype=torch.int32, device=dev),
           torch.full((eng.n, eng.L), 5, dtype=torch.int32, device=dev), torch.full((eng.n, eng.L), -1, dtype=torch.int64, device=dev),
           torch.zeros((eng.n, eng.L), dtype=torch.int32)]
    for p in bad:
        with pytest.raises(ValueError):
            eng.evaluate(p, E, 5)
    with pytest.raises(ValueError):
        eng.evaluate(None, -1, 5)
    with pytest.raises(ValueError):
        eng.evaluate(None, E, 5, out=buf(E + 1))
    with pytest.raises(ValueError):  # a joint-state policy cannot cover L**8 states
        eng4.evaluate(torch.zeros(16, dtype=torch.int32, device=dev), E, 5)
    for T in (0, 1 << 31):
        with pytest.raises(_native.NativeError) as ei:
            eng.evaluate(None, E, T)
        assert ei.value.code == MAPF_ERR_INVALID
    # every valid dtype of a per-agent table is accepted and gives the same episodes
    base = eng.evaluate(torch.ones((eng.n, eng.L), dtype=torch.uint8, device=dev), E, 20, seed=1)
    other = eng.evaluate(torch.ones((eng.n, eng.L), dtype=torch.int64, device=dev), E, 20, seed=1)
    assert all(torch.equal(a, b) for a, b in zip(base, other))


# ---- 10. out-of-range entries through the C ABI are clamped ------------------------------------------------------------
def c_evaluate(eng, policy, E, T, out, scratch=None, gamma=0.95, seed=3, step_index=0, episode_offset=0):
    """One mapf_evaluate (policy = (kind, table)) or mapf_evaluate_groups (policy = (POLICY_GROUPS, tables, group_of))
    call; `out` is (ret, length, outcome) plus, for groups, the conflict output (or None)."""
    import torch
    from gym_mapf_b200._native import POLICY_GROUPS, _ptr, check, lib
    if scratch is None:
        scratch = torch.empty(2, dtype=torch.int64, device=eng.torch_device)
    table = policy[1]
    n = 0 if table is None else table.numel()
    if policy[0] == POLICY_GROUPS:
        gof = (C.c_int32 * eng.n)(*policy[2])
        check(lib().mapf_evaluate_groups(eng._h, gof, _ptr(table), n, E, T, gamma, seed, step_index, episode_offset,
                                         _ptr(scratch), *(_ptr(x) for x in out), eng._stream()))
    else:
        check(lib().mapf_evaluate(eng._h, policy[0], _ptr(table), n, E, T, gamma, seed, step_index, episode_offset,
                                  _ptr(scratch), *(_ptr(x) for x in out), eng._stream()))
    return out


def new_outputs(torch, eng, E, conflict=False):
    dev = eng.torch_device
    out = (torch.empty(E, dtype=torch.float64, device=dev), torch.empty(E, dtype=torch.int32, device=dev),
           torch.empty(E, dtype=torch.uint8, device=dev))
    return out + ((torch.empty(E, dtype=torch.uint8, device=dev),) if conflict else ())


def assert_clamped(torch, eng, make_policy, table, bad, top, rng, E=20000, T=100):
    """Some entries of `table` overwritten with the values `bad` give bit for bit the episodes of the same entries set
    to `top`, the documented maximum; and those entries are read (the episodes differ from the unmodified table's).
    `bad` and `top` hold scalars or per-entry arrays."""
    hit = np.flatnonzero(rng.random(len(table)) < 0.3)
    cand = np.stack([np.broadcast_to(np.asarray(b, np.int64), table.shape) for b in bad])
    worst, capped = table.copy(), table.copy()
    worst[hit] = cand[rng.integers(0, len(bad), len(hit)), hit].astype(table.dtype)
    capped[hit] = np.broadcast_to(top, table.shape)[hit]
    dev = eng.torch_device
    conflict = make_policy(None)[0] == 3
    got = [c_evaluate(eng, make_policy(torch.from_numpy(t).to(dev)), E, T, new_outputs(torch, eng, E, conflict))
           for t in (worst, capped, table)]
    assert all(torch.equal(a, b) for a, b in zip(got[0], got[1]))
    assert not all(torch.equal(a, b) for a, b in zip(got[1], got[2]))


@pytest.mark.parametrize("case", ["joint_c1", "agents_c2", "agents_c4"])
def test_out_of_range_entries_are_clamped(case, torch):
    """JOINT entries >= nA or < 0 act as nA - 1; AGENTS entries above 4 act as 4 (LEFT).  The Python layer rejects such
    tables, so only C callers reach the clamp."""
    from gym_mapf_b200._native import POLICY_AGENTS, POLICY_JOINT
    rng = np.random.default_rng(len(case))
    if case == "joint_c1":
        eng = c1_env(soc=True).engine
        nA = int(eng.nA)
        table = rng.integers(0, nA, int(eng.nS)).astype(np.int32)
        assert_clamped(torch, eng, lambda t: (POLICY_JOINT, t), table, [nA, (1 << 31) - 1, -1], nA - 1, rng)
    else:  # planned tables: with random ones the agents never meet or arrive, and every episode is a timeout alike
        from gym_mapf_b200.envs.utils import independent_policy
        env = env_of(G.load("rows_" + case[-2:])[0])
        eng = env.engine
        table = independent_policy(env).cpu().numpy().astype(np.uint8).reshape(-1)
        assert_clamped(torch, eng, lambda t: (POLICY_AGENTS, t), table, [5, 17, 255], 4, rng)


# ---- 11. the episode queue: lanes refill past the resident threads of a launch -----------------------------------------
QUEUE_CASES = ["random_c1", "agents_c1", "joint_c1", "groups_c2", "groups_c5_n10"]
SENTINEL_RET = 0x7FF4DEADBEEF0001  # the bits of a NaN, which no return is


def queue_policy(torch, case):
    """(engine, oracle, C ABI policy, replay policy, replay kind) of a queue case."""
    from gym_mapf_b200._native import POLICY_AGENTS, POLICY_GROUPS, POLICY_JOINT, POLICY_RANDOM
    from gym_mapf_b200.envs.vec_env import GroupPolicy
    rng = np.random.default_rng(len(case))
    if case.endswith("c1"):
        env = c1_env(soc=True)
        spec = dict(rows=["".join("@" if v else "." for v in r) for r in env.grid.obstacles], n_agents=2,
                    goals=[list(g) for g in env.agents_goals], fail_prob=0.2, r_clash=-1000.0, r_goal=100.0,
                    r_living=-1.0, soc=True)
        eng, ora = env.engine, make_oracle(spec)
    else:
        spec = G.load("rows_" + case[len("groups_"):])[0]
        eng, ora = make_engine(spec), make_oracle(spec)
    dev = eng.torch_device
    if case.startswith("random"):
        return eng, ora, (POLICY_RANDOM, None), None, "random"
    if case.startswith("agents"):
        table = rng.integers(0, 5, (eng.n, eng.L))
        return eng, ora, (POLICY_AGENTS, torch.from_numpy(table.astype(np.uint8)).to(dev)), table, "agents"
    if case.startswith("joint"):
        table = rng.integers(0, eng.nA, int(eng.nS)).astype(np.int32)
        return eng, ora, (POLICY_JOINT, torch.from_numpy(table).to(dev)), table, "joint"
    m = (eng.n + 1) // 2  # pairs of agents i, i + m (and a singleton when n is odd)
    groups = [tuple(range(g, eng.n, m)) for g in range(m)]
    tables = [rng.integers(0, 5 ** len(g), eng.L ** len(g), dtype=np.int32) for g in groups]
    gp = GroupPolicy(groups, [torch.from_numpy(t).to(dev) for t in tables])
    return eng, ora, (POLICY_GROUPS, torch.cat(gp.tables), gp.group_of()), (groups, tables), "groups"


@pytest.mark.timeout(300)
@pytest.mark.parametrize("case", QUEUE_CASES)
def test_episode_queue_hands_out_every_episode_once(case, torch):
    """E = 2**19 + 3 episodes: more than a B200 launch holds resident (148 SMs x 2048 threads = 303 104), so lanes take
    further episodes from the queue.  Every output is written, with the episode the oracle computes for that index
    (sampled up to E - 1), in two calls that share one scratch buffer, and three shards give the same records."""
    from gym_mapf_b200 import sharding
    from gym_mapf_b200._native import POLICY_GROUPS
    from gym_mapf_b200.envs.vec_env import GroupPolicy
    from test_gpu_kernel_matrix import SEED, assert_episodes, replay_episodes
    eng, ora, policy, table, kind = queue_policy(torch, case)
    E, T, gamma, step0, off = (1 << 19) + 3, 64, 0.95, 11, 1 << 33
    groups = policy[0] == POLICY_GROUPS
    scratch = torch.empty(2, dtype=torch.int64, device=eng.torch_device)
    runs = []
    for _ in range(2):
        out = new_outputs(torch, eng, E, groups)
        out[0].view(torch.int64).fill_(SENTINEL_RET)
        out[1].fill_(-1)
        for x in out[2:]:
            x.fill_(0xEE)
        c_evaluate(eng, policy, E, T, out, scratch=scratch, gamma=gamma, seed=SEED, step_index=step0,
                   episode_offset=off)
        assert bool((out[0].view(torch.int64) != SENTINEL_RET).all())
        assert bool(((out[1] >= 1) & (out[1] <= T)).all()) and bool((out[2] <= 3).all())
        if groups:
            assert bool(((out[3] != 0xFF) == (out[2] == 1)).all()) and bool(((out[3] & 15) < (out[3] >> 4)).any())
        runs.append(out)
    assert all(torch.equal(a, b) for a, b in zip(*runs))
    out = runs[0]
    sub = np.unique(np.concatenate([np.arange(0, E, 257), np.arange(303104 - 40, 303104 + 40), [E - 1]]))
    ep = replay_episodes(eng, ora, table, kind, T, gamma, step0, off, sub)
    assert_episodes(out, ep, sub, case)
    if groups:
        assert np.array_equal(out[3].cpu().numpy()[sub], ep.pair) and (ep.outcome == 1).any()
    assert (ep.outcome != ep.outcome[0]).any() and (ep.length < T).any()
    pol = GroupPolicy(table[0], [torch.from_numpy(t).to(eng.torch_device) for t in table[1]]) if groups else policy[1]
    parts = []
    for rank in range(3):
        sh = sharding.split_range(E, 3, rank, begin=off)
        p = new_outputs(torch, eng, sh.count, groups)
        if groups:
            eng.evaluate_groups(pol, sh.count, T, gamma=gamma, seed=SEED, step_index=step0, episode_offset=sh.begin,
                                out=p[:3], conflicts=p[3])
        else:
            eng.evaluate(pol, sh.count, T, gamma=gamma, seed=SEED, step_index=step0, episode_offset=sh.begin, out=p)
        parts.append(p)
    for k in range(len(out)):
        assert torch.equal(torch.cat([p[k] for p in parts]), out[k])
