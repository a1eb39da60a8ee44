"""On-disk formats and heterogeneous batches (SURVEY.md 8f row 4).

CPU part: the oracle's parser restatement against fixtures produced by the unmodified reference parsers
(tests/golden/formats.json, oracle/make_golden_formats.py).  GPU part: the device-side .map parser and
`create_mapf_env_from_text` against the same fixtures, and the grouped step kernel (several specs in one launch)
against the C oracle and against the single-spec step."""
import json
import os

import numpy as np
import pytest

import golden_util as G
from oracle import mapf_oracle as O

with open(os.path.join(G.GOLDEN, "formats.json")) as f:
    CASES = json.load(f)
IDS = [c["name"] for c in CASES]


def _expected_error(case):
    return {"KeyError": KeyError, "ValueError": ValueError}[case["error"]]


def _free_cells(rows):
    return [(r, c) for c in range(len(rows[0])) for r in range(len(rows)) if rows[r][c] == "."]  # column-major (grid.py:37-40)


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_oracle_parsers_match_reference(case):
    m, s = case["map_text"].encode("latin-1"), case["scen_text"].encode("latin-1")

    def build():
        rows = O.parse_map_text(m)
        starts, goals = O.parse_scen_text(s, case["n_agents"])
        cells = {rc: i for i, rc in enumerate(_free_cells(rows))}
        ids = [cells[tuple(x)] for x in starts]
        [cells[tuple(x)] for x in goals]
        return rows, starts, goals, len(cells), O.from_digits(ids, len(cells))

    if "error" in case:
        with pytest.raises(_expected_error(case)) as ei:
            build()
        if case["error"] == "KeyError":
            assert repr(ei.value.args[0]) == case["key"]
        return
    rows, starts, goals, L, s0 = build()
    ok = case["ok"]
    assert rows == ok["rows"] and len(rows) == ok["H"] and len(rows[0]) == ok["W"]
    assert [list(x) for x in starts] == ok["starts"] and [list(x) for x in goals] == ok["goals"]
    assert len(goals) == ok["n_agents"] and L == ok["L"] and str(s0) == ok["s0"]


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_library_scen_parser_matches_reference(case):
    """The C library's host-side .scen parser (no GPU involved) against the reference's parse_scen_file."""
    from gym_mapf_b200 import _native
    s = case["scen_text"].encode("latin-1")
    if case.get("error") == "ValueError":
        with pytest.raises(_native.NativeError) as ei:
            _native.parse_scen_text(s, case["n_agents"])
        assert ei.value.code == _native.MAPF_ERR_INVALID
        return
    starts, goals = _native.parse_scen_text(s, case["n_agents"])
    want = O.parse_scen_text(s, case["n_agents"])
    assert (starts, goals) == want
    if "ok" in case:
        assert [list(x) for x in starts] == case["ok"]["starts"] and [list(x) for x in goals] == case["ok"]["goals"]


# ---------------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu


@gpu
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_device_parser_matches_reference(case):
    from gym_mapf_b200 import _native
    from gym_mapf_b200.envs.mapf_env import OptimizationCriteria
    from gym_mapf_b200.envs.utils import create_mapf_env_from_text
    m, s = case["map_text"].encode("latin-1"), case["scen_text"].encode("latin-1")
    if "error" in case:
        if case["error"] == "KeyError":
            with pytest.raises(KeyError) as ei:
                create_mapf_env_from_text(m, s, case["n_agents"], 0.2, -1000.0, 100.0, -1.0, OptimizationCriteria.SoC)
            assert str(ei.value.args[0]) == case["key"]
        else:  # the reference's ValueError surfaces as the library's invalid-argument error
            with pytest.raises(_native.NativeError) as ei:
                create_mapf_env_from_text(m, s, case["n_agents"], 0.2, -1000.0, 100.0, -1.0, OptimizationCriteria.SoC)
            assert ei.value.code == _native.MAPF_ERR_INVALID
        return
    ok = case["ok"]
    mask = _native.parse_map_text(m)
    want = np.array([[1 if ch == "@" else 0 for ch in row] for row in ok["rows"]], dtype=np.uint8)
    assert mask.shape == (ok["H"], ok["W"]) and np.array_equal(mask, want)
    if ok["n_agents"] > 13:
        return
    env = create_mapf_env_from_text(m, s, case["n_agents"], 0.2, -1000.0, 100.0, -1.0, OptimizationCriteria.SoC)
    assert env.n_agents == ok["n_agents"] and len(env.valid_locations) == ok["L"] and str(env.s) == ok["s0"]
    assert [list(x) for x in env.agents_starts] == ok["starts"] and [list(x) for x in env.agents_goals] == ok["goals"]
    assert np.array_equal(env.grid.obstacles, want)
    assert str(env.engine.s0) == ok["s0"] and env.engine.L == ok["L"]


@gpu
def test_device_parser_every_shipped_map():
    """Every packaged map: the device parse of the materialised .map file equals the packaged obstacle mask (which
    oracle/../maps/build_bundle.py took from the reference's files), and create_mapf_env_from_text == create_mapf_env."""
    from gym_mapf_b200 import _native
    from gym_mapf_b200.envs import map_name_to_files, maps
    from gym_mapf_b200.envs.mapf_env import OptimizationCriteria
    from gym_mapf_b200.envs.utils import create_mapf_env, create_mapf_env_from_text
    for name in maps.map_names():
        map_file, scen_file = map_name_to_files(name, 2)
        with open(map_file, "rb") as f:
            m = f.read()
        with open(scen_file, "rb") as f:
            s = f.read()
        assert np.array_equal(_native.parse_map_text(m), maps.obstacle_mask(name)), name
        if name.startswith("empty"):
            a = create_mapf_env(name, 2, 3, 0.1, -10.0, 5.0, -0.5, OptimizationCriteria.Makespan)
            b = create_mapf_env_from_text(m, s, 3, 0.1, -10.0, 5.0, -0.5, OptimizationCriteria.Makespan)
            assert a.grid == b.grid and a.agents_starts == b.agents_starts and a.agents_goals == b.agents_goals
            assert a.s == b.s and a.nS == b.nS
            assert a.P[a.s][7] == b.P[b.s][7]


@gpu
def test_parse_errors():
    from gym_mapf_b200 import _native
    with pytest.raises(_native.NativeError):   # fewer than five lines: no grid
        _native.parse_map_text(b"type octile\nheight 1\nwidth 1\nmap\n")
    with pytest.raises(_native.NativeError):   # ragged rows
        _native.parse_map_text(b"a\nb\nc\nd\n...\n..\n")
    with pytest.raises(KeyError):
        _native.parse_map_text(b"a\nb\nc\nd\n.x.\n")
    assert _native.parse_map_text(b"a\rb\rc\rd\r.@\r@.").tolist() == [[0, 1], [1, 0]]   # lone CR line ends, no final one


def _spec(rows, starts, goals, fail_prob, r_clash, r_goal, r_living, soc):
    return dict(rows=rows, n_agents=len(starts), starts=starts, goals=goals, fail_prob=fail_prob, r_clash=r_clash,
                r_goal=r_goal, r_living=r_living, soc=soc)


def _shipped_spec(name, scen, n, fail_prob, r_clash, r_goal, r_living, soc):
    from gym_mapf_b200.envs import map_name_to_files
    from gym_mapf_b200.envs.utils import parse_map_file, parse_scen_file
    map_file, scen_file = map_name_to_files(name, scen)
    rows = [ln.strip() for ln in parse_map_file(map_file)]
    starts, goals = parse_scen_file(scen_file, n)
    return _spec(rows, [list(x) for x in starts], [list(x) for x in goals], fail_prob, r_clash, r_goal, r_living, soc)


def _group_case(n):
    specs = [_shipped_spec("room-32-32-4", 1 if n <= 4 else 13, n, 0.2, -1000.0, 100.0, -1.0, True),
             _shipped_spec("empty-32-32", 3, n, 0.3, -50.0, 10.0, -0.5, False),
             _shipped_spec("maze-32-32-4", 10, n, 0.2, -1000.0, 100.0, -1.0, False),
             _shipped_spec("empty-16-16", 7, n, 0.0, -7.0, 3.0, -2.0, True),
             _shipped_spec("empty-8-8", 5, n, 1.0, -1.0, 1.0, -0.125, True)]
    counts = [3000, 1, 2049, 0, 777]
    return specs, counts


@gpu
@pytest.mark.parametrize("n", [2, 4, 6])
def test_group_step_matches_oracle(n):
    """Five specs (different grids, scenarios, slip probabilities, rewards, criteria) in one launch, replayed uniforms:
    every env must equal the C oracle's step for ITS spec, bit for bit; and the single-spec kernel on each segment."""
    import torch
    from engine_util import make_engine, make_oracle, states_tensor, split_states, u64
    from gym_mapf_b200 import _native
    specs, counts = _group_case(n)
    engines = [make_engine(sp) for sp in specs]
    group = _native.Group(engines, counts)
    B = sum(counts)
    assert group.size == B
    rng = np.random.default_rng(40 + n)
    lo = np.zeros(B, np.uint64)
    act = rng.integers(0, 5 ** n, B).astype(np.int32)
    uni = rng.random((B, n))
    at = 0
    for eng, c in zip(engines, counts):
        # a mix of the start state, random states and (for density of terminal / clash cases) states in a small window
        s = rng.integers(0, eng.nS, c, dtype=np.uint64)
        s[: c // 4] = eng.s0
        s[c // 4: c // 2] = eng.goal_state
        lo[at:at + c] = s
        at += c
    states = torch.from_numpy(lo.view(np.int64).copy()).cuda()
    actions = torch.from_numpy(act).cuda()
    uniforms = torch.from_numpy(uni).cuda()
    ns, reward, prob, done, coll = group.step(states, actions, uniforms=uniforms)
    torch.cuda.synchronize()
    at = 0
    for sp, eng, c in zip(specs, engines, counts):
        if c == 0:
            continue
        sl = slice(at, at + c)
        w = make_oracle(sp).step(lo[sl], np.zeros(c, np.uint64), act[sl].astype(np.int64), uni[sl])
        assert np.array_equal(u64(ns[sl]), w["next_lo"])
        assert np.array_equal(u64(reward[sl]), G.f64_to_bits(w["reward"]))
        assert np.array_equal(u64(prob[sl]), G.f64_to_bits(w["prob"]))
        assert np.array_equal(done[sl].cpu().numpy().astype(np.uint8), w["done"])
        assert np.array_equal(coll[sl].cpu().numpy().astype(np.uint8), w["collision"])
        one = eng.step(states[sl].clone(), actions[sl].clone(), uniforms=uniforms[sl].clone())
        for a, b in zip(one, (ns[sl], reward[sl], prob[sl], done[sl], coll[sl])):
            assert torch.equal(a, b)
        at += c
    # device-side sampling: the grouped launch draws the same Philox words as the single-spec kernel, env by env
    g2 = group.step(states, actions, seed=99, step_index=5, env_offset=1000, auto_reset=True)
    at = 0
    for eng, c in zip(engines, counts):
        if c and eng is not engines[3]:
            sl = slice(at, at + c)
            one = eng.step(states[sl].clone(), actions[sl].clone(), seed=99, step_index=5, env_offset=1000 + at, auto_reset=True)
            for a, b in zip(one, g2):
                assert torch.equal(a, b[sl])
        at += c


@gpu
def test_group_two_word_states_and_errors():
    import torch
    from engine_util import make_engine, make_oracle, u64
    from gym_mapf_b200 import _native
    a = _shipped_spec("room-64-64-8", 1, 8, 0.2, -1000.0, 100.0, -1.0, False)
    b = _shipped_spec("room-64-64-16", 2, 8, 0.4, -3.0, 2.0, -1.0, True)
    ea, eb = make_engine(a), make_engine(b)
    assert ea.words == 2 and eb.words == 2
    counts = [1500, 1200]
    group = _native.Group([ea, eb], counts)
    rng = np.random.default_rng(8)
    B = sum(counts)
    lo, hi = np.zeros(B, np.uint64), np.zeros(B, np.uint64)
    cells = np.zeros((B, 8), np.int32)
    cells[:1500] = rng.integers(0, ea.L, (1500, 8))
    cells[1500:] = rng.integers(0, eb.L, (1200, 8))
    for sp, sl in ((a, slice(0, 1500)), (b, slice(1500, B))):
        lo[sl], hi[sl] = make_oracle(sp).encode(cells[sl])
    act = rng.integers(0, 5 ** 8, B).astype(np.int32)
    uni = rng.random((B, 8))
    states = torch.from_numpy(np.stack([lo, hi], 1).view(np.int64).copy()).cuda()
    out = group.step(states, torch.from_numpy(act).cuda(), uniforms=torch.from_numpy(uni).cuda())
    ns = out[0].cpu().numpy().view(np.uint64)
    for sp, sl in ((a, slice(0, 1500)), (b, slice(1500, B))):
        w = make_oracle(sp).step(lo[sl], hi[sl], act[sl].astype(np.int64), uni[sl])
        assert np.array_equal(ns[sl, 0], w["next_lo"]) and np.array_equal(ns[sl, 1], w["next_hi"])
        assert np.array_equal(u64(out[1][sl]), G.f64_to_bits(w["reward"])) and np.array_equal(u64(out[2][sl]), G.f64_to_bits(w["prob"]))
        assert np.array_equal(out[3][sl].cpu().numpy().astype(np.uint8), w["done"])
        assert np.array_equal(out[4][sl].cpu().numpy().astype(np.uint8), w["collision"])
    # mixed agent counts / state widths / unstaged tables are refused with a clear error
    c4 = make_engine(_shipped_spec("room-32-32-4", 1, 4, 0.2, -1000.0, 100.0, -1.0, True))
    with pytest.raises(_native.NativeError) as ei:
        _native.Group([ea, c4], [1, 1])
    assert ei.value.code == _native.MAPF_ERR_UNSUPPORTED
    c2 = make_engine(_shipped_spec("room-32-32-4", 1, 2, 0.2, -1000.0, 100.0, -1.0, True))
    berlin = make_engine(_shipped_spec("Berlin_1_256", 11, 2, 0.2, -1000.0, 100.0, -1.0, True))
    with pytest.raises(_native.NativeError) as ei:
        _native.Group([c2, berlin], [1, 1])
    assert ei.value.code == _native.MAPF_ERR_UNSUPPORTED and "shared memory" in ei.value.text
    with pytest.raises(ValueError):
        group.step(states[:10], torch.zeros(10, dtype=torch.int32, device="cuda"))


@gpu
def test_multimap_vec_env():
    """MultiMapVecEnv: mixed agent counts fall into one group per class; one spec alone equals VecMapfEnv."""
    import torch
    from gym_mapf_b200.envs.mapf_env import OptimizationCriteria
    from gym_mapf_b200.envs.utils import create_mapf_env
    from gym_mapf_b200.envs.vec_env import MultiMapVecEnv, VecMapfEnv
    e1 = create_mapf_env("room-32-32-4", 1, 4, 0.2, -1000.0, 100.0, -1.0, OptimizationCriteria.SoC)
    e2 = create_mapf_env("maze-32-32-4", 10, 4, 0.2, -1000.0, 100.0, -1.0, OptimizationCriteria.Makespan)
    e3 = create_mapf_env("empty-16-16", 1, 2, 0.2, -1000.0, 100.0, -1.0, OptimizationCriteria.SoC)
    e4 = create_mapf_env("Berlin_1_256", 11, 2, 0.2, -1000.0, 100.0, -1.0, OptimizationCriteria.SoC)
    mm = MultiMapVecEnv([e1, e2, e3, e4], [500, 300, 200, 100], seed=3)
    assert mm.num_envs == 1100 and mm.spec_of(0) == 0 and mm.spec_of(799) == 1 and mm.spec_of(800) == 2 and mm.spec_of(1099) == 3
    assert len(mm._parts) == 3
    g = torch.Generator(device="cpu").manual_seed(1)
    singles = []
    for env, c, lo in zip((e1, e2, e3, e4), mm.counts, mm.offsets):
        v = VecMapfEnv(env, c, seed=3)
        v.env_offset = lo
        singles.append(v)
    for _ in range(6):
        acts = torch.cat([torch.randint(0, env.nA, (c,), generator=g, dtype=torch.int32) for env, c in
                          zip((e1, e2, e3, e4), mm.counts)]).cuda()
        ns, r, d, info = mm.step(acts)
        for v, lo, hi in zip(singles, mm.offsets[:-1], mm.offsets[1:]):
            n1, r1, d1, i1 = v.step(acts[lo:hi].contiguous())
            assert torch.equal(n1, ns[lo:hi]) and torch.equal(r1, r[lo:hi]) and torch.equal(d1, d[lo:hi])
            assert torch.equal(i1["prob"], info["prob"][lo:hi]) and torch.equal(i1["collision"], info["collision"][lo:hi])


# ---- the step on conflict-dense states (mapf_step) ------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("n,map_name,scen", [(2, "empty-8-8", 1), (3, "room-32-32-4", 1), (4, "room-32-32-4", 1),
                                             (5, "empty-16-16", 2), (6, "maze-32-32-4", 10), (7, "empty-16-16", 4),
                                             (8, "empty-8-8", 3)])
@pytest.mark.parametrize("soc", [True, False])
@pytest.mark.timeout(180)
def test_step_conflict_dense_matches_oracle(n, map_name, scen, soc):
    """k_step == the C oracle given the uniforms; ragged batch sizes, conflict-dense states."""
    import torch
    from engine_util import make_engine, make_oracle, u64
    sp = _shipped_spec(map_name, scen, n, 0.2, -1000.0, 100.0, -1.0, soc)
    eng = make_engine(sp)
    ora = make_oracle(sp)
    assert eng.words == 1
    rng = np.random.default_rng(100 * n + soc)
    for B in (1, 31, 33, 4099):
        cells = rng.integers(0, eng.L, (B, n)).astype(np.int32)
        # conflict-dense half: every agent inside a few cells around agent 0 (vertex and swap clashes, shared cells)
        near = (cells[:, :1] + rng.integers(0, 3, (B, n))) % eng.L
        cells[B // 2:] = near[B // 2:]
        lo, hi = ora.encode(cells)
        lo[: B // 8] = eng.s0
        lo[B // 8: B // 6] = eng.goal_state
        act = rng.integers(0, 5 ** n, B).astype(np.int32)
        act[::5] = 0   # all STAY: parked agents under SoC
        uni = rng.random((B, n))
        states = torch.from_numpy(lo.view(np.int64).copy()).cuda()
        actions = torch.from_numpy(act).cuda()
        uniforms = torch.from_numpy(uni).cuda()
        got = eng.step(states, actions, uniforms=uniforms)
        w = ora.step(lo, hi, act.astype(np.int64), uni)
        assert np.array_equal(u64(got[0]), w["next_lo"])
        assert np.array_equal(u64(got[1]), G.f64_to_bits(w["reward"])) and np.array_equal(u64(got[2]), G.f64_to_bits(w["prob"]))
        assert np.array_equal(got[3].cpu().numpy().astype(np.uint8), w["done"])
        assert np.array_equal(got[4].cpu().numpy().astype(np.uint8), w["collision"])
        assert w["collision"].sum() > 0 or B < 1000


# ---- exclusive scan of row lengths (mapf_scan_rows): folded and spine paths, aligned and unaligned buffers ------------
@gpu
@pytest.mark.parametrize("B", [1, 2, 511, 512, 513, 2047, 2048, 2049, 100001, (2048 * 2048) + 4097,
                               2 * 4096 * 2048 + 12345])   # the last one: three passes of the spine kernel
def test_scan_rows_matches_cumsum(B):
    import torch
    from engine_util import make_engine
    from gym_mapf_b200._native import _ptr, check, lib
    eng = make_engine(_shipped_spec("empty-8-8", 1, 2, 0.2, -1000.0, 100.0, -1.0, True))
    g = torch.Generator(device="cuda").manual_seed(B)
    for shift in (0, 1):   # shift 1: the arrays start on an odd element, i.e. only 8-byte aligned (scalar path)
        buf_len = torch.randint(1, 6562, (B + 2,), generator=g, device="cuda", dtype=torch.int64)
        buf_ptr = torch.full((B + 3,), -7, device="cuda", dtype=torch.int64)
        row_len, row_ptr = buf_len[shift:shift + B], buf_ptr[shift:shift + B + 1]
        scratch = torch.empty(int(lib().mapf_scan_scratch_bytes(B)) // 8 + 1, dtype=torch.int64, device="cuda")
        check(lib().mapf_scan_rows(eng._h, row_len.data_ptr(), B, row_ptr.data_ptr(), _ptr(scratch), eng._stream()))
        want = torch.zeros(B + 1, dtype=torch.int64, device="cuda")
        want[1:] = torch.cumsum(row_len, 0)
        assert torch.equal(row_ptr, want)
        assert int(buf_ptr[shift + B + 1]) == -7 and (shift == 0 or int(buf_ptr[0]) == -7)   # nothing written outside


@gpu
def test_multimap_shards_equal_the_whole_batch():
    """A heterogeneous batch cut into rank shards (sharding.segment_shard) steps exactly like the whole batch: the Philox
    stream is keyed by the env's index in the global batch."""
    import torch
    from gym_mapf_b200 import sharding
    from gym_mapf_b200.envs.mapf_env import OptimizationCriteria
    from gym_mapf_b200.envs.utils import create_mapf_env
    from gym_mapf_b200.envs.vec_env import MultiMapVecEnv
    envs = [create_mapf_env("room-32-32-4", 1, 4, 0.2, -1000.0, 100.0, -1.0, OptimizationCriteria.SoC),
            create_mapf_env("maze-32-32-4", 10, 4, 0.3, -10.0, 5.0, -0.5, OptimizationCriteria.Makespan),
            create_mapf_env("empty-32-32", 2, 4, 0.2, -1000.0, 100.0, -1.0, OptimizationCriteria.SoC)]
    counts = [700, 45, 1303]
    whole = MultiMapVecEnv(envs, counts, seed=5)
    g = torch.Generator(device="cpu").manual_seed(2)
    acts = [torch.randint(0, 625, (sum(counts),), generator=g, dtype=torch.int32).cuda() for _ in range(4)]
    ref = [tuple(t.clone() for t in (lambda o: (o[0], o[1], o[2], o[3]["prob"], o[3]["collision"]))(whole.step(a))) for a in acts]
    for world in (2, 3):
        for rank in range(world):
            sh, parts = sharding.segment_shard(counts, world, rank)
            mm = MultiMapVecEnv([envs[i] for i, _ in parts], [c for _, c in parts], seed=5, env_offset=sh.begin)
            for a, want in zip(acts, ref):
                ns, r, d, info = mm.step(a[sh.begin:sh.begin + sh.count].contiguous())
                got = (ns, r, d, info["prob"], info["collision"])
                for x, y in zip(got, want):
                    assert torch.equal(x, y[sh.begin:sh.begin + sh.count])


@gpu
@pytest.mark.timeout(300)
def test_fuzz_group_and_step_kernels_every_agent_count():
    """Random small grids (obstacles, coinciding starts/goals, every noise level), 1..13 agents: groups of 2-4 random
    specs per agent count stepped in one launch must equal the C oracle per spec, and each spec's segment must equal
    mapf_step of that spec alone."""
    import torch
    from engine_util import make_engine, make_oracle, u64
    from gym_mapf_b200 import _native
    rng = np.random.default_rng(4711)

    def random_spec(n, H, W):
        while True:
            grid = rng.random((H, W)) < rng.choice([0.0, 0.15, 0.35])
            if (~grid).sum() >= 2:
                break
        free = [(r, c) for r in range(H) for c in range(W) if not grid[r, c]]
        pick = lambda: [list(free[int(rng.integers(0, len(free)))]) for _ in range(n)]  # noqa: E731
        return dict(rows=["".join("@" if v else "." for v in row) for row in grid], n_agents=n, starts=pick(), goals=pick(),
                    fail_prob=float(rng.choice([0.0, 0.1, 0.2, 0.37, 1.0])), r_clash=float(rng.choice([-1000.0, -3.5])),
                    r_goal=float(rng.choice([100.0, 7.25])), r_living=float(rng.choice([-1.0, -0.25, 0.0])),
                    soc=bool(rng.integers(0, 2)))

    for n in range(1, 14):
        for words in (1, 2):
            # grid sizes that give one-word (L**n < 2**63) or two-word states for this agent count
            specs = []
            for _ in range(40):
                H, W = (int(rng.integers(2, 7)), int(rng.integers(2, 7))) if words == 1 else (8, int(rng.integers(7, 9)))
                sp = random_spec(n, H, W)
                L = sum(row.count(".") for row in sp["rows"])
                if (L ** n < 2 ** 63) == (words == 1) and L ** n < 2 ** 127:
                    specs.append(sp)
                if len(specs) == 3:
                    break
            if len(specs) < 2:
                continue
            engines = [make_engine(sp) for sp in specs]
            assert all(e.words == words for e in engines)
            counts = [int(rng.integers(1, 700)) for _ in specs]
            group = _native.Group(engines, counts)
            B = sum(counts)
            lo, hi = np.zeros(B, np.uint64), np.zeros(B, np.uint64)
            act = rng.integers(0, 5 ** n, B).astype(np.int32)
            uni = rng.random((B, n))
            at = 0
            for sp, eng, c in zip(specs, engines, counts):
                cells = rng.integers(0, eng.L, (c, n)).astype(np.int32)
                lo[at:at + c], hi[at:at + c] = make_oracle(sp).encode(cells)
                at += c
            arr = lo.view(np.int64).copy() if words == 1 else np.stack([lo, hi], 1).view(np.int64).copy()
            states = torch.from_numpy(arr).cuda()
            actions, uniforms = torch.from_numpy(act).cuda(), torch.from_numpy(uni).cuda()
            out = group.step(states, actions, uniforms=uniforms)
            ns = out[0].cpu().numpy().view(np.uint64).reshape(B, -1)
            at = 0
            for sp, eng, c in zip(specs, engines, counts):
                sl = slice(at, at + c)
                w = make_oracle(sp).step(lo[sl], hi[sl], act[sl].astype(np.int64), uni[sl])
                assert np.array_equal(ns[sl, 0], w["next_lo"]), (n, words, sp)
                if words == 2:
                    assert np.array_equal(ns[sl, 1], w["next_hi"]), (n, words, sp)
                assert np.array_equal(u64(out[1][sl]), G.f64_to_bits(w["reward"])), (n, words, sp)
                assert np.array_equal(u64(out[2][sl]), G.f64_to_bits(w["prob"])), (n, words, sp)
                assert np.array_equal(out[3][sl].cpu().numpy().astype(np.uint8), w["done"])
                assert np.array_equal(out[4][sl].cpu().numpy().astype(np.uint8), w["collision"])
                one = eng.step(states[sl].clone(), actions[sl].clone(), uniforms=uniforms[sl].clone())
                for x, y in zip(one, out):
                    assert torch.equal(x, y[sl]), (n, sp)
                at += c
            group.close()
            for e in engines:
                e.close()
