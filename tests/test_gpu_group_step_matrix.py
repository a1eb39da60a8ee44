"""The grouped step kernel k_step_group<N, W, TAPE> (mapf_group_step, _native.Group, MultiMapVecEnv) in every
instantiation against the C oracle.

A group needs staged move tables, so its kernels exist for the staged cells of test_gpu_kernel_matrix.py: W = 1 with
N = 1..13 and W = 2 with N = 6..13, 21 cells, each with a replayed-draw (TAPE) and a Philox variant.  Every cell gets
four specs of its agent count and state width: three with distinct L, the fourth with a terminal start state (every
agent on its goal, or two agents on one cell).  Their slip probabilities cycle through 0.2, 0 (one outcome), 1 (two
outcomes) and 0.5, and their criteria and rewards differ, so a segment that ran with its neighbour's staged tables or
DevSpec would step differently.  `test_group_cells_have_the_intended_shape` checks all of this on the host.

What the kernel does beyond k_step is where it could go wrong unnoticed: at each segment change it re-stages the spec's
shared-memory image and DevSpec behind an mbarrier whose phase flips, it finds a CTA's first segment by a binary search
that has to skip empty segments, and it keys the Philox stream by the env's index in the whole batch.  So each cell
runs these layouts (segment i is spec i % 4; a context may appear in a group more than once):
    ragged   [2049, 0, 1, 33, 31, 517]: empty and one-env segments, boundaries off the 32-env chunks, several segments
             inside one CTA, a segment over three CTAs
    full     311 297 envs over five segments: more than one round of the largest grid a group launch can have (two
             512-thread CTAs on each of 148 SMs take 303 104 envs per round), so the grid is full and segments span CTAs
    many     24 segments of 0, 1, 2, 31, 32, 33 or 517 envs, the first and last empty
    empty    every count 0: the step returns OK and writes nothing
in both variants, auto-reset on and off.  The uniforms of the TAPE variant are salted with each spec's exact
cumulative probabilities, their neighbours (np.nextafter) and 0.0 and 1 - 2**-53, where `cumsum > u` decides the
outcome; the Philox words are regenerated on the host at the env's global index.  Step indices are at and around 2**32,
env offsets are >= 2**32 and the low word of the env index wraps inside a segment.  Every env must equal
`make_oracle(spec).step` of its own spec bit for bit, and every segment must equal `Engine.step` of its spec alone at
env_offset + the segment's start.

Also: the outputs are carved from canary-padded buffers (the configurations of test_gpu_guard_bands.py, split over three
segments); mapf_group_step refuses every option but MAPF_OPT_AUTO_RESET before it launches anything (its stores are the
default layout: a compact-sized reward buffer would be overrun); mapf_group_create refuses 2**31 envs or more and
negative counts; and MultiMapVecEnv, interleaving staged and unstaged specs and two agent counts, equals the oracle
driven by the host Philox stream over five steps with auto-reset."""
import math

import numpy as np
import pytest

from engine_util import make_engine, make_oracle, states_tensor
from test_formats import _shipped_spec
from test_gpu_evaluate import env_of
from test_gpu_guard_bands import CANARY, SIZES, SPECS, Guarded, _env
from test_gpu_kernel_matrix import (CELLS, SEED, assert_step_equal, cell_id, cell_ids, cell_spec, philox_uniforms,
                                    reset_to_s0, staged_by_rule, state_batch, words_of)

GROUP_CELLS = [c for c in CELLS if c[2]]
# (r_clash, r_goal, r_living) of a cell's specs 0..3
REWARDS = ((-1000.0, 100.0, -1.5), (-7.25, 3.5, -0.125), (-50.0, 10.0, 0.0), (-1.0, 1.0, -2.0))


def spec_sizes(c):
    """Three distinct L of cell c: below the cell's L for one-word states (L**N stays < 2**63), above it for two-word
    states (L**N stays >= 2**63; every one is far below the staging limit)."""
    n, w, _, L = c
    return (L, L - 4, L - 10) if w == 1 else (L, L * 4 // 3, L * 5 // 3)


def group_specs(c):
    """The four specs of cell c: spec k has fail_prob [0.2, 0, 1, 0.5][k], rewards REWARDS[k] and the criterion of
    cell_spec; spec 3 starts in a terminal state."""
    n = c[0]
    sizes = spec_sizes(c)
    out = []
    for k in range(4):
        terminal = None if k < 3 else ("goal" if n == 1 or GROUP_CELLS.index(c) % 2 else "shared")
        sp = cell_spec(n, sizes[k] if k < 3 else sizes[1], k, terminal)
        sp["r_clash"], sp["r_goal"], sp["r_living"] = REWARDS[k]
        out.append(sp)
    return out


def free_cells(spec):
    return sum(row.count(".") for row in spec["rows"])


def start_is_terminal(spec, ora):
    ids = cell_ids(spec)
    lo, hi = ora.encode(np.array([[ids[tuple(rc)] for rc in spec["starts"]]], np.int32))
    return bool(ora.step(lo, hi, np.zeros(1, np.int64), np.full((1, spec["n_agents"]), 0.5))["terminal"][0])


def test_group_cells_have_the_intended_shape():
    limit = {n: max(L for L in range(1, 6000) if staged_by_rule(n, L)) for n in range(1, 14)}
    reach = {(n, 1) for n in range(1, 14)} | {(n, 2) for n in range(1, 14)
                                              if 65535 ** n >= 2 ** 63 and limit[n] >= math.ceil(2 ** (63 / n))}
    assert sorted((c[0], c[1]) for c in GROUP_CELLS) == sorted(reach) and len(GROUP_CELLS) == 21
    for c in GROUP_CELLS:
        n, w = c[0], c[1]
        specs = group_specs(c)
        assert len({free_cells(sp) for sp in specs}) == 3, c
        assert [sp["fail_prob"] for sp in specs] == [0.2, 0.0, 1.0, 0.5]
        assert {sp["soc"] for sp in specs} == {True, False}
        assert len({(sp["r_clash"], sp["r_goal"], sp["r_living"]) for sp in specs}) == 4
        terminal = []
        for sp in specs:
            L = free_cells(sp)
            assert sp["n_agents"] == n and words_of(n, L) == w and staged_by_rule(n, L) and L ** n < 2 ** 127, (c, L)
            ora = make_oracle(sp)
            assert ora.L == L
            terminal.append(start_is_terminal(sp, ora))
        assert terminal == [False, False, False, True], c


# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


def boundary_uniforms(ora):
    """Every cumulative probability `cumsum > u` compares against in this spec (summed left to right as the oracle
    does), its two fp64 neighbours, 0.0 and 1 - 2**-53: the draws in [0, 1) where an off-by-one ulp flips the outcome."""
    k, _, prob = ora.moves()
    vals = {0.0, 1.0 - 2.0 ** -53}
    acc = None
    for j in range(3):
        acc = prob[:, :, 0] if j == 0 else acc + prob[:, :, j]
        for v in np.unique(acc[k > j]):
            vals |= {float(v), float(np.nextafter(v, 0.0)), float(np.nextafter(v, 2.0))}
    return np.array(sorted(v for v in vals if 0.0 <= v < 1.0))


class Member:
    """One spec of a group with its engine and oracle; shaped like test_gpu_kernel_matrix.Cell for state_batch."""

    def __init__(self, spec):
        self.spec, self.n = spec, spec["n_agents"]
        self.eng, self.ora = make_engine(spec), make_oracle(spec)
        self.L = self.ora.L
        self.edges = boundary_uniforms(self.ora)


def segments(counts):
    at = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    return [(i, int(at[i]), int(at[i + 1])) for i in range(len(counts))]


# (name, spec of each segment, counts, step index, env offset)
LAYOUTS = (("ragged", [0, 1, 2, 3, 0, 1], [2049, 0, 1, 33, 31, 517], (1 << 32) - 1, (3 << 32) - 700),
           ("full", [0, 1, 2, 3, 0], [150001, 1, 0, 65536, 95759], 1 << 32, (5 << 32) - 200000))


def many_segments(rng):
    counts = rng.choice([0, 1, 2, 31, 32, 33, 517], 24)
    counts[0] = counts[-1] = 0
    return ("many", [k % 4 for k in range(24)], [int(x) for x in counts], (1 << 32) + 7, (1 << 32) + 3)


def run_layout(torch, members, layout, rng):
    from gym_mapf_b200._native import Group
    name, order, counts, step, env0 = layout
    n = members[0].n
    eng0 = members[0].eng
    dev = eng0.torch_device
    group = Group([members[k].eng for k in order], counts)
    B = sum(counts)
    assert group.size == B
    segs = [(members[order[i]], a, b) for i, a, b in segments(counts) if b > a]
    lo, hi = np.zeros(B, np.uint64), np.zeros(B, np.uint64)
    act = np.zeros(B, np.int64)
    tape = rng.random((B, n))
    for m, a, b in segs:
        lo[a:b], hi[a:b] = state_batch(m, b - a, rng)
        act[a:b] = rng.integers(0, m.eng.nA, b - a)
        salt = rng.random((b - a, n)) < 0.3
        tape[a:b][salt] = rng.choice(m.edges, int(salt.sum()))
    st = states_tensor(eng0, lo, hi)
    at = torch.from_numpy(act.astype(np.int32)).to(dev)
    env = np.arange(B, dtype=np.uint64) + np.uint64(env0)
    for given in (True, False):
        uni = tape if given else philox_uniforms(SEED, env, step, n)
        want = [m.ora.step(lo[a:b], hi[a:b], act[a:b], uni[a:b], threads=8) for m, a, b in segs]
        ut = torch.from_numpy(tape).to(dev) if given else None
        for auto_reset in (False, True):
            what = (name, "tape" if given else "philox", auto_reset)
            got = group.step(st, at, uniforms=ut, seed=SEED, step_index=step, env_offset=env0, auto_reset=auto_reset)
            host = tuple(x.cpu() for x in got)
            for (m, a, b), w in zip(segs, want):
                assert_step_equal(torch, m.eng, w, tuple(x[a:b] for x in host), auto_reset, what + (a, b))
                one = m.eng.step(st[a:b], at[a:b], uniforms=None if ut is None else ut[a:b], seed=SEED,
                                 step_index=step, env_offset=env0 + a, auto_reset=auto_reset)
                assert all(torch.equal(x, y[a:b]) for x, y in zip(one, got)), what + (a, b, "Engine.step")
    group.close()


@pytest.mark.timeout(600)
@pytest.mark.parametrize("c", [pytest.param(c, id=cell_id(c), marks=pytest.mark.gpu) for c in GROUP_CELLS])
def test_group_step_matches_oracle(c, torch):
    from gym_mapf_b200._native import Group
    members = [Member(sp) for sp in group_specs(c)]
    try:
        e = members[0].eng
        assert all((m.eng.n, m.eng.words, m.eng.moves_in_smem) == (c[0], c[1], True) for m in members)
        rng = np.random.default_rng(c[0] * 100 + c[3])
        for layout in LAYOUTS + (many_segments(rng),):
            run_layout(torch, members, layout, rng)
        # a group of empty segments: OK, and nothing written
        group = Group([m.eng for m in members], [0, 0, 0, 0])
        assert group.size == 0
        g = Guarded(torch)
        st = e.new_states(0)
        at = torch.zeros(0, dtype=torch.int32, device=e.torch_device)
        for ut in (None, torch.zeros((0, c[0]), dtype=torch.float64, device=e.torch_device)):
            out = (g.new(e.state_shape(0), torch.int64), g.new(0, torch.float64), g.new(0, torch.float64),
                   g.new(0, torch.bool), g.new(0, torch.bool))
            group.step(st, at, uniforms=ut, seed=SEED, auto_reset=True, out=out)
            g.check("empty group, tape=%s" % (ut is not None))
        group.close()
    finally:
        for m in members:
            m.eng.close()


# ---- memory safety ----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("spec", SPECS, ids=lambda s: "%s-%d" % (s[0], s[2]))
def test_group_step_writes_only_its_outputs(spec, torch):
    """Three scenarios of the map (1, 13 and 25: some others put an agent on an obstacle) as three segments, split
    unevenly (an empty first segment at B = 1 and 2)."""
    from gym_mapf_b200._native import Group
    name, scen, n, soc = spec
    engines = [_env(name, scen + k, n, soc).engine for k in (0, 12, 24)]
    assert all(e.moves_in_smem and e.words == engines[0].words for e in engines)
    g = Guarded(torch)
    rng = np.random.default_rng(9)
    for B in SIZES:
        counts = [B // 3, B - B // 3 - B // 2, B // 2]
        group = Group(engines, counts)
        st = torch.cat([e.encode(torch.from_numpy(rng.integers(0, min(e.L, 50), (k, n)).astype(np.int32)).cuda())
                        for e, k in zip(engines, counts) if k])
        ac = torch.from_numpy(rng.integers(0, engines[0].nA, B).astype(np.int32)).cuda()
        un = torch.from_numpy(rng.random((B, n))).cuda()
        for uniforms in (None, un):
            out = (g.new(engines[0].state_shape(B), torch.int64), g.new(B, torch.float64), g.new(B, torch.float64),
                   g.new(B, torch.bool), g.new(B, torch.bool))
            group.step(st, ac, uniforms=uniforms, seed=1, step_index=2, auto_reset=True, out=out)
            g.check("group step B=%d %s tape=%s" % (B, counts, uniforms is not None))
        group.close()


@pytest.mark.gpu
def test_group_refuses_what_it_cannot_do(torch):
    """mapf_group_step with any option but MAPF_OPT_AUTO_RESET (the compact layout would get 8-byte rewards in a
    one-byte-per-env buffer) fails before it launches: every byte of the outputs keeps its canary.  mapf_group_create
    refuses groups of 2**31 envs or more (a host check: nothing is allocated for the envs) and negative counts."""
    from gym_mapf_b200._native import (MAPF_ERR_INVALID, MAPF_ERR_UNSUPPORTED, OPT_AUTO_RESET, OPT_COMPACT,
                                       OPT_SHARE_SM, Group, NativeError, _ptr, lib)
    c = GROUP_CELLS[3]
    engines = [make_engine(sp) for sp in group_specs(c)[:2]]
    e, n, dev = engines[0], c[0], engines[0].torch_device
    rng = np.random.default_rng(11)
    stream = torch.cuda.current_stream().cuda_stream
    for counts in ([1000, 1049], [0, 0]):
        group = Group(engines, counts)
        B = group.size
        st = e.states_from_ints([e.s0] * B) if B else e.new_states(0)
        at = torch.from_numpy(rng.integers(0, e.nA, B).astype(np.int32)).to(dev)
        un = torch.from_numpy(rng.random((B, n))).to(dev)
        g = Guarded(torch)
        for opts in (OPT_COMPACT, OPT_COMPACT | OPT_AUTO_RESET, OPT_SHARE_SM, OPT_SHARE_SM | OPT_AUTO_RESET, 8, 1 << 31):
            for uniforms in (None, un):
                narrow = torch.uint8 if opts & OPT_COMPACT else torch.float64  # the compact layout's reward codes
                out = (g.new(e.state_shape(B), torch.int64), g.new(B, narrow), g.new(B, torch.float64),
                       g.new(B, torch.uint8), g.new(B, torch.uint8))
                rc = lib().mapf_group_step(group._h, _ptr(st), _ptr(at), _ptr(uniforms), SEED, 3, 0, opts,
                                           *[_ptr(t) for t in out], stream)
                assert rc == MAPF_ERR_UNSUPPORTED, (counts, opts)
                assert "MAPF_OPT_AUTO_RESET" in lib().mapf_last_error().decode()
                torch.cuda.synchronize()
                assert all(bool((buf == CANARY).all()) for buf, _ in g.raw), (counts, opts)
                g.check("refused options %#x" % opts)
        group.close()
    for counts, code in (([2 ** 30, 2 ** 30], MAPF_ERR_UNSUPPORTED), ([2 ** 31 - 1, 1], MAPF_ERR_UNSUPPORTED),
                         ([-1, 5], MAPF_ERR_INVALID), ([5, -1], MAPF_ERR_INVALID)):
        with pytest.raises(NativeError) as ei:
            Group(engines, counts)
        assert ei.value.code == code, counts
    largest = Group(engines, [2 ** 31 - 2, 1])  # 2**31 - 1 envs: the largest group, never stepped here
    assert largest.size == 2 ** 31 - 1
    largest.close()
    for eng in engines:
        eng.close()


# ---- MultiMapVecEnv ---------------------------------------------------------------------------------------------------
def multimap_specs(words):
    """A staged spec, an unstaged one of the same agent count (it steps alone), another staged one, then a class of a
    larger agent count (two specs, the second with a terminal start).  The slip probabilities of the staged specs are
    0.2, 1 and 0.2, so their draws decide outcomes."""
    if words == 1:
        a, b = group_specs(GROUP_CELLS[1]), group_specs(GROUP_CELLS[3])  # 2 and 4 agents
        unstaged = _shipped_spec("Berlin_1_256", 11, 2, 0.2, -1000.0, 100.0, -1.0, True)
    else:
        a, b = group_specs(GROUP_CELLS[13]), group_specs(GROUP_CELLS[14])  # 6 and 7 agents, two-word states
        unstaged = cell_spec(6, 5000, 1)
    return [a[0], unstaged, a[2], b[0], b[3]]


@pytest.mark.gpu
@pytest.mark.parametrize("words", [1, 2])
def test_multimap_vec_env_matches_oracle(words, torch):
    from gym_mapf_b200.envs.vec_env import MultiMapVecEnv
    specs = multimap_specs(words)
    envs = [env_of(sp) for sp in specs]
    engines = [env.engine for env in envs]
    assert [e.moves_in_smem for e in engines] == [True, False, True, True, True]
    assert {e.words for e in engines} == {words}
    oracles = [make_oracle(sp) for sp in specs]
    counts = [2500, 257, 33, 3001, 1]  # the first and last group span several CTAs
    mm = MultiMapVecEnv(envs, counts, seed=SEED, auto_reset=True, env_offset=(1 << 32) + 5)
    assert [type(p[2]).__name__ for p in mm._parts] == ["Group", "Engine", "Group", "Group"]
    mm.step_count = (1 << 32) - 2  # the step index crosses 2**32
    segs = segments(counts)
    lo, hi = np.zeros(mm.num_envs, np.uint64), np.zeros(mm.num_envs, np.uint64)
    for i, a, b in segs:
        lo[a:b], hi[a:b] = np.uint64(engines[i].s0 & ((1 << 64) - 1)), np.uint64(engines[i].s0 >> 64)
    rng = np.random.default_rng(13 + words)
    resets = 0
    for t in range(5):
        act = np.concatenate([rng.integers(0, engines[i].nA, b - a) for i, a, b in segs])
        step = mm.step_count
        ns, r, d, info = mm.step(torch.from_numpy(act.astype(np.int32)).to(mm.device))
        got = tuple(x.cpu() for x in (ns, r, info["prob"], d, info["collision"]))
        for i, a, b in segs:
            env = np.arange(a, b, dtype=np.uint64) + np.uint64(mm.env_offset)
            w = oracles[i].step(lo[a:b], hi[a:b], act[a:b], philox_uniforms(SEED, env, step, engines[i].n))
            assert_step_equal(torch, engines[i], w, tuple(x[a:b] for x in got), True, (words, t, i))
            lo[a:b], hi[a:b] = reset_to_s0(engines[i], w, True)
            resets += int(w["done"][w["terminal"] == 0].sum())
    assert resets > 0
