"""Every shipped kernel instantiation against the C oracle, cell by cell.

The library compiles its hot kernels once per agent count N (1..13), state width W (1 or 2 words) and move-table
placement (staged in shared memory, or read through __ldg).  The context stages the table when L**4 < 2**50 and
MAPF_SMEM_LUT + 40 L (padded to 16) + 16 sizeof(BackupSlab<N>) fits the opt-in shared memory (232 448 B on a B200,
so L <= (198 672 - 5120 N) / 40: 4838 cells at N = 1, 3302 at N = 13); the L**4 bound never binds first.  A state
takes two words when L**N >= 2**63.  That makes these cells reachable:

    placement  W  N      L used here                          why this L
    staged     1  1..12  34 (6 x 6, two obstacles)            L**N < 2**63 up to N = 12
    staged     1  13     24 (5 x 5, one obstacle)             34**13 >= 2**63
    staged     2  6..13  1500, 520, 240, 130, 80, 54, 40, 30  ceil(2**(63/N)) <= L <= the staging limit
    unstaged   1  1..5   5000                                 above the staging limit, 5000**5 < 2**63
    unstaged   2  4      60000                                L**4 >= 2**63 needs L >= 55 109
    unstaged   2  5      6400                                 L**5 >= 2**63 needs L >= 6208
    unstaged   2  6..10  5000                                 above the staging limit, L**N < 2**127

and leaves these unreachable:
    W = 2 with N <= 3            65535**3 < 2**63
    staged W = 2 with N = 4, 5   the staging limit (4454 / 4326 cells) is below 2**(63/N) (55 109 / 6208)
    unstaged W = 1 with N >= 6   above the staging limit L**N >= 2**63
    unstaged with N >= 11        above the staging limit L**N >= 2**127, which no context accepts
No L below 6000 needs the divisor fix-up (Div32::fix), so that condition of the staging rule never decides a cell.
`test_cells_have_the_intended_shape` checks this table on the host; `test_device_picks_the_intended_kernels` checks
`words` and `moves_in_smem` as the device reports them for every spec built here.

Each cell's spec is a lightly obstructed rectangle with the agents' starts and goals drawn from a small window in its
corner, so vertex and swap clashes are frequent.  fail_prob cycles through 0.2, 0 (one outcome), 1 (two outcomes) and
0.5, the criterion alternates between sum-of-costs and makespan.  Every cell also has a twin whose start state is
terminal (every agent on its goal, or two agents on one cell).

In every cell: step (Philox draws regenerated on the host, given uniforms, one and two envs per thread, compact
results, auto-reset, shared-SM launches and the device-resident host step), rollout (all instantiated variants,
auto-reset on and off, starts from s0, random, conflict-dense, goal and terminal states), evaluate (random and per-agent
policies, joint-state policies where W = 1 and nS <= 2**26, and group policies with their conflict bytes: singletons,
equal to the per-agent kind on the same table; agents dealt round-robin into groups of up to four; {0, N-1} plus
singletons; one group of every agent where the joint table fits, equal to the joint kind on the same table), the table
path (transitions, checksum; table_range on a slab up to N = 6, where a slab of 5**N actions stays small), encode /
decode / project and predecessors (up to N = 8: a state has up to 5**N predecessors).  Step indices cross 2**32 and env
offsets are >= 2**32.

Backup / greedy need one-word states and V of nS doubles, so they run on their own specs: staged N = 1..9 with small
grids (N = 9 on nine cells: nS = 9**9, V = 3.1 GB, rows of permutation states, more batches than warps so a warp's
head cache meets a second batch), unstaged N = 1, 2 on 5000 cells, and staged N = 10..13 on four cells, where L < N
puts two agents on one cell in every state: every row there is terminal.  The staged N = 8 and 9 specs also run one
group of every agent (tables of 9**8 and 9**9 entries): the device then takes digits 0..8 of a group's entry.  Digits
9..12 would need a group of 10 or more agents with L >= 10 (10**10 entries); the host check of the digit arithmetic in
test_groups_host.py covers them."""
import math

import numpy as np
import pytest

import golden_util as G
from engine_util import assert_rows_equal, make_engine, make_oracle, split_states, states_tensor, u64
from test_gpu_evaluate import Episodes, kinds, philox_words

M64 = (1 << 64) - 1
SMEM_OPTIN = 232448  # cudaDevAttrMaxSharedMemoryPerBlockOptin of a B200
SMEM_LUT, BACKUP_WARPS = 6128, 16  # MAPF_SMEM_LUT; 512-thread CTAs when staged


def backup_slab_bytes(n):
    # sizeof(BackupSlab<N>): ExpandSlab<N> (ent, st, rcp, pref, prev, 4 pair lists, parked, flag) + 32 doubles
    return 256 * n + 512 + 256 + 128 + 64 * n + 512 + 32 + 32 + 256


def div_needs_fix(d):
    """Div32::fix of make_div32 (mapf_capi.cu): no exact round-up magic for two-digit chunks."""
    if d <= 1:
        return False
    xmax = d * d - 1
    for s in range(32, 64):
        m = ((1 << s) + d - 1) // d
        if m >> 32:
            break
        if (m * d - (1 << s)) * xmax < (1 << s):
            return False
    return True


def staged_by_rule(n, L):
    lut_pad = (40 * L + 15) // 16 * 16
    return (not div_needs_fix(L) and L ** 4 < 2 ** 50
            and SMEM_LUT + lut_pad + BACKUP_WARPS * backup_slab_bytes(n) <= SMEM_OPTIN)


def words_of(n, L):
    return 1 if L ** n < 2 ** 63 else 2


STAGED_W2_L = {6: 1500, 7: 520, 8: 240, 9: 130, 10: 80, 11: 54, 12: 40, 13: 30}
CELLS = ([(n, 1, True, 34 if n <= 12 else 24) for n in range(1, 14)]
         + [(n, 2, True, STAGED_W2_L[n]) for n in range(6, 14)]
         + [(n, 1, False, 5000) for n in range(1, 6)]
         + [(4, 2, False, 60000), (5, 2, False, 6400)] + [(n, 2, False, 5000) for n in range(6, 11)])
BACKUP_L = {1: 34, 2: 34, 3: 34, 4: 34, 5: 24, 6: 12, 7: 10, 8: 9, 9: 9, 10: 4, 11: 4, 12: 4, 13: 4}
BACKUP_CELLS = [(n, 1, True, BACKUP_L[n]) for n in range(1, 14)] + [(1, 1, False, 5000), (2, 1, False, 5000)]


def cell_id(c):
    return "n%d_w%d_%s_L%d" % (c[0], c[1], "staged" if c[2] else "ldg", c[3])


def grid_rows(L):
    """A rectangle of exactly L free cells: one obstacle inside the agents' window when there is room, the surplus
    cells of the last row blocked."""
    w = max(1, math.isqrt(L - 1) + 1) if L > 1 else 1
    interior = 1 if w >= 5 else 0
    h = -(-(L + interior) // w)
    trim = h * w - interior - L
    cells = [["."] * w for _ in range(h)]
    if interior:
        cells[1][2] = "@"
    for k in range(trim):
        cells[h - 1][w - 1 - k] = "@"
    return ["".join(r) for r in cells]


def cell_spec(n, L, index, terminal=None):
    rows = grid_rows(L)
    rng = np.random.default_rng(1000 * n + L)
    k = min(len(rows[0]), len(rows), max(3, math.isqrt(2 * n) + 2))
    window = [(r, c) for r in range(k) for c in range(k) if rows[r][c] == "."]
    distinct = len(window) >= n
    starts = [window[i] for i in rng.choice(len(window), n, replace=not distinct)]
    goals = [window[i] for i in rng.choice(len(window), n, replace=not distinct)]
    if terminal == "goal":
        starts = list(goals)
    elif terminal == "shared":
        starts[-1] = starts[0]
    return dict(rows=rows, n_agents=n, starts=[list(s) for s in starts], goals=[list(g) for g in goals],
                fail_prob=[0.2, 0.0, 1.0, 0.5][index % 4], r_clash=-1000.0, r_goal=100.0, r_living=-1.5,
                soc=index % 3 != 0)


def cell_ids(spec):
    """(row, col) -> cell id: free cells numbered column by column, as the engine and the oracle number them."""
    rows = spec["rows"]
    free = [(r, c) for c in range(len(rows[0])) for r in range(len(rows)) if rows[r][c] == "."]
    return {rc: i for i, rc in enumerate(free)}


def window_ids(spec, k):
    """Cell ids of the k x k corner window."""
    ids = cell_ids(spec)
    return np.array([ids[(r, c)] for r in range(k) for c in range(k) if (r, c) in ids], np.int64)


def test_cells_have_the_intended_shape():
    reach = {(n, w, s) for n in range(1, 14) for w in (1, 2) for s in (True, False)}
    limit = {n: max(L for L in range(1, 6000) if staged_by_rule(n, L)) for n in range(1, 14)}
    unreachable = set()
    for n in range(1, 14):
        if 65535 ** n < 2 ** 63:
            unreachable.add((n, 2, True)), unreachable.add((n, 2, False))
        if limit[n] < math.ceil(2 ** (63 / n)):
            unreachable.add((n, 2, True))
        if (limit[n] + 1) ** n >= 2 ** 63:
            unreachable.add((n, 1, False))
        if (limit[n] + 1) ** n >= 2 ** 127:
            unreachable.add((n, 2, False))
    assert not any(div_needs_fix(L) for L in range(1, 6000))
    assert sorted((c[0], c[1], c[2]) for c in CELLS) == sorted(reach - unreachable)
    assert limit[1] == 4838 and limit[13] == 3302 and len(CELLS) == 33
    for i, (n, w, staged, L) in enumerate(CELLS + BACKUP_CELLS):
        for terminal in (None, "goal", "shared"):
            spec = cell_spec(n, L, i, terminal)
            assert sum(row.count(".") for row in spec["rows"]) == L
            assert words_of(n, L) == w and staged_by_rule(n, L) == staged, (n, w, staged, L)
            assert make_oracle(spec).L == L
    for n, w, staged, L in BACKUP_CELLS:  # V of nS doubles; N >= 10 only through terminal rows
        assert L ** n <= 9 ** 9 and (n < 10 or L < n)


# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


class Cell:
    def __init__(self, c, index, terminal=None):
        self.n, self.w, self.staged, self.L = c
        self.spec = cell_spec(self.n, self.L, index, terminal)
        self.eng = make_engine(self.spec)
        self.ora = make_oracle(self.spec)


@pytest.fixture(scope="module")
def cells(torch):
    made = {}

    def get(c, terminal=None):
        key = (c, terminal)
        if key not in made:
            made[key] = Cell(c, (CELLS + BACKUP_CELLS).index(c), terminal)
        return made[key]
    yield get
    for cell in made.values():
        cell.eng.close()


def philox_uniforms(seed, env, step, n):
    u = np.zeros((len(env), n))
    for b in range((n + 3) // 4):
        words = philox_words(seed, env, step, b)
        for q in range(4):
            if 4 * b + q < n:
                u[:, 4 * b + q] = words[q].astype(np.float64) * 2.0 ** -32
    return u


def philox_actions(seed, env, step, nA):
    """k_rollout's random action: umul64hi(w0 << 32 | w1, nA) of Philox block 15."""
    w = philox_words(seed, env, step, 15)
    nA = np.uint64(nA)
    return ((w[0] * nA + ((w[1] * nA) >> np.uint64(32))) >> np.uint64(32)).astype(np.int64)


def state_batch(cell, B, rng):
    """s0, the goal state, terminal states (two agents on one cell), conflict-dense states from the start window and
    uniformly random states, shuffled."""
    n, L, ora = cell.n, cell.L, cell.ora
    k = min(len(cell.spec["rows"][0]), max(3, math.isqrt(2 * n) + 2))
    win = window_ids(cell.spec, k)
    # agents on distinct cells where the grid allows it, so that most rows are not terminal
    ids = rng.integers(0, L, (B, n)) if L > 64 or L < n else np.argsort(rng.random((B, L)), 1)[:, :n]
    dense = rng.random(B) < 0.45
    nd = int(dense.sum())
    ids[dense] = (win[np.argsort(rng.random((nd, len(win))), 1)[:, :n]] if len(win) >= n
                  else win[rng.integers(0, len(win), (nd, n))])
    if n >= 2:
        shared = rng.random(B) < 0.1
        ids[shared, 1] = ids[shared, 0]
    lo, hi = ora.encode(ids)
    e = cell.eng
    pick = rng.random(B)
    lo = np.where(pick < 0.1, np.uint64(e.s0 & M64), np.where(pick > 0.93, np.uint64(e.goal_state & M64), lo))
    hi = np.where(pick < 0.1, np.uint64(e.s0 >> 64), np.where(pick > 0.93, np.uint64(e.goal_state >> 64), hi))
    return lo, hi


def split_s0(eng):
    return np.uint64(eng.s0 & M64), np.uint64(eng.s0 >> 64)


def reset_to_s0(eng, w, auto_reset):
    lo, hi = w["next_lo"], w["next_hi"]
    if auto_reset:
        s0_lo, s0_hi = split_s0(eng)
        lo = np.where(w["done"] == 1, s0_lo, lo)
        hi = np.where(w["done"] == 1, s0_hi, hi)
    return lo, hi


def bytes_of(torch, t):
    t = t.detach().cpu()
    return (t.view(torch.uint8) if t.dtype == torch.bool else t).numpy()


def assert_step_equal(torch, eng, w, got, auto_reset, what):
    ns, reward, prob, done, coll = got
    lo, hi = reset_to_s0(eng, w, auto_reset)
    glo, ghi = split_states(eng, ns)
    assert np.array_equal(glo, lo) and np.array_equal(ghi, hi), what
    assert np.array_equal(u64(reward), G.f64_to_bits(w["reward"])), what
    assert np.array_equal(u64(prob), G.f64_to_bits(w["prob"])), what
    assert np.array_equal(bytes_of(torch, done), w["done"]) and np.array_equal(bytes_of(torch, coll), w["collision"]), what


def decode_compact(eng, code, flags):
    code, flags = np.asarray(code), np.asarray(flags)
    assert not np.any(flags & ~np.uint8(3))
    return eng.reward_table()[code], flags & 1, (flags >> 1) & 1


def offset_view(torch, t, offset):
    """`t` itself, or a copy of it that starts one element into a larger buffer (breaks 16-byte alignment of narrow
    element types; two-word states stay aligned, their actions and outputs do not)."""
    if not offset:
        return t
    flat = torch.empty(t.numel() + t[0].numel(), dtype=t.dtype, device=t.device)
    v = flat[t[0].numel():].view(t.shape)
    v.copy_(t)
    return v


SEED = 0x9E3779B97F4A7C15
# seeds of the group-policy tables that give every partition of these cells a collision episode (the default, 1, does
# elsewhere)
GROUP_SEEDS = {(2, 1, True, 34): 250, (3, 1, True, 34): 2, (5, 1, False, 5000): 6}
GPU_CELLS = [pytest.param(c, id=cell_id(c), marks=pytest.mark.gpu) for c in CELLS]


@pytest.mark.parametrize("c", GPU_CELLS)
def test_device_picks_the_intended_kernels(c, cells):
    for terminal in (None, "goal", "shared"):
        cell = cells(c, terminal)
        e = cell.eng
        assert (e.n, e.L, e.words, e.moves_in_smem) == (cell.n, cell.L, cell.w, cell.staged)
        # the engine numbers cells as cell_ids() assumes
        for key, want in (("starts", e.s0), ("goals", e.goal_state)):
            ids = np.array([[cell_ids(cell.spec)[tuple(rc)] for rc in cell.spec[key]]], np.int32)
            lo, hi = cell.ora.encode(ids)
            assert G.big(lo[0], hi[0]) == want



# ---- step -------------------------------------------------------------------------------------------------------------
# (B, offset view, given uniforms, compact, auto_reset, share_sm)
STEP_CASES = [(2048, 0, False, False, False, False), (2047, 0, False, False, False, False),
              (2048, 1, False, False, False, False), (2048, 0, True, False, False, False),
              (2047, 1, True, False, True, False), (2048, 0, False, True, True, False),
              (2047, 0, True, True, False, False), (2048, 1, False, True, False, True),
              (2048, 0, False, False, True, True), (1, 0, False, False, True, False)]


@pytest.mark.timeout(300)
@pytest.mark.parametrize("c", GPU_CELLS)
def test_step_matches_oracle(c, cells, torch):
    cell = cells(c)
    eng, ora, n = cell.eng, cell.ora, cell.n
    rng = np.random.default_rng(cell.L * 31 + n)
    dev = eng.torch_device
    for k, (B, off, tape, compact, auto_reset, share_sm) in enumerate(STEP_CASES):
        lo, hi = state_batch(cell, B, rng)
        act = rng.integers(0, eng.nA, B)
        step, env0 = (1 << 32) - 5 + 2 * k, (1 << 32) + 977 * k
        env = np.arange(B, dtype=np.uint64) + np.uint64(env0)
        uni = rng.random((B, n)) if tape else philox_uniforms(SEED, env, step, n)
        w = ora.step(lo, hi, act, uni)
        st = offset_view(torch, states_tensor(eng, lo, hi), off)
        at = offset_view(torch, torch.from_numpy(act.astype(np.int32)).to(dev), off)
        ut = offset_view(torch, torch.from_numpy(uni).to(dev), off) if tape else None
        what = (cell_id(c), k)
        got = eng.step(st, at, uniforms=ut, seed=SEED, step_index=step, env_offset=env0, auto_reset=auto_reset,
                       share_sm=share_sm, compact=compact)
        if compact:
            ns, code, prob, flags = got
            r, d, co = decode_compact(eng, code.cpu().numpy(), flags.cpu().numpy())
            got = (ns, torch.from_numpy(r), prob, torch.from_numpy(d), torch.from_numpy(co))
        assert_step_equal(torch, eng, w, got, auto_reset, what)
        # the same step with the states resident on the device and the results in host memory (the KEEP kernels)
        ds = states_tensor(eng, lo, hi)
        shape = (B,) if eng.words == 1 else (B, 2)
        hns, hp = np.zeros(shape, np.int64), np.zeros(B)
        if compact:
            hc, hf = np.zeros(B, np.uint8), np.zeros(B, np.uint8)
            eng.step_host_resident(ds, act.astype(np.int32), (hns, hc, hp, hf), uniforms=uni if tape else None,
                                   seed=SEED, step_index=step, env_offset=env0, auto_reset=auto_reset, compact=True)
            r, d, co = decode_compact(eng, hc, hf)
        else:
            hr, d, co = np.zeros(B), np.zeros(B, np.uint8), np.zeros(B, np.uint8)
            eng.step_host_resident(ds, act.astype(np.int32), (hns, hr, hp, d, co), uniforms=uni if tape else None,
                                   seed=SEED, step_index=step, env_offset=env0, auto_reset=auto_reset)
            r = hr
        torch.cuda.synchronize()
        for states in (torch.from_numpy(hns), ds):
            assert_step_equal(torch, eng, w, (states, torch.from_numpy(np.asarray(r)), torch.from_numpy(hp),
                                              torch.from_numpy(np.asarray(d)), torch.from_numpy(np.asarray(co))),
                              auto_reset, what + ("resident",))


# ---- rollout ----------------------------------------------------------------------------------------------------------
def chain_oracle(cell, lo, hi, T, step0, env0, actions, uniforms, auto_reset):
    eng, ora = cell.eng, cell.ora
    env = np.arange(len(lo), dtype=np.uint64) + np.uint64(env0)
    out = []
    for t in range(T):
        a = actions[t].astype(np.int64) if actions is not None else philox_actions(SEED, env, step0 + t, eng.nA)
        u = uniforms[t] if uniforms is not None else philox_uniforms(SEED, env, step0 + t, cell.n)
        w = ora.step(lo, hi, a, u)
        out.append(w)
        lo, hi = reset_to_s0(eng, w, auto_reset)
    return out, lo, hi


def assert_rollout_equal(torch, cell, got, states, want, auto_reset, what):
    eng = cell.eng
    ns, reward, prob, done, coll = got
    for t, w in enumerate(want[0]):
        assert_step_equal(torch, eng, w, (ns[t], reward[t], prob[t], done[t], coll[t]), auto_reset, what + (t,))
    glo, ghi = split_states(eng, states)
    assert np.array_equal(glo, want[1]) and np.array_equal(ghi, want[2]), what


def rollout_out(torch, eng, T, B, off):
    dev = eng.torch_device
    shapes = [((T,) + eng.state_shape(B), torch.int64), ((T, B), torch.float64), ((T, B), torch.float64),
              ((T, B), torch.bool), ((T, B), torch.bool)]
    # offset by one env: one state (16 bytes for two-word states, which must stay 16-byte aligned), one flag byte
    return tuple(offset_view(torch, torch.zeros(s, dtype=d, device=dev).view((-1,) + s[2:]), off).view(s)
                 for s, d in shapes)


# (T, B, offset view, given uniforms, given actions): EPT = 2 where B is even and nothing is offset (N <= 6, Philox)
ROLLOUT_CASES = [(37, 1024, 0, False, True), (37, 1024, 0, False, False), (37, 1025, 0, False, True),
                 (37, 1024, 1, False, False), (37, 1024, 0, True, True), (37, 1025, 0, True, False),
                 (2, 33, 0, False, True), (1, 1, 0, False, False), (37, 4097, 0, False, False)]


@pytest.mark.timeout(300)
@pytest.mark.parametrize("c", GPU_CELLS)
def test_rollout_matches_oracle(c, cells, torch):
    cell = cells(c)
    eng, n = cell.eng, cell.n
    dev = eng.torch_device
    rng = np.random.default_rng(cell.L * 7 + n)
    step0 = (1 << 32) - 3
    for k, (T, B, off, tape, given) in enumerate(ROLLOUT_CASES):
        for auto_reset in (True, False):
            lo, hi = state_batch(cell, B, rng)
            env0 = (1 << 32) + 101 * k
            acts = rng.integers(0, eng.nA, (T, B)).astype(np.int32) if given else None
            uni = rng.random((T, B, n)) if tape else None
            want = chain_oracle(cell, lo, hi, T, step0, env0, acts, uni, auto_reset)
            st = offset_view(torch, states_tensor(eng, lo, hi), off)
            at = None if acts is None else offset_view(torch, torch.from_numpy(acts).to(dev).view(-1), off).view(T, B)
            ut = None if uni is None else offset_view(torch, torch.from_numpy(uni).to(dev).view(-1), off).view(T, B, n)
            got = eng.rollout(st, at, T, uniforms=ut, seed=SEED, step_index=step0, env_offset=env0,
                              auto_reset=auto_reset, out=rollout_out(torch, eng, T, B, off))
            assert_rollout_equal(torch, cell, got, st, want, auto_reset, (cell_id(c), k, auto_reset))
            if k == 0 and auto_reset:  # the rollout is T steps with consecutive step indices
                s = states_tensor(eng, lo, hi)
                for t in range(T):
                    one = eng.step(s, at[t].contiguous(), seed=SEED, step_index=step0 + t, env_offset=env0,
                                   auto_reset=True)
                    for x, y in zip(one, got):
                        assert torch.equal(x, y[t])
                    s = one[0]
    # a terminal start state under auto-reset: every step is a no-op from s0 (prob 0, done, not a collision)
    for terminal in ("goal", "shared"):
        tw = cells(c, terminal)
        if tw.n == 1 and terminal == "shared":
            continue
        te = tw.eng
        for B in (1024, 1025):
            lo = np.full(B, np.uint64(te.s0 & M64))
            hi = np.full(B, np.uint64(te.s0 >> 64))
            T = 5
            want = chain_oracle(tw, lo, hi, T, step0, 7, None, None, True)
            st = states_tensor(te, lo, hi)
            got = te.rollout(st, None, T, seed=SEED, step_index=step0, env_offset=7, auto_reset=True)
            assert_rollout_equal(torch, tw, got, st, want, True, (cell_id(c), terminal, B))
            assert all(w["done"].all() and not w["prob"].any() for w in want[0])


# ---- evaluate ---------------------------------------------------------------------------------------------------------
def gather(table, idx):
    """table[idx] as int64 numpy, from a host array or a device tensor (tables too large to copy back)."""
    if isinstance(table, np.ndarray):
        return table[idx].astype(np.int64)
    import torch
    return table[torch.from_numpy(idx).to(table.device)].cpu().numpy().astype(np.int64)


def group_actions(cells_, L, groups, tables):
    """The joint action of a group policy: each group's entry at its local state sum_k cell[g_k] * L**k, split into
    base-5 digits, agent g_k's at 5**k."""
    actions = np.zeros(len(cells_), np.int64)
    for g, table in zip(groups, tables):
        entry = gather(table, sum(cells_[:, a] * L ** k for k, a in enumerate(g)))
        for k, a in enumerate(g):
            actions += entry // 5 ** k % 5 * 5 ** a
    return actions


def replay_episodes(eng, ora, policy, kind, T, gamma, step0, off, sub):
    """Episodes `sub` of an evaluate call, stepped through the oracle with the host Philox draws.  kind "groups" takes
    policy = (groups, tables) and also gives ep.pair, the conflict byte of every replayed episode (host_pair of the
    oracle-decoded cells before and after a collision episode's last step, NO_CONFLICT for every other episode)."""
    from test_gpu_groups import host_pair
    env = sub.astype(np.uint64) + np.uint64(off)
    s0_lo, s0_hi = split_s0(eng)
    lo, hi = np.full(len(sub), s0_lo), np.full(len(sub), s0_hi)
    ep = Episodes(len(sub), gamma)
    ep.pair = np.full(len(sub), 0xFF, np.uint8)
    if kind == "groups":
        group_of = [next(gi for gi, g in enumerate(policy[0]) if a in g) for a in range(eng.n)]
    for t in range(T):
        if kind in ("agents", "groups"):
            cells_ = ora.decode(lo, hi).astype(np.int64)
        if kind == "agents":
            actions = sum(policy[i][cells_[:, i]] * 5 ** i for i in range(eng.n))
        elif kind == "groups":
            actions = group_actions(cells_, eng.L, *policy)
        elif kind == "joint":
            actions = gather(policy, lo.astype(np.int64))
        else:
            actions = philox_actions(SEED, env, step0 + t, eng.nA)
        w = ora.step(lo, hi, actions, philox_uniforms(SEED, env, step0 + t, eng.n))
        k = np.where(w["collision"] == 1, 1, np.where(w["terminal"] == 1, 3, 2)).astype(np.uint8)
        if kind == "groups":
            hit = np.flatnonzero(ep.active & (w["done"] == 1) & (w["collision"] == 1))
            nxt = ora.decode(w["next_lo"][hit], w["next_hi"][hit])
            for h, row in zip(hit, nxt):
                ep.pair[h] = host_pair(cells_[h], row, group_of)
        if not ep.add(t, w["reward"], w["done"].astype(bool), k):
            break
        lo, hi = w["next_lo"], w["next_hi"]
    return ep


def cell_partitions(n, L, joint):
    """The agent partitions a cell's group policies use: singletons; agents dealt round-robin into groups of at most
    k <= 4 agents with L**k <= 2**25 entries (non-contiguous groups such as (0, 4, 8, 12) at 13 agents, so the whole
    N x N multiplier matrix is used); {0, n-1} plus singletons; one group of every agent where a joint table fits.
    Duplicates (small n) are dropped."""
    k = max(k for k in range(1, min(n, 4) + 1) if L ** k <= 1 << 25)
    m = -(-n // k)
    out = [tuple((i,) for i in range(n)), tuple(tuple(range(g, n, m)) for g in range(m))]
    if n >= 2 and L ** 2 <= 1 << 25:
        out.append(((0, n - 1),) + tuple((i,) for i in range(1, n - 1)))
    if joint:
        out.append((tuple(range(n)),))
    return list(dict.fromkeys(out))


def assert_episodes(got, ep, sub, what):
    assert np.array_equal(u64(got[0])[sub], ep.G.view(np.uint64)), what
    assert np.array_equal(got[1].cpu().numpy()[sub], ep.length), what
    assert np.array_equal(got[2].cpu().numpy()[sub], ep.outcome), what


@pytest.mark.timeout(300)
@pytest.mark.parametrize("c", GPU_CELLS)
def test_evaluate_matches_oracle(c, cells, torch):
    from gym_mapf_b200.envs.vec_env import GroupPolicy
    cell = cells(c)
    eng, ora, n, L = cell.eng, cell.ora, cell.n, cell.L
    dev = eng.torch_device
    rng = np.random.default_rng(cell.L + 5 * cell.n)
    policies = [("random", None, None), ("agents", None, rng.integers(0, 5, (eng.n, eng.L)))]
    joint = eng.words == 1 and eng.nS <= 1 << 26
    if joint:
        policies.append(("joint", None, rng.integers(0, eng.nA, int(eng.nS))))
    step0, off, gamma = (1 << 32) - 7, (1 << 32) + 3, 0.95
    cases = ((1500, 50), (257, 1))
    results = {}
    for kind, _, table in policies:
        pol = None if table is None else torch.from_numpy(table.astype(np.int32)).to(dev)
        for E, T in cases:
            got = eng.evaluate(pol, E, T, gamma=gamma, seed=SEED, step_index=step0, episode_offset=off)
            sub = np.arange(E) if E < 1000 else np.arange(0, E, 3)
            ep = replay_episodes(eng, ora, table, kind, T, gamma, step0, off, sub)
            assert_episodes(got, ep, sub, (kind, E, T))
            results[kind, E] = got
    # group policies: singletons act as AGENTS on the same table, one group of every agent as JOINT on the same table
    grng = np.random.default_rng(cell.L + 7 * cell.n + GROUP_SEEDS.get(c, 1))
    for groups in cell_partitions(n, L, joint):
        if len(groups) == 1 and joint:
            tables = [policies[2][2].astype(np.int32)]
        else:
            tables = [grng.integers(0, 5 ** len(g), L ** len(g), dtype=np.int32) for g in groups]
        gp = GroupPolicy(groups, [torch.from_numpy(t).to(dev) for t in tables])
        for E, T in cases:
            what = (groups, E, T)
            pairs = torch.full((E,), 0xEE, dtype=torch.uint8, device=dev)
            got = eng.evaluate_groups(gp, E, T, gamma=gamma, seed=SEED, step_index=step0, episode_offset=off,
                                      conflicts=pairs)
            plain = eng.evaluate_groups(gp, E, T, gamma=gamma, seed=SEED, step_index=step0, episode_offset=off)
            assert all(torch.equal(a, b) for a, b in zip(got, plain)), what  # conflicts=None changes nothing else
            if len(groups) == n:
                same = eng.evaluate(torch.stack(gp.tables), E, T, gamma=gamma, seed=SEED, step_index=step0,
                                    episode_offset=off)
                assert all(torch.equal(a, b) for a, b in zip(got, same)), what
            elif len(groups) == 1 and joint:
                assert all(torch.equal(a, b) for a, b in zip(got, results["joint", E])), what
            sub = np.arange(E) if E < 1000 else np.arange(0, E, 3)
            ep = replay_episodes(eng, ora, (groups, tables), "groups", T, gamma, step0, off, sub)
            assert_episodes(got, ep, sub, what)
            assert np.array_equal(pairs.cpu().numpy()[sub], ep.pair), what
            if n >= 2 and T > 1:  # attribution is tested only where something collides
                assert (ep.outcome == 1).any(), what
    for terminal in ("goal", "shared"):
        tw = cells(c, terminal)
        if tw.n == 1 and terminal == "shared":
            continue
        ret, length, outcome = tw.eng.evaluate(None, 300, 20, gamma=gamma, seed=SEED)
        assert np.all(u64(ret) == 0) and bool((length == 1).all()) and bool((outcome == 3).all())
        gp = GroupPolicy([(i,) for i in range(n)], [torch.from_numpy(t).to(dev) for t in
                                                     grng.integers(0, 5, (n, L), dtype=np.int32)])
        pairs = torch.zeros(300, dtype=torch.uint8, device=dev)
        ret, length, outcome = tw.eng.evaluate_groups(gp, 300, 20, gamma=gamma, seed=SEED, conflicts=pairs)
        assert np.all(u64(ret) == 0) and bool((length == 1).all()) and bool((outcome == 3).all())
        assert bool((pairs == 0xFF).all())


@pytest.mark.timeout(300)
@pytest.mark.parametrize("c", [pytest.param(c, id=cell_id(c), marks=pytest.mark.gpu) for c in BACKUP_CELLS
                               if c[0] in (8, 9)])
def test_one_group_takes_every_digit(c, cells, torch):
    """One group of all 8 or 9 agents on nine cells: entries of 9**n states, so the device takes digits 0..8 of an entry
    (positions 9..12 are covered by the host check of the arithmetic in test_groups_host.py: a group of 10 agents needs
    L >= 10 for a non-terminal start, and 10**10 entries).  Against JOINT on the same table, and against the oracle
    with conflict bytes.  Each digit is STAY with probability 3/4: with uniform digits nearly every agent moves on a
    full grid, and nearly every episode would end on its first step, having read the entry of s0 only.  (At 9 agents
    the grid is full and fail_prob is 0: every episode is that one step, and its conflict byte names the movers.)"""
    from gym_mapf_b200.envs.vec_env import GroupPolicy
    cell = cells(c)
    eng, ora, n = cell.eng, cell.ora, cell.n
    dev = eng.torch_device
    nS = int(eng.nS)
    assert eng.words == 1 and nS == 9 ** n
    gen = torch.Generator(device=dev)
    gen.manual_seed(77 + n)
    table = torch.zeros(nS, dtype=torch.int32, device=dev)
    for k in range(n):
        d = torch.randint(1, 5, (nS,), dtype=torch.int32, device=dev, generator=gen)
        d.masked_fill_(torch.rand(nS, device=dev, generator=gen) < 0.75, 0)
        table += d * 5 ** k
        del d
    gp = GroupPolicy([tuple(range(n))], [table])
    E, T, gamma, step0, off = 100003, 40, 0.95, (1 << 32) - 3, (1 << 32) + 11
    pairs = torch.full((E,), 0xEE, dtype=torch.uint8, device=dev)
    got = eng.evaluate_groups(gp, E, T, gamma=gamma, seed=SEED, step_index=step0, episode_offset=off, conflicts=pairs)
    want = eng.evaluate(table, E, T, gamma=gamma, seed=SEED, step_index=step0, episode_offset=off)
    assert all(torch.equal(a, b) for a, b in zip(got, want))
    sub = np.concatenate([np.arange(0, E, 331), [E - 1]])
    ep = replay_episodes(eng, ora, (gp.groups, [table]), "groups", T, gamma, step0, off, sub)
    assert_episodes(got, ep, sub, c)
    assert np.array_equal(pairs.cpu().numpy()[sub], ep.pair)
    assert (ep.outcome == 1).any() and (n == 9 or (ep.length > 1).any())


# ---- table path -------------------------------------------------------------------------------------------------------
def mostly_stay_actions(n, B, rng, max_movers=7):
    """Joint actions with at most `max_movers` agents moving, so rows stay within 3**max_movers records."""
    movers = np.argsort(rng.random((B, n)), 1) < rng.integers(0, min(n, max_movers) + 1, (B, 1))
    digits = np.where(movers, rng.integers(1, 5, (B, n)), 0)
    return (digits * 5 ** np.arange(n, dtype=np.int64)).sum(1)


CS_KEYS = ["count", "n_collision", "n_done", "sum_next_lo", "sum_next_hi", "sum_prob_bits", "sum_reward_bits", "ordered"]


@pytest.mark.timeout(300)
@pytest.mark.parametrize("c", GPU_CELLS)
def test_table_path_matches_oracle(c, cells, torch):
    cell = cells(c)
    eng, ora, n = cell.eng, cell.ora, cell.n
    rng = np.random.default_rng(cell.L * 3 + n)
    B = 600
    lo, hi = state_batch(cell, B, rng)
    act = mostly_stay_actions(n, B, rng)
    want = ora.rows(lo, hi, act, threads=8)
    got = eng.transitions(states_tensor(eng, lo, hi), torch.from_numpy(act.astype(np.int32)).to(eng.torch_device))
    assert_rows_equal(eng, got, want["row_ptr"], want["next_lo"], want["next_hi"], G.f64_to_bits(want["prob"]),
                      G.f64_to_bits(want["reward"]), want["done"], want["collision"])
    lens = np.diff(want["row_ptr"])
    terminal_row = (lens == 1) & (want["done"][want["row_ptr"][:-1]] == 1) & (want["prob"][want["row_ptr"][:-1]] == 1.0)
    if n >= 4 and cell.spec["fail_prob"] not in (0.0, 1.0):
        assert (lens > 32).any(), "rows longer than 32 records"
    assert (~terminal_row).any()
    cs = eng.checksum(got[1], got[2], got[3], got[4]).cpu().numpy().view(np.uint64)
    wcs = G.checksums(want["next_lo"], want["next_hi"], G.f64_to_bits(want["prob"]), G.f64_to_bits(want["reward"]),
                      want["done"], want["collision"])
    assert {k: int(v) for k, v in zip(CS_KEYS, cs)} == wcs
    if n > 6:
        return
    n_states = min(int(eng.nS), max(1, 30000 // 13 ** n))
    s_begin = int(rng.integers(0, int(eng.nS) - n_states + 1)) if eng.nS < (1 << 62) else (int(eng.nS) // 7) * 3 + 11
    got = eng.table_range(s_begin, n_states)
    s = np.repeat(np.array([s_begin + i for i in range(n_states)], dtype=object), int(eng.nA))
    s_lo = np.array([int(x) & M64 for x in s], np.uint64)
    s_hi = np.array([int(x) >> 64 for x in s], np.uint64)
    a = np.tile(np.arange(int(eng.nA), dtype=np.int64), n_states)
    want = ora.rows(s_lo, s_hi, a, threads=8)
    assert_rows_equal(eng, got, want["row_ptr"], want["next_lo"], want["next_hi"], G.f64_to_bits(want["prob"]),
                      G.f64_to_bits(want["reward"]), want["done"], want["collision"])
    cs = eng.checksum(got[1], got[2], got[3], got[4]).cpu().numpy().view(np.uint64)
    assert {k: int(v) for k, v in zip(CS_KEYS, cs)} == ora.table_checksums(s_begin, n_states)


# ---- encode / decode / project / predecessors -------------------------------------------------------------------------
@pytest.mark.parametrize("c", GPU_CELLS)
def test_encodings_match_oracle(c, cells, torch):
    cell = cells(c)
    eng, ora, n = cell.eng, cell.ora, cell.n
    rng = np.random.default_rng(cell.L * 11 + n)
    lo, hi = state_batch(cell, 3001, rng)
    st = states_tensor(eng, lo, hi)
    ids = ora.decode(lo, hi)
    assert np.array_equal(eng.decode(st).cpu().numpy(), ids)
    elo, ehi = split_states(eng, eng.encode(torch.from_numpy(ids).to(eng.torch_device)))
    assert np.array_equal(elo, lo) and np.array_equal(ehi, hi)
    for k in range(1, n + 1):
        sub = [int(x) for x in rng.permutation(n)[:k]]
        got = eng.project(st, sub).cpu().numpy().view(np.uint64).reshape(len(lo), -1)
        wlo, whi = ora.project(lo, hi, sub)
        assert np.array_equal(got[:, 0], wlo) and (got.shape[1] == 1 and not whi.any() or np.array_equal(got[:, 1], whi))
    if n > 8:
        return
    m = max(2, 64 // 5 ** max(0, n - 5))
    wp = ora.predecessors(lo[:m], hi[:m])
    row_ptr, pred = eng.predecessors(st[:m])
    assert np.array_equal(row_ptr.cpu().numpy(), wp["row_ptr"])
    plo, phi = split_states(eng, pred)
    for b in range(m):
        sl = slice(int(wp["row_ptr"][b]), int(wp["row_ptr"][b + 1]))
        order = np.lexsort((plo[sl], phi[sl]))
        assert np.array_equal(plo[sl][order], wp["pred_lo"][sl]) and np.array_equal(phi[sl][order], wp["pred_hi"][sl])


# ---- backup / greedy --------------------------------------------------------------------------------------------------
@pytest.mark.timeout(300)
@pytest.mark.parametrize("c", [pytest.param(c, id=cell_id(c), marks=pytest.mark.gpu) for c in BACKUP_CELLS])
def test_backup_matches_oracle(c, cells, torch):
    cell = cells(c)
    eng, ora, n = cell.eng, cell.ora, cell.n
    assert (eng.words, eng.moves_in_smem) == (1, cell.staged)
    dev = eng.torch_device
    nS, gamma = int(eng.nS), 0.95
    gen = torch.Generator(device=dev)
    gen.manual_seed(n)
    Vt = torch.randn(nS, dtype=torch.float64, device=dev, generator=gen) * 30.0
    V = Vt.cpu().numpy()
    rng = np.random.default_rng(n * 17 + cell.L)
    lo, _ = state_batch(cell, 5000, rng)
    act = rng.integers(0, eng.nA, len(lo)) if n <= 6 else mostly_stay_actions(n, len(lo), rng)
    if n == 9:  # all 9! placements of nine agents on nine cells (non-terminal rows): more batches than warps
        import itertools
        perm = np.array(list(itertools.permutations(range(9))), np.int32)
        plo, _ = ora.encode(perm)
        lo = np.concatenate([lo, plo])
        act = np.concatenate([act, mostly_stay_actions(9, len(plo), rng, max_movers=2)])
    z = np.zeros_like(lo)
    q = eng.backup(states_tensor(eng, lo, z), torch.from_numpy(act.astype(np.int32)).to(dev), Vt, gamma)
    assert np.array_equal(u64(q), G.f64_to_bits(ora.backup(lo, z, act, V, gamma, threads=8)))
    if n >= 10:
        assert np.all(ora.rows(lo[:50], z[:50], act[:50])["done"] == 1)  # L < N: every row is terminal
    if n <= 5:
        n_states = min(nS, max(1, 4000 // int(eng.nA)))
        s_begin = int(rng.integers(0, nS - n_states + 1))
        Q = eng.backup_range(s_begin, n_states, Vt, gamma)
        s = np.repeat(np.arange(s_begin, s_begin + n_states, dtype=np.uint64), int(eng.nA))
        a = np.tile(np.arange(int(eng.nA), dtype=np.int64), n_states)
        want = ora.backup(s, np.zeros_like(s), a, V, gamma, threads=8)
        assert np.array_equal(u64(Q).reshape(-1), G.f64_to_bits(want))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [3, 4, 5])
@pytest.mark.parametrize("n_states", [1, 33, 1001])
def test_greedy_is_the_first_argmax(n, n_states, cells, torch):
    eng = cells(CELLS[n - 1]).eng
    rng = np.random.default_rng(n_states + n)
    Q = rng.integers(-2, 2, (n_states, int(eng.nA))).astype(np.float64) * 0.5  # ties across all 32 lanes
    V, pi = eng.greedy(torch.from_numpy(Q).to(eng.torch_device))
    assert np.array_equal(u64(V), G.f64_to_bits(Q.max(1)))
    assert np.array_equal(pi.cpu().numpy(), Q.argmax(1))


@pytest.mark.gpu
def test_misaligned_two_word_states_are_rejected(cells, torch):
    """Two-word states are read and written as 16-byte vectors: an array of them that is only 8-byte aligned (a valid
    contiguous tensor that starts one int64 into its buffer) is an argument error, not a fault in the kernel."""
    from gym_mapf_b200._native import MAPF_ERR_INVALID, NativeError
    eng = cells(CELLS[13]).eng
    assert eng.words == 2
    B, dev = 64, eng.torch_device
    good = eng.states_from_ints([eng.s0] * B)
    bad = torch.empty(2 * B + 1, dtype=torch.int64, device=dev)[1:].view(B, 2)
    bad.copy_(good)
    acts = torch.zeros(B, dtype=torch.int32, device=dev)
    out_bad = torch.empty(2 * B + 1, dtype=torch.int64, device=dev)[1:].view(1, B, 2)
    calls = [lambda: eng.step(bad, acts), lambda: eng.rollout(bad, None, 1),
             lambda: eng.rollout(good.clone(), None, 1, out=(out_bad,) + eng.rollout(good.clone(), None, 1)[1:]),
             lambda: eng.decode(bad), lambda: eng.transitions(bad, acts), lambda: eng.predecessors(bad),
             lambda: eng.project(bad, [0])]
    for call in calls:
        with pytest.raises(NativeError) as ei:
            call()
        assert ei.value.code == MAPF_ERR_INVALID
    torch.cuda.synchronize()
    assert torch.equal(bad, good)
