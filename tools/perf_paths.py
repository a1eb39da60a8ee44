"""Device-side timing of every kernel family on the BASELINE.json configs other than the bench line
(C2 expand, C3 table slab, C4 128-bit step, C5 agent-count sweep, rollout).  Prints one JSON line per measurement.

    python tools/perf_paths.py [c2_expand] [c3_table] [c4_step] [c5_sweep] [c2_rollout] [c2_step]

Achieved GB/s uses the algorithmic bytes of SURVEY.md 8d / DESIGN.md 3 (W = state bytes, R = mean row length):
expand W+17 per record + (W+12) per row; table slab W+17 per record + 8 per row; step 2W+22 per env-step.
Inputs/outputs are sized well above the 126 MB L2 (or cycled over a ring), timing is CUDA events on the launching
stream after warm-up."""
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from gym_mapf_b200 import _native  # noqa: E402
from gym_mapf_b200._native import _ptr, check, lib  # noqa: E402
from gym_mapf_b200.envs.mapf_env import OptimizationCriteria  # noqa: E402
from gym_mapf_b200.envs.utils import create_mapf_env  # noqa: E402

PEAK = 6436.1
if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")):
    PEAK = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
DEV = torch.device("cuda", 0)
TARGET_RECORDS = int(os.environ.get("PERF_RECORDS", 1 << 26))


def timed(fn, reps=5, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e-3)
    ts.sort()
    return ts[len(ts) // 2]


def emit(**kw):
    print(json.dumps(kw), flush=True)


def make(map_name, scen, n, soc=True):
    crit = OptimizationCriteria.SoC if soc else OptimizationCriteria.Makespan
    return create_mapf_env(map_name, scen, n, 0.2, -1000.0, 100.0, -1.0, crit, device=0)


def random_states(eng, B, rng):
    cells = torch.from_numpy(rng.integers(0, eng.L, (B, eng.n)).astype(np.int32)).to(DEV)
    return eng.encode(cells)


def expand_case(tag, env, B_guess, rng, window=None):
    """count -> scan -> expand on B random (s, a) pairs, each phase timed."""
    eng = env.engine
    W = eng.words * 8
    # calibrate B so that the number of records is about TARGET_RECORDS
    def draw(B):
        if window is None:
            st = random_states(eng, B, rng)
        else:  # conflict-density sweep: every agent inside a w x w corner window of the (empty) map
            H = len(env.grid)
            r = rng.integers(0, window, (B, eng.n))
            c = rng.integers(0, window, (B, eng.n))
            st = eng.encode(torch.from_numpy((c * H + r).astype(np.int32)).to(DEV))
        ac = torch.from_numpy(rng.integers(0, eng.nA, B).astype(np.int32)).to(DEV)
        return st, ac
    st, ac = draw(4096)
    rl = torch.empty(4096, dtype=torch.int64, device=DEV)
    check(lib().mapf_count_rows(eng._h, _ptr(st), _ptr(ac), 4096, _ptr(rl), eng._stream()))
    R = float(rl.double().mean().item())
    B = max(1024, int(TARGET_RECORDS / R))
    st, ac = draw(B)
    row_len = torch.empty(B, dtype=torch.int64, device=DEV)
    row_ptr = torch.empty(B + 1, dtype=torch.int64, device=DEV)
    scratch = torch.empty(int(lib().mapf_scan_scratch_bytes(B)) // 8 + 1, dtype=torch.int64, device=DEV)
    s = eng._stream()
    t_count = timed(lambda: check(lib().mapf_count_scan_rows(eng._h, _ptr(st), _ptr(ac), B, _ptr(row_len), _ptr(row_ptr),
                                                             _ptr(scratch), s)))
    t_scan = 0.0  # fused into the count call
    total = int(row_ptr[-1].item())
    ns, prob, reward, flags = eng._alloc_records(total)
    t_exp = timed(lambda: check(lib().mapf_expand(eng._h, _ptr(st), _ptr(ac), B, _ptr(row_ptr), _ptr(ns), _ptr(prob),
                                                  _ptr(reward), _ptr(flags), s)))
    cs = eng.checksum(ns, prob, reward, flags)
    words = cs.cpu().numpy().view(np.uint64)
    by = total * (W + 17) + B * (W + 12)
    t_all = t_count + t_scan + t_exp
    emit(case=tag, n_agents=eng.n, L=eng.L, state_bytes=W, rows=B, records=total, mean_row=total / B,
         clash_frac=float(words[1]) / total, moves_in_smem=eng.moves_in_smem,
         ms=dict(count=t_count * 1e3, scan=t_scan * 1e3, expand=t_exp * 1e3),
         records_per_s=total / t_all, expand_only_records_per_s=total / t_exp,
         gbs=by / t_all / 1e9, frac=by / t_all / 1e9 / PEAK,
         expand_only_gbs=total * (W + 17) / t_exp / 1e9, expand_only_frac=total * (W + 17) / t_exp / 1e9 / PEAK)


def c2_expand():
    expand_case("c2_expand room-32-32-4 n=4 SoC", make("room-32-32-4", 1, 4), 1 << 20, np.random.default_rng(2))


def c5_sweep():
    rng = np.random.default_rng(5)
    only = [int(x) for x in os.environ.get("PERF_N", "").split(",") if x]
    for n in range(2, 11):
        if only and n not in only:
            continue
        expand_case("c5_expand empty-32-32 n=%d" % n, make("empty-32-32", 1, n), 1 << 16, rng)
    for w in (16, 8, 4, 2):
        if only and 6 not in only:
            continue
        expand_case("c5_density empty-32-32 n=6 window=%d" % w, make("empty-32-32", 1, 6), 1 << 16, rng, window=w)


def c3_table():
    env = make("maze-32-32-4", 10, 6)
    eng = env.engine
    W = eng.words * 8
    s_begin = eng.s0  # consecutive states from the start state: agent 0 sweeps its cells, the others stay put
    n_states = int(os.environ.get("PERF_C3_STATES", 16))
    sb = (C.c_uint64 * 2)(s_begin & ((1 << 64) - 1), s_begin >> 64)
    B = n_states * eng.nA
    row_len = torch.empty(B, dtype=torch.int64, device=DEV)
    row_ptr = torch.empty(B + 1, dtype=torch.int64, device=DEV)
    scratch = torch.empty(int(lib().mapf_scan_scratch_bytes(B)) // 8 + 1, dtype=torch.int64, device=DEV)
    s = eng._stream()
    t_count = timed(lambda: check(lib().mapf_count_scan_range(eng._h, C.byref(sb), n_states, _ptr(row_len), _ptr(row_ptr),
                                                              _ptr(scratch), s)))
    t_scan = 0.0  # fused into the count call
    total = int(row_ptr[-1].item())
    ns, prob, reward, flags = eng._alloc_records(total)
    t_exp = timed(lambda: check(lib().mapf_expand_range(eng._h, C.byref(sb), n_states, _ptr(row_ptr), _ptr(ns),
                                                        _ptr(prob), _ptr(reward), _ptr(flags), s)))
    by = total * (W + 17) + B * 8
    t_all = t_count + t_scan + t_exp
    emit(case="c3_table maze-32-32-4 scen 10 n=6 slab", n_agents=eng.n, L=eng.L, state_bytes=W, states=n_states, rows=B,
         records=total, mean_row=total / B, ms=dict(count=t_count * 1e3, scan=t_scan * 1e3, expand=t_exp * 1e3),
         records_per_s=total / t_all, gbs=by / t_all / 1e9, frac=by / t_all / 1e9 / PEAK,
         expand_only_gbs=total * (W + 17) / t_exp / 1e9, expand_only_frac=total * (W + 17) / t_exp / 1e9 / PEAK)


def step_case(tag, env, B, ring):
    eng = env.engine
    W = eng.words * 8
    g = torch.Generator(device=DEV)
    g.manual_seed(4)
    states = [eng.states_from_ints([eng.s0]).expand(*eng.state_shape(B)).contiguous()]
    actions = [torch.randint(0, env.nA, (B,), generator=g, device=DEV, dtype=torch.int32) for _ in range(ring)]
    outs = []
    for j in range(ring):
        out = (eng.new_states(B), torch.empty(B, dtype=torch.float64, device=DEV),
               torch.empty(B, dtype=torch.float64, device=DEV), torch.empty(B, dtype=torch.bool, device=DEV),
               torch.empty(B, dtype=torch.bool, device=DEV))
        outs.append(out)
        eng.step(states[j], actions[j], seed=1, step_index=j, auto_reset=True, out=out)
        if j + 1 < ring:
            states.append(out[0].clone())
    K = ring * 4

    def run():
        for i in range(K):
            j = i % ring
            eng.step(states[j], actions[j], seed=1, step_index=100 + i, auto_reset=True, out=outs[j])
    t = timed(run, reps=5, warm=1) / K
    by = B * (2 * W + 22)
    emit(case=tag, n_agents=eng.n, L=eng.L, state_bytes=W, envs=B, moves_in_smem=eng.moves_in_smem, us_per_step=t * 1e6,
         steps_per_s=B / t, gbs=by / t / 1e9, frac=by / t / 1e9 / PEAK)


def mappings():
    """The same batched step through (a) the shipped thread-per-env kernel and (b) the grouped kernel of heterogeneous
    batches with 1, 4 and 64 specs (mapf_group_step).  Stream launches, ring of buffers > L2."""
    for map_name, scen, n, B in (("room-32-32-4", 1, 4, 1 << 20), ("empty-32-32", 1, 2, 1 << 20),
                                 ("room-32-32-4", 13, 6, 1 << 20), ("empty-16-16", 1, 7, 1 << 20)):
        env = make(map_name, scen, n)
        eng = env.engine
        W = eng.words * 8
        ring = 16
        g = torch.Generator(device=DEV)
        g.manual_seed(4)
        rng = np.random.default_rng(3)
        states = [random_states(eng, B, rng) for _ in range(ring)]
        actions = [torch.randint(0, env.nA, (B,), generator=g, device=DEV, dtype=torch.int32) for _ in range(ring)]
        outs = [(eng.new_states(B), torch.empty(B, dtype=torch.float64, device=DEV),
                 torch.empty(B, dtype=torch.float64, device=DEV), torch.empty(B, dtype=torch.bool, device=DEV),
                 torch.empty(B, dtype=torch.bool, device=DEV)) for _ in range(ring)]
        ref = eng.step(states[0], actions[0], seed=1, step_index=7)
        by = B * (2 * W + 22)
        K = ring * 4
        variants = [("thread-per-env (k_step)", lambda j, i: eng.step(states[j], actions[j], seed=1, step_index=i, out=outs[j]))]
        for n_specs in (1, 4, 64):
            # copies of the same spec with different rewards: every CTA re-stages when its tile run crosses a segment
            envs = [create_mapf_env(map_name, scen, n, 0.2, -1000.0 - k, 100.0, -1.0, OptimizationCriteria.SoC, device=0)
                    for k in range(n_specs)]
            grp = _native.Group([e.engine for e in envs], [B // n_specs] * n_specs)
            variants.append(("grouped, %d specs (k_step_group)" % n_specs,
                             lambda j, i, grp=grp: grp.step(states[j], actions[j], seed=1, step_index=i, out=outs[j])))
        for tag, fn in variants:
            got = fn(0, 7)
            same = all(torch.equal(a, b) for a, b in zip(got[:1] + got[2:4], ref[:1] + ref[2:4]))  # rewards differ per spec

            def run():
                for i in range(K):
                    fn(i % ring, 100 + i)
            t = timed(run, reps=5, warm=1) / K
            emit(case="mapping %s n=%d: %s" % (map_name, n, tag), envs=B, us_per_step=t * 1e6, steps_per_s=B / t,
                 gbs=by / t / 1e9, frac=by / t / 1e9 / PEAK, same_states_probs_dones=bool(same))


def c4_step():
    step_case("c4_step room-64-64-8 n=8 Makespan 2**24 envs", make("room-64-64-8", 1, 8, soc=False), 1 << 24, 2)


def c2_step():
    step_case("c2_step room-32-32-4 n=4 SoC 2**20 envs (stream launches)", make("room-32-32-4", 1, 4), 1 << 20, 32)
    step_case("c2_step room-32-32-4 n=4 SoC 2**23 envs", make("room-32-32-4", 1, 4), 1 << 23, 4)


def c2_rollout():
    env = make("room-32-32-4", 1, 4)
    eng = env.engine
    W = eng.words * 8
    B, T = 1 << 20, 32
    states = eng.states_from_ints([eng.s0]).expand(B).contiguous()
    out = (torch.empty((T, B), dtype=torch.int64, device=DEV), torch.empty((T, B), dtype=torch.float64, device=DEV),
           torch.empty((T, B), dtype=torch.float64, device=DEV), torch.empty((T, B), dtype=torch.bool, device=DEV),
           torch.empty((T, B), dtype=torch.bool, device=DEV))
    t = timed(lambda: eng.rollout(states, None, T, seed=5, auto_reset=True, out=out), reps=5, warm=1)
    by = B * T * (W + 18)
    emit(case="c2_rollout room-32-32-4 n=4 random policy T=32", envs=B, T=T, us_per_step=t / T * 1e6,
         steps_per_s=B * T / t, gbs=by / t / 1e9, frac=by / t / 1e9 / PEAK)


def backup_case():
    """Fused Bellman backup (no table written): records consumed per second, beside the table-writing path.  (Bit
    identity with the CPU oracle is a test: tests/test_gpu_parity.py::test_backup_large_vs_oracle.)"""
    for map_name, n in (("empty-32-32", 2), ("empty-16-16", 3)):
        env = make(map_name, 1, n, soc=False)
        eng = env.engine
        nS, nA = eng.nS, eng.nA
        g = torch.Generator(device=DEV)
        g.manual_seed(6)
        V = torch.randn(nS, generator=g, device=DEV, dtype=torch.float64) * 30
        n_states = min(nS, (1 << 28) // nA // 8)
        s0 = (nS - n_states) // 2
        Q = torch.empty((n_states, nA), dtype=torch.float64, device=DEV)
        t_b = timed(lambda: eng.backup_range(s0, n_states, V, 0.95, out=Q), reps=5, warm=1)
        t_g = timed(lambda: eng.greedy(Q), reps=5, warm=1)
        # how many records did the sweep consume?  (count kernel, not timed)
        sb = (C.c_uint64 * 2)(s0, 0)
        B = n_states * nA
        row_len = torch.empty(B, dtype=torch.int64, device=DEV)
        check(lib().mapf_count_range(eng._h, C.byref(sb), n_states, _ptr(row_len), eng._stream()))
        records = int(row_len.sum().item())
        # the same slab through count + scan + expand (table written), for comparison
        row_ptr = torch.empty(B + 1, dtype=torch.int64, device=DEV)
        scratch = torch.empty(int(lib().mapf_scan_scratch_bytes(B)) // 8 + 1, dtype=torch.int64, device=DEV)
        ns, prob, reward, flags = eng._alloc_records(records)
        s = eng._stream()

        def table():
            check(lib().mapf_count_range(eng._h, C.byref(sb), n_states, _ptr(row_len), s))
            check(lib().mapf_scan_rows(eng._h, _ptr(row_len), B, _ptr(row_ptr), _ptr(scratch), s))
            check(lib().mapf_expand_range(eng._h, C.byref(sb), n_states, _ptr(row_ptr), _ptr(ns), _ptr(prob),
                                          _ptr(reward), _ptr(flags), s))
        t_t = timed(table, reps=3, warm=1)
        emit(case="backup %s n=%d (Makespan), slab of %d states x %d actions" % (map_name, n, n_states, nA),
             rows=B, records=records, mean_row=records / B, ms=dict(backup=t_b * 1e3, greedy=t_g * 1e3, table=t_t * 1e3),
             records_per_s=records / t_b, rows_per_s=B / t_b, table_records_per_s=records / t_t,
             table_bytes_avoided=records * 25, q_bytes_written=B * 8)


CASES = dict(mappings=mappings, backup=backup_case, c2_expand=c2_expand, c3_table=c3_table, c4_step=c4_step, c5_sweep=c5_sweep, c2_rollout=c2_rollout,
             c2_step=c2_step)

if __name__ == "__main__":
    for name in (sys.argv[1:] or list(CASES)):
        CASES[name]()
