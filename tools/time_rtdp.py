"""RTDP on the headline workload C2 (room-32-32-4, 4 agents, SoC, fail_prob 0.2): the cost of the value-table Bellman
update, the driver's progress per iteration, and the TablePolicy against its fallback GroupPolicy.

    python tools/time_rtdp.py [--out profiles/r06_rtdp.txt] [--episodes 4194304]

Records: k_rtdp_backup's records/s against k_backup on the same rows (room-32-32-4 with 2 agents, the largest space of
that map whose V fits, both with CUDA events over a warmed-up launch; on C2 k_backup cannot run, V would need 2.2e11
values); the per-iteration log of `VecMapfEnv.rtdp` on C2 with two heuristics (the singleton values, and the group
values of independence detection's final groups); success and collision rates of each TablePolicy and its fallback over
the same Philox streams.  The card's name and power limit are read in the same run."""
import argparse
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def timed(torch, fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / 1e3 / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_rtdp.txt"))
    ap.add_argument("--episodes", type=int, default=1 << 22)
    ap.add_argument("--trials", type=int, default=1024)
    ap.add_argument("--depth", type=int, default=256)
    ap.add_argument("--iterations", type=int, default=12)
    args = ap.parse_args()
    import numpy as np
    import torch
    from gym_mapf_b200.envs.mapf_env import OptimizationCriteria
    from gym_mapf_b200.envs.utils import create_mapf_env, group_values, independence_detection
    from gym_mapf_b200.envs.vec_env import ValueTable, VecMapfEnv, evaluation_summary
    lines = ["# tools/time_rtdp.py on %s" % gpu_info(), ""]
    say = lambda s: (print(s, flush=True), lines.append(s))  # noqa: E731
    soc = OptimizationCriteria.SoC

    # 1. records/s of the value-table update against k_backup on the same rows
    env2 = create_mapf_env("room-32-32-4", 1, 2, 0.2, -1000.0, 100.0, -1.0, soc, device=0)
    vec2 = VecMapfEnv(env2, 1)
    eng2 = vec2.engine
    rng = np.random.default_rng(0)
    B = 1 << 14
    S = torch.from_numpy(rng.choice(int(eng2.nS), B, replace=False).astype(np.int64)).cuda()
    acts = torch.arange(eng2.nA, dtype=torch.int32, device="cuda").repeat(B)
    rows_s = S.repeat_interleave(eng2.nA)
    records = int(eng2.transitions(rows_s, acts)[0][-1])
    V = torch.zeros(int(eng2.nS), dtype=torch.float64, device="cuda")
    hv2 = group_values(env2, [(0,), (1,)])
    empty2 = ValueTable(eng2, 64)
    full2 = ValueTable(eng2, 1 << 21)
    full2.store(torch.arange(int(eng2.nS), dtype=torch.int64, device="cuda"), V,
                torch.zeros(int(eng2.nS), dtype=torch.int32, device="cuda"))
    t_backup = timed(torch, lambda: eng2.backup(rows_s, acts, V, 1.0), 20)
    t_empty = timed(torch, lambda: eng2.rtdp_backup(S, hv2, empty2, 1.0), 20)
    t_full = timed(torch, lambda: eng2.rtdp_backup(S, hv2, full2, 1.0), 20)
    say("## value-table update vs k_backup, room-32-32-4 2 agents, %d states x %d actions = %d records" % (B, eng2.nA, records))
    say("k_backup (V[s2] gather)                 %8.3f ms  %.3e records/s" % (t_backup * 1e3, records / t_backup))
    say("k_rtdp_backup, empty table (heuristic)  %8.3f ms  %.3e records/s" % (t_empty * 1e3, records / t_empty))
    say("k_rtdp_backup, every state stored       %8.3f ms  %.3e records/s" % (t_full * 1e3, records / t_full))
    del full2, V

    # 2. RTDP on C2 with two heuristics
    env = create_mapf_env("room-32-32-4", 1, 4, 0.2, -1000.0, 100.0, -1.0, soc, device=0)
    vec = VecMapfEnv(env, 1, seed=0)
    eng = vec.engine
    Sc = torch.from_numpy(rng.integers(0, int(eng.nS), 1024).astype(np.int64)).cuda()
    t0 = time.perf_counter()
    single = group_values(env, [(i,) for i in range(env.n_agents)])
    t_single = time.perf_counter() - t0
    t0 = time.perf_counter()
    idr = independence_detection(env)
    grouped = group_values(env, idr.policy.groups)
    t_id = time.perf_counter() - t0
    c_rows = int(eng.transitions(Sc.repeat_interleave(eng.nA),
                                 torch.arange(eng.nA, dtype=torch.int32, device="cuda").repeat(1024))[0][-1])
    say("")
    say("## C2 (room-32-32-4, 4 agents): %d random states x %d actions = %d records (%.0f per state)"
        % (1024, eng.nA, c_rows, c_rows / 1024))
    for name, hv in (("singletons", single), ("ID groups %s" % (idr.policy.groups,), grouped)):
        t = timed(torch, lambda: eng.rtdp_backup(Sc, hv, ValueTable(eng, 64), 1.0), 10)
        say("k_rtdp_backup, empty table, %-28s %8.3f ms  %.3e records/s  %.3e state backups/s"
            % (name, t * 1e3, c_rows / t, 1024 / t))
    say("heuristic set-up: singleton values %.2f s; ID (resolved=%s, %d rounds) + group values %.2f s"
        % (t_single, idr.resolved, len(idr.log), t_id))
    for name, hv in (("singletons", single), ("ID groups", grouped)):
        say("")
        say("## rtdp on C2, heuristic = %s: %d trials, max_depth %d, gamma 1" % (name, args.trials, args.depth))
        res = vec.rtdp(hv, args.trials, args.depth, args.iterations, gamma=1.0, eps=1e-6, capacity=1 << 26)
        say("%4s %12s %14s %10s %10s %9s %12s" % ("it", "residual", "V(s0)", "table", "backups", "s/iter", "backups/s"))
        for i, r in enumerate(res.log):
            say("%4d %12.4g %14.6f %10d %10d %9.3f %12.4g" % (i, r["residual"], r["v_s0"], r["table_size"], r["backups"],
                                                              r["seconds"], r["backups"] / r["seconds"]))
        say("table occupancy %d of %d slots (%.2f %% of the 1/2 cap)" % (len(res.table), res.table.capacity,
                                                                      100.0 * len(res.table) / (res.table.capacity / 2)))
        for label, pol in (("TablePolicy", res.policy), ("fallback GroupPolicy", hv.policy)):
            s = evaluation_summary(vec.evaluate(pol, args.episodes, 256, seed=1))
            say("%-22s %d episodes: success %.4f  collision %.4f  timeout %.4f  mean return %.3f"
                % (label, args.episodes, s["success_rate"], s["collision_rate"], s["timeout_rate"], s["mean_return"]))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
