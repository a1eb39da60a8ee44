"""Closed-loop policy evaluation (`k_evaluate`, mapf_evaluate) timed with CUDA events (profiles/r03_evaluate.txt).

    python tools/time_evaluate.py

Workloads (SoC, fail 0.2, scenario 1, max_steps 256, 2**22 episodes, gamma 1):
  (a) room-32-32-4, 4 agents, the product of single-agent value-iteration policies (independent_policy)
  (b) the same env with the uniformly random policy, next to k_rollout's random policy (2**20 envs, T = 32, auto-reset)
  (c) room-32-32-4, 2 agents, the joint value-iteration policy (nS = 465 124); value iteration timed on its own
  (d) room-64-64-8, 8 agents (128-bit states), independent_policy
  (e) the loop a user writes without mapf_evaluate on workload (a): `vec.step(policy(states))` + torch accumulators
Each call is warmed up twice and timed seven times between its own pair of events; median [min, max] are reported.
The policy tables are small (2.7 KB for (a), 1.9 MB for (c)) and stay in L2 after the first step, as they do in use.
"""
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from gym_mapf_b200.envs.mapf_env import OptimizationCriteria  # noqa: E402
from gym_mapf_b200.envs.utils import create_mapf_env, independent_policy  # noqa: E402
from gym_mapf_b200.envs.vec_env import Evaluation, VecMapfEnv, evaluation_summary  # noqa: E402

E, T = 1 << 22, 256


def env_of(map_name, n):
    return create_mapf_env(map_name, 1, n, 0.2, -1000.0, 100.0, -1.0, OptimizationCriteria.SoC, device=0)


def timed(fn, reps=7, warm=2):
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) * 1e-3)
    ts.sort()
    return ts[len(ts) // 2], ts[0], ts[-1]


def report(tag, t, ev):
    med, lo, hi = t
    steps = int(ev.lengths.sum(dtype=torch.int64))
    st = evaluation_summary(ev)
    print("%s: %.3f ms [%.3f, %.3f]  %.3e env-steps/s  %.3e episodes/s  (%d env-steps, %.2f ps per env-step)"
          % (tag, med * 1e3, lo * 1e3, hi * 1e3, steps / med, ev.returns.numel() / med, steps, med * 1e12 / steps))
    print("    success %.4f  collision %.4f  timeout %.4f  mean length %.2f  mean return %.3f"
          % (st["success_rate"], st["collision_rate"], st["timeout_rate"], st["mean_length"], st["mean_return"]))
    return steps, med


def run_eval(vec, policy):
    out = vec.engine.evaluate(policy, E, T, seed=vec.seed)
    return lambda: vec.engine.evaluate(policy, E, T, seed=vec.seed, out=out), Evaluation(*out)


def workload_a(c2, table_c2):
    fn, ev = run_eval(c2, table_c2)
    report("(a) C2 AGENTS, independent_policy", timed(fn), ev)
    return ev


def workload_b(c2):
    fn, ev = run_eval(c2, None)
    steps, med = report("(b) C2 RANDOM", timed(fn), ev)
    eng = c2.engine
    B, TR = 1 << 20, 32
    states = eng.states_from_ints([eng.s0] * B)
    out = eng.rollout(states, None, TR, seed=1, auto_reset=True)
    t = timed(lambda: eng.rollout(states, None, TR, seed=1, auto_reset=True, out=out))
    print("    k_rollout, random policy, 2**20 envs x T=32, auto-reset: %.3f ms [%.3f, %.3f]  %.3e env-steps/s  "
          "(%.2f ps per env-step; k_evaluate %.2f, ratio %.3f)" % (t[0] * 1e3, t[1] * 1e3, t[2] * 1e3, B * TR / t[0],
                                                                  t[0] * 1e12 / (B * TR), med * 1e12 / steps,
                                                                  (med / steps) / (t[0] / (B * TR))))


def main():
    gpu = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print("GPU: %s" % gpu)
    print("%d episodes, max_steps %d, gamma 1.0, SoC, fail 0.2; median [min, max] of 7 timed calls" % (E, T))
    env2 = env_of("room-32-32-4", 4)
    c2 = VecMapfEnv(env2, 1, seed=11)
    table_c2 = independent_policy(env2)
    ev_a = workload_a(c2, table_c2)
    workload_b(c2)
    env = env_of("room-32-32-4", 2)
    vec = VecMapfEnv(env, 1, seed=11)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    _, pi, iters = vec.value_iteration(gamma=1.0)
    torch.cuda.synchronize()
    print("(c) value_iteration, room-32-32-4, 2 agents (nS = %d): %d sweeps in %.3f s" % (env.nS, iters,
                                                                                        time.perf_counter() - t0))
    fn, ev = run_eval(vec, pi)
    report("(c) JOINT 2 agents, value_iteration policy", timed(fn), ev)
    env = env_of("room-64-64-8", 8)
    vec = VecMapfEnv(env, 1, seed=11)
    fn, ev = run_eval(vec, independent_policy(env))
    report("(d) C4 AGENTS 8 agents (128-bit states), independent_policy", timed(fn), ev)
    user_loop(env2, table_c2, ev_a)


def user_loop(env, table, ev_a):
    """What a caller writes today: per step, the policy's joint action from the decoded cells, one `step`, and torch
    accumulators masked at each env's first done (the envs that are done keep stepping until the slowest one ends)."""
    vec = VecMapfEnv(env, E, seed=11, auto_reset=False)
    n = env.n_agents
    pw = torch.tensor([5 ** i for i in range(n)], dtype=torch.int64, device=vec.device)
    tl = table.to(torch.int64)

    def run():
        vec.reset()
        vec.step_count = 0
        G = torch.zeros(E, dtype=torch.float64, device=vec.device)
        length = torch.zeros(E, dtype=torch.int32, device=vec.device)
        active = torch.ones(E, dtype=torch.bool, device=vec.device)
        for t in range(T):
            cells = vec.state_to_cells(vec.states).to(torch.int64)
            a = (tl.gather(1, cells.t().contiguous()).t() * pw).sum(1).to(torch.int32)
            _, r, done, _ = vec.step(a)
            G = torch.where(active, G + r, G)  # gamma = 1
            length += active.to(torch.int32)
            active &= ~done
        return G, length
    t = timed(run, reps=3, warm=1)
    G, length = run()
    steps = int(length.sum(dtype=torch.int64))
    same = ev_a is not None and torch.equal(G, ev_a.returns) and torch.equal(length, ev_a.lengths)
    print("(e) user loop on (a): vec.step(policy(states)) x %d + torch accumulators: %.1f ms [%.1f, %.1f]  %.3e useful "
          "env-steps/s  (%d env-steps; same returns and lengths as k_evaluate: %s)"
          % (T, t[0] * 1e3, t[1] * 1e3, t[2] * 1e3, steps / t[0], steps, same))
    if ev_a is not None:
        fn = lambda: vec.engine.evaluate(table, E, T, seed=11)  # noqa: E731
        t_eval = timed(fn)[0]
        print("    speedup of mapf_evaluate over the loop: %.1fx" % (t[0] / t_eval))


if __name__ == "__main__":
    main()
