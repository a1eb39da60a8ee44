"""Products of group policies (`k_evaluate_groups`, mapf_evaluate_groups) and independence detection, timed with CUDA
events (profiles/r05_groups.txt).

    python tools/time_groups.py

Workloads (SoC, fail 0.2, scenario 1, max_steps 256, 2**22 episodes, gamma 1):
  (f) C2 = room-32-32-4, 4 agents: the independent_policy table as AGENTS and as singleton GROUPS, timed alternately
  (g) C2 with groups {0,1},{2,3} from group_policy (two 1.9 MB tables), with and without the conflict output
  (h) C4 = room-64-64-8, 8 agents (128-bit states), groups {0,1},{2,3},{4,5},{6,7} from group_policy (about 167 MB of
      tables, more than L2 holds), next to AGENTS with independent_policy
  (i) independence_detection on C2 (2**20 episodes per round): wall time, rounds, groups, collision rate per round
Each call is warmed up twice and timed seven times between its own pair of events; median [min, max] are reported.
"""
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # noqa: E402

from gym_mapf_b200.envs.utils import group_policy, independence_detection, independent_policy  # noqa: E402
from gym_mapf_b200.envs.vec_env import Evaluation, GroupPolicy  # noqa: E402
from time_evaluate import E, T, env_of, report, timed  # noqa: E402


def run(eng, policy, seed=11, conflicts=False):
    out = eng.evaluate(policy, E, T, seed=seed)
    if conflicts:
        pairs = torch.empty(E, dtype=torch.uint8, device=eng.torch_device)
        fn = lambda: eng.evaluate_groups(policy, E, T, seed=seed, out=out, conflicts=pairs)  # noqa: E731
    else:
        fn = lambda: eng.evaluate(policy, E, T, seed=seed, out=out)  # noqa: E731
    return fn, Evaluation(*out)


def planned(env, groups, **kw):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    gp = group_policy(env, groups, **kw)
    torch.cuda.synchronize()
    mb = sum(t.numel() for t in gp.tables) * 4 / 1e6
    print("    group_policy %s: %.2f s of value iteration, %.1f MB of tables" % (gp.groups, time.perf_counter() - t0, mb))
    return gp


def main():
    import subprocess
    gpu = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print("GPU: %s" % gpu)
    print("%d episodes, max_steps %d, gamma 1.0, SoC, fail 0.2; median [min, max] of 7 timed calls" % (E, T))
    env2 = env_of("room-32-32-4", 4)
    eng2 = env2.engine
    table = independent_policy(env2)
    single = GroupPolicy([(i,) for i in range(4)], list(table))
    fa, eva = run(eng2, table)
    fg, evg = run(eng2, single)
    for rnd in range(2):
        report("(f) C2 AGENTS, independent_policy [round %d]" % rnd, timed(fa), eva)
        report("(f) C2 GROUPS, singletons of the same table [round %d]" % rnd, timed(fg), evg)
    print("    same returns, lengths and outcomes: %s" % all(torch.equal(a, b) for a, b in zip(eva, evg)))

    pairs2 = planned(env2, [(0, 1), (2, 3)])
    fn, ev = run(eng2, pairs2)
    report("(g) C2 GROUPS {0,1},{2,3}", timed(fn), ev)
    fn, ev = run(eng2, pairs2, conflicts=True)
    report("(g) C2 GROUPS {0,1},{2,3} with the conflict output", timed(fn), ev)

    env4 = env_of("room-64-64-8", 8)
    eng4 = env4.engine
    fn, ev = run(eng4, independent_policy(env4))
    report("(h) C4 AGENTS, independent_policy", timed(fn), ev)
    pairs4 = planned(env4, [(0, 1), (2, 3), (4, 5), (6, 7)], max_iter=400)
    fn, ev = run(eng4, pairs4)
    report("(h) C4 GROUPS, four pairs", timed(fn), ev)
    del pairs4, fn, ev

    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = independence_detection(env2)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    print("(i) independence_detection, C2, 2**20 episodes per round: %.2f s, %d rounds, resolved %s, final groups %s"
          % (wall, len(res.log), res.resolved, res.policy.groups))
    for k, rec in enumerate(res.log):
        s = rec["summary"]
        c = rec["counts"]
        top = sorted(((int(c[i, j]), (i, j)) for i in range(4) for j in range(i + 1, 4) if int(c[i, j])), reverse=True)
        print("    round %d: groups %s  collision %.4f  success %.4f  mean return %.3f  attributed pairs %s"
              % (k, rec["groups"], s["collision_rate"], s["success_rate"], s["mean_return"], top))


if __name__ == "__main__":
    main()
