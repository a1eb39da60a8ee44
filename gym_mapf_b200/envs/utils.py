"""Factories and parsers (reference gym_mapf/envs/utils.py): MovingAI `.map` / `.scen` parsing, env construction
by map name, the synthetic multi-room "sanity" env and agent-subset views.  Host-side setup only."""
import collections

from . import map_name_to_files
from .grid import MapfGrid
from .mapf_env import MapfEnv


def parse_scen_file(scen_file, n_agents):
    """(starts, goals) of the first `n_agents` scenario lines.  Fields 4..7 of a line are used as
    (row, col) pairs in file order, exactly as the reference does (utils.py:8-30)."""
    starts, goals = [], []
    with open(scen_file, "r") as f:
        f.readline()  # "version 1"
        for line in f:
            fields = line.split("\t")
            if len(fields) != 9:
                raise ValueError("not enough values to unpack (expected 9, got %d)" % len(fields))
            starts.append((int(fields[4]), int(fields[5])))
            goals.append((int(fields[6]), int(fields[7])))
            if len(starts) == n_agents:
                break
    return tuple(starts), tuple(goals)


def parse_map_file(map_file):
    """The grid lines of a MovingAI map: everything after the 4 header lines (utils.py:33-37)."""
    with open(map_file, "r") as f:
        return f.readlines()[4:]


def create_sanity_mapf_env(n_rooms, room_size, n_agents, fail_prob, reward_of_clash, reward_of_goal, reward_of_living,
                           optimization_criteria, **kwargs):
    """`n_rooms` empty rooms side by side, separated by a 2-wide wall that is open on the bottom row; room i takes
    its agents from scenario (i % 25) + 1 of empty-<room_size>-<room_size> (utils.py:40-98)."""
    per_room = int(n_agents / n_rooms)
    last_room = n_agents - per_room * (n_rooms - 1)
    if last_room == 0 or per_room == 0:
        raise ValueError(
            f"asked for a sanity env with {n_rooms} rooms  and {n_agents} agents, There are redundant rooms")
    stride = room_size + 2
    lines = []
    for r in range(room_size):
        gap = ".." if r == room_size - 1 else "@@"
        lines.append(gap.join(["." * room_size] * n_rooms))
    starts, goals = (), ()
    for i in range(n_rooms):
        _, scen_file = map_name_to_files(f"empty-{room_size}-{room_size}", i % 25 + 1)
        room_starts, room_goals = parse_scen_file(scen_file, per_room if i != n_rooms - 1 else last_room)
        starts += tuple((r, c + i * stride) for r, c in room_starts)
        goals += tuple((r, c + i * stride) for r, c in room_goals)
    return MapfEnv(MapfGrid(lines), n_agents, starts, goals, fail_prob, reward_of_clash, reward_of_goal,
                   reward_of_living, optimization_criteria, **kwargs)


def create_mapf_env(map_name, scen_id, n_agents, fail_prob, reward_of_clash, reward_of_goal, reward_of_living,
                    optimization_criteria, **kwargs):
    """Env for a shipped map + scenario, or for a 'sanity-<rooms>-<size>' name (utils.py:101-135).  `n_agents` is
    truncated to the scenario's length.  Extra keyword arguments (device=...) go to MapfEnv."""
    if map_name.startswith("sanity"):
        n_rooms, room_size = [int(x) for x in map_name.split("-")[1:]]
        return create_sanity_mapf_env(n_rooms, room_size, n_agents, fail_prob, reward_of_clash, reward_of_goal,
                                      reward_of_living, optimization_criteria, **kwargs)
    map_file, scen_file = map_name_to_files(map_name, scen_id)
    grid = MapfGrid(parse_map_file(map_file))
    starts, goals = parse_scen_file(scen_file, n_agents)
    return MapfEnv(grid, len(goals), starts, goals, fail_prob, reward_of_clash, reward_of_goal, reward_of_living,
                   optimization_criteria, **kwargs)


def create_mapf_env_from_text(map_text, scen_text, n_agents, fail_prob, reward_of_clash, reward_of_goal, reward_of_living,
                              optimization_criteria, device=None):
    """`create_mapf_env` for file CONTENTS (bytes or str) instead of a shipped map name: the .map text is parsed on the
    GPU straight into the obstacle bitmap and move table (C ABI `mapf_ctx_create_from_text`; same rules as
    utils.py:8-37 and grid.py:17-25, same KeyError for an unknown cell character or a start/goal on an obstacle).
    The returned MapfEnv's grid / starts / goals are read back from the device context."""
    from .. import _native
    from .mapf_env import OptimizationCriteria
    eng = _native.Engine.from_text(map_text, scen_text, n_agents, fail_prob, reward_of_clash, reward_of_goal,
                                   reward_of_living, optimization_criteria == OptimizationCriteria.Makespan,
                                   device=0 if device is None else device)
    obstacles, starts, goals = eng.grid()
    grid = MapfGrid(["".join("@" if v else "." for v in row) for row in obstacles])
    env = MapfEnv(grid, eng.n, starts, goals, fail_prob, reward_of_clash, reward_of_goal, reward_of_living,
                  optimization_criteria, device=device)
    env._engine_obj = eng
    return env


def get_local_view(env: MapfEnv, agent_indexes: list, **kwargs):
    """The env restricted to a subset of its agents (utils.py:138-157)."""
    keep = [i for i in range(env.n_agents) if i in agent_indexes]
    return MapfEnv(env.grid, len(agent_indexes), tuple(env.agents_starts[i] for i in keep),
                   tuple(env.agents_goals[i] for i in keep), kwargs.get("fail_prob", env.fail_prob),
                   env.reward_of_clash, env.reward_of_goal, env.reward_of_living, env.optimization_criteria,
                   device=env.device)


def independent_policy(env: MapfEnv, gamma=1.0, eps=1e-6, max_iter=1000):
    """The product of single-agent optimal policies: for each agent i, `value_iteration` of the one-agent view
    `get_local_view(env, [i])` (same grid, so its states are the joint env's cell ids).  Returns int32[n_agents, L]:
    agent i on cell c intends action [i, c] -- the per-agent policy `VecMapfEnv.evaluate` takes."""
    import torch
    from .vec_env import VecMapfEnv
    rows = []
    for i in range(env.n_agents):
        _, pi, _ = VecMapfEnv(get_local_view(env, [i]), 1).value_iteration(gamma=gamma, eps=eps, max_iter=max_iter)
        rows.append(pi)
    return torch.stack(rows).contiguous()


def _solve_group(env, group, gamma, eps, max_iter, slab):
    from .vec_env import VecMapfEnv
    V, pi, _ = VecMapfEnv(get_local_view(env, list(group)), 1).value_iteration(gamma=gamma, eps=eps, max_iter=max_iter,
                                                                              slab=slab)
    return V, pi


def _plan_group(env, group, gamma, eps, max_iter, slab):
    return _solve_group(env, group, gamma, eps, max_iter, slab)[1]


def group_policy(env: MapfEnv, groups, gamma=1.0, eps=1e-6, max_iter=1000, slab=None):
    """The product of jointly optimal group policies: for each group g, `value_iteration` of the agent-subset env
    `get_local_view(env, g)`, whose policy is indexed by g's local state.  `independent_policy` with any grouping:
    singleton groups give tables equal to its rows.  `slab` bounds the states of one backup launch.  Returns a
    GroupPolicy (groups in canonical order)."""
    from .vec_env import GroupPolicy
    groups = [tuple(sorted(int(a) for a in g)) for g in groups]
    return GroupPolicy(groups, [_plan_group(env, g, gamma, eps, max_iter, slab) for g in groups])


def group_values(env: MapfEnv, groups, gamma=1.0, eps=1e-6, max_iter=1000, slab=None):
    """`group_policy` that also keeps each group's values: the same per-group `value_iteration`, returned as
    GroupValues(groups, values, policy) with values[g] = V of `get_local_view(env, g)` (float64[L**|g|]) and `policy`
    equal to `group_policy(env, groups, ...)`.  The heuristic of `VecMapfEnv.rtdp`."""
    from .vec_env import GroupPolicy, GroupValues
    groups = [tuple(sorted(int(a) for a in g)) for g in groups]
    solved = [_solve_group(env, g, gamma, eps, max_iter, slab) for g in groups]
    return GroupValues(groups, [V for V, _ in solved], GroupPolicy(groups, [pi for _, pi in solved]))


IndependenceDetection = collections.namedtuple("IndependenceDetection", "policy resolved log")


def independence_detection(env: MapfEnv, n_episodes=1 << 20, max_steps=256, gamma=1.0, seed=0, max_group_size=3,
                           max_table_entries=1 << 28, eps=1e-6, max_iter=1000):
    """Independence detection: plan every agent alone, then repeatedly evaluate the product of the group policies
    (`VecMapfEnv.find_conflicts`, `n_episodes` episodes of at most `max_steps` steps from Philox stream `seed`), merge
    the two groups with the most episodes whose collision is attributed to a pair of agents across them (ties: the
    lowest group ids), and re-plan the merged group jointly with `value_iteration`.  Stops when no episode collides
    across groups (resolved=True), or when the next merge would make a group of more than `max_group_size` agents or a
    table of more than `max_table_entries` entries (resolved=False).

    Detection is sampled: a conflict is found only if it occurs in the evaluated episodes, so resolved=True means that
    none of them collided across groups, not that no reachable state does.  The run is deterministic for a seed.
    Returns IndependenceDetection(policy: GroupPolicy, resolved, log), with one log record per evaluation round:
    {"groups", "counts" (int64[n, n] attributed collision episodes per agent pair, on the CPU), "summary"
    (`evaluation_summary`)}."""
    from .vec_env import GroupPolicy, VecMapfEnv, evaluation_summary
    vec = VecMapfEnv(env, 1, seed=seed, auto_reset=False)
    L = len(env.valid_locations)
    plans = {(i,): _plan_group(env, (i,), gamma, eps, max_iter, None) for i in range(env.n_agents)}
    log = []
    while True:
        groups = sorted(plans, key=lambda g: g[0])
        policy = GroupPolicy(groups, [plans[g] for g in groups])
        found = vec.find_conflicts(policy, n_episodes, max_steps, gamma=gamma)
        counts = found.counts.cpu()
        log.append(dict(groups=policy.groups, counts=counts, summary=evaluation_summary(found.evaluation)))
        gid = policy.group_of()
        across = collections.Counter()
        for i in range(env.n_agents):
            for j in range(i + 1, env.n_agents):
                if gid[i] != gid[j] and int(counts[i, j]):
                    across[(min(gid[i], gid[j]), max(gid[i], gid[j]))] += int(counts[i, j])
        if not across:
            return IndependenceDetection(policy, True, log)
        ga, gb = min(across, key=lambda k: (-across[k], k))
        merged = tuple(sorted(policy.groups[ga] + policy.groups[gb]))
        if len(merged) > max_group_size or L ** len(merged) > max_table_entries:
            return IndependenceDetection(policy, False, log)
        del plans[policy.groups[ga]], plans[policy.groups[gb]]
        plans[merged] = _plan_group(env, merged, gamma, eps, max_iter, None)


def mapf_env_load_from_json(json_str: str) -> MapfEnv:
    raise NotImplementedError()


def manhattan_distance(env: MapfEnv, s, a1, a2):
    """Manhattan distance between two agents in joint state `s` (utils.py:164-167)."""
    locs = env.state_to_locations(s)
    return abs(locs[a1][0] - locs[a2][0]) + abs(locs[a1][1] - locs[a2][1])
