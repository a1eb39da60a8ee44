"""Host side of group policies: GroupPolicy canonical order and validation, the table sizes mapf_evaluate_groups
expects, the digit arithmetic of k_evaluate_groups, and the new C entry point.  No GPU needed."""
import ctypes as C

import numpy as np
import pytest


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


def tables_for(torch, groups, L, value=0):
    return [torch.full((L ** len(g),), value, dtype=torch.int32) for g in groups]


def test_group_policy_canonical_order(torch):
    from gym_mapf_b200.envs.vec_env import GroupPolicy
    L = 5
    a = torch.arange(L * L, dtype=torch.int32) % 25
    b = torch.full((L,), 3, dtype=torch.int32)
    c = torch.full((L,), 1, dtype=torch.int32)
    gp = GroupPolicy([[3], (1, 2), [0]], [b, a, c])  # groups are put in order of their lowest agent, with their tables
    assert gp.groups == ((0,), (1, 2), (3,))
    assert gp.tables[0] is c and gp.tables[1] is a and gp.tables[2] is b
    assert gp.group_of() == [0, 1, 1, 2] and gp.n_agents == 4 and gp.n_cells == L
    # the tables' total is what mapf_evaluate_groups checks tables_len against: sum_g L**|g|
    assert sum(t.numel() for t in gp.tables) == sum(L ** len(g) for g in gp.groups)
    assert GroupPolicy(gp.groups, gp.tables) == gp


@pytest.mark.parametrize("groups", [[], [(0,), (0,)], [(0, 2)], [(1,), (2,)], [(1, 0)], [(0, 0)], [()], [(0,), (2,)]])
def test_group_policy_rejects_bad_partitions(groups, torch):
    from gym_mapf_b200.envs.vec_env import GroupPolicy
    with pytest.raises(ValueError):
        GroupPolicy(groups, tables_for(torch, groups, 4))


def test_group_policy_rejects_bad_tables(torch):
    from gym_mapf_b200.envs.vec_env import GroupPolicy
    L = 6
    ok = tables_for(torch, [(0, 1), (2,)], L)
    GroupPolicy([(0, 1), (2,)], ok)
    bad = [
        [ok[0]],                                                      # one table short
        [ok[0].long(), ok[1]],                                        # dtype
        [ok[0].float(), ok[1]],
        [ok[0].view(L, L), ok[1]],                                    # shape
        [ok[0][:-1], ok[1]],                                          # not L**2 entries
        [ok[0], torch.zeros(L + 1, dtype=torch.int32)],               # the groups disagree on L
        [ok[0], torch.zeros(0, dtype=torch.int32)],                   # empty
        [ok[0].clone().fill_(25), ok[1]],                             # entries must lie in [0, 5**|g|)
        [ok[0].clone().fill_(-1), ok[1]],
        [ok[0], torch.full((L,), 5, dtype=torch.int32)],
        [ok[0].numpy(), ok[1]],                                       # not a tensor
    ]
    for tables in bad:
        with pytest.raises(ValueError):
            GroupPolicy([(0, 1), (2,)], tables)
    # the largest valid entry is fine
    GroupPolicy([(0, 1), (2,)], [ok[0].clone().fill_(24), torch.full((L,), 4, dtype=torch.int32)])


def test_digit_extraction_arithmetic():
    """k_evaluate_groups takes digit k of an entry v < 5**13 as umulhi(hi32(v * ceil(2**64 / 5**(k + 1))) + 1, 5)."""
    rng = np.random.default_rng(0)
    for size in range(1, 14):
        top = 5 ** size
        vals = set(int(x) for x in rng.integers(0, top, 3000))
        for k in range(size):
            for q in list(range(0, 200)) + list(range(top // 5 ** k - 200, top // 5 ** k)):
                for v in (q * 5 ** k, q * 5 ** k - 1):
                    if 0 <= v < top:
                        vals.add(v)
        for k in range(size):
            frac = (2 ** 64 - 1) // 5 ** (k + 1) + 1
            for v in vals:
                fhi = (v * frac % 2 ** 64) >> 32
                assert ((fhi + 1) * 5) >> 32 == v // 5 ** k % 5, (size, k, v)


def test_evaluate_groups_is_exported_and_checks_its_context():
    from gym_mapf_b200 import _native
    lib = _native.lib()
    assert "mapf_evaluate_groups" in _native.EXPORTS and lib.mapf_evaluate_groups is not None
    assert _native.POLICY_GROUPS == 3 and _native.NO_CONFLICT == 0xFF
    group_of = (C.c_int32 * 2)(0, 0)
    rc = lib.mapf_evaluate_groups(None, group_of, None, 0, 0, 1, 1.0, 0, 0, 0, None, None, None, None, None, None)
    assert rc == _native.MAPF_ERR_INVALID
