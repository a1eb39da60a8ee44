"""Host-side parts of RTDP that need no GPU: argument validation of GroupValues, ValueTable and TablePolicy, and the
restatements the GPU tests compare against (the table's slot hash, the group order of the additive heuristic)."""
import types

import numpy as np
import pytest

torch = pytest.importorskip("torch")

M64 = (1 << 64) - 1


def policy(groups, L):
    from gym_mapf_b200.envs.vec_env import GroupPolicy
    return GroupPolicy(groups, [torch.zeros(L ** len(g), dtype=torch.int32) for g in groups])


def values(groups, L, dtype=torch.float64):
    return [torch.zeros(L ** len(g), dtype=dtype) for g in groups]


def test_group_values_canonicalises_and_validates():
    from gym_mapf_b200.envs.vec_env import GroupValues
    gv = GroupValues([(1,), (0, 2)], [torch.full((4,), 1.0, dtype=torch.float64), torch.full((16,), 2.0, dtype=torch.float64)],
                     policy([(0, 2), (1,)], 4))
    assert gv.groups == ((0, 2), (1,)) and gv.values[0].numel() == 16 and float(gv.values[1][0]) == 1.0
    with pytest.raises(ValueError, match="one value table per group"):
        GroupValues([(0,), (1,)], values([(0,)], 4), policy([(0,), (1,)], 4))
    with pytest.raises(ValueError, match="partition"):
        GroupValues([(0,), (2,)], values([(0,), (2,)], 4), policy([(0,), (1,)], 4))
    with pytest.raises(ValueError, match="ascending"):
        GroupValues([(1, 0)], values([(0, 1)], 4), policy([(0, 1)], 4))
    with pytest.raises(ValueError, match="float64"):
        GroupValues([(0,), (1,)], values([(0,), (1,)], 4, torch.float32), policy([(0,), (1,)], 4))
    with pytest.raises(ValueError, match="entries"):
        GroupValues([(0,), (1,)], [torch.zeros(4, dtype=torch.float64), torch.zeros(5, dtype=torch.float64)],
                    policy([(0,), (1,)], 4))
    with pytest.raises(ValueError, match="GroupPolicy of the groups"):
        GroupValues([(0,), (1,)], values([(0,), (1,)], 4), policy([(0, 1)], 4))
    with pytest.raises(ValueError, match="GroupPolicy of the groups"):
        GroupValues([(0,), (1,)], values([(0,), (1,)], 4), policy([(0,), (1,)], 5))
    with pytest.raises(ValueError, match="GroupPolicy of the groups"):
        GroupValues([(0,), (1,)], values([(0,), (1,)], 4), None)


def test_value_table_and_table_policy_reject_bad_arguments():
    from gym_mapf_b200.envs.vec_env import TablePolicy, ValueTable
    one_word = types.SimpleNamespace(words=1)
    for cap in (0, 32, 63, 100, 1000):
        with pytest.raises(ValueError, match="power of two"):
            ValueTable(one_word, cap)
    with pytest.raises(ValueError, match="one-word"):
        ValueTable(types.SimpleNamespace(words=2), 64)
    with pytest.raises(ValueError, match="ValueTable"):
        TablePolicy(object(), policy([(0,)], 4))
    table = object.__new__(ValueTable)
    with pytest.raises(ValueError, match="GroupPolicy"):
        TablePolicy(table, None)
    assert TablePolicy(table, policy([(0,)], 4)).table is table


def home_slot(s, cap):
    """The table's home slot of key s: the splitmix64 finalizer masked to the capacity."""
    z = s
    z = ((z ^ (z >> 30)) * 0xbf58476d1ce4e5b9) & M64
    z = ((z ^ (z >> 27)) * 0x94d049bb133111eb) & M64
    return (z ^ (z >> 31)) & (cap - 1)


def test_slot_hash_restatement_spreads_keys():
    # the finalizer is a bijection of 64-bit words: consecutive states spread over the slots
    cap = 1 << 12
    slots = np.bincount([home_slot(s, cap) for s in range(cap // 2)], minlength=cap)
    assert slots.max() <= 8 and (slots > 0).sum() > cap // 3
    assert home_slot(0, cap) == 0 and home_slot(1, 1 << 63) != 1


def test_group_of_and_heads_follow_canonical_order():
    from gym_mapf_b200.envs.vec_env import GroupValues
    gv = GroupValues([(3,), (0, 2), (1,)], values([(3,), (0, 2), (1,)], 3), policy([(0, 2), (1,), (3,)], 3))
    assert gv.groups == ((0, 2), (1,), (3,))
    # the heuristic sums the groups in this order: the first agent of each group, walked in agent order
    heads = [g[0] for g in gv.groups]
    assert heads == sorted(heads)
