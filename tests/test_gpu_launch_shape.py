"""k_step sizes its CTAs from the batch (mapf_capi.cu: plan_step_cta), so one batch size runs with other CTA sizes,
grids and grid-stride round counts than another.  An env's result depends only on its index: a batch stepped in one
call must equal the same envs stepped as slices with matching env_offset, bit for bit, and a sample must equal the C
oracle.  The sizes cover one-warp launches (2, 66), one round at every CTA size (131 072), several rounds with and
without a short last one (2**19, 2**19 + 2, 2**20), and an odd batch that runs one env per thread; each with and without
MAPF_OPT_SHARE_SM, in Philox, TAPE (given uniforms) and COMPACT modes, for C2 (4 agents) and C4 (8 agents, 128-bit
states, the wide one-env-per-thread CTAs)."""
import numpy as np
import pytest

import golden_util as G
from engine_util import make_engine, make_oracle, split_states, u64
from test_gpu_evaluate import philox_words

pytestmark = pytest.mark.gpu

SIZES = (2, 66, 131072, 1 << 19, (1 << 19) + 2, 1 << 20, 393217)
SEED, STEP, OFFSET = 0x5eed, 7, 1000


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


@pytest.fixture(scope="module", params=["rows_c2", "rows_c4"])
def case(request):
    spec, _ = G.load(request.param)
    return make_engine(spec), make_oracle(spec)


def bits(t):
    import torch
    return t.view(torch.int64) if t.dtype == torch.float64 else t


def step(eng, states, actions, uniforms, share_sm, compact, env_offset):
    return eng.step(states, actions, uniforms=uniforms, seed=SEED, step_index=STEP, env_offset=env_offset,
                    share_sm=share_sm, compact=compact)


def philox_uniforms(n, env):
    """The slip draws k_step generates for envs `env` (Philox blocks 0.. of (seed, env, step), 2**-32 units)."""
    u = np.zeros((len(env), n))
    for b in range((n + 3) // 4):
        words = philox_words(SEED, env, STEP, b)
        for q in range(4):
            if 4 * b + q < n:
                u[:, 4 * b + q] = words[q].astype(np.float64) * 2.0 ** -32
    return u


@pytest.mark.parametrize("B", SIZES)
def test_batch_equals_slices_and_oracle(case, B, torch):
    eng, ora = case
    rng = np.random.default_rng(B)
    dev = eng.torch_device
    states = eng.encode(torch.from_numpy(rng.integers(0, eng.L, (B, eng.n)).astype(np.int32)).to(dev))
    actions = torch.from_numpy(rng.integers(0, eng.nA, B).astype(np.int32)).to(dev)
    given = torch.from_numpy(rng.random((B, eng.n))).to(dev)
    # slices start at even and odd envs, so they also run the other EPT and other CTA sizes
    cuts = sorted({0, min(B, 1), B // 3 & ~1, (2 * B // 3) | 1, B})
    sub = np.unique(rng.integers(0, B, min(B, 1500)))
    lo, hi = split_states(eng, states)
    acts = actions.cpu().numpy().astype(np.int64)
    for mode in ("philox", "tape", "compact"):
        uniforms = given if mode == "tape" else None
        compact = mode == "compact"
        for share_sm in (False, True):
            whole = step(eng, states, actions, uniforms, share_sm, compact, OFFSET)
            parts = [step(eng, states[a:b], actions[a:b], None if uniforms is None else uniforms[a:b], share_sm,
                          compact, OFFSET + a) for a, b in zip(cuts, cuts[1:])]
            for k, got in enumerate(whole):
                assert torch.equal(bits(got), torch.cat([bits(p[k]) for p in parts])), (mode, share_sm, k)
        # a sample of the envs against the C oracle
        u = given.cpu().numpy()[sub] if mode == "tape" else philox_uniforms(eng.n, sub.astype(np.uint64) + np.uint64(OFFSET))
        want = ora.step(lo[sub], hi[sub], acts[sub], u)
        if compact:
            ns, code, prob, flags = whole
            reward = eng.reward_table()[code.cpu().numpy()[sub]]
            f = flags.cpu().numpy()[sub]
            done, coll = f & 1, (f >> 1) & 1
        else:
            ns, r, prob, d, c = whole
            reward = r.cpu().numpy()[sub]
            done, coll = d.cpu().numpy()[sub].astype(np.uint8), c.cpu().numpy()[sub].astype(np.uint8)
        glo, ghi = split_states(eng, ns)
        assert np.array_equal(glo[sub], want["next_lo"]) and np.array_equal(ghi[sub], want["next_hi"]), mode
        assert np.array_equal(reward.view(np.uint64), G.f64_to_bits(want["reward"])), mode
        assert np.array_equal(u64(prob)[sub], G.f64_to_bits(want["prob"])), mode
        assert np.array_equal(done, want["done"]) and np.array_equal(coll, want["collision"]), mode
