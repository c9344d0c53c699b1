"""CPU checks of PolicyPool.plan: the rows, indices and masks it lays out for league duel batches, without a device.
The grouped trunk and the heads themselves are checked on the GPU in test_gpu_policy_pool."""
from types import SimpleNamespace

import pytest
import torch

from helpers import compiled
from marl_ctf_development_b200 import _native
from marl_ctf_development_b200.fused_policy import N_ACTIONS, PolicyPool, trunk_dims
from marl_ctf_development_b200.league import pool_segments
from marl_ctf_development_b200.policy import CtfPolicy


def _env(exp, B):
    ce = compiled(exp)
    N = ce.N_AGENTS
    return SimpleNamespace(
        n_channels=ce.n_channels, GRID_SIZE=ce.GRID_SIZE, meta_size=ce.meta_size, N_AGENTS=N, num_envs=B,
        device=torch.device("cpu"), AGENT_TEAMS=ce.AGENT_TEAMS, obs_bits=None,
        use_action_mask=torch.tensor([float(ce.AGENT_TYPE_ACTION_MASK[ce.AGENT_TYPES[i]]) for i in range(N)]))


def _policies(env, n, unmasked=()):
    torch.manual_seed(0)
    return [CtfPolicy(N_ACTIONS, env.n_channels, env.GRID_SIZE, env.meta_size, use_masking=i not in unmasked)
            for i in range(n)]


def _pairs(kind, pols):
    if kind == "symmetric":        # generate_metrics_symmetric: every ordered pair, self-play included
        return [(a, o) for a in pols for o in pols]
    if kind == "lower":            # winrate_matrix_symmetric: i > j
        return [(a, o) for i, a in enumerate(pols) for j, o in enumerate(pols) if i > j]
    if kind == "non_symmetric":    # two disjoint groups
        return [(a, o) for a in pols[:2] for o in pols[2:]]
    if kind == "self_play":
        return [(p, p) for p in pols]
    raise AssertionError(kind)


@pytest.mark.parametrize("D", [1, 3])
@pytest.mark.parametrize("kind", ["symmetric", "lower", "non_symmetric", "self_play"])
@pytest.mark.parametrize("exp", ["0_the_split", "8_arena"])
def test_league_plan_covers_every_agent_once(exp, kind, D):
    probe = _env(exp, 1)
    pols = _policies(probe, 4, unmasked=(1,))
    pairs = _pairs(kind, pols)
    env = _env(exp, len(pairs) * D)
    B, N = env.num_envs, env.N_AGENTS
    team_ids = [[i for i in range(N) if env.AGENT_TEAMS[i] == t] for t in (0, 1)]
    uniq, segments = pool_segments(pairs, D, team_ids)
    assert len({id(p) for p in uniq}) == len(uniq)
    pool = PolicyPool(env, uniq)
    plan = pool.plan(segments)
    S = plan.n_outputs
    assert S == B * N

    # every (env, agent) of the batch maps to exactly one valid row
    flat = plan.flat_index.tolist()
    assert sorted(flat) == list(range(B * N))
    # that row belongs to the policy that plays the agent: team t of pair p is pairs[p][t]
    for r, f in enumerate(flat):
        e, a = divmod(f, N)
        t = env.AGENT_TEAMS[a]
        assert uniq[int(plan.policy_of_row[r])] is pairs[e // D][t]
    # rows of a policy are contiguous, start at p * s_max, and the pad rows are never gathered or scattered
    rows = plan.row_index.tolist()
    assert len(set(rows)) == S
    for p in range(len(uniq)):
        mine = sorted(rows[r] for r in range(S) if int(plan.policy_of_row[r]) == p)
        assert mine == list(range(p * plan.s_max, p * plan.s_max + plan.n_samples[p]))
    assert plan.s_max == max(plan.n_samples)
    assert plan.features.shape == (len(uniq) * plan.s_max, trunk_dims(env.n_channels, env.GRID_SIZE, env.meta_size)[1])
    assert not plan.features.any()
    # outputs are in plan order: segment after segment, sample e*k + j
    for (pol, e0, e1, ids), (r0, r1) in zip(plan.segments, plan.seg_rows):
        k = len(ids)
        assert r1 - r0 == (e1 - e0) * k
        assert flat[r0:r1] == [(e0 + s // k) * N + ids[s % k] for s in range(r1 - r0)]

    # the additive mask: (mask_5 - 1) * 1e9 on masked agent types of masking policies, zeros elsewhere
    for r, f in enumerate(flat):
        pol = uniq[int(plan.policy_of_row[r])]
        flag = env.use_action_mask[f % N].reshape(1)
        want = pol.masked_logits(torch.zeros(1, N_ACTIONS), flag)[0]
        assert torch.equal(plan.mask_add[r], want)


def test_kernel_tables_are_policy_major_and_rows_match():
    env = _env("8_arena", 6)
    pols = _policies(env, 3)
    pool = PolicyPool(env, pols)
    segs = [(2, slice(0, 2), (0, 1)), (0, slice(2, 6), (4,)), (2, slice(3, 3), (1,)), (1, slice(1, 4), (7, 6, 5)),
            (0, slice(0, 1), (2, 3))]
    plan = pool.plan(segs)
    (arr, n), = plan._tables
    assert n == len(segs)
    assert [arr[i].policy for i in range(n)] == [0, 0, 1, 2, 2]
    assert plan.n_samples == [4 + 2, 9, 4]
    assert plan.s_max == 9
    # segment 4 (policy 0) comes after segment 1 in policy 0's block
    want = {(0, 2, 4): 0, (0, 0, 2): 4, (1, 1, 7): 9, (2, 0, 0): 18, (2, 3, 1): 22}
    got = {(arr[i].policy, arr[i].env_begin, arr[i].agent_ids[0]): arr[i].out_row for i in range(n)}
    assert got == want
    assert plan.seg_rows == [(0, 4), (4, 8), (8, 8), (8, 17), (17, 19)]


def test_plans_with_many_segments_are_split_into_kernel_calls():
    env = _env("0_the_split", 1200)
    pool = PolicyPool(env, _policies(env, 2))
    plan = pool.plan([(i % 2, slice(i, i + 1), (0,)) for i in range(1200)])
    assert [n for _, n in plan._tables] == [512, 512, 176]
    assert plan.n_samples == [600, 600]


def test_bad_pools_and_segments_are_rejected():
    env = _env("8_arena", 4)
    pols = _policies(env, 2)
    with pytest.raises(ValueError, match="only once"):
        PolicyPool(env, [pols[0], pols[1], pols[0]])
    with pytest.raises(ValueError):
        PolicyPool(env, [])
    with pytest.raises(ValueError):
        PolicyPool(env, [CtfPolicy(N_ACTIONS, env.n_channels + 1, env.GRID_SIZE, env.meta_size)])
    pool = PolicyPool(env, pols)
    for seg in ((2, slice(0, 4), (0,)), (-1, slice(0, 4), (0,)), (0, slice(0, 4, 2), (0,)), (0, slice(0, 4), ()),
                (0, slice(0, 4), tuple(range(9))), (0, slice(0, 4), (8,)), (0, slice(3, 1), (0,))):
        with pytest.raises(ValueError):
            pool.plan([seg])
    assert _native.GROUPED_MAX_POLICIES == 64 and _native.GROUPED_MAX_SEGMENTS == 512


def test_league_segments_count_a_module_and_its_views_once():
    env = _env("8_arena", 4)
    a, b = _policies(env, 2)
    from marl_ctf_development_b200 import league

    class View(league.FusedPolicy):      # a FusedPolicy without device buffers: only .policy matters here
        def __init__(self, policy):
            self.policy = policy

    pairs = [(View(a), b), (a, View(a)), (b, View(b))]
    team_ids = [[0, 1, 2, 3], [4, 5, 6, 7]]
    uniq, segments = pool_segments(pairs, 2, team_ids)
    assert uniq == [a, b] and [s[0] for s in segments] == [0, 1, 0, 0, 1, 1]
    PolicyPool(env, uniq).plan(segments)
