"""ctf_sample_actions (k_sample_actions): seeded policy draws on the device, against the float64 host statement
(draws.sample_action) and against itself, and the policy_seed paths of FusedPolicy, PolicyPool, the rollout and duel
adapters, league.duel_pairs and PackedPPO."""
import ctypes as C
import types

import numpy as np
import pytest
import torch
from scipy.stats import chi2

from marl_ctf_development_b200 import _native, draws, experiment_env_config, league
from marl_ctf_development_b200.env import GridworldCtfGPU
from marl_ctf_development_b200.fused_policy import FusedPolicy, PolicyPool, sample_actions
from marl_ctf_development_b200.policy import CtfPolicy
from marl_ctf_development_b200.ppo import PackedPPO
from marl_ctf_development_b200.rollout import batched_duel, collect_rollout

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
EC = experiment_env_config("8_arena")


def _env(B, base=0, seed=5, **kw):
    kw = {**dict(packed_obs=True, dense_obs=False), **kw}
    return GridworldCtfGPU(**EC, num_envs=B, device=DEV, seed=seed, env_id_base=base, reverse_team1_actions=True, **kw)


def _policy(env, seed, use_masking=True):
    torch.manual_seed(seed)
    return CtfPolicy(9, env.n_channels, env.GRID_SIZE, env.meta_size, use_masking=use_masking).to(env.device).eval()


def _team(env, t):
    return [i for i in range(env.N_AGENTS) if env.AGENT_TEAMS[i] == t]


def _set_counts(env, step, episode):
    """Sets every env's step and episode counters (arrays [B]) through get_state / set_state."""
    st = env.get_state()
    env.set_state(st["grid"], st["pos"], st["hp_q"], st["has_flag"], st["inventory"], step, episode, st["captures"])


def _ptr(t):
    return C.c_void_p(None if t is None else t.data_ptr())


def _raw(env, head, masked, flat, seed, actions=None, aout=None, lp=None, ent=None, stride=None, n=None, state=None,
         handle=None):
    """ctf_sample_actions on raw pointers (ints are addresses); returns the return code."""
    p = lambda x: C.c_void_p(x) if isinstance(x, int) else _ptr(x)
    return env._lib.ctf_sample_actions(
        env._handle if handle is None else handle, env._state_struct if state is None else state, p(head),
        head.stride(0) if stride is None else stride, p(masked), p(flat), flat.numel() if n is None else n, seed,
        p(actions), p(aout), p(lp), p(ent), C.c_void_p(torch.cuda.current_stream().cuda_stream))


# ---------------------------------------------------------------------------------------------------- 1. host statement
def _host(env, head, masked, flat, seed):
    """draws.sample_action with the Philox words of every row, and the rows whose u*Z lies within 1e-5 (relative) of a
    CDF boundary, all in float64 from the device's fp32 logits."""
    N = env.N_AGENTS
    f = flat.cpu().numpy()
    b, a = f // N, f % N
    counts = env._envs.cpu().numpy().view(np.uint32)
    u = draws.policy_uniform(draws.policy_words(seed, env.env_id_base + b, counts[b, 1], counts[b, 0], a))
    x = head[:, 1:10].double().cpu().numpy()
    m = masked.cpu().numpy().astype(bool) if masked is not None else np.zeros(len(f), bool)
    act, lp, ent = draws.sample_action(x, m, u)
    xm = x.copy()
    xm[m, 5:] += -1e9
    e = np.exp(xm - xm.max(1, keepdims=True))
    c = np.cumsum(e, 1)
    z = c[:, -1]
    near = (np.abs((u * z)[:, None] - c) <= 1e-5 * z[:, None]).any(1)
    return act, lp, ent, near


def test_matches_host_statement_on_2_18_rows():
    B = 1 << 15                       # 8 agents: 2^18 (env, agent) rows
    env = _env(B, base=12345)
    rng = np.random.default_rng(1)
    _set_counts(env, rng.integers(0, 500, B), rng.integers(0, 1 << 20, B))
    S = B * env.N_AGENTS
    g = torch.Generator(device="cpu").manual_seed(2)
    head = torch.randn((S, 12), generator=g) * torch.tensor([1.0] + [2.5] * 9 + [1.0] * 2)
    head[: S // 8, 1:10] *= 8         # some very peaked rows
    head = head.to(DEV)
    masked = (torch.rand(S, generator=g) < 0.5).to(torch.uint8).to(DEV)
    flat = torch.randperm(S, generator=g).to(DEV)
    near_total = 0
    for i, seed in enumerate((0, 7, 0xDEADBEEFCAFEF00D)):
        sl = slice(i * S // 3, (i + 1) * S // 3)
        h, mk, fl = head[sl], masked[sl], flat[sl]
        a, lp, ent = sample_actions(env, h, mk, fl, seed)
        act, lp64, ent64, near = _host(env, h, mk, fl, seed)
        a = a.cpu().numpy()
        ok = ~near
        near_total += int(near.sum())
        assert np.array_equal(a[ok], act[ok]), f"seed {seed}: {(a[ok] != act[ok]).sum()} actions differ"
        assert np.abs(lp.cpu().numpy()[ok] - lp64[ok]).max() <= 1e-5
        assert np.abs(ent.cpu().numpy() - ent64).max() <= 1e-5
        assert not (a[mk.cpu().numpy() == 1] >= 5).any()
    print(f"rows within 1e-5 of a CDF boundary (not compared): {near_total} of {S}")
    assert near_total < S // 1000
    assert env.take_faults() == 0


def test_reruns_are_bit_identical_and_leave_torch_rng_alone():
    env = _env(512, base=3)
    S = 512 * 8
    head = torch.randn((S, 10), device=DEV) * 3
    flat = torch.arange(S, device=DEV)
    rng = torch.cuda.get_rng_state()
    first = sample_actions(env, head, None, flat, 99)
    for _ in range(3):
        again = sample_actions(env, head, None, flat, 99)
        assert all(torch.equal(x, y) for x, y in zip(first, again))
    assert torch.equal(torch.cuda.get_rng_state(), rng)
    assert not torch.equal(sample_actions(env, head, None, flat, 100)[0], first[0])


# ---------------------------------------------------------------------------------------------------- 2. range and mask
def test_non_finite_logits_stay_in_range_and_masked_rows_stay_below_5():
    env = _env(1024)
    S = 1024 * 8
    g = torch.Generator(device="cpu").manual_seed(3)
    head = torch.randn((S, 10), generator=g) * 4
    special = torch.tensor([float("nan"), float("inf"), -float("inf"), 3e38, -3e38])
    pick = torch.rand((S, 10), generator=g) < 0.3
    head = torch.where(pick, special[torch.randint(0, 5, (S, 10), generator=g)], head).to(DEV)
    masked = (torch.rand(S, generator=g) < 0.5).to(torch.uint8).to(DEV)
    flat = torch.arange(S, device=DEV)
    actions = torch.full((1024, 8), 255, dtype=torch.uint8, device=DEV)
    a, lp, ent = sample_actions(env, head, masked, flat, 5, actions)
    assert bool(((a >= 0) & (a <= 8)).all()) and torch.equal(actions.view(-1).long(), a)
    # the host statement gives the same action on every row (non-finite rows included) not near a boundary
    act, _, _, near = _host(env, head, masked, flat, 5)
    assert np.array_equal(a.cpu().numpy()[~near], act[~near])
    finite = torch.isfinite(head[:, 1:6]).all(1) & (head[:, 1:6].abs() < 1e30).all(1) \
        & (head[:, 6:10].abs() < 1e30).all(1) & torch.isfinite(head[:, 6:10]).all(1)
    assert int((finite & (masked == 1)).sum()) > 100
    assert not bool((a[finite & (masked == 1)] >= 5).any())
    env.step(actions)        # every action is valid for the step kernel
    assert env.take_faults() == 0


def test_bad_flat_index_sets_the_fault_bit_and_writes_nothing():
    env = _env(16)
    head = torch.randn((6, 10), device=DEV)
    flat = torch.tensor([0, -1, 127, 128, 1 << 40, 5], dtype=torch.int64, device=DEV)
    actions = torch.full((16, 8), 200, dtype=torch.uint8, device=DEV)
    aout = torch.full((6,), -7, dtype=torch.int64, device=DEV)
    lp, ent = torch.full((6,), 42.0, device=DEV), torch.full((6,), 42.0, device=DEV)
    assert env.take_faults() == 0
    assert _raw(env, head, None, flat, 1, actions, aout, lp, ent) == 0
    assert env.take_faults() == _native.FAULT_BAD_INDEX and env.take_faults() == 0
    bad = torch.tensor([False, True, False, True, True, False], device=DEV)
    assert bool((aout[bad] == -7).all()) and bool((lp[bad] == 42).all()) and bool((ent[bad] == 42).all())
    assert bool((aout[~bad] >= 0).all())
    written = torch.zeros(128, dtype=torch.bool, device=DEV)
    written[[0, 127, 5]] = True
    assert bool((actions.view(-1)[~written] == 200).all()) and bool((actions.view(-1)[written] <= 8).all())
    with pytest.raises(IndexError):
        _raw(env, head, None, flat, 1, actions, aout, lp, ent)
        env.raise_on_faults()


# ---------------------------------------------------------------------------------------------------- 3. distribution
def test_draws_follow_softmax_g_test():
    B = 1 << 14
    env = _env(B, base=777)
    S = B * 8                        # 2^17 draws per launch, 32 launches (episodes): 2^22 per logit row
    rows = torch.tensor([[0.0] * 9, [2.0, 1.0, 0.0, -1.0, -2.0, 0.5, 0.25, 3.0, -5.0],
                         [-1.0, 4.0, 0.0, 1.0, 2.0, 9.0, 9.0, 9.0, 9.0]])
    masked_row = [False, False, True]
    flat = torch.arange(S, device=DEV)
    st = env._envs
    for r, (x, mk) in enumerate(zip(rows, masked_row)):
        head = torch.cat((torch.zeros(1), x)).to(DEV).expand(S, 10).contiguous()
        masked = torch.full((S,), int(mk), dtype=torch.uint8, device=DEV)
        counts = torch.zeros(9, dtype=torch.int64, device=DEV)
        for ep in range(32):
            st[:, 1] = ep
            a = sample_actions(env, head, masked, flat, 1234 + r)[0]
            counts += torch.bincount(a, minlength=9)
        obs = counts.cpu().numpy().astype(np.float64)
        xm = x.double().numpy().copy()
        if mk:
            xm[5:] += -1e9
        p = np.exp(xm - xm.max())
        p /= p.sum()
        assert obs.sum() == 1 << 22
        assert obs[p == 0].sum() == 0
        o, e = obs[p > 0], p[p > 0] * obs.sum()
        nz = o > 0
        G = 2 * (o[nz] * np.log(o[nz] / e[nz])).sum()
        pval = chi2.sf(G, df=len(o) - 1)
        print(f"row {r}: G = {G:.2f}, p = {pval:.3g}")
        assert pval > 1e-6


# ---------------------------------------------------------------------------------------------------- 4. layout
def test_results_do_not_depend_on_batch_layout_or_row_order():
    one = _env(64, base=0)
    halves = [_env(32, base=0), _env(32, base=32)]
    steps, eps = np.arange(64) % 7 + 3, np.arange(64) % 3
    _set_counts(one, steps, eps)
    _set_counts(halves[0], steps[:32], eps[:32])
    _set_counts(halves[1], steps[32:], eps[32:])
    g = torch.Generator(device="cpu").manual_seed(4)
    head = (torch.randn((512, 10), generator=g) * 3).to(DEV)
    masked = (torch.rand(512, generator=g) < 0.5).to(torch.uint8).to(DEV)
    flat = torch.arange(512, device=DEV)
    acts = torch.zeros((64, 8), dtype=torch.uint8, device=DEV)
    want = sample_actions(one, head, masked, flat, 31, acts)
    got = [torch.empty_like(t) for t in want]
    for h, env in enumerate(halves):
        perm = torch.randperm(256, generator=g).to(DEV)
        rows = h * 256 + perm
        part = torch.zeros((32, 8), dtype=torch.uint8, device=DEV)
        out = sample_actions(env, head[rows], masked[rows], perm, 31, part)
        for full, o in zip(got, out):
            full[rows] = o
        assert torch.equal(part, acts[h * 32 : (h + 1) * 32])
    for x, y in zip(want, got):
        assert torch.equal(x.view(torch.int32) if x.dtype == torch.float32 else x,
                           y.view(torch.int32) if y.dtype == torch.float32 else y)


# ---------------------------------------------------------------------------------------------------- 5. no torch RNG
def _twice(fn):
    """fn() under two different torch seeds; returns both results."""
    out = []
    for s in (1, 2):
        torch.manual_seed(s)
        out.append(fn())
    return out


def _same(x, y):
    if isinstance(x, torch.Tensor):   # NaN equals NaN (episode statistics are NaN when no episode ended)
        return x.shape == y.shape and x.dtype == y.dtype and bool(((x == y) | (x.isnan() & y.isnan())).all()) \
            if x.is_floating_point() else torch.equal(x, y)
    if isinstance(x, dict):
        return x.keys() == y.keys() and all(_same(x[k], y[k]) for k in x)
    if isinstance(x, (list, tuple)):
        return len(x) == len(y) and all(_same(a, b) for a, b in zip(x, y))
    return x == y or (x != x and y != y)


def test_fused_policy_seeded_call_leaves_torch_rng_alone():
    env = _env(256)
    fp = FusedPolicy(env, _policy(env, 1))
    ids = _team(env, 0)
    flags = env.use_action_mask[ids].repeat(256)
    rng = torch.cuda.get_rng_state()
    a1 = fp.get_action_and_value(flags, agent_ids=ids, seed=8)
    assert torch.equal(torch.cuda.get_rng_state(), rng)
    torch.rand(5, device=DEV)
    a2 = fp.get_action_and_value(flags, agent_ids=ids, seed=8)
    assert _same(a1, a2)
    assert torch.equal(fp.get_action(flags, agent_ids=ids, seed=8), a1[0])
    # the same value head and log-probs as the torch path evaluates for these actions
    _, lp, ent, v = fp.get_action_and_value(flags, a1[0], agent_ids=ids)
    assert torch.equal(v, a1[3])
    assert float((lp - a1[1]).abs().max()) < 1e-5 and float((ent - a1[2]).abs().max()) < 1e-5


def test_batched_duel_and_rollouts_are_functions_of_their_seeds():
    probe = _env(1)
    pa, pb = _policy(probe, 1), _policy(probe, 2)

    def duel():
        env = _env(128, base=9)
        return batched_duel(env, FusedPolicy(env, pa), FusedPolicy(env, pb), max_steps=40, policy_seed=3)

    r1, r2 = _twice(duel)
    assert torch.equal(r1, r2)

    def metrics():
        env = _env(128, base=9, stats="counters")
        return batched_duel(env, FusedPolicy(env, pa), FusedPolicy(env, pb), max_steps=40, return_result=False,
                            policy_seed=3)

    m1, m2 = _twice(metrics)
    assert _same(m1, m2)

    for reset in (True, False):
        def rollout():
            env = _env(128, base=9)
            ro = collect_rollout(env, FusedPolicy(env, pa), FusedPolicy(env, pb), num_env_steps=30,
                                 obs_storage_dtype="packed", reset=reset, policy_seed=11)
            if not reset:   # continue into a second rollout from where the first stopped
                ro2 = collect_rollout(env, FusedPolicy(env, pa), FusedPolicy(env, pb), num_env_steps=30,
                                      obs_storage_dtype="packed", reset=False, policy_seed=11)
                return [ro.__dict__, ro2.__dict__]
            return ro.__dict__

        x, y = _twice(rollout)
        assert _same(x, y), f"reset={reset}"


@pytest.mark.parametrize("grouped", [False, True])
def test_duel_pairs_are_functions_of_their_seeds(grouped):
    probe = _env(1)
    pols = [FusedPolicy(probe, _policy(probe, s)) for s in (1, 2, 3)]
    pairs = [(x, y) for x in pols for y in pols]
    r1, r2 = _twice(lambda: league.duel_pairs(EC, pairs, 16, max_steps=30, device=DEV, seed=2, env_id_base=40,
                                              collect_metrics=True, per_duel_metrics=True, grouped=grouped,
                                              policy_seed=17))
    assert _same(r1, r2)


def test_packed_ppo_collect_is_a_function_of_its_seeds():
    probe = _env(1)
    agent, opp = _policy(probe, 1), _policy(probe, 2)

    def collect():
        env = _env(128)
        tr = PackedPPO(env, agent, types.SimpleNamespace(learning_rate=1e-4), rollout_steps=20, policy_seed=5)
        a = tr.collect(FusedPolicy(env, opp)).__dict__
        torch.randperm(1000, device=DEV)       # what optimise draws between collects
        b = tr.collect(FusedPolicy(env, opp)).__dict__
        return [a, b]

    x, y = _twice(collect)
    assert _same(x, y)


# ---------------------------------------------------------------------------------------------------- 6. graph replay
def test_cuda_graph_replay_equals_the_eager_seeded_loop():
    B, T = 256, 50
    probe = _env(1)
    pa, pb = _policy(probe, 1), _policy(probe, 2)
    teams = [_team(probe, 0), _team(probe, 1)]

    def setup():
        env = _env(B, base=100)
        fps = [FusedPolicy(env, pa), FusedPolicy(env, pb)]
        flags = [env.use_action_mask[ids].repeat(B) for ids in teams]
        actions = torch.zeros((B, env.N_AGENTS), dtype=torch.uint8, device=DEV)

        def step():
            for fp, ids, f in zip(fps, teams, flags):
                fp.get_action_and_value(f, agent_ids=ids, env=env, seed=77, actions=actions)
            env.step(actions)

        return env, actions, step

    env, actions, step = setup()
    eager = []
    for _ in range(T + 1):
        step()
        eager.append(actions.clone())
    want_state = env.get_state()

    env, actions, step = setup()
    step()                                    # warm-up, eager: step 1
    got = [actions.clone()]
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    for _ in range(T):
        graph.replay()
        got.append(actions.clone())
    torch.cuda.synchronize()
    assert all(torch.equal(x, y) for x, y in zip(eager, got))
    st = env.get_state()
    for k in ("grid", "pos", "hp_q", "has_flag", "captures", "step", "episode"):
        assert np.array_equal(st[k], want_state[k]), k


# ---------------------------------------------------------------------------------------------------- 7. grouped vs per pair
class _RecordingPool(PolicyPool):
    log = []

    def act(self, plan, actions, env=None, seed=None):
        a = super().act(plan, actions, env, seed)
        _RecordingPool.log.append(actions.clone())
        return a


class _RecordingFused(FusedPolicy):
    log = []

    def get_action_and_value(self, *args, **kw):
        out = super().get_action_and_value(*args, **kw)
        _RecordingFused.log.append(kw["actions"].clone())
        return out


def test_grouped_duel_pairs_equal_replay_and_per_pair_draws(monkeypatch):
    D, seed, base, max_steps, ps = 12, 4, 21, 40, 1234
    probe = _env(1)
    mods = [_policy(probe, s) for s in (1, 2, 3, 4)]
    # cuBLAS sums the random policies' heads in another order on the two paths, so their logits may differ in the last
    # bits on every row; the last policy's logits are its action-head bias on every row, exact on both paths
    with torch.no_grad():
        mods[3].action_head.weight.zero_()
    fps = [_RecordingFused(probe, m) for m in mods]
    pairs = [(x, y) for x in fps for y in fps]
    P = len(pairs)
    monkeypatch.setattr(league, "PolicyPool", _RecordingPool)
    _RecordingPool.log = []
    results, _ = league.duel_pairs(EC, pairs, D, max_steps=max_steps, device=DEV, seed=seed, env_id_base=base,
                                   grouped=True, policy_seed=ps)
    log = _RecordingPool.log
    dense = GridworldCtfGPU(**EC, num_envs=P * D, device=DEV, seed=seed, env_id_base=base, reverse_team1_actions=True)
    dense.reset()
    for a in log:
        dense.step(a)
    caps = dense.flag_captures()
    assert torch.equal(results, torch.sign(caps[:, 0] - caps[:, 1]).reshape(P, D))

    # per-pair path: its step-1 actions are the buffer after the last policy call of step 1
    _RecordingFused.log = []
    league.duel_pairs(EC, pairs, D, max_steps=0, device=DEV, seed=seed, env_id_base=base, policy_seed=ps)
    per_pair = _RecordingFused.log[2 * P - 1]
    # logits of both paths at step 1, from a fresh env laid out as duel_pairs lays it out
    env = _env(P * D, base=base, seed=seed)
    team_ids = [_team(env, 0), _team(env, 1)]
    uniq, segments = league.pool_segments(pairs, D, team_ids)
    pool = PolicyPool(env, uniq)
    plan = pool.plan(segments)
    _, grouped_logits = pool.forward(plan)
    rows = []
    for p, pair in enumerate(pairs):
        for ids, pol in zip(team_ids, pair):
            rows.append(pol.forward_from_env(ids, env=env, envs=slice(p * D, (p + 1) * D))[1])
    equal = (torch.cat(rows).view(torch.int32) == grouped_logits.view(torch.int32)).all(1)
    n_equal = int(equal.sum())
    const = plan.policy_of_row == uniq.index(mods[3])
    print(f"rows with bitwise-equal logits: {n_equal} of {equal.numel()} "
          f"({int(equal[~const].sum())} of them of random-weight policies)")
    assert n_equal > 0 and bool(equal[const].all())
    f = plan.flat_index[equal]
    assert torch.equal(per_pair.view(-1)[f], log[0].view(-1)[f])


# ---------------------------------------------------------------------------------------------------- 8. rejections
def test_host_side_rejections():
    env = _env(8)
    head = torch.randn((16, 12), device=DEV)
    flat = torch.arange(16, device=DEV)
    masked = torch.zeros(16, dtype=torch.uint8, device=DEV)
    aout = torch.empty(16, dtype=torch.int64, device=DEV)
    lp, ent = torch.empty(16, device=DEV), torch.empty(16, device=DEV)
    actions = torch.empty((8, 8), dtype=torch.uint8, device=DEV)
    spare = torch.empty(64, dtype=torch.int64, device=DEV)
    st = env._state_struct
    good = dict(handle=env._handle, state=st, head=head.data_ptr(), stride=12, masked=masked.data_ptr(),
                flat=flat.data_ptr(), n=16, actions=actions.data_ptr(), aout=aout.data_ptr(), lp=lp.data_ptr(),
                ent=ent.data_ptr())

    def call(**over):
        a = {**good, **over}
        v = lambda x: C.c_void_p(x or None)
        return env._lib.ctf_sample_actions(a["handle"], a["state"], v(a["head"]), a["stride"], v(a["masked"]),
                                           v(a["flat"]), a["n"], 1, v(a["actions"]), v(a["aout"]), v(a["lp"]),
                                           v(a["ent"]), C.c_void_p(torch.cuda.current_stream().cuda_stream))

    assert call() == 0
    state_with = lambda envs: _native.CtfState(st.grid, st.agents, envs, st.stats, st.visits, st.hp)
    bad = {
        "null handle": dict(handle=C.c_void_p(None)),
        "null state.envs": dict(state=state_with(None)),
        "null head": dict(head=0),
        "null flat_index": dict(flat=0),
        "n_rows < 0": dict(n=-1),
        "head_stride < 10": dict(stride=9),
        "misaligned state.envs": dict(state=state_with(st.envs + 4)),
        "misaligned head": dict(head=head.data_ptr() + 2),
        "misaligned flat_index": dict(flat=spare.data_ptr() + 4),
        "misaligned action_out": dict(aout=spare.data_ptr() + 4 + 8 * 20),
        "misaligned logprob": dict(lp=lp.data_ptr() + 2),
        "misaligned entropy": dict(ent=ent.data_ptr() + 1),
        "logprob overlaps head": dict(lp=head.data_ptr() + 4 * 50),
        "entropy overlaps head": dict(ent=head.data_ptr()),
        "action_out overlaps flat_index": dict(aout=flat.data_ptr() + 8 * 15),
        "actions overlap masked": dict(actions=masked.data_ptr()),
        "logprob overlaps entropy": dict(lp=ent.data_ptr() + 4 * 3),
        "action_out overlaps actions": dict(aout=actions.data_ptr() + 8),
        "actions overlap logprob": dict(actions=lp.data_ptr() - 32),
    }
    for name, over in bad.items():
        assert call(**over) == -1, name
        assert env._lib.ctf_last_error().startswith(b"ctf_sample_actions: "), name
    # every output is optional, and zero rows launch nothing
    assert call(masked=0, actions=0, aout=0, lp=0, ent=0) == 0
    assert call(n=0) == 0
    assert env.take_faults() == 0


def test_value_errors():
    env = _env(8)
    pol = _policy(env, 1)
    fp = FusedPolicy(env, pol)
    ids = _team(env, 0)
    flags = env.use_action_mask[ids].repeat(8)
    bits = env.obs_bits[:, ids].reshape(-1, env.bits_words_per_agent)
    meta = env.meta[:, ids].reshape(-1, env.meta_size)
    with pytest.raises(ValueError):
        fp.get_action_and_value(flags, bits=bits, meta=meta, seed=1)
    with pytest.raises(ValueError):
        fp.get_action(flags, bits=bits, meta=meta, seed=1)
    with pytest.raises(ValueError):
        fp.get_action_and_value(flags, torch.zeros(len(flags), dtype=torch.long, device=DEV), agent_ids=ids, seed=1)
    with pytest.raises(ValueError):
        fp.get_action_and_value(flags, agent_ids=ids, seed=-1)
    with pytest.raises(ValueError):
        fp.get_action_and_value(flags, agent_ids=ids, seed=1 << 64)
    with pytest.raises(ValueError):
        fp.get_action_and_value(flags, agent_ids=ids, actions=torch.zeros((8, 8), dtype=torch.uint8, device=DEV))
    with pytest.raises(ValueError):
        fp.get_action_and_value(flags, agent_ids=ids, seed=1, actions=torch.zeros((8, 7), dtype=torch.uint8, device=DEV))
    dense = _env(8, dense_obs=True)
    with pytest.raises(ValueError):
        collect_rollout(dense, FusedPolicy(dense, pol), pol, num_env_steps=2, policy_seed=1)
    with pytest.raises(ValueError):
        collect_rollout(dense, pol, FusedPolicy(dense, pol), num_env_steps=2, policy_seed=1)
    with pytest.raises(ValueError):
        batched_duel(dense, FusedPolicy(dense, pol), pol, max_steps=2, policy_seed=1)
    with pytest.raises(ValueError):
        league.duel_pairs(EC, [(fp, pol)], 2, max_steps=2, device=DEV, policy_seed=1)
    with pytest.raises(ValueError):
        PackedPPO(env, pol, types.SimpleNamespace(learning_rate=1e-4), policy_seed=-3)
    pool = PolicyPool(env, [pol])
    plan = pool.plan([(0, slice(0, 8), ids)])
    with pytest.raises(ValueError):
        pool.act(plan, torch.zeros((8, 8), dtype=torch.uint8, device=DEV), seed=-1)
