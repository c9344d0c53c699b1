"""PolicyPool and ctf_policy_features_grouped (k_policy_trunk_grouped) on the GPU.

Rows are checked bit for bit against FusedPolicy.trunk_from_env of the segment's policy (the kernels share the
per-sample code); the heads against fp32 CtfPolicy within the inference contract (twice torch's own bf16 autocast error
+ 1e-3); the grouped league path by replaying the actions it took on a dense env.
"""
import ctypes as C

import pytest
import torch

from random_scenarios import random_env_config
from marl_ctf_development_b200 import _native, experiment_env_config
from marl_ctf_development_b200.env import GridworldCtfGPU, metrics_dict
from marl_ctf_development_b200.fused_policy import FusedPolicy, PolicyPool
from marl_ctf_development_b200 import league
from marl_ctf_development_b200.policy import CtfPolicy

from test_gpu_fused_policy import SCENARIOS, _bound, _policy, _stepped_env, _team

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
SENTINEL = 7.0   # no trunk row is all 7.0 (its pad columns are zeros)


def _ctas(env):
    """(k_policy_trunk, k_policy_trunk_grouped) CTAs per launch on this env's handle, from ctf_create's occupancy."""
    t, g = C.c_int(), C.c_int()
    _native.check(env._lib.ctf_policy_trunk_ctas(env._handle, C.byref(t), C.byref(g)))
    return t.value, g.value


def _envs_needed(ec):
    probe = GridworldCtfGPU(**ec, num_envs=1, device=DEV, packed_obs=True, dense_obs=False)
    return 8 * max(_ctas(probe)) + 16


def _segments(env, L):
    """Out-of-order segments over 3..5 policies: k from 1 to N, one env, an empty one, all envs, and 8 * CTAs +- 1
    samples for the CTA counts of both trunk kernels (one sample per warp of every CTA, plus or minus one)."""
    B, N = env.num_envs, env.N_AGENTS
    everyone = list(range(N))[::-1]
    t, g = _ctas(env)
    assert B >= 8 * max(t, g) + 2
    segs = [
        (2 % L, slice(5, 6), [N - 1]),
        (0, slice(0, B), everyone),
        (1, slice(0, 8 * t - 1), [0]),
        (3 % L, slice(1, 2 + 8 * t), [N - 1]),
        (0, slice(7, 7), [0]),
        (1, slice(2, 2 + 8 * g + 1), [N // 2]),
        (L - 1, slice(0, 8 * g - 1), [0]),
    ]
    for k in range(1, N + 1):
        segs.append(((k * 3) % L, slice(3 * k, 3 * k + 7), everyone[:k]))
    return segs


def _pool(env, L, seed=11, **kw):
    pols = [_policy(env, seed + i) for i in range(L)]
    for i, p in enumerate(pols):
        p.use_masking = kw.get("unmasked") != i
    return pols, PolicyPool(env, pols)


def _check_rows(env, pols, pool, plan):
    plan.features.fill_(SENTINEL)
    feat = pool.trunk(plan).clone()
    torch.cuda.synchronize()
    for (p, e0, e1, ids), (r0, r1) in zip(plan.segments, plan.seg_rows):
        if r0 == r1:
            continue
        want = FusedPolicy(env, pols[p]).trunk_from_env(ids, envs=slice(e0, e1))
        got = feat[plan.row_index[r0:r1]]
        assert torch.equal(got.view(torch.int16), want.view(torch.int16)), (p, e0, e1, ids)
    untouched = torch.ones(feat.shape[0], dtype=torch.bool, device=DEV)
    untouched[plan.row_index] = False
    assert bool((feat[untouched] == SENTINEL).all())
    return feat


# ---------------------------------------------------------------------------------------------------- 1. trunk rows
@pytest.mark.parametrize("steps", [0, 50])
@pytest.mark.parametrize("name", list(SCENARIOS))
def test_grouped_rows_equal_single_policy_rows(name, steps):
    ec = SCENARIOS[name]()
    env = _stepped_env(ec, _envs_needed(ec), steps)
    L = 3 + (len(name) + steps) % 3          # 3..5 policies
    pols, pool = _pool(env, L)
    plan = pool.plan(_segments(env, L))
    _check_rows(env, pols, pool, plan)
    # a rerun is bit-identical
    again = pool.trunk(plan).clone()
    assert torch.equal(again.view(torch.int16), pool.trunk(plan).view(torch.int16))


# ---------------------------------------------------------------------------------------------------- 2. heads
@pytest.mark.parametrize("name", ["8_arena", "random-4-G16", "random-29-G7"])
def test_heads_within_the_inference_contract(name):
    env = _stepped_env(SCENARIOS[name](), 37, 50)
    L = 4
    pols, pool = _pool(env, L)
    N = env.N_AGENTS
    segs = [(p, slice(3 * p, 3 * p + 20), list(range(N))[p % 2 :: 2] or [0]) for p in range(L)][::-1]
    plan = pool.plan(segs)
    value, logits = pool.forward(plan)
    assert value.shape == (plan.n_outputs, 1) and logits.shape == (plan.n_outputs, 9)
    assert value.dtype == logits.dtype == torch.float32
    for (p, e0, e1, ids), (r0, r1) in zip(plan.segments, plan.seg_rows):
        bits = env.obs_bits[e0:e1][:, ids].reshape(-1, env.bits_words_per_agent)
        meta = env.meta[e0:e1][:, ids].reshape(-1, env.meta_size)
        (ev, bv), (el, bl) = _bound(pols[p], env.unpack_obs(bits), meta, value[r0:r1], logits[r0:r1])
        assert ev <= bv, f"policy {p}: value error {ev} > {bv}"
        assert el <= bl, f"policy {p}: logit error {el} > {bl}"


# ---------------------------------------------------------------------------------------------------- 3. masking
def test_each_policy_masks_as_its_own_use_masking_says():
    env = _stepped_env(SCENARIOS["8_arena"](), 256, 10)
    B, N = env.num_envs, env.N_AGENTS
    masked_agents = [i for i in range(N) if float(env.use_action_mask[i]) == 1]
    assert masked_agents
    pols, pool = _pool(env, 3, unmasked=1)
    plan = pool.plan([(p, slice(p * 80, p * 80 + 80), list(range(N))) for p in range(3)])
    actions = torch.full((B, N), 255, dtype=torch.uint8, device=DEV)
    high_unmasked = 0
    for _ in range(20):
        a = pool.act(plan, actions)
        for p in range(3):
            sub = actions[p * 80 : p * 80 + 80][:, masked_agents]
            if p == 1:
                high_unmasked += int((sub > 4).sum())
            else:
                assert bool((sub <= 4).all()), p
        assert torch.equal(actions.view(-1)[plan.flat_index], a.to(torch.uint8))
    assert high_unmasked > 0                     # the unmasked policy does use actions 5..8 on those agents
    assert bool((actions[240:] == 255).all())    # envs outside every segment are not written


# ---------------------------------------------------------------------------------------------------- 4. duels
class _RecordingPool(PolicyPool):
    log = []

    def act(self, plan, actions, env=None):
        a = super().act(plan, actions, env)
        _RecordingPool.log.append(actions.clone())
        return a


def _replay(ec, log, B, seed):
    dense = GridworldCtfGPU(**ec, num_envs=B, device=DEV, seed=seed, reverse_team1_actions=True, stats="counters")
    dense.reset()
    for a in log:
        dense.step(a)
    return dense


@pytest.mark.parametrize("kind", ["symmetric_self_play", "non_symmetric"])
def test_grouped_duel_pairs_match_replay(kind, monkeypatch):
    ec = experiment_env_config("8_arena")
    D, seed, max_steps = 12, 4, 60
    probe = GridworldCtfGPU(**ec, num_envs=1, device=DEV, packed_obs=True, dense_obs=False)
    a, b, c = _policy(probe, 1), _policy(probe, 2), _policy(probe, 3)
    fa = FusedPolicy(probe, a)           # the pool runs a FusedPolicy's own CtfPolicy
    if kind == "symmetric_self_play":
        pairs = [(x, y) for x in (fa, b, c) for y in (fa, b, c)]
    else:
        pairs = [(x, y) for x in (fa, b) for y in (c,)] + [(c, b)]
    monkeypatch.setattr(league, "PolicyPool", _RecordingPool)
    _RecordingPool.log = []
    results, metrics = league.duel_pairs(ec, pairs, D, max_steps=max_steps, device=DEV, seed=seed,
                                         collect_metrics=True, per_duel_metrics=True, grouped=True)
    log = _RecordingPool.log
    P = len(pairs)
    assert results.shape == (P, D) and len(log) == min(max_steps + 1, probe.GAME_STEPS)
    dense = _replay(ec, log, P * D, seed)
    caps = dense.flag_captures()
    assert torch.equal(results, torch.sign(caps[:, 0] - caps[:, 1]).reshape(P, D))
    c_ = dense.counters().reshape(P, D, *dense.counters().shape[1:]).cpu().numpy()
    for p in range(P):
        for d in range(D):
            want = {k: v for k, v in metrics_dict(dense.ce, c_[p, d]).items() if k != "agent_visitation_maps"}
            got = {k: v for k, v in metrics[p][d].items() if k != "agent_visitation_maps"}
            assert got == want
    # the same structures as the per-pair path
    ref, ref_m = league.duel_pairs(ec, pairs, D, max_steps=5, device=DEV, seed=seed, collect_metrics=True)
    got, got_m = league.duel_pairs(ec, pairs, D, max_steps=5, device=DEV, seed=seed, collect_metrics=True, grouped=True)
    assert got.shape == ref.shape and got.dtype == ref.dtype
    assert [sorted(m) for m in got_m] == [sorted(m) for m in ref_m]


class _Harvest:
    def __init__(self):
        self.calls = []

    def harvest_metrics(self, metrics, label, iteration, scale, team_idx=None):
        self.calls.append((label, iteration, scale, team_idx, tuple(sorted(metrics))))


def test_league_entry_points_run_grouped():
    ec = experiment_env_config("0_the_split")
    probe = GridworldCtfGPU(**ec, num_envs=1, device=DEV, packed_obs=True, dense_obs=False)
    t1 = [FusedPolicy(probe, _policy(probe, i)) for i in range(3)]
    t2 = [_policy(probe, 10 + i) for i in range(2)]
    kw = dict(max_steps=20, device=DEV, seed=3)
    for fn, args in ((league.winrate_matrix_symmetric, (ec, t1, 4)), (league.winrate_matrix_non_symmetric, (ec, t1, t2, 4))):
        assert sorted(fn(*args, grouped=True, **kw)) == sorted(fn(*args, **kw))
    for fn, args in ((league.generate_metrics_symmetric, (ec, t1, 0, 3, 0, 1, 1, 1)),
                     (league.generate_metrics_non_symmetric, (ec, t1, t2, 0, 0, 3, 0, 1, 1, 1))):
        h_ref, h_grp = _Harvest(), _Harvest()
        n_ref, n_grp = fn(h_ref, *args, **kw), fn(h_grp, *args, grouped=True, **kw)
        assert n_ref == n_grp and h_ref.calls == h_grp.calls
    # a module and FusedPolicy views of it are one pool entry
    view = FusedPolicy(probe, t1[0].policy)
    res, _ = league.duel_pairs(ec, [(t1[0], view), (t1[0].policy, t1[1])], 2, grouped=True, **kw)
    assert res.shape == (2, 2)
    with pytest.raises(ValueError, match="grouped=True"):
        league.duel_pairs(ec, [(t1[0], object())], 2, grouped=True, **kw)


# ---------------------------------------------------------------------------------------------------- 5. CUDA graph
def test_graph_replay_is_bit_identical_and_follows_refresh():
    env = _stepped_env(SCENARIOS["8_arena"](), 64, 10)
    pols, pool = _pool(env, 3)
    N = env.N_AGENTS
    plan = pool.plan([(p, slice(16 * p, 16 * p + 30), list(range(N))) for p in range(3)])
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        pool.forward(plan)                        # warm-up outside the capture (cuBLAS handles, workspaces)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        gv, gl = pool.forward(plan)
    graph.replay()
    ev, el = pool.forward(plan)
    torch.cuda.synchronize()
    assert torch.equal(gl, el) and torch.equal(gv, ev)
    with torch.no_grad():
        for p in pols[1].parameters():
            p.mul_(-1.5)
    pool.refresh()
    graph.replay()
    ev2, el2 = pool.forward(plan)
    torch.cuda.synchronize()
    assert torch.equal(gl, el2) and torch.equal(gv, ev2)
    r0, r1 = plan.seg_rows[1]
    assert not torch.equal(el2[r0:r1], el[r0:r1])
    assert torch.equal(el2[: plan.seg_rows[0][1]], el[: plan.seg_rows[0][1]])   # other policies unchanged


# ---------------------------------------------------------------------------------------------------- 6. argument checks
def test_bad_arguments_are_rejected():
    env = _stepped_env(SCENARIOS["8_arena"](), 4, 0)
    N = env.N_AGENTS
    pols, pool = _pool(env, 2)
    lib = _native.load()
    stride = pool.stride
    feat = torch.zeros((40, stride), dtype=torch.bfloat16, device=DEV)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def seg(policy=0, e0=0, n=2, row=0, ids=(0, 1)):
        s = _native.CtfPolicySegment()
        s.env_begin, s.n_envs, s.out_row, s.policy, s.k = e0, n, row, policy, len(ids)
        for j, a in enumerate(ids[:8]):
            s.agent_ids[j] = a
        return s

    def call(segs=None, weights=None, n_pol=2, n_envs=4, out=None, st=stride, rows=40, packed=None, k=None):
        segs = [seg(), seg(policy=1, row=4)] if segs is None else segs
        arr = (_native.CtfPolicySegment * max(len(segs), 1))(*segs)
        if k is not None:
            arr[0].k = k
        return lib.ctf_policy_features_grouped(
            env._handle, pool._weights if weights is None else weights, n_pol, arr, len(segs),
            C.c_void_p(env.obs_bits.data_ptr() if packed is None else packed), C.c_void_p(env.meta.data_ptr()), n_envs,
            N, C.c_void_p(feat.data_ptr() if out is None else out), st, rows, stream)

    assert call() == 0
    assert call(segs=[seg(n=0), seg(policy=1, n=0, row=40)]) == 0     # empty segments: nothing is launched
    torch.cuda.synchronize()
    w = pool._weights
    null_w = (_native.CtfPolicyWeights * 2)(w[0], _native.CtfPolicyWeights(w[1].conv1_w, None, w[1].conv2_w, w[1].conv2_b))
    odd_w = (_native.CtfPolicyWeights * 2)(w[0], _native.CtfPolicyWeights(w[1].conv1_w + 4, w[1].conv1_b, w[1].conv2_w,
                                                                           w[1].conv2_b))
    bad = {
        "policy index": dict(segs=[seg(policy=2)]),
        "negative policy": dict(segs=[seg(policy=-1)]),
        "k = 0": dict(k=0),
        "k = 9": dict(k=9),
        "agent id": dict(segs=[seg(ids=(0, N))]),
        "env range": dict(segs=[seg(e0=3, n=2)]),
        "negative env": dict(segs=[seg(e0=-1, n=2)]),
        "rows outside": dict(segs=[seg(row=37)]),
        "negative row": dict(segs=[seg(row=-1)]),
        "overlap": dict(segs=[seg(), seg(policy=1, row=3)]),
        "stride": dict(st=stride - 8),
        "stride not multiple of 8": dict(st=stride + 4),
        "misaligned features": dict(out=feat.data_ptr() + 2),
        "null features": dict(out=0),
        "null packed": dict(packed=0),
        "null weight": dict(weights=null_w),
        "misaligned weight": dict(weights=odd_w),
        "too many policies": dict(n_pol=65),
        "no policies": dict(n_pol=0),
        "too many segments": dict(segs=[seg(n=0)] * 513),
    }
    for what, kw in bad.items():
        assert call(**kw) == -1, what
        assert lib.ctf_last_error().startswith(b"ctf_policy_features_grouped"), (what, lib.ctf_last_error())
    assert lib.ctf_policy_features_grouped(env._handle, None, 2, None, 0, None, None, 4, N, None, stride, 40, stream) == -1
    with pytest.raises(ValueError):
        pool.act(pool.plan([(0, slice(0, 4), [0])]), torch.zeros((4, N), dtype=torch.int64, device=DEV))
    with pytest.raises(ValueError):
        PolicyPool(env, [pols[0], pols[0]])


# ---------------------------------------------------------------------------------------------------- 7. scale
def test_all_pairs_of_8_policies_at_1024_duels():
    ec = experiment_env_config("8_arena")
    D, L = 1024, 8
    env = GridworldCtfGPU(**ec, num_envs=L * L * D, device=DEV, seed=1, reverse_team1_actions=True, dense_obs=False,
                          packed_obs=True)
    B, N = env.num_envs, env.N_AGENTS
    assert B == 65536
    g = torch.Generator(device=DEV).manual_seed(0)
    for _ in range(5):
        env.step(torch.randint(0, 9, (B, N), generator=g, device=DEV, dtype=torch.int64).to(torch.uint8))
    pols = [_policy(env, 30 + i) for i in range(L)]
    pairs = [(a, o) for a in pols for o in pols]
    uniq, segs = league.pool_segments(pairs, D, [_team(env, 0), _team(env, 1)])
    pool = PolicyPool(env, uniq)
    plan = pool.plan(segs)
    value, logits = pool.forward(plan)
    assert value.shape == (B * N, 1)
    assert bool(torch.isfinite(value).all()) and bool(torch.isfinite(logits).all())
    sub = torch.randperm(B * N, generator=g, device=DEV)[:512]
    flat = plan.flat_index[sub]
    bits = env.obs_bits.reshape(B * N, -1)[flat]
    meta = env.meta.reshape(B * N, -1)[flat]
    dense = env.unpack_obs(bits)
    pol_of = plan.policy_of_row[sub]
    for p in range(L):
        m = pol_of == p
        if bool(m.any()):
            (ev, bv), (el, bl) = _bound(uniq[p], dense[m], meta[m], value[sub][m], logits[sub][m])
            assert ev <= bv and el <= bl, (p, ev, bv, el, bl)
    actions = torch.empty((B, N), dtype=torch.uint8, device=DEV)
    pool.act(plan, actions)
    assert int(actions.max()) <= 8
