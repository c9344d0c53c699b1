"""FusedPolicy and ctf_policy_features (k_policy_trunk) on the GPU.

The trunk is checked against fused_policy.reference_features (its torch statement) to one bf16 ulp; the full forward
against fp32 CtfPolicy within twice torch's own bf16 autocast error on the same samples; the adapters by replaying the
actions the fused policies sampled on a dense env.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from hash_policy import HashPolicy, flag_targets
from random_scenarios import random_env_config
from marl_ctf_development_b200 import _native, experiment_env_config
from marl_ctf_development_b200.env import GridworldCtfGPU, metrics_dict
from marl_ctf_development_b200.fused_policy import FusedPolicy, reference_conv1, reference_features, trunk_dims
from marl_ctf_development_b200.league import duel_pairs
from marl_ctf_development_b200.policy import CtfPolicy
from marl_ctf_development_b200.rollout import batched_duel, collect_rollout

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
ULP = 2.0 ** -8   # one bf16 ulp of a value in [0.5, 1): tanh outputs lie in (-1, 1)
SCENARIOS = {
    "0_the_split": lambda: experiment_env_config("0_the_split"),
    "7_gridlocked": lambda: experiment_env_config("7_gridlocked"),
    "8_arena": lambda: experiment_env_config("8_arena"),
    "random-4-G16": lambda: random_env_config(4),
    "random-29-G7": lambda: random_env_config(29),
}


def _team(env, t):
    return [i for i in range(env.N_AGENTS) if env.AGENT_TEAMS[i] == t]


def _policy(env, seed):
    torch.manual_seed(seed)
    return CtfPolicy(9, env.n_channels, env.GRID_SIZE, env.meta_size).to(env.device).eval()


def _stepped_env(ec, B, steps, seed=3, **kw):
    """Dense + packed env after ``steps`` steps of HashPolicy actions (captures, mined blocks, respawns)."""
    env = GridworldCtfGPU(**ec, num_envs=B, device=DEV, seed=seed, reverse_team1_actions=True, packed_obs=True, **kw)
    B, N, Cn, G, M = env.num_envs, env.N_AGENTS, env.n_channels, env.GRID_SIZE, env.meta_size
    pol = HashPolicy(Cn * G * G, M, 11, flag_targets(env)).to(env.device)
    flags = env.use_action_mask.unsqueeze(0).expand(B, N).reshape(-1)
    for _ in range(steps):
        a = pol.get_action(env.obs.reshape(B * N, Cn, G, G).float(), env.meta.reshape(B * N, M), flags)
        env.step(a.reshape(B, N).to(torch.uint8))
    return env


def _samples(env, ids):
    """Dense float32 observations (unpacked from obs_bits) and metadata of agents ``ids`` of every env, env-major."""
    k = len(ids)
    bits = env.obs_bits[:, ids].reshape(-1, env.bits_words_per_agent)
    return env.unpack_obs(bits), env.meta[:, ids].reshape(env.num_envs * k, env.meta_size)


def _bound(pol, dense, meta, got_v, got_l):
    """max|fused - fp32| and the contract bound 2 * max|autocast_bf16 - fp32| + 1e-3, for value and logits."""
    with torch.no_grad():
        v32, l32 = pol(dense, meta)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            va, la = pol(dense, meta)
    out = []
    for got, ref, amp in ((got_v, v32, va.float()), (got_l, l32, la.float())):
        out.append((float((got - ref).abs().max()), 2 * float((amp - ref).abs().max()) + 1e-3))
    return out


class Recording(FusedPolicy):
    """Records every sampled batch (agent ids, env slice, actions) in one log shared by several policies."""

    def __init__(self, env, policy, log):
        super().__init__(env, policy)
        self.log = log

    def get_action_and_value(self, use_action_mask, action=None, **kw):
        out = super().get_action_and_value(use_action_mask, action, **kw)
        self.log.append((list(kw["agent_ids"]), kw.get("envs"), out[0].clone()))
        return out


def _assert_trunk_close(feat, pol, dense, meta):
    """Trunk rows against reference_features, per element: conv1 is the same ordered fp32 sum as the kernel's, so what
    remains is conv2's fp32 tensor-core accumulation (bounded by 144 * 2^-22 * sum|terms|, twice the worst case of
    round-to-nearest, as the hardware's alignment may truncate) plus one bf16 rounding (one ulp of the larger value).
    The contract's global bound, 2^-8, must hold as well; metadata columns are exact and pad columns zero."""
    M = meta.shape[1]
    ref = reference_features(pol, dense, meta)
    K1 = ref.shape[1]
    got = feat[:, :K1].float()
    h1 = reference_conv1(pol, dense)
    abs_sum = torch.nn.functional.conv2d(h1.abs().double(), pol.conv2.weight.detach().bfloat16().double().abs())
    abs_sum = (abs_sum + pol.conv2.bias.detach().double().abs().view(1, -1, 1, 1)).reshape(len(ref), -1).float()
    g, r = got[:, : K1 - M], ref[:, : K1 - M]
    big = torch.maximum(g.abs(), r.abs()).clamp_min(2.0**-126)
    ulp = torch.exp2(torch.floor(torch.log2(big)) - 7)
    allowed = ulp + 144 * 2.0**-22 * abs_sum
    excess = (g - r).abs() - allowed
    worst = int(excess.argmax())
    assert float(excess.max()) <= 0, (f"element {divmod(worst, K1 - M)}: got {float(g.reshape(-1)[worst])}, "
                                      f"want {float(r.reshape(-1)[worst])}, allowed {float(allowed.reshape(-1)[worst])}")
    assert float((g - r).abs().max()) <= ULP
    assert torch.equal(got[:, K1 - M :], meta.bfloat16().float())
    assert not feat[:, K1:].any()


# ---------------------------------------------------------------------------------------------------- 1. trunk vs spec
@pytest.mark.parametrize("steps", [0, 50])
@pytest.mark.parametrize("name", list(SCENARIOS))
def test_trunk_matches_reference_features(name, steps):
    env = _stepped_env(SCENARIOS[name](), 37, steps)
    K1 = trunk_dims(env.n_channels, env.GRID_SIZE, env.meta_size)[0]
    M = env.meta_size
    for t in (0, 1):
        ids = _team(env, t)
        pol = _policy(env, 5 + t)
        fp = FusedPolicy(env, pol)
        feat = fp.trunk_from_env(ids).clone()
        assert feat.shape == (37 * len(ids), fp.stride) and feat.dtype == torch.bfloat16
        dense, meta = _samples(env, ids)
        assert torch.equal(dense, env.obs[:, ids].reshape(dense.shape))   # packed copy == dense observations
        assert feat.shape[1] >= K1 and meta.shape[1] == M
        _assert_trunk_close(feat, pol, dense, meta)


def test_trunk_is_exact_for_any_binary_input():
    """Every bit pattern, not only one-hot cells: random words through the contiguous-buffer path (G = 16)."""
    env = _stepped_env(SCENARIOS["random-4-G16"](), 8, 0)
    pol = _policy(env, 2)
    fp = FusedPolicy(env, pol)
    g = torch.Generator(device=DEV).manual_seed(0)
    S, wpa = 300, env.bits_words_per_agent
    bits = torch.randint(-(2**31), 2**31 - 1, (S, wpa), generator=g, device=DEV, dtype=torch.int64).to(torch.int32)
    bits[:100] &= torch.randint(0, 2**31 - 1, (100, wpa), generator=g, device=DEV, dtype=torch.int64).to(torch.int32)
    meta = torch.randn((S, env.meta_size), generator=g, device=DEV)
    feat = fp.trunk_packed(bits, meta)
    _assert_trunk_close(feat, pol, env.unpack_obs(bits), meta)


# ---------------------------------------------------------------------------------------------------- 2. full forward
@pytest.mark.parametrize("name", ["8_arena", "random-4-G16", "random-29-G7"])
def test_forward_and_log_probs_against_fp32_ctf_policy(name):
    env = _stepped_env(SCENARIOS[name](), 37, 50)
    B = env.num_envs
    for t in (0, 1):
        ids = _team(env, t)
        k = len(ids)
        pol = _policy(env, 7 + t)
        fp = FusedPolicy(env, pol)
        value, logits = fp.forward_from_env(ids)
        assert value.shape == (B * k, 1) and logits.shape == (B * k, 9) and value.dtype == logits.dtype == torch.float32
        dense, meta = _samples(env, ids)
        (ev, bv), (el, bl) = _bound(pol, dense, meta, value, logits)
        assert ev <= bv, f"value error {ev} > {bv}"
        assert el <= bl, f"logit error {el} > {bl}"
        flags = env.use_action_mask[ids].unsqueeze(0).expand(B, k).reshape(-1)
        g = torch.Generator(device=DEV).manual_seed(t)
        act = torch.where(flags == 1, torch.randint(0, 5, flags.shape, generator=g, device=DEV),
                          torch.randint(0, 9, flags.shape, generator=g, device=DEV))
        a, lp, ent, v = fp.get_action_and_value(flags, act, agent_ids=ids)
        with torch.no_grad():
            _, lp32, _, _ = pol.get_action_and_value(dense, meta, flags, act)
        assert torch.equal(a, act) and torch.equal(v, value)
        # log-softmax moves by at most twice the largest logit change
        assert float((lp - lp32).abs().max()) <= 2 * el + 1e-4
        assert bool(torch.isfinite(ent).all())


# ---------------------------------------------------------------------------------------------------- 3. addressing
def test_in_place_and_contiguous_addressing_give_identical_rows():
    env = _stepped_env(SCENARIOS["8_arena"](), 37, 50)
    pol = _policy(env, 1)
    fp = FusedPolicy(env, pol)
    for t in (0, 1):
        ids = _team(env, t)
        a = fp.trunk_from_env(ids).clone()
        b = fp.trunk_from_env(ids).clone()
        assert torch.equal(a.view(torch.int16), b.view(torch.int16))          # deterministic
        bits = env.obs_bits[:, ids].reshape(-1, env.bits_words_per_agent).contiguous()
        meta = env.meta[:, ids].reshape(-1, env.meta_size).contiguous()
        c = fp.trunk_packed(bits, meta).clone()
        assert torch.equal(a.view(torch.int16), c.view(torch.int16))
        part = fp.trunk_from_env(ids, envs=slice(5, 20)).clone()               # an env sub-range
        assert torch.equal(part.view(torch.int16), a[5 * len(ids) : 20 * len(ids)].view(torch.int16))
    # a different id order is a different sample order
    ids = _team(env, 0)[::-1]
    r = fp.trunk_from_env(ids).clone()
    assert torch.equal(r.view(torch.int16)[: len(ids)], fp.trunk_packed(
        env.obs_bits[0, ids].contiguous(), env.meta[0, ids].contiguous()).view(torch.int16))


# ---------------------------------------------------------------------------------------------------- 4. rollout
@pytest.mark.parametrize("built_on", ["rollout_env", "other_env_same_B", "other_env_8_envs"])
def test_rollout_on_a_packed_only_env(built_on):
    """The fused policies may have been built on any env of the same shapes: the rollout reads the env it is given."""
    ec = experiment_env_config("8_arena")
    B, T, seed = 64, 40, 5
    env = GridworldCtfGPU(**ec, num_envs=B, device=DEV, seed=seed, reverse_team1_actions=True, dense_obs=False,
                          packed_obs=True)
    assert env.obs is None
    home = env
    if built_on != "rollout_env":
        # another env whose buffers hold different observations (stepped with random actions)
        home = GridworldCtfGPU(**ec, num_envs=B if built_on == "other_env_same_B" else 8, device=DEV, seed=seed + 1,
                               reverse_team1_actions=True, dense_obs=False, packed_obs=True)
        g = torch.Generator(device=DEV).manual_seed(1)
        for _ in range(7):
            home.step(torch.randint(0, 9, (home.num_envs, home.N_AGENTS), generator=g, device=DEV).to(torch.uint8))
    log = []
    pol_a, pol_b = _policy(env, 1), _policy(env, 2)
    agent, opponent = Recording(home, pol_a, log), Recording(home, pol_b, log)
    with pytest.raises(ValueError, match="dense_obs=True"):
        collect_rollout(env, pol_a, opponent, num_env_steps=2, obs_storage_dtype="packed")
    with pytest.raises(ValueError, match="packed"):
        collect_rollout(env, agent, opponent, num_env_steps=2)
    log.clear()
    ro = collect_rollout(env, agent, opponent, num_env_steps=T, obs_storage_dtype="packed")
    mine, theirs = _team(env, 0), _team(env, 1)
    apt = len(mine)
    assert len(log) == 2 * T

    # replay both sides' sampled actions on a dense env: the stored rewards and actions come back exactly
    dense = GridworldCtfGPU(**ec, num_envs=B, device=DEV, seed=seed, reverse_team1_actions=True)
    dense.reset()
    actions = torch.empty((B, env.N_AGENTS), dtype=torch.uint8, device=DEV)
    for t in range(T):
        (ids_a, _, a), (ids_o, _, o) = log[2 * t], log[2 * t + 1]
        assert ids_a == mine and ids_o == theirs
        actions[:, mine] = a.reshape(B, apt).to(torch.uint8)
        actions[:, theirs] = o.reshape(B, len(theirs)).to(torch.uint8)
        assert torch.equal(ro.actions[t * apt : (t + 1) * apt], a.reshape(B, apt).t().float())
        assert torch.equal(ro.metadata_states[t * apt : (t + 1) * apt], dense.meta[:, mine].transpose(0, 1))
        _, _, rewards, _, _ = dense.step(actions)
        assert torch.equal(ro.rewards[t * apt : (t + 1) * apt], rewards[:, mine].t()), f"rewards differ at step {t}"
    assert torch.equal(ro.next_grid_state, dense.obs[:, min(mine)].float())

    # fp32 CtfPolicy on the unpacked stored observations: values and log-probs within the contract
    g = ro.unpack_grid_states(env).reshape(T * apt * B, env.n_channels, env.GRID_SIZE, env.GRID_SIZE)
    m = ro.metadata_states.reshape(T * apt * B, -1)
    f = ro.use_action_mask.reshape(-1)
    act = ro.actions.reshape(-1).long()
    with torch.no_grad():
        _, lp32, _, v32 = pol_a.get_action_and_value(g, m, f, act)
        v32, l32 = pol_a(g, m)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            va, la = pol_a(g, m)
    bound_v = 2 * float((va.float() - v32).abs().max()) + 1e-3
    bound_l = 2 * float((la.float() - l32).abs().max()) + 1e-3
    assert float((ro.values.reshape(-1) - v32.reshape(-1)).abs().max()) <= bound_v
    assert float((ro.logprobs.reshape(-1) - lp32).abs().max()) <= 2 * bound_l + 1e-4
    masked = ro.use_action_mask == 1
    assert bool(masked.any()) and bool((ro.actions[masked] <= 4).all())


# ---------------------------------------------------------------------------------------------------- 5. duels
def _no_maps(m):
    return {k: v for k, v in m.items() if k != "agent_visitation_maps"}


def test_batched_duel_with_fused_policies_matches_replay():
    ec = experiment_env_config("8_arena")
    B, seed = 48, 8
    env = GridworldCtfGPU(**ec, num_envs=B, device=DEV, seed=seed, reverse_team1_actions=True, dense_obs=False,
                          packed_obs=True, stats="counters")
    log = []
    result = batched_duel(env, Recording(env, _policy(env, 3), log), Recording(env, _policy(env, 4), log), max_steps=60)
    dense = GridworldCtfGPU(**ec, num_envs=B, device=DEV, seed=seed, reverse_team1_actions=True, stats="counters")
    dense.reset()
    actions = torch.empty((B, env.N_AGENTS), dtype=torch.uint8, device=DEV)
    assert len(log) % 2 == 0 and len(log) // 2 == min(61, env.GAME_STEPS)
    for s in range(len(log) // 2):
        for ids, _, a in log[2 * s : 2 * s + 2]:
            actions[:, ids] = a.reshape(B, len(ids)).to(torch.uint8)
        dense.step(actions)
    caps = dense.flag_captures()
    assert torch.equal(result, torch.sign(caps[:, 0] - caps[:, 1]))
    assert torch.equal(env.counters(), dense.counters())


def test_duel_pairs_with_fused_policies_matches_replay():
    ec = experiment_env_config("0_the_split")
    D, seed, max_steps = 16, 6, 50
    probe = GridworldCtfGPU(**ec, num_envs=1, device=DEV, packed_obs=True, dense_obs=False)
    log = []
    a, b = Recording(probe, _policy(probe, 1), log), Recording(probe, _policy(probe, 2), log)
    pairs = [(a, b), (b, a)]
    results, metrics = duel_pairs(ec, pairs, D, max_steps=max_steps, device=DEV, seed=seed, collect_metrics=True)
    P = len(pairs)
    dense = GridworldCtfGPU(**ec, num_envs=P * D, device=DEV, seed=seed, reverse_team1_actions=True, stats="counters")
    dense.reset()
    actions = torch.empty((P * D, dense.N_AGENTS), dtype=torch.uint8, device=DEV)
    per_step = 2 * P
    assert len(log) % per_step == 0
    for s in range(len(log) // per_step):
        for ids, sl, act in log[per_step * s : per_step * (s + 1)]:
            actions[sl, ids] = act.reshape(D, len(ids)).to(torch.uint8)
        dense.step(actions)
    caps = dense.flag_captures()
    assert torch.equal(results, torch.sign(caps[:, 0] - caps[:, 1]).reshape(P, D))
    c = dense.counters().reshape(P, D, *dense.counters().shape[1:]).cpu().numpy()
    for p in range(P):
        assert _no_maps(metrics[p]) == _no_maps(metrics_dict(dense.ce, c[p].sum(0)))


def test_stock_policy_on_a_packed_only_env_is_refused():
    ec = experiment_env_config("8_arena")
    env = GridworldCtfGPU(**ec, num_envs=4, device=DEV, reverse_team1_actions=True, dense_obs=False, packed_obs=True)
    pol = _policy(env, 0)
    with pytest.raises(ValueError, match="dense_obs=True"):
        batched_duel(env, FusedPolicy(env, pol), pol, max_steps=2)


# ---------------------------------------------------------------------------------------------------- 6. CUDA graph
def test_graph_replay_is_bit_identical_and_follows_refresh():
    env = _stepped_env(SCENARIOS["8_arena"](), 64, 10)
    pol = _policy(env, 9)
    fp = FusedPolicy(env, pol)
    ids = _team(env, 1)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fp.forward_from_env(ids)                    # warm-up outside the capture (cuBLAS handles, workspaces)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        gv, gl = fp.forward_from_env(ids)
    graph.replay()
    ev, el = fp.forward_from_env(ids)
    torch.cuda.synchronize()
    assert torch.equal(gl, el) and torch.equal(gv, ev)
    with torch.no_grad():
        for p in pol.parameters():
            p.mul_(-1.5)
    fp.refresh()
    graph.replay()
    ev2, el2 = fp.forward_from_env(ids)
    torch.cuda.synchronize()
    assert torch.equal(gl, el2) and torch.equal(gv, ev2)
    assert not torch.equal(el2, el)


# ---------------------------------------------------------------------------------------------------- 7. argument checks
def test_bad_arguments_are_rejected():
    env = _stepped_env(SCENARIOS["8_arena"](), 4, 0)
    Cn, G, M, N, wpa = env.n_channels, env.GRID_SIZE, env.meta_size, env.N_AGENTS, env.bits_words_per_agent
    pol = _policy(env, 0)
    fp = FusedPolicy(env, pol)
    for ids in ([N], [-1], [], [0] * 9):
        with pytest.raises(ValueError):
            fp.forward_from_env(ids)
    ok_bits, ok_meta = env.obs_bits[:, 0].contiguous(), env.meta[:, 0].contiguous()
    for bits, meta in ((ok_bits.float(), ok_meta), (ok_bits[:, 1:], ok_meta), (ok_bits, ok_meta[:, 1:]),
                       (ok_bits, ok_meta.double()), (ok_bits, ok_meta[:2])):
        with pytest.raises(ValueError):
            fp.forward_packed(bits, meta)
    for shape in ((9, Cn + 1, G, M), (9, Cn, G + 1, M), (9, Cn, G, M + 1), (8, Cn, G, M)):
        with pytest.raises(ValueError):
            FusedPolicy(env, CtfPolicy(*shape).to(DEV))
    with pytest.raises(ValueError):
        FusedPolicy(env, pol).forward_from_env([0], env=GridworldCtfGPU(**experiment_env_config("0_the_split"),
                                                                       num_envs=2, device=DEV, packed_obs=True))
    dense_only = GridworldCtfGPU(**experiment_env_config("8_arena"), num_envs=2, device=DEV)
    with pytest.raises(ValueError, match="packed_obs"):
        FusedPolicy(dense_only, pol).forward_from_env([0])

    # the C entry point validates on its own
    lib = _native.load()
    k1, stride = trunk_dims(Cn, G, M)
    feat = torch.zeros((4 * 2, stride + 8), dtype=torch.bfloat16, device=DEV)
    ids2 = (C.c_uint8 * 2)(0, 2)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    w = fp._weights

    def call(packed=env.obs_bits.data_ptr(), meta=env.meta.data_ptr(), ape=N, ids=ids2, k=2, out=feat.data_ptr(),
             st=stride, weights=C.byref(w)):
        return lib.ctf_policy_features(env._handle, weights, C.c_void_p(packed), C.c_void_p(meta), 4, ape, ids, k,
                                       C.c_void_p(out), st, stream)

    assert call() == 0
    torch.cuda.synchronize()
    bad = [
        dict(k=0), dict(k=9), dict(ape=2), dict(st=k1), dict(st=stride - 8), dict(out=feat.data_ptr() + 2),
        dict(packed=0), dict(meta=0), dict(out=0), dict(ids=None), dict(weights=None),
        dict(weights=C.byref(_native.CtfPolicyWeights(w.conv1_w, w.conv1_b + 2, w.conv2_w, w.conv2_b))),
        dict(weights=C.byref(_native.CtfPolicyWeights(w.conv1_w, w.conv1_b, w.conv2_w, w.conv2_b + 2))),
    ]
    for kw in bad:
        assert call(**kw) == -1, kw
        assert lib.ctf_last_error().startswith(b"ctf_policy_features"), kw
    null_w = _native.CtfPolicyWeights(w.conv1_w, None, w.conv2_w, w.conv2_b)
    assert call(weights=C.byref(null_w)) == -1


# ---------------------------------------------------------------------------------------------------- 8. scale
def test_one_forward_per_team_at_65536_envs():
    ec = experiment_env_config("8_arena")
    B = 65536
    env = GridworldCtfGPU(**ec, num_envs=B, device=DEV, seed=1, reverse_team1_actions=True, dense_obs=False,
                          packed_obs=True)
    g = torch.Generator(device=DEV).manual_seed(0)
    for _ in range(5):
        env.step(torch.randint(0, 9, (B, env.N_AGENTS), generator=g, device=DEV, dtype=torch.int64).to(torch.uint8))
    for t in (0, 1):
        ids = _team(env, t)
        k = len(ids)
        pol = _policy(env, 20 + t)
        fp = FusedPolicy(env, pol)
        value, logits = fp.forward_from_env(ids)
        assert value.shape == (B * k, 1) and bool(torch.isfinite(value).all()) and bool(torch.isfinite(logits).all())
        sub = torch.randperm(B * k, generator=g, device=DEV)[:512]
        bits = env.obs_bits[:, ids].reshape(B * k, -1)[sub]
        meta = env.meta[:, ids].reshape(B * k, -1)[sub]
        (ev, bv), (el, bl) = _bound(pol, env.unpack_obs(bits), meta, value[sub], logits[sub])
        assert ev <= bv and el <= bl, (ev, bv, el, bl)
    assert np.isfinite(float(value.double().sum()))
