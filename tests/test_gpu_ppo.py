"""ppo.py on the GPU: ctf_gae (k_gae) bit for bit against reference_advantages, its rejections and graph replay, the
bootstrap of PackedPPO.collect, the gradient of a chunked PackedPPO minibatch against fp32 CtfPolicy, early stopping,
and an update that learns and leaves the inference weights in sync."""
import ctypes as C
import math
import types

import pytest
import torch

from test_gpu_fused_policy import DEV, _bound, _policy, _team
from marl_ctf_development_b200 import PackedPPO, experiment_env_config
from marl_ctf_development_b200.env import GridworldCtfGPU
from marl_ctf_development_b200.fused_policy import FusedPolicy
from marl_ctf_development_b200.ppo import advantages, ppo_loss, reference_advantages

pytestmark = pytest.mark.gpu


def _env(B, game_steps=None, **kw):
    ec = experiment_env_config("8_arena")
    if game_steps is not None:
        ec = dict(ec, GAME_STEPS=game_steps)
    kw = dict(dict(seed=2, reverse_team1_actions=True, dense_obs=False, packed_obs=True), **kw)
    return GridworldCtfGPU(**ec, num_envs=B, device=DEV, **kw)


def _args(**kw):
    a = dict(num_minibatches=4, update_epochs=4, gamma=0.99, gae_lambda=0.95, norm_adv=True, clip_coef=0.2,
             clip_vloss=True, ent_coef=0.01, vf_coef=0.5, max_grad_norm=0.5, target_kl=None, learning_rate=2.5e-4,
             gae=True)
    a.update(kw)
    return types.SimpleNamespace(**a)


@pytest.fixture(scope="module")
def small_env():
    return _env(2)


# ---------------------------------------------------------------------------------------------------- 1. bit equality
def _gae_inputs(T, apt, B, seed, zero_bootstrap):
    """Rewards and values with exact zeros and magnitudes from 1e-4 to 1e20 mixed in."""
    g = torch.Generator(device=DEV).manual_seed(seed)

    def one(shape):
        x = torch.randn(shape, generator=g, device=DEV)
        scale = 10.0 ** torch.randint(-4, 21, shape, generator=g, device=DEV).float()
        x = torch.where(torch.rand(shape, generator=g, device=DEV) < 0.2, x * scale, x)
        return torch.where(torch.rand(shape, generator=g, device=DEV) < 0.1, torch.zeros_like(x), x)

    r, v = one((T * apt, B)), one((T * apt, B))
    nv = torch.zeros((apt, B), device=DEV) if zero_bootstrap else one((apt, B))
    return r, v, nv


def _ro(r, v):
    return types.SimpleNamespace(rewards=r, values=v)


@pytest.mark.parametrize("zero_bootstrap", [True, False])
@pytest.mark.parametrize("gamma,lam", [(0.99, 0.95), (1.0, 1.0), (0.9, 0.0)])
@pytest.mark.parametrize("shape", [(1, 1, 1), (7, 3, 33), (32, 4, 4101), (500, 4, 65536)])
def test_gae_is_bit_equal_to_the_reference(small_env, shape, gamma, lam, zero_bootstrap):
    T, apt, B = shape
    r, v, nv = _gae_inputs(T, apt, B, T * 7 + B, zero_bootstrap)
    adv, ret = advantages(small_env, _ro(r, v), nv, gamma, lam)
    want_adv, want_ret = reference_advantages(r, v, nv, gamma, lam)
    assert adv.shape == (T * apt, B) and ret.shape == (T * apt, B)
    assert torch.equal(adv, want_adv)
    assert torch.equal(ret, want_ret)


# ---------------------------------------------------------------------------------------------------- 2. graph replay
def test_gae_graph_replay(small_env):
    T, apt, B = 40, 4, 1000
    r, v, nv = _gae_inputs(T, apt, B, 5, False)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        advantages(small_env, _ro(r, v), nv, 0.99, 0.95)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        adv, ret = advantages(small_env, _ro(r, v), nv, 0.99, 0.95)
    for seed in (6, 7):
        r2, v2, nv2 = _gae_inputs(T, apt, B, seed, False)
        r.copy_(r2), v.copy_(v2), nv.copy_(nv2)
        graph.replay()
        torch.cuda.synchronize()
        want_adv, want_ret = reference_advantages(r, v, nv, 0.99, 0.95)
        assert torch.equal(adv, want_adv) and torch.equal(ret, want_ret)


# ---------------------------------------------------------------------------------------------------- 3. rejections
def test_gae_rejections(small_env):
    lib, h = small_env._lib, small_env._handle
    T, apt, B = 3, 2, 5
    n = T * apt * B
    buf = torch.zeros(5 * n + 2 * apt * B + 8, device=DEV)
    base = buf.data_ptr()
    # byte addresses: rewards, values, next_value, advantages and returns, apart and 16-byte aligned
    r, v, nv = base, base + 4 * n, base + 8 * n
    adv, ret = nv + 4 * apt * B + 64, nv + 4 * n + 4 * apt * B + 128
    ok = dict(r=r, v=v, nv=nv, adv=adv, ret=ret, T=T, apt=apt, B=B, g=0.99, gl=0.95)

    def call(**kw):
        a = dict(ok, **kw)
        return lib.ctf_gae(h, C.c_void_p(a["r"]), C.c_void_p(a["v"]), C.c_void_p(a["nv"]), C.c_void_p(a["adv"]),
                           C.c_void_p(a["ret"]), a["T"], a["apt"], a["B"], a["g"], a["gl"], None)

    assert call() == 0
    torch.cuda.synchronize()
    bad = [dict(r=None), dict(v=None), dict(nv=None), dict(adv=None), dict(ret=None),
           dict(T=0), dict(T=-1), dict(apt=0), dict(apt=9), dict(B=0), dict(B=-3),
           dict(g=math.nan), dict(g=math.inf), dict(g=-0.1), dict(g=1.5),
           dict(gl=math.nan), dict(gl=-math.inf), dict(gl=-1e-3), dict(gl=1.01),
           dict(adv=r), dict(adv=r + 4 * (n - 1)), dict(ret=v + 4), dict(adv=v - 4 * (n - 1)), dict(ret=nv + 4),
           dict(adv=nv - 4 * n + 4), dict(ret=adv), dict(ret=adv + 4 * (n - 1)), dict(adv=adv + 2)]
    for kw in bad:
        lib.ctf_get_sizes(None, None)   # leaves a message that does not start with ctf_gae
        rc = call(**kw)
        assert rc == -1, kw
        assert lib.ctf_last_error().startswith(b"ctf_gae"), (kw, lib.ctf_last_error())


# ---------------------------------------------------------------------------------------------------- 4. bootstrap
def test_collect_bootstrap_and_advantages_from_a_rollout():
    env = _env(64, game_steps=12)
    pol, opp = _policy(env, 11), _policy(env, 12)
    tr = PackedPPO(env, pol, _args())
    opponent = FusedPolicy(env, opp)
    B = env.num_envs
    for train_team1 in (True, False):
        mine = _team(env, 0 if train_team1 else 1)
        apt = len(mine)
        ro = tr.collect(opponent, train_team1=train_team1)
        assert ro.packed and ro.rewards.shape == (12 * apt, B)
        assert torch.equal(ro.next_value, torch.zeros((apt, B), device=DEV))
        ro = tr.collect(opponent, train_team1=train_team1, num_env_steps=5)
        assert ro.rewards.shape == (5 * apt, B)
        v, _ = FusedPolicy(env, pol).forward_from_env(mine)
        assert torch.equal(ro.next_value, v.reshape(B, apt).t())
        assert bool(ro.next_value.abs().sum() > 0)
        adv, ret = tr.advantages(ro)
        want_adv, want_ret = reference_advantages(ro.rewards, ro.values, ro.next_value, 0.99, 0.95)
        assert torch.equal(adv, want_adv) and torch.equal(ret, want_ret)
    with pytest.raises(ValueError):
        tr.collect(opponent, num_env_steps=13)


def test_trainer_rejects_unsupported_setups():
    with pytest.raises(ValueError):
        PackedPPO(_env(4, dense_obs=True, packed_obs=False), _policy(_env(4), 1), _args())
    with pytest.raises(ValueError):
        env = _env(4, reverse_team1_actions=False)
        PackedPPO(env, _policy(env, 1), _args())
    env = _env(4)
    with pytest.raises(ValueError):
        PackedPPO(env, FusedPolicy(env, _policy(env, 1)), _args())
    with pytest.raises(ValueError):
        PackedPPO(env, _policy(env, 1), _args(gae=False))


# ---------------------------------------------------------------------------------------------------- 5. gradients
class _GradRecorder:
    """An optimiser that records the gradients it is asked to step with and changes nothing."""

    def __init__(self, params):
        self.params, self.grads = list(params), []

    def zero_grad(self):
        for p in self.params:
            p.grad = None

    def step(self):
        self.grads.append([p.grad.clone() for p in self.params])


def test_chunked_minibatch_gradient_against_fp32_ctf_policy():
    env = _env(64)
    pol, opp = _policy(env, 21), _policy(env, 22)
    args = _args(num_minibatches=1, update_epochs=1, max_grad_norm=math.inf)
    tr = PackedPPO(env, pol, args, optimizer=_GradRecorder(pol.parameters()))
    ro = tr.collect(FusedPolicy(env, opp), num_env_steps=16)
    adv, ret = tr.advantages(ro)
    n = ro.rewards.numel()
    tr.chunk = n // 3 + 7                                  # three uneven chunks
    tr.optimise(ro, adv, ret)
    got = dict(zip([k for k, _ in pol.named_parameters()], tr.optimizer.grads[0]))
    dense = env.unpack_obs(ro.grid_states.reshape(-1, env.bits_words_per_agent))
    meta = ro.metadata_states.reshape(-1, env.meta_size)
    flat = [x.reshape(-1) for x in (ro.use_action_mask, ro.logprobs, ro.values, adv, ret)]
    act = ro.actions.reshape(-1).long()
    ref = []
    for amp in (False, True):
        pol.zero_grad()
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
            _, lp, ent, v = pol.get_action_and_value(dense, meta, flat[0], act)
        ppo_loss(lp.float(), ent.float(), v.float(), flat[1], flat[2], flat[3], flat[4], args)[0].backward()
        ref.append({k: p.grad.clone() for k, p in pol.named_parameters()})
    pol.zero_grad()
    g32, gamp = ref
    for k, _ in pol.named_parameters():
        err = float((got[k] - g32[k]).norm())
        allowed = 2 * float((gamp[k] - g32[k]).norm()) + 1e-3 * float(g32[k].norm())
        assert err <= allowed, f"{k}: |packed - fp32| = {err} > {allowed}"


# ---------------------------------------------------------------------------------------------------- 6. precision
def test_rollout_and_update_log_probs_agree_within_the_inference_contract():
    """The rollout's log-probs come from the bf16 inference head, the update's from train_head (bf16 fc1/fc2, fp32
    heads).  Each side's logits are within the logit bound bl of fp32 CtfPolicy (the contract of
    test_gpu_fused_policy), so the two logit vectors differ by at most 2 bl and a log-softmax, which moves by at most
    twice the largest logit change, by 4 bl."""
    env = _env(64)
    pol, opp = _policy(env, 31), _policy(env, 32)
    tr = PackedPPO(env, pol, _args())
    ro = tr.collect(FusedPolicy(env, opp), num_env_steps=16)
    bits = ro.grid_states.reshape(-1, env.bits_words_per_agent)
    meta = ro.metadata_states.reshape(-1, env.meta_size)
    with torch.no_grad():
        new_lp, _, _ = tr.fused.evaluate_actions(bits, meta, ro.use_action_mask.reshape(-1), ro.actions.reshape(-1).long())
        value, logits = tr.fused.forward_packed(bits, meta)
        _, (_, bl) = _bound(pol, env.unpack_obs(bits), meta, value, logits)
    diff = float((new_lp - ro.logprobs.reshape(-1)).abs().max())
    assert diff <= 4 * bl + 1e-4, (diff, bl)


# ---------------------------------------------------------------------------------------------------- 7. early stop
def test_target_kl_stops_early():
    env = _env(32)
    pol, opp = _policy(env, 41), _policy(env, 42)
    for target_kl, epochs in ((0.0, 1), (None, 3)):
        tr = PackedPPO(env, pol, _args(update_epochs=3, target_kl=target_kl))
        ro = tr.collect(FusedPolicy(env, opp), num_env_steps=8)
        out = tr.optimise(ro, *tr.advantages(ro))
        assert out["epochs_run"] == epochs
        assert out["first_approx_kl"] >= 0 and 0 <= out["first_clipfrac"] <= 1


# ---------------------------------------------------------------------------------------------------- 8. learning
@torch.no_grad()
def _value_loss(tr, ro, ret):
    bits = ro.grid_states.reshape(-1, tr.env.bits_words_per_agent)
    meta = ro.metadata_states.reshape(-1, tr.env.meta_size)
    value, _ = tr.fused.train_head(tr.fused.trunk_packed(bits, meta).clone())
    return float(0.5 * ((value.reshape(-1) - ret.reshape(-1)) ** 2).mean())


def test_it_learns_and_stays_in_sync():
    """Eight epochs of optimise on one fixed rollout lower the value loss over the whole rollout; then update()
    changes every parameter, keeps them finite, and refreshes the FusedPolicy's inference weights.

    A random policy on 8_arena scores almost nothing in 64 steps, so its values already sit within about 1e-2 of the
    GAE returns and the value loss has nowhere to go.  The returns given to optimise are therefore the rollout's
    values + 1: a target the value head has to move to, 0.5 away in value loss.  At lr 2.5e-4, 32 Adam steps move the
    value by well under that distance, so the loss falls without overshooting."""
    env = _env(256)
    pol, opp = _policy(env, 51), _policy(env, 52)
    tr = PackedPPO(env, pol, _args(update_epochs=8, clip_vloss=False))
    opponent = FusedPolicy(env, opp)
    ro = tr.collect(opponent, num_env_steps=64)
    adv, _ = tr.advantages(ro)
    ret = ro.values + 1
    before = _value_loss(tr, ro, ret)
    out = tr.optimise(ro, adv, ret)
    assert out["epochs_run"] == 8 and all(math.isfinite(x) for x in out.values())
    after = _value_loss(tr, ro, ret)
    assert after < 0.9 * before, (before, after)
    del ro, adv, ret
    params = [p.detach().clone() for p in pol.parameters()]
    out = tr.update(opponent)
    assert out["epochs_run"] == 8 and all(math.isfinite(x) for x in out.values())
    assert all(bool(torch.isfinite(p).all()) for p in pol.parameters())
    assert all(not torch.equal(a, b.detach()) for a, b in zip(params, pol.parameters()))
    mine = _team(env, 0)
    got_v, got_l = tr.fused.forward_from_env(mine)
    got_v, got_l = got_v.clone(), got_l.clone()
    want_v, want_l = FusedPolicy(env, pol).forward_from_env(mine)
    assert torch.equal(got_v, want_v) and torch.equal(got_l, want_l)
