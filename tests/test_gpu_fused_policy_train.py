"""Training through FusedPolicy: ctf_policy_features_backward (k_policy_trunk_backward) and evaluate_actions on the GPU.

The kernel's gradients are checked against fused_policy.reference_trunk_grads (its torch statement) within a bound
derived from fp32 accumulation (DESIGN §4); the PPO loss gradients of evaluate_actions against fp32 CtfPolicy within
twice torch's own bf16 autocast error, the form of the inference contract.
"""
import ctypes as C
import math

import pytest
import torch
from torch.nn.grad import conv2d_input, conv2d_weight

from test_gpu_fused_policy import DEV, SCENARIOS, _bound, _policy, _stepped_env, _team
from marl_ctf_development_b200 import _native, experiment_env_config
from marl_ctf_development_b200.env import GridworldCtfGPU
from marl_ctf_development_b200.fused_policy import FusedPolicy, _PackedTrunk, reference_conv1, reference_trunk_grads
from marl_ctf_development_b200.rollout import collect_rollout

pytestmark = pytest.mark.gpu

NAMES = ("conv1.weight", "conv1.bias", "conv2.weight", "conv2.bias")
U = 2.0 ** -22    # error of one fp32 accumulation step, relative to the sum of |terms| (twice round-to-nearest's 2^-23)


def _conv_params(pol):
    return [pol.conv1.weight, pol.conv1.bias, pol.conv2.weight, pol.conv2.bias]


def _trunk_grads(fp, bits, meta, grad_rows):
    """(rows, [dconv1.w, dconv1.b, dconv2.w, dconv2.b]) through the autograd function over the two kernels."""
    pol = fp.policy
    rows = _PackedTrunk.apply(bits, *_conv_params(pol), fp, meta)
    grads = torch.autograd.grad(rows, _conv_params(pol), grad_rows)
    return rows.detach(), grads


def _n_ctas(fp):
    """CTAs of a backward with at least that many samples (= workspace rows), from the handle's workspace size."""
    n_grad = 32 * 144 + 32 + fp.env.n_channels * 9 * 16 + 16
    return fp._train_state()["workspace"].numel() // n_grad


def _parts(fp, S):
    """CTAs (= partial rows) of a backward over S samples: sample s goes to CTA s mod min(S, n_ctas)."""
    return min(S, _n_ctas(fp))


def _assert_grads_close(fp, dense, grad_rows, rows, got):
    """Kernel gradients against reference_trunk_grads (given the kernel's rows), per element, within
        dW2, db2: L * U * sum|dz2 * h1|                                  (fp32 sums of L terms on one path)
        dh1:      288 * U * sum|dz2 * W2|                                (9 taps x 32 channels)
        dz1:      err(dh1) * (1 - h1^2) + U * |dz1|                      (the product's rounding)
        dW1, db1: sum err(dz1) * x + L * U * sum|dz1 * x|
    L = samples per CTA * max(padded conv2 positions, cells) + CTAs (the fixed-order sum of the partial rows); each
    bound gets 2^-23 |reference| more for the reference's own rounding to fp32.  dz2 carries no error term: kernel
    and statement compute it from the same bf16 inputs with the same three correctly rounded fp32 operations and one
    round-to-nearest-even to bf16, so it is the same value (a term of one bf16 ulp per dz2, summed over a chunk, would
    be larger than the random-sign sums it bounds and would hide a lost sample)."""
    pol = fp.policy
    S, Cn, G, _ = dense.shape
    S2 = G - 4
    parts = _parts(fp, S)
    L = -(-S // parts) * max((S2 * S2 + 15) // 16 * 16, G * G) + parts
    ref = reference_trunk_grads(pol, dense, grad_rows, features=rows)
    with torch.no_grad():
        x = dense.double()
        h1 = reference_conv1(pol, dense).double()
        h2 = rows[:, : 32 * S2 * S2].double().reshape(S, 32, S2, S2)
        d = grad_rows[:, : 32 * S2 * S2].float().reshape(S, 32, S2, S2)
        dz2 = (d * (1 - h2.float() * h2.float())).bfloat16().double()
        w2 = pol.conv2.weight.detach().bfloat16().double()
        dh1 = conv2d_input(h1.shape, w2, dz2)
        dz1 = (dh1 * (1 - h1 * h1)).abs()
        e_dh1 = 288 * U * conv2d_input(h1.shape, w2.abs(), dz2.abs())
        e_dz1 = e_dh1 * (1 - h1 * h1) + U * dz1
        bounds = (
            conv2d_weight(x, pol.conv1.weight.shape, e_dz1) + L * U * conv2d_weight(x, pol.conv1.weight.shape, dz1),
            e_dz1.sum((0, 2, 3)) + L * U * dz1.sum((0, 2, 3)),
            L * U * conv2d_weight(h1.abs(), w2.shape, dz2.abs()),
            L * U * dz2.abs().sum((0, 2, 3)),
        )
    for name, g, r, b in zip(NAMES, got, ref, bounds):
        assert g.dtype == torch.float32 and g.shape == r.shape, name
        excess = (g.double() - r.double()).abs() - (b + 2.0**-23 * r.double().abs())
        worst = int(excess.argmax())
        assert float(excess.max()) <= 0, (f"{name} element {worst}: got {float(g.reshape(-1)[worst])}, want "
                                          f"{float(r.reshape(-1)[worst])}, allowed {float(b.reshape(-1)[worst])}")


def _grad_rows(S, stride, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.randn((S, stride), generator=g, device=DEV) * 0.05).bfloat16()


def _packed(env, ids):
    bits = env.obs_bits[:, ids].reshape(-1, env.bits_words_per_agent).contiguous()
    meta = env.meta[:, ids].reshape(-1, env.meta_size).contiguous()
    return bits, meta


# ---------------------------------------------------------------------------------------------------- 1. kernel vs spec
@pytest.mark.parametrize("steps", [0, 50])
@pytest.mark.parametrize("name", list(SCENARIOS))
def test_trunk_grads_match_reference(name, steps):
    env = _stepped_env(SCENARIOS[name](), 37, steps)
    for t in (0, 1):
        ids = _team(env, t)
        fp = FusedPolicy(env, _policy(env, 5 + t))
        bits, meta = _packed(env, ids)
        dF = _grad_rows(len(bits), fp.stride, t)
        rows, got = _trunk_grads(fp, bits, meta, dF)
        _assert_grads_close(fp, env.unpack_obs(bits), dF, rows, got)


def test_trunk_grads_for_any_binary_input():
    """Every bit pattern, not only one-hot cells (G = 16, C = 10; the largest plan, G = 16, C = 14, is a row of
    test_gpu_trunk_geometry)."""
    env = _stepped_env(SCENARIOS["random-4-G16"](), 8, 0)
    fp = FusedPolicy(env, _policy(env, 2))
    g = torch.Generator(device=DEV).manual_seed(0)
    S, wpa = 300, env.bits_words_per_agent
    bits = torch.randint(-(2**31), 2**31 - 1, (S, wpa), generator=g, device=DEV, dtype=torch.int64).to(torch.int32)
    bits[:100] &= torch.randint(0, 2**31 - 1, (100, wpa), generator=g, device=DEV, dtype=torch.int64).to(torch.int32)
    meta = torch.randn((S, env.meta_size), generator=g, device=DEV)
    dF = _grad_rows(S, fp.stride, 1)
    rows, got = _trunk_grads(fp, bits, meta, dF)
    _assert_grads_close(fp, env.unpack_obs(bits), dF, rows, got)


# ---------------------------------------------------------------------------------------------------- 2. model vs fp32
def _ppo_loss(logprob, entropy, value, old_logprob, adv, ret, clip=0.2):
    ratio = torch.exp(logprob - old_logprob)
    pg = torch.max(-adv * ratio, -adv * torch.clamp(ratio, 1 - clip, 1 + clip)).mean()
    return pg + 0.5 * ((value.reshape(-1) - ret) ** 2).mean() - 0.01 * entropy.mean()


def _minibatch(env, ids, seed):
    bits, meta = _packed(env, ids)
    B, k = env.num_envs, len(ids)
    flags = env.use_action_mask[ids].unsqueeze(0).expand(B, k).reshape(-1)
    g = torch.Generator(device=DEV).manual_seed(seed)
    act = torch.where(flags == 1, torch.randint(0, 5, flags.shape, generator=g, device=DEV),
                      torch.randint(0, 9, flags.shape, generator=g, device=DEV))
    adv = torch.randn(flags.shape, generator=g, device=DEV)
    ret = torch.randn(flags.shape, generator=g, device=DEV)
    return bits, meta, flags, act, adv, ret


def _fp32_and_autocast_grads(pol, dense, meta, flags, act, old, adv, ret):
    out = []
    for amp in (False, True):
        pol.zero_grad()
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
            _, lp, ent, v = pol.get_action_and_value(dense, meta, flags, act)
        _ppo_loss(lp.float(), ent.float(), v.float(), old, adv, ret).backward()
        out.append({n: p.grad.clone() for n, p in pol.named_parameters()})
    pol.zero_grad()
    return out


def _assert_model_grads(pol, got, g32, gamp):
    for n, _ in pol.named_parameters():
        err = float((got[n] - g32[n]).norm())
        allowed = 2 * float((gamp[n] - g32[n]).norm()) + 1e-3 * float(g32[n].norm())
        assert err <= allowed, f"{n}: |fused - fp32| = {err} > {allowed}"


@pytest.mark.parametrize("name", ["8_arena", "random-4-G16", "random-29-G7"])
def test_ppo_loss_gradients_against_fp32_ctf_policy(name):
    env = _stepped_env(SCENARIOS[name](), 37, 50)
    for t in (0, 1):
        ids = _team(env, t)
        pol = _policy(env, 7 + t)
        fp = FusedPolicy(env, pol)
        bits, meta, flags, act, adv, ret = _minibatch(env, ids, t)
        dense = env.unpack_obs(bits)
        with torch.no_grad():
            _, old, _, _ = pol.get_action_and_value(dense, meta, flags, act)
        g32, gamp = _fp32_and_autocast_grads(pol, dense, meta, flags, act, old, adv, ret)
        lp, ent, v = fp.evaluate_actions(bits, meta, flags, act)
        _ppo_loss(lp, ent, v, old, adv, ret).backward()
        got = {n: p.grad.clone() for n, p in pol.named_parameters()}
        pol.zero_grad()
        _assert_model_grads(pol, got, g32, gamp)
        # outputs within the inference contract: value within its bound, log-probs within twice the logit bound (as
        # test_gpu_fused_policy), entropy within 5x (|dH/dlogits|_1 <= 2 log 9)
        with torch.no_grad():
            value, logits = fp.forward_packed(bits, meta)
            (_, bv), (_, bl) = _bound(pol, dense, meta, value, logits)
            _, _, ent32, v32 = pol.get_action_and_value(dense, meta, flags, act)
        assert float((v.detach() - v32).abs().max()) <= bv
        assert float((lp.detach() - old).abs().max()) <= 2 * bl + 1e-4
        assert float((ent.detach() - ent32).abs().max()) <= 5 * bl + 1e-4


# ---------------------------------------------------------------------------------------------------- 3. many samples per CTA
# Every CTA of the backward works on samples blockIdx.x, + n_ctas, ... and keeps its gradient sums in registers across
# them; these tests put 3 or more samples on every CTA, with S not a multiple of n_ctas, so that some CTAs get one more
# sample than others.
def _many(n):
    """3 n + 37 rounded up to a multiple of 4 (one 8_arena team per env) that is not a multiple of n."""
    S = (3 * n + 37 + 3) // 4 * 4
    return S if S % n else S + 4


def _backward_in_place(fp, env, ids, rows, dF):
    """Trunk gradients read in place from env.obs_bits (agents_per_env = N with ids) for rows / dF of those samples."""
    tr = fp._train_state()
    grads = [torch.empty_like(t, dtype=torch.float32) for t in _conv_params(fp.policy)]
    gs = _native.CtfPolicyGrads(*(g.data_ptr() for g in grads))
    ids_arr = (C.c_uint8 * len(ids))(*ids)
    ws = tr["workspace"]
    lib = _native.load()
    rc = lib.ctf_policy_features_backward(
        env._handle, C.byref(tr["weights"]), C.c_void_p(tr["c2wt"].data_ptr()), C.c_void_p(env.obs_bits.data_ptr()),
        env.num_envs, env.N_AGENTS, ids_arr, len(ids), C.c_void_p(rows.data_ptr()), C.c_void_p(dF.data_ptr()), fp.stride,
        C.c_void_p(ws.data_ptr()), ws.numel() * 4, C.byref(gs), C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, lib.ctf_last_error()
    return grads


def test_many_samples_per_cta_match_reference_and_are_deterministic_in_place_and_contiguous():
    probe = _stepped_env(SCENARIOS["8_arena"](), 4, 0)
    n = _n_ctas(FusedPolicy(probe, _policy(probe, 1)))
    S = _many(n)
    env = _stepped_env(SCENARIOS["8_arena"](), S // 4, 50)
    ids = _team(env, 1)
    fp = FusedPolicy(env, _policy(env, 1))
    assert _n_ctas(fp) == n and len(ids) == 4 and S > 3 * n and S % n
    bits, meta = _packed(env, ids)
    assert len(bits) == S
    dF = _grad_rows(S, fp.stride, 3)
    rows, a = _trunk_grads(fp, bits, meta, dF)
    _assert_grads_close(fp, env.unpack_obs(bits), dF, rows, a)
    _, b = _trunk_grads(fp, bits, meta, dF)
    for x, y in zip(a, b):
        assert torch.equal(x, y)                                    # rerun: bit-identical
    for x, y in zip(a, _backward_in_place(fp, env, ids, rows, dF)):
        assert torch.equal(x, y)                                    # in place in env.obs_bits: bit-identical
    # the same samples in another order land on other CTAs: the sums differ in rounding only, within the bound
    perm = torch.randperm(S, generator=torch.Generator(device=DEV).manual_seed(0), device=DEV)
    rows_p, c = _trunk_grads(fp, bits[perm].contiguous(), meta[perm].contiguous(), dF[perm].contiguous())
    assert torch.equal(rows_p.view(torch.int16), rows[perm].view(torch.int16))
    _assert_grads_close(fp, env.unpack_obs(bits[perm]), dF[perm], rows_p, c)


def test_many_samples_per_cta_for_any_binary_input():
    """Random non-one-hot words at G = 16, C = 10, 3 n_ctas + 37 samples."""
    env = _stepped_env(SCENARIOS["random-4-G16"](), 8, 0)
    fp = FusedPolicy(env, _policy(env, 2))
    n = _n_ctas(fp)
    S = 3 * n + 37
    g = torch.Generator(device=DEV).manual_seed(5)
    wpa = env.bits_words_per_agent
    bits = torch.randint(-(2**31), 2**31 - 1, (S, wpa), generator=g, device=DEV, dtype=torch.int64).to(torch.int32)
    bits[: S // 3] &= torch.randint(0, 2**31 - 1, (S // 3, wpa), generator=g, device=DEV, dtype=torch.int64).to(torch.int32)
    meta = torch.randn((S, env.meta_size), generator=g, device=DEV)
    dF = _grad_rows(S, fp.stride, 2)
    rows, got = _trunk_grads(fp, bits, meta, dF)
    _assert_grads_close(fp, env.unpack_obs(bits), dF, rows, got)
    _, again = _trunk_grads(fp, bits, meta, dF)
    for x, y in zip(got, again):
        assert torch.equal(x, y)


# ---------------------------------------------------------------------------------------------------- 4. edges
def test_sample_counts_around_the_cta_count():
    """S = 0 (zero gradients), 1, and S just below, at and above n_ctas and 2 n_ctas: CTAs with one sample more than
    others, and CTAs with none (those write zero partial rows)."""
    probe = _stepped_env(SCENARIOS["random-29-G7"](), 2, 0)
    n = _n_ctas(FusedPolicy(probe, _policy(probe, 4)))
    counts = (0, 1, n - 1, n, n + 1, 2 * n + 5)
    env = _stepped_env(SCENARIOS["random-29-G7"](), -(-max(counts) // probe.N_AGENTS), 20)
    fp = FusedPolicy(env, _policy(env, 4))
    bits, meta = _packed(env, list(range(env.N_AGENTS)))
    for S in counts:
        dF = _grad_rows(S, fp.stride, S)
        rows, got = _trunk_grads(fp, bits[:S].contiguous(), meta[:S].contiguous(), dF)
        if S == 0:
            assert all(not bool(g.any()) for g in got)
        else:
            _assert_grads_close(fp, env.unpack_obs(bits[:S]), dF, rows, got)


# ---------------------------------------------------------------------------------------------------- 5. refresh
def test_training_forwards_leave_captured_inference_graphs_alone_until_refresh():
    env = _stepped_env(SCENARIOS["8_arena"](), 64, 10)
    pol = _policy(env, 9)
    fp = FusedPolicy(env, pol)
    ids = _team(env, 0)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fp.forward_from_env(ids)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        gv, gl = fp.forward_from_env(ids)
    graph.replay()
    v0, l0 = gv.clone(), gl.clone()
    # a training step: new parameters, training forward + backward with them
    with torch.no_grad():
        for p in pol.parameters():
            p.mul_(-1.5)
    bits, meta, flags, act, adv, ret = _minibatch(env, ids, 0)
    lp, ent, v = fp.evaluate_actions(bits, meta, flags, act)
    _ppo_loss(lp, ent, v, lp.detach(), adv, ret).backward()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(gv, v0) and torch.equal(gl, l0)
    fp.refresh()
    graph.replay()
    torch.cuda.synchronize()
    assert not torch.equal(gl, l0)
    ev, _ = fp.forward_packed(bits, meta)        # inference after refresh() sees the trained parameters
    torch.testing.assert_close(ev, v.detach(), rtol=0, atol=1e-2)


# ---------------------------------------------------------------------------------------------------- 6. argument checks
def test_backward_bad_arguments_are_rejected():
    env = _stepped_env(SCENARIOS["8_arena"](), 4, 0)
    N = env.N_AGENTS
    fp = FusedPolicy(env, _policy(env, 0))
    bits, meta = _packed(env, [0, 2])
    dF = _grad_rows(len(bits), fp.stride, 0)
    rows, ok = _trunk_grads(fp, bits, meta, dF)
    tr = fp._train_state()
    ws = tr["workspace"]
    lib = _native.load()
    n = C.c_size_t()
    assert lib.ctf_policy_grad_workspace_size(env._handle, C.byref(n)) == 0 and n.value == ws.numel() * 4
    assert lib.ctf_policy_grad_workspace_size(env._handle, None) == -1
    grads = [torch.empty_like(g) for g in ok]
    gs = _native.CtfPolicyGrads(*(g.data_ptr() for g in grads))
    ids2 = (C.c_uint8 * 2)(0, 2)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    big = torch.zeros(len(rows) * fp.stride + 8, dtype=torch.bfloat16, device=DEV)

    def call(weights=C.byref(tr["weights"]), w2t=tr["c2wt"].data_ptr(), packed=env.obs_bits.data_ptr(), ape=N,
             ids=ids2, k=2, feat=rows.data_ptr(), dfeat=dF.data_ptr(), st=fp.stride, wsp=ws.data_ptr(),
             wsb=ws.numel() * 4, g=C.byref(gs)):
        return lib.ctf_policy_features_backward(env._handle, weights, C.c_void_p(w2t), C.c_void_p(packed), 4, ape, ids,
                                                k, C.c_void_p(feat), C.c_void_p(dfeat), st, C.c_void_p(wsp), wsb, g,
                                                stream)

    assert call() == 0
    torch.cuda.synchronize()
    bad = [
        dict(k=0), dict(k=9), dict(ape=2), dict(st=fp.k1), dict(st=fp.stride - 8), dict(feat=big.data_ptr() + 2),
        dict(dfeat=big.data_ptr() + 8), dict(wsb=ws.numel() * 4 - 4), dict(wsp=ws.data_ptr() + 4), dict(w2t=0),
        dict(packed=0), dict(feat=0), dict(dfeat=0), dict(wsp=0), dict(ids=None), dict(weights=None), dict(g=None),
    ]
    for kw in bad:
        assert call(**kw) == -1, kw
        assert lib.ctf_last_error().startswith(b"ctf_policy_features_backward"), kw
    w = tr["weights"]
    assert call(weights=C.byref(_native.CtfPolicyWeights(w.conv1_w, None, w.conv2_w, w.conv2_b))) == -1
    assert call(g=C.byref(_native.CtfPolicyGrads(gs.conv1_w, gs.conv1_b, None, gs.conv2_b))) == -1
    assert lib.ctf_last_error().startswith(b"ctf_policy_features_backward")
    with pytest.raises(ValueError):
        fp.evaluate_actions(bits.float(), meta, torch.zeros(len(bits), device=DEV), torch.zeros(len(bits), device=DEV))


# ---------------------------------------------------------------------------------------------------- 7. end to end
def _gae(rewards, values, next_value, gamma=0.99, lam=0.95):
    T = rewards.shape[0]
    adv = torch.zeros_like(rewards)
    last = torch.zeros_like(next_value)
    for t in reversed(range(T)):
        nv = next_value if t == T - 1 else values[t + 1]
        delta = rewards[t] + gamma * nv - values[t]
        last = delta + gamma * lam * last
        adv[t] = last
    return adv, adv + values


def test_ppo_update_on_a_packed_rollout():
    """Packed-only 8_arena env, fused policies, torch GAE, 2 epochs x 4 minibatches of Adam in chunks."""
    ec = experiment_env_config("8_arena")
    B, T = 64, 32
    env = GridworldCtfGPU(**ec, num_envs=B, device=DEV, seed=2, reverse_team1_actions=True, dense_obs=False,
                          packed_obs=True)
    pol, opp = _policy(env, 11), _policy(env, 12)
    agent, opponent = FusedPolicy(env, pol), FusedPolicy(env, opp)
    ro = collect_rollout(env, agent, opponent, num_env_steps=T, obs_storage_dtype="packed")
    apt = len(_team(env, 0))
    wpa, M = env.bits_words_per_agent, env.meta_size
    # per-agent time series [T, apt*B] (bootstrap value 0: the rollout is cut, not ended, but any value serves the test)
    rew = ro.rewards.reshape(T, apt * B)
    val = ro.values.reshape(T, apt * B)
    adv, ret = _gae(rew, val, torch.zeros_like(val[0]))
    bits_all = ro.grid_states.reshape(-1, wpa)
    meta_all = ro.metadata_states.reshape(-1, M)
    n = bits_all.shape[0]
    flat = dict(act=ro.actions.reshape(-1).long(), mask=ro.use_action_mask.reshape(-1), lp=ro.logprobs.reshape(-1),
                adv=adv.reshape(-1), ret=ret.reshape(-1))
    before = [p.detach().clone() for p in pol.parameters()]
    optim = torch.optim.Adam(pol.parameters(), lr=2.5e-4, eps=1e-5)
    g = torch.Generator(device=DEV).manual_seed(0)
    mb, chunk = n // 4, n // 4 // 3 + 1
    first = True
    for _ in range(2):
        perm = torch.randperm(n, generator=g, device=DEV)
        for start in range(0, n, mb):
            idx = perm[start : start + mb]
            optim.zero_grad()
            total = 0.0
            for c0 in range(0, len(idx), chunk):
                ci = idx[c0 : c0 + chunk]
                lp, ent, v = agent.evaluate_actions(bits_all[ci], meta_all[ci], flat["mask"][ci], flat["act"][ci])
                loss = _ppo_loss(lp, ent, v, flat["lp"][ci], flat["adv"][ci], flat["ret"][ci]) * (len(ci) / len(idx))
                loss.backward()
                total += float(loss.detach())
            assert math.isfinite(total)
            if first:
                got = {k: p.grad.clone() for k, p in pol.named_parameters()}
                dense = env.unpack_obs(bits_all[idx])
                g32, gamp = _fp32_and_autocast_grads(pol, dense, meta_all[idx], flat["mask"][idx], flat["act"][idx],
                                                     flat["lp"][idx], flat["adv"][idx], flat["ret"][idx])
                _assert_model_grads(pol, got, g32, gamp)
                for k, p in pol.named_parameters():
                    p.grad = got[k]
                first = False
            optim.step()
            agent.refresh()
    assert all(not torch.equal(a, b.detach()) for a, b in zip(before, pol.parameters()))
    assert all(bool(torch.isfinite(p).all()) for p in pol.parameters())


# ---------------------------------------------------------------------------------------------------- 8. scale
def test_one_full_size_chunk():
    """262 144 samples (8_arena, B = 65 536, one team) through forward and backward."""
    ec = experiment_env_config("8_arena")
    B = 65536
    env = GridworldCtfGPU(**ec, num_envs=B, device=DEV, seed=1, reverse_team1_actions=True, dense_obs=False,
                          packed_obs=True)
    g = torch.Generator(device=DEV).manual_seed(0)
    for _ in range(5):
        env.step(torch.randint(0, 9, (B, env.N_AGENTS), generator=g, device=DEV, dtype=torch.int64).to(torch.uint8))
    ids = _team(env, 0)
    pol = _policy(env, 3)
    fp = FusedPolicy(env, pol)
    bits, meta, flags, act, adv, ret = _minibatch(env, ids, 0)
    assert len(bits) == 262144
    lp, ent, v = fp.evaluate_actions(bits, meta, flags, act)
    _ppo_loss(lp, ent, v, lp.detach(), adv, ret).backward()
    for n, p in pol.named_parameters():
        assert bool(torch.isfinite(p.grad).all()), n
        assert bool(p.grad.any()), n
    # the whole chunk's trunk gradients (about 590 samples per CTA) against the statement, and bit-identical when the
    # same samples are read in place from env.obs_bits
    dF = _grad_rows(len(bits), fp.stride, 9)
    rows, got = _trunk_grads(fp, bits, meta, dF)
    assert -(-len(bits) // _parts(fp, len(bits))) >= 100
    for x, y in zip(got, _backward_in_place(fp, env, ids, rows, dF)):
        assert torch.equal(x, y)
    _assert_grads_close(fp, env.unpack_obs(bits), dF, rows, got)
