"""CPU statements of the PPO trainer (ppo.py): the GAE reference, the clipped loss, chunking and the minibatch plan."""
import math
import types

import pytest
import torch

from marl_ctf_development_b200.ppo import minibatches, ppo_loss, reference_advantages


def _gae64(rewards, values, next_value, gamma, lam):
    """The recurrence in float64, one (agent, env) column at a time."""
    apt, B = next_value.shape
    T = rewards.shape[0] // apt
    r, v, nv = (x.double().numpy() for x in (rewards.reshape(T, apt, B), values.reshape(T, apt, B), next_value))
    adv = torch.zeros((T, apt, B), dtype=torch.float64)
    for j in range(apt):
        for b in range(B):
            last, nxt = 0.0, float(nv[j, b])
            for t in reversed(range(T)):
                delta = r[t, j, b] + gamma * nxt - v[t, j, b]
                last = delta + gamma * lam * last
                adv[t, j, b] = last
                nxt = v[t, j, b]
    return adv.reshape(T * apt, B)


def _inputs(T, apt, B, seed, zero_bootstrap=False):
    g = torch.Generator().manual_seed(seed)
    r = torch.randn((T * apt, B), generator=g)
    v = torch.randn((T * apt, B), generator=g)
    nv = torch.zeros((apt, B)) if zero_bootstrap else torch.randn((apt, B), generator=g)
    return r, v, nv


@pytest.mark.parametrize("gamma,lam", [(0.99, 0.95), (1.0, 1.0), (0.9, 0.0)])
@pytest.mark.parametrize("shape", [(1, 1, 1), (7, 3, 5), (16, 4, 3)])
def test_reference_advantages_against_float64(shape, gamma, lam):
    T, apt, B = shape
    r, v, nv = _inputs(T, apt, B, T + apt + B)
    adv, ret = reference_advantages(r, v, nv, gamma, lam)
    want = _gae64(r, v, nv, gamma, lam)
    scale = float(want.abs().max()) + float(v.abs().max()) + 1
    assert adv.dtype == torch.float32 and adv.shape == r.shape
    assert float((adv.double() - want).abs().max()) <= 4 * T * 2.0 ** -24 * scale
    assert torch.allclose(ret.double(), want + v.double(), atol=4 * (T + 1) * 2.0 ** -24 * scale, rtol=0)


def test_lambda_zero_is_the_one_step_td_error():
    T, apt, B, gamma = 6, 2, 3, 0.9
    r, v, nv = _inputs(T, apt, B, 1)
    adv, _ = reference_advantages(r, v, nv, gamma, 0.0)
    nxt = torch.cat((v[apt:], nv))
    assert torch.equal(adv, r + gamma * nxt - v)


def test_lambda_one_with_zero_bootstrap_is_the_discounted_return_minus_the_value():
    T, apt, B, gamma = 9, 3, 4, 0.97
    r, v, nv = _inputs(T, apt, B, 2, zero_bootstrap=True)
    adv, ret = reference_advantages(r, v, nv, gamma, 1.0)
    r3 = r.double().reshape(T, apt, B)
    disc = torch.zeros_like(r3)
    acc = torch.zeros((apt, B), dtype=torch.float64)
    for t in reversed(range(T)):
        acc = r3[t] + gamma * acc
        disc[t] = acc
    disc = disc.reshape(T * apt, B)
    assert torch.allclose(adv.double(), disc - v.double(), atol=1e-5, rtol=0)
    assert torch.allclose(ret.double(), disc, atol=1e-5, rtol=0)


# ---------------------------------------------------------------------------------------------------- loss
def _args(norm_adv, clip_vloss, clip=0.2):
    return types.SimpleNamespace(norm_adv=norm_adv, clip_vloss=clip_vloss, clip_coef=clip, ent_coef=0.01, vf_coef=0.5)


LP_NEW = [0.0, math.log(1.5), math.log(0.5), math.log(1.1)]   # ratios 1, 1.5, 0.5, 1.1 against old log-probs 0
ADV = [1.0, 2.0, -1.0, -3.0]
V_NEW, V_OLD, RET = [0.5, 1.0, -0.5, 2.0], [0.0, 1.5, -0.4, 1.0], [1.0, 0.0, 0.0, 3.0]
ENT = [1.0, 2.0, 0.5, 0.5]


@pytest.mark.parametrize("norm_adv", [False, True])
@pytest.mark.parametrize("clip_vloss", [False, True])
def test_ppo_loss_against_hand_computed_values(norm_adv, clip_vloss):
    t = lambda x: torch.tensor(x, dtype=torch.float64)
    loss, st = ppo_loss(t(LP_NEW), t(ENT), t(V_NEW).reshape(-1, 1), torch.zeros(4, dtype=torch.float64), t(V_OLD),
                        t(ADV), t(RET), _args(norm_adv, clip_vloss))
    ratio = [1.0, 1.5, 0.5, 1.1]
    a = ADV
    if norm_adv:
        mean = sum(a) / 4
        std = math.sqrt(sum((x - mean) ** 2 for x in a) / 3)
        a = [(x - mean) / (std + 1e-8) for x in a]
    clipped = [min(max(r, 0.8), 1.2) for r in ratio]
    pg = sum(max(-x * r, -x * c) for x, r, c in zip(a, ratio, clipped)) / 4
    if clip_vloss:
        vc = [o + min(max(n - o, -0.2), 0.2) for n, o in zip(V_NEW, V_OLD)]
        v = 0.5 * sum(max((n - r) ** 2, (c - r) ** 2) for n, c, r in zip(V_NEW, vc, RET)) / 4
    else:
        v = 0.5 * sum((n - r) ** 2 for n, r in zip(V_NEW, RET)) / 4
    ent = sum(ENT) / 4
    assert float(st["pg_loss"]) == pytest.approx(pg, abs=1e-12)
    assert float(st["v_loss"]) == pytest.approx(v, abs=1e-12)
    assert float(st["entropy"]) == pytest.approx(ent, abs=1e-12)
    assert float(loss) == pytest.approx(pg - 0.01 * ent + 0.5 * v, abs=1e-12)
    kl = sum((r - 1) - math.log(r) for r in ratio) / 4
    assert float(st["approx_kl"]) == pytest.approx(kl, abs=1e-12)
    assert float(st["clipfrac"]) == pytest.approx(0.5)   # |ratio - 1| > 0.2 for 1.5 and 0.5


@pytest.mark.parametrize("clip_vloss", [False, True])
def test_chunked_loss_has_the_gradients_of_the_one_piece_loss(clip_vloss):
    """A small linear model: a minibatch cut into uneven chunks, advantages normalised over the whole minibatch and
    each chunk's loss scaled by its share, accumulates the gradients of the loss over the minibatch in one piece."""
    torch.manual_seed(0)
    S, D, A = 101, 6, 9
    model = torch.nn.Linear(D, A + 1)
    x = torch.randn(S, D)
    act = torch.randint(0, A, (S,))
    old_lp = torch.randn(S) * 0.1 - 2.2
    old_v, ret, adv = torch.randn(S), torch.randn(S), torch.randn(S) * 3 + 1
    args = _args(True, clip_vloss)

    def run(rows, stats):
        out = model(x[rows])
        dist = torch.distributions.Categorical(logits=out[:, 1:])
        return ppo_loss(dist.log_prob(act[rows]), dist.entropy(), out[:, :1], old_lp[rows], old_v[rows], adv[rows],
                        ret[rows], args, stats)

    model.zero_grad()
    run(torch.arange(S), None)[0].backward()
    whole = [p.grad.clone() for p in model.parameters()]
    model.zero_grad()
    stats = (adv.mean(), adv.std())
    bounds = [0, 7, 40, 41, 90, S]
    for a, b in zip(bounds, bounds[1:]):
        (run(torch.arange(a, b), stats)[0] * ((b - a) / S)).backward()
    for g, w in zip((p.grad for p in model.parameters()), whole):
        assert torch.allclose(g, w, atol=1e-6, rtol=1e-5)


@pytest.mark.parametrize("n,k", [(16, 4), (17, 4), (103, 4), (5, 8), (1, 1), (2000, 3)])
def test_minibatch_plan_visits_every_sample_once(n, k):
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(n))
    mbs = minibatches(perm, k)
    size = max(n // k, 1)
    assert all(m.numel() == size for m in mbs[:-1]) and 1 <= mbs[-1].numel() <= size
    assert len(mbs) == -(-n // size)
    assert torch.equal(torch.sort(torch.cat(mbs)).values, torch.arange(n))
