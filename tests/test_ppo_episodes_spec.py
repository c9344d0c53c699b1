"""CPU statements of GAE across episode boundaries (ppo.reference_advantages with dones, what ctf_gae_dones computes):
CleanRL's recurrence in float64, bit equality with dones=None when no episode starts, and no information crossing a
boundary."""
import pytest
import torch

from marl_ctf_development_b200.ppo import reference_advantages


def _cleanrl64(rewards, values, next_value, dones, gamma, lam):
    """CleanRL's loop (ppo.py of CleanRL: nextnonterminal = 1 - dones[t + 1]) in float64, one (agent, env) column at a
    time.  next_value already carries the bootstrap of the last row, so the last row's nextnonterminal is 1."""
    apt, B = next_value.shape
    T = rewards.shape[0] // apt
    r, v, d = (x.double().reshape(T, apt, B) for x in (rewards, values, dones))
    adv = torch.zeros((T, apt, B), dtype=torch.float64)
    for j in range(apt):
        for b in range(B):
            last = 0.0
            for t in reversed(range(T)):
                if t == T - 1:
                    nnt, nxt = 1.0, float(next_value[j, b])
                else:
                    nnt, nxt = 1.0 - float(d[t + 1, j, b] != 0), float(v[t + 1, j, b])
                delta = float(r[t, j, b]) + gamma * nxt * nnt - float(v[t, j, b])
                last = delta + gamma * lam * nnt * last
                adv[t, j, b] = last
    return adv.reshape(T * apt, B)


def _inputs(T, apt, B, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn((T * apt, B), generator=g), torch.randn((T * apt, B), generator=g),
            torch.randn((apt, B), generator=g), g)


def _dones(kind, T, apt, B, g):
    d = torch.zeros((T, apt, B))
    if kind == "all":
        d[:] = 1
    elif kind == "random":
        d = (torch.rand((T, apt, B), generator=g) < 0.2).float()
    else:
        d[kind] = 1
    return d.reshape(T * apt, B)


@pytest.mark.parametrize("gamma,lam", [(0.99, 0.95), (1.0, 1.0), (0.9, 0.0)])
@pytest.mark.parametrize("kind", [0, 1, 5, 6, "all", "random"])
def test_dones_statement_against_cleanrl_in_float64(kind, gamma, lam):
    T, apt, B = 7, 3, 5
    r, v, nv, g = _inputs(T, apt, B, 11 if kind == "random" else 3)
    d = _dones(kind, T, apt, B, g)
    adv, ret = reference_advantages(r, v, nv, gamma, lam, dones=d)
    want = _cleanrl64(r, v, nv, d, gamma, lam)
    scale = float(want.abs().max()) + float(v.abs().max()) + 1
    assert adv.dtype == torch.float32 and adv.shape == r.shape
    assert float((adv.double() - want).abs().max()) <= 4 * T * 2.0 ** -24 * scale
    assert torch.allclose(ret.double(), want + v.double(), atol=4 * (T + 1) * 2.0 ** -24 * scale, rtol=0)


@pytest.mark.parametrize("row", range(7))
def test_a_boundary_at_every_row(row):
    """Each single boundary row of a (7, 2, 3) rollout, λ = 0.95, and with λ = 0 the one-step TD error that drops the
    bootstrap across the boundary."""
    T, apt, B = 7, 2, 3
    r, v, nv, g = _inputs(T, apt, B, row)
    d = _dones(row, T, apt, B, g)
    adv, _ = reference_advantages(r, v, nv, 0.99, 0.95, dones=d)
    want = _cleanrl64(r, v, nv, d, 0.99, 0.95)
    assert float((adv.double() - want).abs().max()) <= 4 * T * 2.0 ** -24 * (float(want.abs().max()) + 4)
    td, _ = reference_advantages(r, v, nv, 0.9, 0.0, dones=d)
    nxt = torch.cat((v[apt:], nv))
    if row > 0:
        nxt[(row - 1) * apt : row * apt] = 0
    assert torch.equal(td, r + 0.9 * nxt - v)


@pytest.mark.parametrize("gamma,lam", [(0.99, 0.95), (1.0, 1.0), (0.9, 0.0)])
@pytest.mark.parametrize("shape", [(1, 1, 1), (9, 4, 6)])
def test_zero_dones_are_bit_equal_to_no_dones(shape, gamma, lam):
    T, apt, B = shape
    r, v, nv, _ = _inputs(T, apt, B, 5)
    r[0, 0], v[-1, -1] = -0.0, float("nan")           # signed zeros and NaN pass through the select untouched
    a0, r0 = reference_advantages(r, v, nv, gamma, lam)
    a1, r1 = reference_advantages(r, v, nv, gamma, lam, dones=torch.zeros_like(r))
    assert torch.equal(a0.view(torch.int32), a1.view(torch.int32))
    assert torch.equal(r0.view(torch.int32), r1.view(torch.int32))


@pytest.mark.parametrize("row", [1, 4, 8])
def test_nothing_after_a_boundary_reaches_the_rows_before_it(row):
    """Rewards, values and the bootstrap from the boundary row onward may change arbitrarily: every earlier row's
    advantage and return stays the same, bit for bit."""
    T, apt, B = 9, 4, 5
    r, v, nv, g = _inputs(T, apt, B, 20 + row)
    d = _dones(row, T, apt, B, g)
    adv, ret = reference_advantages(r, v, nv, 0.99, 0.95, dones=d)
    k = row * apt
    r2, v2 = r.clone(), v.clone()
    r2[k:] = torch.randn(r2[k:].shape, generator=g) * 1e6
    v2[k:] = torch.randn(v2[k:].shape, generator=g) * 1e6
    adv2, ret2 = reference_advantages(r2, v2, nv * -3 + 7, 0.99, 0.95, dones=d)
    assert torch.equal(adv2[:k], adv[:k]) and torch.equal(ret2[:k], ret[:k])
    assert not torch.equal(adv2[k:], adv[k:])
