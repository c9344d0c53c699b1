"""CPU checks of the training statement of the fused trunk (fused_policy.reference_trunk_grads) and of the transposed
conv2 layout the backward kernel reads.  The kernel itself is checked against reference_trunk_grads in
test_gpu_fused_policy_train."""
import pytest
import torch

from helpers import compiled
from test_fused_policy_spec import GEOMETRY_SHAPES
from marl_ctf_development_b200.fused_policy import (conv2_kernel_layout_index, conv2_transpose_layout_index,
                                                    reference_features, reference_trunk_grads, trunk_dims)
from marl_ctf_development_b200.policy import CtfPolicy

SHAPES = [(4, 6, 10)] + [
    (ce.n_channels, ce.GRID_SIZE, ce.meta_size) for ce in (compiled(e) for e in ("0_the_split", "7_gridlocked", "8_arena"))
] + GEOMETRY_SHAPES


def _case(C, G, M, S, seed):
    torch.manual_seed(seed)
    pol = CtfPolicy(9, C, G, M)
    g = torch.Generator().manual_seed(seed)
    obs = (torch.rand((S, C, G, G), generator=g) < 0.3).float()
    stride = trunk_dims(C, G, M)[1]
    grad_rows = torch.randn((S, stride), generator=g)
    return pol, obs, grad_rows


def _autograd_trunk_grads(pol, obs, grad_rows):
    """float64 autograd of CtfPolicy's conv trunk (conv1 -> tanh -> conv2 -> tanh -> flatten) against grad_rows."""
    p64 = {k: v.detach().double().requires_grad_(True) for k, v in pol.named_parameters() if k.startswith("conv")}
    x = torch.tanh(torch.nn.functional.conv2d(obs.double(), p64["conv1.weight"], p64["conv1.bias"]))
    x = torch.tanh(torch.nn.functional.conv2d(x, p64["conv2.weight"], p64["conv2.bias"])).reshape(len(obs), -1)
    (x * grad_rows[:, : x.shape[1]].double()).sum().backward()
    return [p64[k].grad for k in ("conv1.weight", "conv1.bias", "conv2.weight", "conv2.bias")]


@pytest.mark.parametrize("C,G,M", SHAPES, ids=[f"C{c}G{g}M{m}" for c, g, m in SHAPES])
def test_unrounded_reference_trunk_grads_equal_float64_autograd(C, G, M):
    pol, obs, grad_rows = _case(C, G, M, 7, C + G)
    got = reference_trunk_grads(pol, obs, grad_rows, round_bf16=False)
    want = _autograd_trunk_grads(pol, obs, grad_rows)
    for name, a, b in zip(("conv1.weight", "conv1.bias", "conv2.weight", "conv2.bias"), got, want):
        assert a.dtype == torch.float64 and a.shape == b.shape, name
        torch.testing.assert_close(a, b, rtol=1e-12, atol=1e-12, msg=name)


def test_rounded_reference_trunk_grads_are_close_to_fp32_and_use_the_given_rows():
    C, G, M = 14, 15, 22
    pol, obs, grad_rows = _case(C, G, M, 9, 3)
    got = reference_trunk_grads(pol, obs, grad_rows)
    want = _autograd_trunk_grads(pol, obs, grad_rows)
    for a, b in zip(got, want):
        assert a.dtype == torch.float32
        # bf16 activations, weights and dz2: about 2^-8 relative
        assert float((a.double() - b).norm()) <= 2e-2 * float(b.norm())
    # the conv2 part of the rows is h2: passing reference_features' rows reproduces the default
    meta = torch.randn((9, M))
    rows = reference_features(pol, obs, meta)
    again = reference_trunk_grads(pol, obs, grad_rows, features=rows)
    for a, b in zip(got, again):
        assert torch.equal(a, b)


def test_conv2_transpose_layout_holds_the_mma_b_fragments():
    """Lane 4g + t of n-tile j in k-half h at tap (dy, dx): input channel 8j + g, output channels 16h + 2t, 2t+1, 2t+8,
    2t+9."""
    w = torch.arange(32 * 16 * 9).reshape(32, 16, 3, 3)
    lay = w.reshape(-1)[conv2_transpose_layout_index()].reshape(9, 2, 2, 32, 4)
    for tap in range(9):
        dy, dx = divmod(tap, 3)
        for h in range(2):
            for j in range(2):
                for lane in range(32):
                    g, t = divmod(lane, 4)
                    want = [int(w[16 * h + co, 8 * j + g, dy, dx]) for co in (2 * t, 2 * t + 1, 2 * t + 8, 2 * t + 9)]
                    assert lay[tap, h, j, lane].tolist() == want
    assert sorted(lay.reshape(-1).tolist()) == list(range(32 * 16 * 9))   # a permutation of conv2.weight
    assert conv2_transpose_layout_index().numel() == conv2_kernel_layout_index().numel()
