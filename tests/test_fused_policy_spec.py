"""CPU checks of the torch statement of the fused policy trunk (fused_policy.reference_features) and of the conv2
weight layout the kernel reads.  The GPU kernel itself is checked against reference_features in test_gpu_fused_policy."""
import pytest
import torch

from helpers import compiled
from marl_ctf_development_b200.fused_policy import conv2_kernel_layout_index, reference_features, trunk_dims
from marl_ctf_development_b200.policy import CtfPolicy

# (C, G, M) of three shipped maps and of the rows of test_gpu_trunk_geometry.GEOMETRY: every G from 5 to 16, C = 5 and 14
GEOMETRY_SHAPES = [(5, 5, 10), (14, 5, 22), (11, 6, 16), (5, 6, 12), (9, 7, 16), (5, 8, 10), (14, 8, 22), (14, 9, 20),
                   (11, 10, 16), (7, 12, 14), (14, 12, 22), (11, 14, 18), (5, 16, 10), (11, 16, 16), (14, 16, 22)]
SHAPES = [(4, 6, 10)] + [
    (ce.n_channels, ce.GRID_SIZE, ce.meta_size) for ce in (compiled(e) for e in ("0_the_split", "7_gridlocked", "8_arena"))
] + GEOMETRY_SHAPES


def _inputs(C, G, M, S, seed):
    g = torch.Generator().manual_seed(seed)
    obs = (torch.rand((S, C, G, G), generator=g) < 0.3).float()
    meta = torch.randn((S, M), generator=g)
    return obs, meta


@pytest.mark.parametrize("C,G,M", SHAPES, ids=[f"C{c}G{g}M{m}" for c, g, m in SHAPES])
def test_unrounded_reference_features_reproduce_ctf_policy_in_fp32(C, G, M):
    torch.manual_seed(C * 100 + G)
    pol = CtfPolicy(9, C, G, M)
    obs, meta = _inputs(C, G, M, 13, G)
    feats = reference_features(pol, obs, meta, round_bf16=False)
    assert feats.shape == (13, trunk_dims(C, G, M)[0]) == (13, pol.fc1.in_features)
    with torch.no_grad():
        x = torch.tanh(pol.fc2(torch.tanh(pol.fc1(feats))))
        value, logits = pol.value_head(x), pol.action_head(x)
        want_v, want_l = pol(obs, meta)
    torch.testing.assert_close(value, want_v, rtol=0, atol=2e-5)
    torch.testing.assert_close(logits, want_l, rtol=0, atol=2e-5)
    # the metadata sits after the conv2 outputs, unchanged
    assert torch.equal(feats[:, -M:], meta)


@pytest.mark.parametrize("C,G,M", SHAPES, ids=[f"C{c}G{g}M{m}" for c, g, m in SHAPES])
def test_rounded_reference_features_are_bf16_values(C, G, M):
    torch.manual_seed(1)
    pol = CtfPolicy(9, C, G, M)
    obs, meta = _inputs(C, G, M, 5, 3)
    f = reference_features(pol, obs, meta)
    assert torch.equal(f, f.bfloat16().float())
    assert torch.equal(f[:, -M:], meta.bfloat16().float())
    assert float(f[:, :-M].abs().max()) <= 1.0


def test_trunk_dims_of_8_arena():
    assert trunk_dims(14, 15, 22) == (3894, 3896)
    for C, G, M in SHAPES:
        k1, stride = trunk_dims(C, G, M)
        assert stride % 8 == 0 and k1 <= stride < k1 + 8


def test_conv2_layout_holds_the_mma_b_fragments():
    """Lane 4g + t of n-tile j at tap (dy, dx): output channel 8j + g, input channels 2t, 2t+1, 2t+8, 2t+9."""
    w = torch.arange(32 * 16 * 9).reshape(32, 16, 3, 3)
    lay = w.reshape(-1)[conv2_kernel_layout_index()].reshape(9, 4, 32, 4)
    for tap in range(9):
        dy, dx = divmod(tap, 3)
        for j in range(4):
            for lane in range(32):
                g, t = divmod(lane, 4)
                want = [int(w[8 * j + g, ci, dy, dx]) for ci in (2 * t, 2 * t + 1, 2 * t + 8, 2 * t + 9)]
                assert lay[tap, j, lane].tolist() == want
    assert sorted(lay.reshape(-1).tolist()) == list(range(32 * 16 * 9))   # a permutation of conv2.weight
