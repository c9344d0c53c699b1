"""The policy trunk kernels (k_policy_trunk, k_policy_trunk_grouped, k_policy_trunk_backward + k_policy_grad_reduce) and
k_unpack across the geometry FusedPolicy accepts: every G from 5 to 16, C from 5 to 14, N from 2 to 8.

The kernels' tiling follows the plan: conv2 runs ceil((G-4)^2 / 16) m-tiles over padded rows, the backward pads the
conv2 positions to K2 rows and runs ceil((G-2)^2 / 16) dh1 m-tiles, shared memory per CTA runs from 15 KB to 91.6 KB,
and C*G*G often leaves stray bits ("tail bits") after the last element of the last packed word.  GEOMETRY holds small
scenarios that compile to the corner cases of those rules.  Every dense input here comes from ``host_unpack``, a CPU
statement of the packed layout, not from the CUDA unpack kernel; the envs are only reset, never stepped.
"""
import numpy as np
import pytest
import torch

from marl_ctf_development_b200.env import GridworldCtfGPU
from marl_ctf_development_b200.fused_policy import FusedPolicy

from test_gpu_fused_policy import DEV, _assert_trunk_close, _bound, _policy
from test_gpu_fused_policy_train import (_assert_grads_close, _assert_model_grads, _fp32_and_autocast_grads, _grad_rows,
                                         _n_ctas, _ppo_loss, _trunk_grads)
from test_gpu_policy_pool import _check_rows, _ctas, _pool, _segments

pytestmark = pytest.mark.gpu

# (G, N, all agent types, block + destructible tile) -> (C, M, words per agent) that compile_config gives.  Comments:
# conv2 positions (G-4)^2 -> K2, tail bits, fc1 inputs K1 / row stride, shared memory of the forward / backward CTA.
GEOMETRY = [
    (5, 2, False, False, 5, 10, 4),      # 1 -> 16, 3 tail bits, K1 42 / 48, 15.0 / 13.8 KB: the smallest plan
    (5, 8, True, True, 14, 22, 11),      # 1 -> 16, 2, 54 / 56, 20.3 / 18.8 KB
    (6, 5, True, True, 11, 16, 13),      # 4 -> 16, 20, 144 / 144 (M % 8 == 0: no pad columns), 21.0 / 17.8 KB
    (6, 3, False, False, 5, 12, 6),      # 4 -> 16, 12, 140 / 144, 17.4 / 14.4 KB
    (7, 5, True, False, 9, 16, 14),      # 9 -> 16, 7, 304 / 304, 23.0 / 17.5 KB
    (8, 2, False, False, 5, 10, 10),     # 16 -> 16, 0, 522 / 528, 24.4 / 16.3 KB
    (8, 8, True, True, 14, 22, 28),      # 16 -> 16, 0, 534 / 536, 29.9 / 21.4 KB
    (9, 7, True, True, 14, 20, 36),      # 25 -> 32, 18, 820 / 824, 34.9 / 23.7 KB
    (10, 5, True, True, 11, 16, 35),     # 36 -> 48, 20, 1168 / 1168, 38.6 / 24.4 KB
    (12, 4, False, True, 7, 14, 32),     # 64 -> 64, 16, 2062 / 2064, 49.4 / 26.5 KB
    (12, 8, True, True, 14, 22, 63),     # 64 -> 64, 0, 2070 / 2072, 54.3 / 30.6 KB
    (14, 6, True, True, 11, 18, 68),     # 100 -> 112, 20, 3218 / 3224, 69.1 / 36.0 KB
    (16, 2, False, False, 5, 10, 40),    # 144 -> 144, 0, 4618 / 4624, 84.2 / 39.4 KB
    (16, 5, True, True, 11, 16, 88),     # 144 -> 144, 0, 4624 / 4624, 89.1 / 43.0 KB
    (16, 8, True, True, 14, 22, 112),    # 144 -> 144, 0, 4630 / 4632, 91.6 / 44.8 KB: the largest plan
]
IDS = [f"G{r[0]}-N{r[1]}-C{r[4]}" for r in GEOMETRY]
FAMILIES = ("uniform", "sparse", "one_hot", "ones", "zeros")


def geometry_config(G, N, all_types, tiles):
    """The smallest scenario compile_config accepts at any G >= 5: agents start on the first cells in row-major order,
    flags (also the capture cells) in the last row, spawns at (1, 1) and (G-2, G-2); team i % 2, type min(i // 2, N-1)
    (types must be agent ids) or 0; optionally one block and one destructible tile in the last row."""
    flags = {0: (G - 1, G - 1), 1: (G - 1, G - 2)}
    scenario = dict(
        SCENARIO_NAME=f"geometry-G{G}-N{N}", GRID_SIZE=G, FLIP_AXIS=None, FLAG_POSITIONS=flags, CAPTURE_POSITIONS=flags,
        SPAWN_POSITIONS={0: (1, 1), 1: (G - 2, G - 2)}, AGENT_STARTING_POSITIONS={i: (i // G, i % G) for i in range(N)},
        BLOCK_TILE_SLICES=[(G - 1, 0)] if tiles else [], DESTRUCTIBLE_TILE_SLICES=[(G - 1, 1)] if tiles else [],
    )
    agents = {i: {"team": i % 2, "type": min(i // 2, N - 1) if all_types else 0} for i in range(N)}
    return dict(AGENT_CONFIG=agents, SCENARIO=scenario, MAP_SYMMETRY_CHECK=False)


def _env(row, B, dense_obs=False):
    G, N, all_types, tiles, C, M, wpa = row
    env = GridworldCtfGPU(**geometry_config(G, N, all_types, tiles), num_envs=B, device=DEV, seed=1, packed_obs=True,
                          dense_obs=dense_obs)
    assert (env.GRID_SIZE, env.N_AGENTS, env.n_channels, env.meta_size, env.bits_words_per_agent) == (G, N, C, M, wpa)
    return env


def host_unpack(words, C, G):
    """{0,1} float32 [S, C, G, G] on the CPU from packed int32 words [S, wpa] (the layout of outputs.obs_bits in
    include/ctf_b200.h): element c*G*G + p is bit el % 32 of word el // 32; bits at or after C*G*G are ignored."""
    w = words.cpu().numpy().view(np.uint32)
    bits = (w[:, :, None] >> np.arange(32, dtype=np.uint32)) & 1        # [S, wpa, 32]: element 32 * word + bit
    flat = bits.reshape(len(w), -1)[:, : C * G * G]
    return torch.from_numpy(flat.reshape(len(w), C, G, G).astype(np.float32))


def host_pack(dense, wpa):
    """The inverse of host_unpack for {0,1} [S, C, G, G]: int32 [S, wpa] words with zero tail bits."""
    flat = dense.reshape(len(dense), -1).numpy().astype(np.uint32)
    flat = np.pad(flat, ((0, 0), (0, 32 * wpa - flat.shape[1]))).reshape(len(dense), wpa, 32)
    words = (flat << np.arange(32, dtype=np.uint32)).sum(axis=2, dtype=np.uint32)
    return torch.from_numpy(words.view(np.int32))


def tail_mask(C, G, wpa):
    """The tail bits of the last word as an int32 value (0 when C*G*G fills it)."""
    used = C * G * G - 32 * (wpa - 1)
    m = (0xFFFFFFFF << used) & 0xFFFFFFFF
    return m - (1 << 32) if m >= 1 << 31 else m


def _words(family, S, C, G, wpa, seed):
    """int32 [S, wpa] packed words on the device: uniform random words (tail bits included), sparse ones (the AND of
    three), one channel per cell (env-like, zero tail bits), all ones (the longest conv1 sums: C*9 columns per window)
    or all zeros (bias only)."""
    g = torch.Generator().manual_seed(seed)

    def rand():
        return torch.randint(-(2**31), 2**31, (S, wpa), generator=g, dtype=torch.int64).to(torch.int32)

    if family == "uniform":
        w = rand()
    elif family == "sparse":
        w = rand() & rand() & rand()
    elif family == "one_hot":
        ch = torch.randint(0, C, (S, 1, G * G), generator=g)
        w = host_pack(torch.zeros((S, C, G * G)).scatter_(1, ch, 1.0), wpa)
    elif family == "ones":
        w = torch.full((S, wpa), -1, dtype=torch.int32)
    else:
        w = torch.zeros((S, wpa), dtype=torch.int32)
    return w.to(DEV)


def _meta(S, M, seed):
    return torch.randn((S, M), generator=torch.Generator(device=DEV).manual_seed(seed), device=DEV)


def _randomise(env, seed):
    """Random words (tail bits included) and metadata in every env's buffers, so each block differs from the others."""
    B, N, wpa, M = env.num_envs, env.N_AGENTS, env.bits_words_per_agent, env.meta_size
    env.obs_bits.copy_(_words("uniform", B * N, env.n_channels, env.GRID_SIZE, wpa, seed).reshape(B, N, wpa))
    env.meta.copy_(_meta(B * N, M, seed).reshape(B, N, M))


# ---------------------------------------------------------------------------------------------------- 1. unpack
@pytest.mark.parametrize("row", GEOMETRY, ids=IDS)
def test_host_unpack_reads_the_env_and_k_unpack_matches_it(row):
    G, N, C, wpa = row[0], row[1], row[4], row[6]
    env = _env(row, 37, dense_obs=True)
    words = env.obs_bits.reshape(-1, wpa)
    assert torch.equal(host_unpack(words, C, G), env.obs.reshape(-1, C, G, G).cpu())   # the env's own dense writer
    tail = tail_mask(C, G, wpa)
    assert not bool((words[:, -1] & tail).any())                                        # the env writes no tail bit
    S = 389                      # prime: not a multiple of k_unpack's chunk of agent blocks (unless that is 1)
    bits = _words("uniform", S, C, G, wpa, G)
    assert tail == 0 or bool((bits[:, -1] & tail).any())
    want = host_unpack(bits, C, G)
    n = C * G * G
    for dtype in (torch.float32, torch.bfloat16, torch.float16, torch.uint8):
        assert torch.equal(env.unpack_obs(bits, dtype=dtype).cpu().float(), want), dtype
        buf = torch.full((S * n + 2,), 7, dtype=dtype, device=DEV)
        out = buf[1:-1].view(S, C, G, G)                 # one element past an aligned address
        env.unpack_obs(bits, dtype=dtype, out=out)
        assert torch.equal(out.cpu().float(), want), dtype
        assert float(buf[0]) == 7 and float(buf[-1]) == 7, dtype


# ---------------------------------------------------------------------------------------------------- 2. forward rows
@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("row", GEOMETRY, ids=IDS)
def test_trunk_rows_match_reference_features(row, family):
    """8 * CTAs + 1 samples (the grid-stride loop wraps) against the statement; 1, 7, 9 and 8 * CTAs - 1 samples give
    the same rows bit for bit."""
    G, C, M, wpa = row[0], row[4], row[5], row[6]
    env = _env(row, 1)
    n = _ctas(env)[0]
    pol = _policy(env, 3)
    fp = FusedPolicy(env, pol)
    S = 8 * n + 1
    bits, meta = _words(family, S, C, G, wpa, FAMILIES.index(family)), _meta(S, M, 1)
    full = fp.trunk_packed(bits, meta).clone()
    _assert_trunk_close(full, pol, host_unpack(bits, C, G).to(DEV), meta)
    for s in (1, 7, 9, 8 * n - 1):
        part = fp.trunk_packed(bits[:s], meta[:s])
        assert torch.equal(part.view(torch.int16), full[:s].view(torch.int16)), s


# ---------------------------------------------------------------------------------------------------- 3. tail bits
TAIL_ROWS = [r for r in GEOMETRY if tail_mask(r[4], r[0], r[6])]


@pytest.mark.parametrize("row", TAIL_ROWS, ids=[IDS[GEOMETRY.index(r)] for r in TAIL_ROWS])
def test_tail_bits_change_no_row_and_no_gradient(row):
    G, C, M, wpa = row[0], row[4], row[5], row[6]
    env = _env(row, 1)
    fp = FusedPolicy(env, _policy(env, 4))
    S = 2 * _n_ctas(fp) + 5
    bits, meta = _words("uniform", S, C, G, wpa, 2), _meta(S, M, 2)
    bits[::2] = -1                                       # every other sample all ones, up to the last element
    tail = tail_mask(C, G, wpa)
    with_tail, without = bits.clone(), bits.clone()
    with_tail[:, -1] |= tail
    without[:, -1] &= ~tail
    dF = _grad_rows(S, fp.stride, 2)
    rows_a, a = _trunk_grads(fp, with_tail, meta, dF)
    rows_b, b = _trunk_grads(fp, without, meta, dF)
    assert torch.equal(rows_a.view(torch.int16), rows_b.view(torch.int16))
    for x, y in zip(a, b):
        assert torch.equal(x, y)


# ---------------------------------------------------------------------------------------------------- 4. addressing
@pytest.mark.parametrize("row", GEOMETRY, ids=IDS)
def test_in_place_addressing_at_every_agent_count(row):
    """trunk_from_env with k = 1..N shuffled ids (agents_per_env = N, metadata rows of M floats) against trunk_packed
    on the gathered words."""
    G, N, M, wpa = row[0], row[1], row[5], row[6]
    B = 37
    env = _env(row, B)
    _randomise(env, G)
    fp = FusedPolicy(env, _policy(env, 5))
    rng = np.random.default_rng(G * 10 + N)
    for k in range(1, N + 1):
        ids = [int(i) for i in rng.permutation(N)[:k]]
        got = fp.trunk_from_env(ids).clone()
        want = fp.trunk_packed(env.obs_bits[:, ids].reshape(-1, wpa), env.meta[:, ids].reshape(-1, M)).clone()
        assert torch.equal(got.view(torch.int16), want.view(torch.int16)), ids
        part = fp.trunk_from_env(ids, envs=slice(3, 20))
        assert torch.equal(part.view(torch.int16), want[3 * k : 20 * k].view(torch.int16)), ids


# ---------------------------------------------------------------------------------------------------- 5. grouped
@pytest.mark.parametrize("row", GEOMETRY, ids=IDS)
def test_grouped_rows_equal_single_policy_rows(row):
    """A 3-policy PolicyPool over empty segments, 8 * CTAs +- 1 samples and k = 1..N, bit for bit against FusedPolicy."""
    B = 8 * max(_ctas(_env(row, 1))) + 16
    env = _env(row, B)
    _randomise(env, 7)
    pols, pool = _pool(env, 3)
    _check_rows(env, pols, pool, pool.plan(_segments(env, 3)))


# ---------------------------------------------------------------------------------------------------- 6. backward
@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("row", GEOMETRY, ids=IDS)
def test_trunk_grads_match_reference(row, family):
    """S = 1, 37, n + 1 and 2 n + 5 for n backward CTAs (one CTA with two or three samples more than its neighbours);
    a rerun is bit-identical."""
    G, C, M, wpa = row[0], row[4], row[5], row[6]
    env = _env(row, 1)
    fp = FusedPolicy(env, _policy(env, 6))
    n = _n_ctas(fp)
    f = FAMILIES.index(family)
    for S in (1, 37, n + 1, 2 * n + 5):
        bits, meta = _words(family, S, C, G, wpa, 100 * f + S), _meta(S, M, S)
        dF = _grad_rows(S, fp.stride, S)
        rows, got = _trunk_grads(fp, bits, meta, dF)
        _assert_grads_close(fp, host_unpack(bits, C, G).to(DEV), dF, rows, got)
    _, again = _trunk_grads(fp, bits, meta, dF)
    for x, y in zip(got, again):
        assert torch.equal(x, y)


# ---------------------------------------------------------------------------------------------------- 7. whole model
MODEL_ROWS = [r for r in GEOMETRY if r[0] in (5, 6, 8)]


@pytest.mark.parametrize("row", MODEL_ROWS, ids=[IDS[GEOMETRY.index(r)] for r in MODEL_ROWS])
def test_forward_and_ppo_gradients_at_small_k1(row):
    """fc1 with 42 to 534 inputs and 0 to 6 zero pad columns: forward_packed within the inference contract and the PPO
    loss gradients of evaluate_actions within twice autocast's, both against fp32 CtfPolicy."""
    G, N, C, M, wpa = row[0], row[1], row[4], row[5], row[6]
    env = _env(row, 1)
    S = 300
    bits, meta = _words("one_hot", S, C, G, wpa, 3), _meta(S, M, 3)
    dense = host_unpack(bits, C, G).to(DEV)
    pol = _policy(env, 7)
    fp = FusedPolicy(env, pol)
    value, logits = fp.forward_packed(bits, meta)
    (ev, bv), (el, bl) = _bound(pol, dense, meta, value, logits)
    assert ev <= bv, f"value error {ev} > {bv}"
    assert el <= bl, f"logit error {el} > {bl}"
    g = torch.Generator(device=DEV).manual_seed(G)
    flags = env.use_action_mask[torch.arange(S, device=DEV) % N]
    act = torch.where(flags == 1, torch.randint(0, 5, (S,), generator=g, device=DEV),
                      torch.randint(0, 9, (S,), generator=g, device=DEV))
    adv = torch.randn(S, generator=g, device=DEV)
    ret = torch.randn(S, generator=g, device=DEV)
    with torch.no_grad():
        _, old, _, _ = pol.get_action_and_value(dense, meta, flags, act)
    g32, gamp = _fp32_and_autocast_grads(pol, dense, meta, flags, act, old, adv, ret)
    lp, ent, v = fp.evaluate_actions(bits, meta, flags, act)
    _ppo_loss(lp, ent, v, old, adv, ret).backward()
    got = {name: p.grad.clone() for name, p in pol.named_parameters()}
    pol.zero_grad()
    _assert_model_grads(pol, got, g32, gamp)
