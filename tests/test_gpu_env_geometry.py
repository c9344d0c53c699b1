"""The env's step path (k_reset, k_step, k_observe, store_packed, k_unpack) against the CPU oracle on the rows of
tests/edge_geometry.py: 2x2 to 16x16 maps, one agent, 14 channels, spawns on the last row and column, packed words with
and without tail bits.  Each row runs at B = 1, 5 (one full CTA of four env warps plus a ragged one) and 37 (with a
nonzero env_id_base), over a whole episode, two steps past its end, a reset and ten steps of a second episode.

Observations are compared in all four dtypes: float32 in the env's own buffer, uint8 / float16 / bfloat16 in caller
buffers that start one element past an aligned address, with a guard element on each side that must stay untouched.
"""
import numpy as np
import pytest
import torch

from edge_geometry import EDGE_IDS, EDGE_ROWS, builder_actions, check_step, policy
from helpers import bits
from marl_ctf_development_b200 import GridworldCtfGPU
from oracle.ctf_oracle import OracleBatch
from test_gpu_parity import _assert_batch_state, _pack_reference
from test_gpu_trunk_geometry import tail_mask

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
SEED = 29
DTYPES = (torch.float32, torch.uint8, torch.float16, torch.bfloat16)
GUARD = 7
SECOND_EPISODE = 10
CASES = [(row, B) for row in EDGE_ROWS for B in (1, 5, 37)]
CASE_IDS = [f"{i}-B{B}" for i in EDGE_IDS for B in (1, 5, 37)]


def _base(B):
    return 1000 if B == 37 else 0


def _env(row, B, **kw):
    return GridworldCtfGPU(**row.config, num_envs=B, device=DEV, seed=SEED, env_id_base=_base(B), **kw)


def _guarded(shape, dtype):
    """A buffer of GUARD values and the view of ``shape`` inside it that starts one element past its aligned start."""
    buf = torch.full((int(np.prod(shape)) + 2,), GUARD, dtype=dtype, device=DEV)
    return buf, buf[1:-1].view(shape)


def _assert_guards(buf, where):
    assert float(buf[0]) == GUARD and float(buf[-1]) == GUARD, f"{where}: {buf.dtype} store outside the output"


def _assert_same(got, want, where, what):
    """Equality of [B, X, ...] arrays (X: agents, or metrics for the statistics); the message names the first [b, x]
    that differs."""
    if not np.array_equal(got, want):
        b, i = np.argwhere((got != want).reshape(got.shape[0], got.shape[1], -1).any(-1))[0]
        raise AssertionError(f"{where}: {what} differs at env {b}, index {i}\n got={got[b, i]}\nwant={want[b, i]}")


def _masks(N):
    return ([1] * N, [0] * N, [i % 2 for i in range(N)])


@pytest.mark.parametrize("row,B", CASES, ids=CASE_IDS)
def test_step_path_matches_oracle(row, B):
    """Rewards, dones and the fault word every step; the whole state (float HP included), the observations in all four
    dtypes, the metadata and observe(reverse_flags=...) at every seventh step and the last ones; statistics, visitation
    maps and stats_sum at the end of each episode."""
    main = _env(row, B, stats="full")
    G, N, C = row.plan[:3]
    assert (main.GRID_SIZE, main.N_AGENTS, main.n_channels, main.meta_size) == row.plan[:4]
    bufs, envs = [], [main]
    for dtype in DTYPES[1:]:
        buf, view = _guarded((B, N, C, G, G), dtype)
        bufs.append(buf)
        envs.append(_env(row, B, obs_dtype=dtype, obs_out=view))
    orc = OracleBatch(main.ce, B, seed=SEED, env_id_base=_base(B))
    pol, rng = policy(main.ce), np.random.default_rng(SEED)

    def check(where):
        _assert_batch_state(main, orc, where)
        o_ref, m_ref = orc.observe()
        for env in envs:
            _assert_same(env.obs.float().cpu().numpy(), o_ref, where, f"{env.obs_dtype} observation")
            _assert_same(bits(env.meta.cpu().numpy()), bits(m_ref), where, f"metadata (next to {env.obs_dtype})")
        for buf in bufs:
            _assert_guards(buf, where)
        for flags in _masks(N):
            obs, meta = main.observe(reverse_flags=flags, into_new=True)
            o_ref, m_ref = orc.observe(reverse_flags=flags)
            _assert_same(obs.cpu().numpy(), o_ref, where, f"observe(reverse_flags={flags})")
            _assert_same(bits(meta.cpu().numpy()), bits(m_ref), where, f"observe(reverse_flags={flags}) metadata")

    def check_stats(where):
        st, so = main.get_state(), orc.state()
        _assert_same(st["stats"], so["stats"], where, "statistics")
        _assert_same(st["visits"], so["visits"], where, "visitation maps")
        assert np.array_equal(main.stats_sum(all_reduce=False).cpu().numpy(), so["stats"].sum(0)), f"{where}: stats_sum"

    check(f"{row.id} B={B} reset")
    for episode, steps in enumerate((main.GAME_STEPS + 2, SECOND_EPISODE)):
        if episode:
            for env in envs:
                env.reset()
            orc.reset()
            check(f"{row.id} B={B} reset {episode}")
        for t in range(steps):
            where = f"{row.id} B={B} episode {episode} step {t}"
            a = builder_actions(pol, rng, orc.state())
            a_dev = torch.from_numpy(a).to(DEV)
            for env in envs:
                env.step(a_dev)
            r_ref, d_ref = orc.step(a)
            for env in envs:
                _assert_same(bits(env.rewards.cpu().numpy()), bits(r_ref), where, "rewards")
                assert np.array_equal(env.dones.cpu().numpy(), d_ref), f"{where}: dones differ"
            assert main.take_faults() == orc.take_faults(), f"{where}: fault word differs"
            if check_step(t + 1, main.GAME_STEPS) or t == steps - 1:
                check(where)
        check_stats(f"{row.id} B={B} end of episode {episode}")


@pytest.mark.parametrize("row,B", CASES, ids=CASE_IDS)
def test_packed_words_and_unpack_match_oracle(row, B):
    """obs_bits is the little-endian packbits of the oracle's observation with every tail bit 0, a dense_obs=False env
    writes the same words, and unpack_obs turns them back into the oracle's observation in all four dtypes."""
    env = _env(row, B, packed_obs=True)
    packed = _env(row, B, packed_obs=True, dense_obs=False)
    G, N, C, _, wpa, _ = row.plan
    assert env.bits_words_per_agent == wpa
    tail = tail_mask(C, G, wpa)
    orc = OracleBatch(env.ce, B, seed=SEED, env_id_base=_base(B))
    pol, rng = policy(env.ce), np.random.default_rng(SEED + 1)

    def check(where):
        o_ref, _ = orc.observe(u8=True)
        words = env.obs_bits.cpu().numpy().astype(np.int64) & 0xFFFFFFFF
        _assert_same(words, _pack_reference(o_ref, wpa), where, "packed observation")
        assert not bool((env.obs_bits[..., -1] & tail).any()), f"{where}: a tail bit is set"
        assert torch.equal(packed.obs_bits, env.obs_bits), f"{where}: the dense_obs=False env wrote other words"
        for dtype in DTYPES:
            buf, out = _guarded((B, N, C, G, G), dtype)
            packed.unpack_obs(packed.obs_bits, dtype=dtype, out=out)
            _assert_same(out.float().cpu().numpy(), o_ref.astype(np.float32), where, f"{dtype} unpack_obs")
            _assert_guards(buf, where)

    check(f"{row.id} B={B} reset")
    for episode, steps in enumerate((env.GAME_STEPS + 2, SECOND_EPISODE)):
        if episode:
            env.reset()
            packed.reset()
            orc.reset()
            check(f"{row.id} B={B} reset {episode}")
        for t in range(steps):
            a = builder_actions(pol, rng, orc.state())
            a_dev = torch.from_numpy(a).to(DEV)
            env.step(a_dev)
            packed.step(a_dev)
            orc.step(a)
            if check_step(t + 1, env.GAME_STEPS) or t == steps - 1:
                check(f"{row.id} B={B} episode {episode} step {t}")
