"""CPU checks of the edge-geometry table (tests/edge_geometry.py): every row compiles to the plan it names, the oracle's
observation equals a plain numpy statement of standardise_state at every row, and each row's episode still produces
the events its comment claims.  At these shapes the kernel and the oracle are two restatements by the same authors; the
numpy statement below is the third opinion.  No GPU needed."""
import numpy as np
import pytest

from edge_geometry import EDGE_IDS, EDGE_ROWS, EVENTS, builder_actions, check_step, policy
from marl_ctf_development_b200._native import FAULT_RESPAWN_BLOCKED
from marl_ctf_development_b200.config import compile_config
from oracle.ctf_oracle import OracleBatch, OracleEnv

B, SEED = 9, 5

# reverse_grid of standardise_state (gridworld_ctf.py:1003-1007) per FLIP_AXIS, on [..., G, G]
FLIPS = {
    None: lambda x: np.flip(x, (-2, -1)),
    0: lambda x: np.flip(x, -2),
    1: lambda x: np.flip(x, -1),
    2: lambda x: np.rot90(np.swapaxes(x, -2, -1), 2, axes=(-2, -1)),      # rot90(x.T, 2) of every plane
}


def numpy_observation(ce, st, reverse_flags=None):
    """uint8 [B, N, C, G, G] from an oracle state: plane 0 is the agent's own cell, plane chan_lut[team][tile] holds
    every non-open cell whose tile has a channel, and the planes are flipped per FLIP_AXIS where the agent's reverse flag is set."""
    grid, pos = st["grid"], st["pos"]
    N, C, G = ce.N_AGENTS, ce.n_channels, ce.GRID_SIZE
    lut = np.array([list(ce.cfg.chan_lut[t]) for t in (0, 1)])
    rev = [ce.cfg.obs_reverse[i] for i in range(N)] if reverse_flags is None else reverse_flags
    out = np.zeros((len(grid), N, C, G, G), dtype=np.uint8)
    for b in range(len(grid)):
        r, c = np.nonzero(grid[b])
        for i in range(N):
            ch = lut[ce.AGENT_TEAMS[i]][grid[b, r, c]]
            seen = ch > 0            # a tile outside TILES_USED (a flag's home block on a map without blocks) is unseen
            out[b, i, ch[seen], r[seen], c[seen]] = 1
            out[b, i, 0, pos[b, i, 0], pos[b, i, 1]] = 1
            if rev[i]:
                out[b, i] = FLIPS[ce.FLIP_AXIS](out[b, i].copy())
    return out


def _episode(row):
    """Yields (t, ce, orc) before each step of a GAME_STEPS + 2 step episode of B envs with the builder policy, then
    once more after the last step; returns the OR of the fault words."""
    ce = compile_config(**row.config)
    orc = OracleBatch(ce, B, seed=SEED, env_id_base=3)
    pol, rng = policy(ce), np.random.default_rng(SEED)
    faults = 0
    for t in range(ce.GAME_STEPS + 2):
        yield t, ce, orc
        orc.step(builder_actions(pol, rng, orc.state()))
        faults |= orc.take_faults()
    yield ce.GAME_STEPS + 2, ce, orc
    return faults


@pytest.mark.parametrize("row", EDGE_ROWS, ids=EDGE_IDS)
def test_row_compiles_to_its_plan(row):
    ce = compile_config(**row.config)
    G, N, C = ce.GRID_SIZE, ce.N_AGENTS, ce.n_channels
    wpa = -(-C * G * G // 32)
    assert (G, N, C, ce.meta_size, wpa, 32 * wpa - C * G * G) == row.plan


@pytest.mark.parametrize("row", EDGE_ROWS, ids=EDGE_IDS)
def test_oracle_observation_equals_numpy_statement(row):
    N = row.plan[1]
    masks = [None, [1] * N, [0] * N, [i % 2 for i in range(N)], [1 - i % 2 for i in range(N)]]
    for t, ce, orc in _episode(row):
        if not check_step(t, ce.GAME_STEPS):
            continue
        st = orc.state()
        for rf in masks:
            want = numpy_observation(ce, st, rf)
            got, _ = orc.observe(reverse_flags=rf, u8=True)
            assert np.array_equal(got, want), f"{row.id} t={t} reverse_flags={rf}: observation differs"
            got_f, _ = orc.observe(reverse_flags=rf)
            assert np.array_equal(got_f, want.astype(np.float32)), f"{row.id} t={t} reverse_flags={rf}: float observation"


@pytest.mark.parametrize("row", EDGE_ROWS, ids=EDGE_IDS)
def test_observe_fast_equals_observe(row):
    """The CPU baseline's writer (observe_fast) gives observe()'s bytes at these shapes too."""
    ce = compile_config(**row.config)
    envs = [OracleEnv(ce, seed=SEED, env_id=3 + b) for b in range(B)]
    pol, rng = policy(ce), np.random.default_rng(SEED)
    for t in range(ce.GAME_STEPS + 3):
        if check_step(t, ce.GAME_STEPS):
            for b, env in enumerate(envs):
                obs, meta = env.observe()
                o_f, m_f = env.observe_fast()
                assert np.array_equal(o_f, obs), f"{row.id} t={t} env {b}: observe_fast observation differs"
                assert np.array_equal(m_f.view(np.uint32), meta.view(np.uint32)), f"{row.id} t={t} env {b}: metadata"
        if t < ce.GAME_STEPS + 2:
            for env in envs:
                st = env.state()
                env.step(pol(rng, st["pos"], st["has_flag"]))


@pytest.mark.parametrize("row", EDGE_ROWS, ids=EDGE_IDS)
def test_row_episode_reaches_its_edge(row):
    """The events named in the row's comment fire in its episode; a row that claims none produces none."""
    gen = _episode(row)
    try:
        while True:
            _, _, orc = next(gen)
    except StopIteration as stop:
        faults = stop.value
    counts = orc.state()["stats"].sum(axis=(0, 2))[: len(EVENTS)]
    for ev in row.events:
        if ev == "fault":
            assert faults & FAULT_RESPAWN_BLOCKED, f"{row.id}: no respawn found its spawn window full"
        else:
            assert counts[EVENTS[ev]] > 0, f"{row.id}: no {ev} ({dict(zip(EVENTS, counts))})"
    if not row.events:
        assert not counts.any() and not faults, f"{row.id}: events fired ({dict(zip(EVENTS, counts))})"
