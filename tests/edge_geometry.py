"""Small scenarios at the edges of the geometry the env's step path accepts: maps from 2x2 to 16x16, one agent, 14
channels, spawns on the last row or column, and packed words with and without tail bits.

``EDGE_ROWS`` is shared by tests/test_edge_geometry_spec.py (the CPU oracle and a numpy statement of the observation)
and tests/test_gpu_env_geometry.py (the CUDA env against the oracle).  Each row names the edge it reaches and the
events its episode must produce; the CPU spec checks that they still fire, so an edit of the table cannot silently
stop reaching its edge.  Importable without a GPU.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

import traces

GAME_STEPS = 40

# stats rows of the counters (config.METRIC_NAMES) that an event check may name
EVENTS = {"tags": 0, "respawns": 1, "pickups": 2, "captures": 3, "dispossessions": 4, "laid": 5, "mined": 6}


def edge_config(G, N, *, teams=None, types=None, flip=None, spawns=None, flags=None, starts=None, blocks=(), destr=(),
                **kw):
    """Env kwargs of a small scenario.  Defaults: agent i starts at (i // G, i % G), team i % 2, type 0; flags (also the
    capture cells) at (G-1, G-1) / (G-1, G-2); spawns at (1, 1) / (G-2, G-2); GAME_STEPS 40.  ``kw`` overrides any
    other constructor keyword."""
    teams = [i % 2 for i in range(N)] if teams is None else list(teams)
    types = [0] * N if types is None else list(types)
    flags = {0: (G - 1, G - 1), 1: (G - 1, G - 2)} if flags is None else flags
    scenario = dict(
        SCENARIO_NAME=f"edge-G{G}-N{N}", GRID_SIZE=G, FLIP_AXIS=flip, FLAG_POSITIONS=flags, CAPTURE_POSITIONS=flags,
        SPAWN_POSITIONS={0: (1, 1), 1: (G - 2, G - 2)} if spawns is None else spawns,
        AGENT_STARTING_POSITIONS={i: (i // G, i % G) for i in range(N)} if starts is None else starts,
        BLOCK_TILE_SLICES=list(blocks), DESTRUCTIBLE_TILE_SLICES=list(destr),
    )
    ec = dict(AGENT_CONFIG={i: {"team": teams[i], "type": types[i]} for i in range(N)}, SCENARIO=scenario,
              MAP_SYMMETRY_CHECK=False, GAME_STEPS=GAME_STEPS)
    ec.update(kw)
    return ec


@dataclass(frozen=True)
class EdgeRow:
    id: str
    config: dict
    plan: tuple                  # (G, N, C, M, words per agent, tail bits) that compile_config must give
    events: tuple = ()           # EVENTS keys, and "fault" for CTF_FAULT_RESPAWN_BLOCKED, that the episode must produce


def _all(v):
    return {t: v for t in range(4)}


EDGE_ROWS = [
    # smallest map: C = 5, one word per agent with 12 tail bits, 20-element env blocks (shorter than a uint8 store
    # vector: stream_env's head and tail scalar stores carry the whole block); the agent cannot move, so nothing fires
    EdgeRow("G2-N1", edge_config(2, 1, flags={0: (1, 0), 1: (0, 1)}, spawns={0: (1, 1), 1: (1, 1)}),
            (2, 1, 5, 8, 1, 12)),
    # a lone team-1 observer (C = 4) with the rows flipped (flip 0) on 3x3; N = 1: no opponents, M = 8
    EdgeRow("G3-N1-team1-flip0", edge_config(3, 1, teams=[1], flip=0), (3, 1, 4, 8, 2, 28), ("pickups", "captures")),
    # lethal tags every few steps on 3x3: both spawn windows are the whole map
    EdgeRow("G3-N2-lethal", edge_config(3, 2, AGENT_TYPE_DAMAGE=_all(100), TAG_PROBABILITY=1.0), (3, 2, 5, 10, 2, 19),
            ("respawns", "dispossessions")),
    # 8 agents on 16 cells, C = 11, 6 words per agent: full spawn windows raise the respawn-blocked fault bit
    EdgeRow("G4-N8", edge_config(4, 8, types=[min(i // 2, 3) for i in range(8)]), (4, 8, 11, 22, 6, 16),
            ("respawns", "fault")),
    # unbalanced teams (two against one), columns flipped (flip 1), C * G * G = 96: no tail bits
    EdgeRow("G4-N3-teams001-flip1", edge_config(4, 3, teams=[0, 0, 1], types=[0, 0, 1], flip=1), (4, 3, 6, 12, 3, 0),
            ("respawns", "captures")),
    # spawns on the last row and column, the anti-diagonal flip (flip 2), C * G * G = 225: 31 tail bits
    EdgeRow("G5-N4-flip2-border", edge_config(5, 4, types=[0, 1, 2, 3], flip=2, spawns={0: (4, 4), 1: (1, 4)}),
            (5, 4, 9, 14, 8, 31), ("respawns", "fault")),
    # border spawns with HP as IEEE doubles (1.15 / 0.3 / 0.05 are not dyadic)
    EdgeRow("G6-N4-hpfloat-border", edge_config(6, 4, spawns={0: (5, 5), 1: (1, 5)}, AGENT_TYPE_HP=_all(1.15),
                                                AGENT_TYPE_DAMAGE=_all(0.3), AGENT_HP_HEALING_PER_STEP=0.05),
            (6, 4, 5, 14, 6, 12), ("respawns", "fault")),
    # a flag dropped at the victim's cell, home-flag capture and adjusted rewards on a small map
    EdgeRow("G6-N5-dropflag", edge_config(6, 5, DROP_FLAG_WHEN_NO_HP=True, HOME_FLAG_CAPTURE=True, USE_ADJUSTED_REWARDS=True,
                                          TAG_PROBABILITY=1.0), (6, 5, 5, 16, 6, 12), ("dispossessions", "captures")),
    # the largest plan: G = 16, N = 8, C = 14 (channel codes up to 13), 28 672 bits per env, the most non-open cells;
    # the destructible row 2 lies in the miners' path, so blocks are mined and laid within the episode
    EdgeRow("G16-N8-C14", edge_config(16, 8, types=[min(i // 2, 3) for i in range(8)],
                                      blocks=[(r, slice(2, 8)) for r in range(4, 15, 2)],
                                      destr=[(r, slice(9, 14)) for r in range(4, 15, 2)] + [(2, slice(3, 12))]),
            (16, 8, 14, 22, 112, 0), ("laid", "mined")),
    # one agent on the largest map: 40 words per agent, M = 8, every tag site without opponents; its spawn in the
    # corner (15, 15) is accepted but never used (no one tags a lone agent: the next row respawns there)
    EdgeRow("G16-N1-corner", edge_config(16, 1, spawns={0: (15, 15), 1: (1, 1)}, starts={0: (15, 0)},
                                         flags={0: (15, 8), 1: (8, 0)}), (16, 1, 5, 8, 40, 0), ("pickups", "captures")),
    # respawns into windows clipped by the last row and the last column of a 16x16 map, whose 16-cell rows leave no
    # padding column in the shared grid
    EdgeRow("G16-N2-corner-lethal", edge_config(16, 2, spawns={0: (15, 15), 1: (15, 14)}, starts={0: (15, 15), 1: (15, 13)},
                                                flags={0: (0, 1), 1: (0, 0)}, AGENT_TYPE_DAMAGE=_all(100),
                                                TAG_PROBABILITY=1.0), (16, 2, 5, 10, 40, 0), ("respawns",)),
]
EDGE_IDS = [r.id for r in EDGE_ROWS]


def builder_actions(pol, rng, st):
    """uint8 [B, N]: the 'builder' policy (traces.make_policy) for every env of an oracle state."""
    return np.stack([pol(rng, st["pos"][b], st["has_flag"][b]) for b in range(len(st["pos"]))])


def policy(ce):
    return traces.make_policy("builder", ce)


def check_step(t, game_steps):
    """Whether the whole state and the observations are compared before step t (t = game_steps + 2: after the last)."""
    return t % 7 == 0 or t >= game_steps - 1
