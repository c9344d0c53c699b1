"""Counter-based random draws of the step path (host restatement).

The reference draws from two global Mersenne Twisters with data-dependent draw
counts (gridworld_ctf.py:740 ``random.shuffle``, :815 ``np.random.rand``, :771
``np.random.randint``).  The B200 path replaces them with Philox4x32-10 draws
addressed by *site*, so that the same draws can be injected into the reference
(oracle/ref_shim.py) and results compared bit for bit.

Draw addressing (identical in csrc/ctf_kernels.cu and oracle/ctf_oracle.c):

    key     = (seed & 0xffffffff, seed >> 32)
    counter = (global env id, episode, env_step_count after increment, site)
    site    = 4 * acting_agent_id + opponent_slot        (32 sites per step)

    word 0 of site (a, j): tag roll of actor a against OPPONENTS[team(a)][j];
                           hit  <=>  word0 < tag_threshold  (== word0 / 2**32 < TAG_PROBABILITY)
    word 1 of site (a, j): respawn cell of that opponent if the hit is lethal;
                           pick = (word1 * k) >> 32 among the k open cells
    word 2 of site i (1 <= i < N): Fisher-Yates draw i of the move order:
                           j = (word2 * (i + 1)) >> 32, swap(order[i], order[j]), i = N-1 .. 1,
                           starting from the identity order.

Policy draws (``ctf_sample_actions``, ``k_sample_actions``; opt-in through ``policy_seed``) use the same key layout
with their own seed and one counter per (env, step, agent):

    key     = (policy_seed & 0xffffffff, policy_seed >> 32)
    counter = (global env id, episode, env_step_count before the step, 0x80000000 | agent)

    word 0:  u = (word0 >> 8) * 2**-24, the uniform of the agent's categorical draw (``sample_action``)

The top bit of the site word keeps every policy counter apart from the env's sites 0..31, so the two streams never
share a word even when the policy seed equals the env seed.

This module is host logic (numpy); the product path never calls it — the CUDA
kernels generate the same words on the device.
"""
from __future__ import annotations

import numpy as np

PHILOX_M0 = 0xD2511F53
PHILOX_M1 = 0xCD9E8D57
PHILOX_W0 = 0x9E3779B9
PHILOX_W1 = 0xBB67AE85

SITES_PER_STEP = 32
MAX_OPP_SLOTS = 4
POLICY_SITE = 0x80000000
N_ACTIONS = 9
NO_OP_ACTION = 4


def philox4x32_10(counter: np.ndarray, key: np.ndarray) -> np.ndarray:
    """Philox4x32 with 10 rounds. counter: uint32[..., 4]; key: uint32[..., 2] (broadcastable)."""
    c = np.asarray(counter, dtype=np.uint64)
    k = np.asarray(key, dtype=np.uint64)
    c0, c1, c2, c3 = (c[..., i].copy() for i in range(4))
    k0 = np.broadcast_to(k[..., 0], c0.shape).copy()
    k1 = np.broadcast_to(k[..., 1], c0.shape).copy()
    mask = np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0 = np.uint64(PHILOX_M0) * c0
        p1 = np.uint64(PHILOX_M1) * c2
        hi0, lo0 = p0 >> np.uint64(32), p0 & mask
        hi1, lo1 = p1 >> np.uint64(32), p1 & mask
        c0, c1, c2, c3 = (hi1 ^ c1 ^ k0) & mask, lo1, (hi0 ^ c3 ^ k1) & mask, lo0
        k0 = (k0 + np.uint64(PHILOX_W0)) & mask
        k1 = (k1 + np.uint64(PHILOX_W1)) & mask
    return np.stack([c0, c1, c2, c3], axis=-1).astype(np.uint32)


def step_words(seed: int, env_id: int, episode: int, step: int) -> np.ndarray:
    """All 32 sites x 4 words of one (env, episode, step). Returns uint32[32, 4]."""
    ctr = np.empty((SITES_PER_STEP, 4), dtype=np.uint32)
    ctr[:, 0] = np.uint32(env_id & 0xFFFFFFFF)
    ctr[:, 1] = np.uint32(episode & 0xFFFFFFFF)
    ctr[:, 2] = np.uint32(step & 0xFFFFFFFF)
    ctr[:, 3] = np.arange(SITES_PER_STEP, dtype=np.uint32)
    key = np.array([seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF], dtype=np.uint32)
    return philox4x32_10(ctr, key)


def move_order(words: np.ndarray, n_agents: int) -> list[int]:
    """Move order of one step from its site words (see module docstring)."""
    order = list(range(n_agents))
    for i in range(n_agents - 1, 0, -1):
        j = (int(words[i, 2]) * (i + 1)) >> 32
        order[i], order[j] = order[j], order[i]
    return order


def tag_site(actor: int, opp_slot: int) -> int:
    return MAX_OPP_SLOTS * actor + opp_slot


def tag_roll_uniform(words: np.ndarray, actor: int, opp_slot: int) -> float:
    """The value ``np.random.rand()`` must return at this site (exact in fp64)."""
    return int(words[tag_site(actor, opp_slot), 0]) / 4294967296.0


def respawn_pick(words: np.ndarray, actor: int, opp_slot: int, k: int) -> int:
    """The value ``np.random.randint(k)`` must return at this site."""
    return (int(words[tag_site(actor, opp_slot), 1]) * k) >> 32


def policy_words(seed: int, env_id, episode, step, agent) -> np.ndarray:
    """The Philox words of the policy draw of (env_id, episode, step, agent), each an int or an integer array (they
    broadcast).  Returns uint32[..., 4]; word 0 is the draw's (see the module docstring)."""
    env_id, episode, step, agent = np.broadcast_arrays(*(np.asarray(v, dtype=np.int64) for v in (env_id, episode, step, agent)))
    ctr = np.stack([env_id & 0xFFFFFFFF, episode & 0xFFFFFFFF, step & 0xFFFFFFFF, POLICY_SITE | (agent & 0x7FFFFFFF)],
                   axis=-1).astype(np.uint32)
    key = np.array([seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF], dtype=np.uint32)
    return philox4x32_10(ctr, key)


def policy_uniform(words: np.ndarray) -> np.ndarray:
    """u = (word0 >> 8) * 2**-24 in [0, 1), exact in float64 (and in float32)."""
    return (np.asarray(words)[..., 0] >> np.uint32(8)).astype(np.float64) * 2.0 ** -24


def sample_action(logits, masked, u):
    """What ``k_sample_actions`` computes, in float64: (action int64, logprob, entropy), each of shape [...].

    ``logits`` [..., 9], ``masked`` [...] (truthy: ``CtfPolicy.masked_logits`` adds -1e9 to actions 5..8), ``u`` [...]
    the draw's uniform.  m = max x, e_i = exp(x_i - m), c_i = e_0 + ... + e_i, Z = c_8; the action is the smallest i
    with u*Z < c_i, else (rounding) the largest i with e_i > 0, else (no positive mass: NaN or infinite logits) the
    no-op 4.  logprob = (x_action - m) - log Z; entropy = log Z - sum_{e_i > 0} e_i (x_i - m) / Z."""
    x = np.array(logits, dtype=np.float64)
    masked = np.broadcast_to(np.asarray(masked, dtype=bool), x.shape[:-1])
    x[..., 5:] += np.where(masked[..., None], -1e9, 0.0)
    u = np.broadcast_to(np.asarray(u, dtype=np.float64), x.shape[:-1])
    with np.errstate(invalid="ignore", over="ignore"):
        m = np.fmax.reduce(x, axis=-1)
        d = x - m[..., None]
        e = np.exp(d)
        c = np.cumsum(e, axis=-1)
        z = c[..., -1]
        hit = (u * z)[..., None] < c
        pos = e > 0
        idx = np.arange(N_ACTIONS)
        last_pos = np.where(pos.any(-1), np.where(pos, idx, -1).max(-1), NO_OP_ACTION)
        action = np.where(hit.any(-1), hit.argmax(-1), last_pos).astype(np.int64)
        log_z = np.log(z)
        logprob = np.take_along_axis(d, action[..., None], -1)[..., 0] - log_z
        entropy = log_z - np.where(pos, e * d, 0.0).sum(-1) / z
    return action, logprob, entropy
