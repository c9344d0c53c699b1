"""Batched versions of the reference's two callers of the step path (SURVEY.md §8f row N1).

``collect_rollout``  mirrors ``PPOTrainer.get_single_rollout`` (ppo.py:31-131) for B envs at once;
``batched_duel``     mirrors ``utils.duel`` (utils.py:500-573).

Instead of a Python loop over agents that builds one observation at a time, the step kernel has already
written every agent's observation and metadata into ``env.obs`` / ``env.meta``; one policy forward per team
handles ``B * agents_per_team`` samples.  Team-1 policies act in the flipped frame and their actions are mapped
back by the kernel (``reverse_team1_actions=True``), as ppo.py:84-93 and utils.py:549 do with
``get_reversed_action`` on the host.

Policies are any module with the reference ``Agent.get_action_and_value(grid, meta, use_action_mask)`` on batched
inputs — the reference ``Agent`` itself (agent_network.py:63-81 is batch-safe) or ``policy.CtfPolicy``.  The duel
adapters sample through the same method: ``Agent.get_action`` ends in ``action.item()`` (agent_network.py:58) and
only takes one sample at a time.  A ``fused_policy.FusedPolicy`` on either side reads the packed observations
``env.obs_bits`` and ``env.meta`` in place instead; an env created packed-only (``dense_obs=False, packed_obs=True``)
is accepted when every policy on it is fused.

``policy_seed`` (an int) makes both adapters reproducible: every action of both sides is drawn by
``ctf_sample_actions`` from a Philox word keyed by (policy_seed, global env id, episode, step, agent), so the result
is a function of the env seed and the policy seed alone, whatever else uses torch's random generator and however the
envs are batched.  It needs a ``FusedPolicy`` on every side that acts (the stock dense path hands out actions, not
logits).  ``policy_seed=None`` samples with torch's ``Categorical`` as before.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import torch

from .fused_policy import FusedPolicy


@dataclass
class Rollout:
    """Layout of ppo.py:298-305 with the env axis batched: index [step * apt + agent_offset, env]."""

    grid_states: torch.Tensor      # [T*apt, B, C, G, G]  (or packed: [T*apt, B, words_per_agent] int32, see unpack_grid_states)
    metadata_states: torch.Tensor  # [T*apt, B, M]
    actions: torch.Tensor          # [T*apt, B]
    use_action_mask: torch.Tensor  # [T*apt, B]
    logprobs: torch.Tensor         # [T*apt, B]
    rewards: torch.Tensor          # [T*apt, B]
    dones: torch.Tensor            # [T*apt, B]  (never written by the reference, ppo.py:53 — zero unless reset=False:
                                   # 1 on the rows of an observation that starts a new episode, CleanRL's convention)
    values: torch.Tensor           # [T*apt, B]
    next_grid_state: torch.Tensor  # [B, C, G, G]
    next_metadata_state: torch.Tensor  # [B, M]
    next_done: torch.Tensor        # [B]
    packed: bool = False
    next_value: torch.Tensor | None = None  # [apt, B] bootstrap V(s_T) per (agent, env), set by ppo.PackedPPO.collect
    # reset=False: (t, env.flag_captures() [B, 2] read after step t) for every step t at which the episodes ended
    episode_ends: list = field(default_factory=list)
    episode_stats: dict | None = None  # episodes ended in this rollout, set by ppo.PackedPPO.collect in continuing mode

    def as_reference_arrays(self):
        """The eleven values ``train_ppo`` keeps per update (ppo.py:298-305, 362-376), in the reference's order.

        The first eight are already ``[num_steps, num_envs, ...]``.  The reference overwrites next_grid_state /
        next_metadata_state / next_done with those of the *last* rollout only (ppo.py:372-374) and bootstraps every
        env from that one value; the last env's row is returned to reproduce it — use the full ``next_*`` tensors
        for a per-env bootstrap instead.
        """
        return (self.grid_states, self.metadata_states, self.actions, self.use_action_mask, self.logprobs, self.rewards,
                self.dones, self.values, self.next_grid_state[-1:], self.next_metadata_state[-1:], self.next_done[-1:])

    def unpack_grid_states(self, env, index=slice(None), dtype=torch.float32) -> torch.Tensor:
        """grid_states[index] as [..., C, G, G] of ``dtype`` — expands packed storage with the CUDA unpack kernel
        (the PPO update gathers minibatches this way, ppo.py:440-449, without a float32 rollout buffer)."""
        g = self.grid_states[index]
        return env.unpack_obs(g, dtype=dtype) if self.packed else g.to(dtype)


def _require_folded_reversal(env):
    if not env.ce.cfg.reverse_team1_actions:
        raise ValueError("create the env with reverse_team1_actions=True: team-1 policies act in the flipped frame")


def _team_indices(env, team):
    return [i for i in range(env.N_AGENTS) if env.AGENT_TEAMS[i] == team]


def _require_dense_obs(env, *policies):
    """Stock policies read env.obs; when every policy given is a FusedPolicy, a packed-only env is fine."""
    if env.obs is None and not (policies and all(isinstance(p, FusedPolicy) for p in policies)):
        raise ValueError("this adapter feeds policies from env.obs: create the env with dense_obs=True")


def _require_fused_for_seed(policy_seed, *policies):
    if policy_seed is not None and not all(isinstance(p, FusedPolicy) for p in policies):
        raise ValueError("policy_seed draws actions from the logits of a FusedPolicy: every policy that acts must be one")


def batched_action(policy, grid, meta, use_action_mask) -> torch.Tensor:
    """Actions for a batch of samples from a reference-style policy: ``get_action_batch`` when the policy has one,
    else ``get_action_and_value(...)[0]`` (same Categorical sample as ``Agent.get_action``, which is scalar-only)."""
    fn = getattr(policy, "get_action_batch", None)
    if fn is not None:
        return fn(grid, meta, use_action_mask)
    return policy.get_action_and_value(grid, meta, use_action_mask)[0]


@torch.no_grad()
def collect_rollout(env, agent, opponent, train_team1=True, num_env_steps=None, obs_storage_dtype=torch.float32,
                    reset=True, policy_seed=None) -> Rollout:
    """One rollout of every env (ppo.py:31-131).  ``train_team1=True`` trains team 0 (ppo.py:274-279).

    num_env_steps defaults to GAME_STEPS (one episode per rollout, as num_steps == GAME_STEPS in every
    experiment).  obs_storage_dtype=torch.uint8 stores the {0,1} observations 4x smaller; obs_storage_dtype="packed"
    stores the kernel's 1-bit-per-element copy (env created with packed_obs=True), 32x smaller than float32.

    ``reset=True`` starts every env from ``env.reset()`` (ppo.py:57) and leaves ``dones`` zero.  ``reset=False``
    continues from the env's current state, so a rollout may be shorter than an episode or cross one: the envs must be
    in lock-step (one ``env.step_counts()`` read on entry; unequal counts raise ValueError).  When a step reaches
    ``GAME_STEPS`` its rewards are recorded as usual, ``episode_ends`` gets (t, ``env.flag_captures()``), and
    ``env.reset()`` runs before the next policy call, whose rows get ``dones = 1``.  An env already at ``GAME_STEPS`` on
    entry (the previous rollout ended the episode) is reset first and row 0 gets ``dones = 1``; an env never reset is
    reset first.  ``next_done`` marks a last step that ended the episode.

    ``policy_seed``: both sides draw with ``ctf_sample_actions`` (see the module docstring); the rollout's ``actions``
    and ``logprobs`` come from it.
    """
    _require_folded_reversal(env)
    team = 0 if train_team1 else 1
    mine, theirs = _team_indices(env, team), _team_indices(env, 1 - team)
    _require_dense_obs(env, agent, *([opponent] if theirs else []))
    _require_fused_for_seed(policy_seed, agent, *([opponent] if theirs else []))
    fused_agent, fused_opponent = isinstance(agent, FusedPolicy), isinstance(opponent, FusedPolicy)
    apt = len(mine)
    T = env.GAME_STEPS if num_env_steps is None else int(num_env_steps)
    B, N, dev = env.num_envs, env.N_AGENTS, env.device
    C, G, M = env.n_channels, env.GRID_SIZE, env.meta_size
    mine_t = torch.tensor(mine, device=dev)
    theirs_t = torch.tensor(theirs, device=dev)
    mask_flags = env.use_action_mask  # [N] float, AGENT_TYPE_ACTION_MASK per agent

    packed = obs_storage_dtype == "packed"
    if packed and env.obs_bits is None:
        raise ValueError('obs_storage_dtype="packed" needs an env created with packed_obs=True')
    if env.obs is None and not packed:
        raise ValueError('an env created with dense_obs=False stores its rollout with obs_storage_dtype="packed"')
    out = Rollout(
        grid_states=(torch.zeros((T * apt, B, env.bits_words_per_agent), dtype=torch.int32, device=dev) if packed
                     else torch.zeros((T * apt, B, C, G, G), dtype=obs_storage_dtype, device=dev)),
        metadata_states=torch.zeros((T * apt, B, M), device=dev),
        actions=torch.zeros((T * apt, B), device=dev),
        use_action_mask=torch.zeros((T * apt, B), device=dev),
        logprobs=torch.zeros((T * apt, B), device=dev),
        rewards=torch.zeros((T * apt, B), device=dev),
        dones=torch.zeros((T * apt, B), device=dev),
        values=torch.zeros((T * apt, B), device=dev),
        next_grid_state=torch.empty(0), next_metadata_state=torch.empty(0), next_done=torch.empty(0), packed=packed,
    )
    step = 0
    if reset or env._first:
        obs, meta, _ = env.reset()                                                # ppo.py:57
    else:
        lo, hi = torch.aminmax(env.step_counts())
        step, hi = int(lo), int(hi)
        if step != hi:
            raise ValueError(f"reset=False continues envs in lock-step, but their step counts range from {step} to {hi}")
        if step >= env.GAME_STEPS:
            obs, meta, _ = env.reset()
            out.dones[:apt] = 1
            step = 0
        else:
            obs, meta = env.obs, env.meta
    actions = torch.empty((B, N), dtype=torch.uint8, device=dev)
    for t in range(T):
        sl = slice(t * apt, (t + 1) * apt)
        # trained team: [B, apt, ...] -> [apt, B, ...] so that buffer row = step*apt + agent_offset (ppo.py:74-79)
        if not (fused_agent and packed):
            g = obs[:, mine_t].transpose(0, 1).contiguous()
        m = meta[:, mine_t].transpose(0, 1).contiguous()
        flags = mask_flags[mine_t].unsqueeze(1).expand(apt, B)
        if fused_agent:
            # samples come env-major (b * apt + j): reorder to the buffer's agent-major rows
            fe = mask_flags[mine_t].unsqueeze(0).expand(B, apt).reshape(B * apt)
            # seeded: the kernel also writes the actions into the env's action buffer
            seeded = dict(seed=policy_seed, actions=actions) if policy_seed is not None else {}
            a, logp, _, v = agent.get_action_and_value(fe, agent_ids=mine, env=env, **seeded)
            a, logp, v = (x.reshape(B, apt).t().reshape(apt * B) for x in (a, logp, v.reshape(-1)))
        else:
            a, logp, _, v = agent.get_action_and_value(
                g.reshape(apt * B, C, G, G).float(), m.reshape(apt * B, M), flags.reshape(apt * B)
            )
        if packed:
            out.grid_states[sl] = env.obs_bits[:, mine_t].transpose(0, 1)
        else:
            out.grid_states[sl] = g.to(obs_storage_dtype)
        out.metadata_states[sl] = m
        out.values[sl] = v.reshape(apt, B)
        out.actions[sl] = a.reshape(apt, B).float()
        out.use_action_mask[sl] = flags
        out.logprobs[sl] = logp.reshape(apt, B)
        if policy_seed is None:
            actions[:, mine_t] = a.reshape(apt, B).t().to(torch.uint8)
        if theirs:
            k = len(theirs)
            fo = mask_flags[theirs_t].unsqueeze(0).expand(B, k).reshape(B * k)
            if policy_seed is not None:
                opponent.get_action_and_value(fo, agent_ids=theirs, env=env, seed=policy_seed, actions=actions)
            else:
                if fused_opponent:
                    ao = opponent.get_action_and_value(fo, agent_ids=theirs, env=env)[0]
                else:
                    go = obs[:, theirs_t].reshape(B * k, C, G, G).float()
                    mo = meta[:, theirs_t].reshape(B * k, M)
                    ao = opponent.get_action_and_value(go, mo, fo)[0]
                actions[:, theirs_t] = ao.reshape(B, k).to(torch.uint8)
        obs, meta, rewards, dones, _ = env.step(actions)                          # ppo.py:98
        out.rewards[sl] = rewards[:, mine_t].t()                                  # ppo.py:106-109
        step += 1
        if not reset and step >= env.GAME_STEPS:
            out.episode_ends.append((t, env.flag_captures().clone()))
            if t + 1 < T:
                obs, meta, _ = env.reset()
                out.dones[(t + 1) * apt : (t + 2) * apt] = 1
                step = 0
    first = min(mine)
    if obs is None:                                                               # packed-only env
        out.next_grid_state = env.unpack_obs(env.obs_bits[:, first])
    else:
        out.next_grid_state = obs[:, first].clone().float()                       # ppo.py:116-118
    out.next_metadata_state = meta[:, first].clone()
    out.next_done = dones.float().clone()                                         # ppo.py:111
    return out


@torch.no_grad()
def batched_duel(env, agent, opponent, max_steps=256, return_result=True, policy_seed=None):
    """utils.duel (utils.py:500-573) for every env of the batch.

    Team 0 acts with ``agent``, team 1 with ``opponent``.  Stops when the envs are done or after
    max_steps + 1 steps (the reference's ``step_count > max_steps`` check runs after the step, :559-560).
    Returns int tensor [B] of +1 / 0 / -1 (team-0 win / draw / loss by flag captures, :562-569), or the
    all-reduced ``env.metrics`` dict when return_result=False (:571).  ``policy_seed``: both sides draw with
    ``ctf_sample_actions`` (see the module docstring).
    """
    _require_folded_reversal(env)
    _require_dense_obs(env, agent, opponent)
    B, N, dev = env.num_envs, env.N_AGENTS, env.device
    C, G, M = env.n_channels, env.GRID_SIZE, env.meta_size
    team_ids = [_team_indices(env, t) for t in (0, 1)]
    _require_fused_for_seed(policy_seed, *(p for p, ids in zip((agent, opponent), team_ids) if ids))
    teams = [torch.tensor(ids, device=dev) for ids in team_ids]
    policies = (agent, opponent)
    obs, meta, _ = env.reset()
    actions = torch.empty((B, N), dtype=torch.uint8, device=dev)
    step_count = 0
    while True:
        step_count += 1
        for idx, ids, pol in zip(teams, team_ids, policies):
            k = idx.numel()
            if k == 0:
                continue
            flags = env.use_action_mask[idx].unsqueeze(0).expand(B, k).reshape(B * k)
            if policy_seed is not None:
                pol.get_action_and_value(flags, agent_ids=ids, env=env, seed=policy_seed, actions=actions)
                continue
            if isinstance(pol, FusedPolicy):
                a = pol.get_action_and_value(flags, agent_ids=ids, env=env)[0]
            else:
                a = batched_action(pol, obs[:, idx].reshape(B * k, C, G, G).float(), meta[:, idx].reshape(B * k, M), flags)
            actions[:, idx] = a.reshape(B, k).to(torch.uint8)
        obs, meta, _, dones, _ = env.step(actions)
        if step_count > max_steps or step_count >= env.GAME_STEPS:  # all envs finish in lock-step
            break
    if return_result:
        caps = env.flag_captures()
        return torch.sign(caps[:, 0] - caps[:, 1])
    return env.episode_stats()
