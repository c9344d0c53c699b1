"""PPO from packed rollouts: advantages on the device (``ctf_gae``) and a CleanRL-style update (``PackedPPO``).

``PackedPPO(env, agent, args)`` joins what the package already has into one trainer: ``collect_rollout`` with
``FusedPolicy`` on both sides and packed observation storage, ``ctf_gae`` (``k_gae`` in csrc/ctf_kernels.cu) for the
advantages and returns, and ``FusedPolicy.evaluate_actions`` for the forward and backward of every minibatch, cut into
chunks whose gradients accumulate.  ``args`` carries the reference's ``TrainingConfig`` names (``num_minibatches``,
``update_epochs``, ``gamma``, ``gae_lambda``, ``norm_adv``, ``clip_coef``, ``clip_vloss``, ``ent_coef``, ``vf_coef``,
``max_grad_norm``, ``target_kl``, ``learning_rate``).  The optimiser is torch's: ``Adam(lr, eps=1e-5)`` unless the
caller passes one.

Two deliberate differences from the reference's ``PPOTrainer`` (ppo.py): every (trained agent, env) pair is its own
sequence over the T steps, where the reference chains the apt agents' rows of an env into one sequence of T*apt rows;
and every (agent, env) bootstraps from its own V(s_T), where the reference bootstraps every env from the last env's
state.  The reference's exact update stays available through ``Rollout.as_reference_arrays``.

``PackedPPO(..., rollout_steps=T)`` trains on rollouts of T <= GAME_STEPS steps that continue the env's episodes
across updates (CleanRL's and Isaac Gym's scheme), where the reference resets the envs at every rollout: the env is reset
when its episodes end, and GAE (``ctf_gae_dones``) stops at every episode boundary.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _native
from .fused_policy import FusedPolicy
from .policy import CtfPolicy
from .rollout import Rollout, _team_indices, collect_rollout


# ---------------------------------------------------------------------------------------------------- advantages
@torch.no_grad()
def reference_advantages(rewards: torch.Tensor, values: torch.Tensor, next_value: torch.Tensor, gamma: float,
                         lam: float, dones: torch.Tensor | None = None):
    """What ``ctf_gae`` (``ctf_gae_dones`` with ``dones``) computes, in eager torch: (advantages, returns), fp32
    [T*apt, B].

    ``rewards`` / ``values`` fp32 [T*apt, B] (row t*apt + j = trained agent j at step t), ``next_value`` fp32 [apt, B].
    Each (agent, env) column is one sequence over t; one rounding per operation, in the kernel's order, with the
    Python scalars ``gamma`` and ``gamma * lam``.  ``dones`` fp32 [T*apt, B]: a nonzero ``dones[t*apt + j, b]`` means
    observation t starts a new episode (CleanRL's convention), so below row t the bootstrap and the running advantage
    are both exactly 0.  ``dones=None`` or all zeros give the same bits."""
    apt, B = next_value.shape
    T = rewards.shape[0] // apt
    r, v = rewards.reshape(T, apt, B), values.reshape(T, apt, B)
    start = None if dones is None else dones.reshape(T, apt, B) != 0
    adv = torch.empty_like(r)
    gl = gamma * lam
    nv, last = next_value, torch.zeros_like(next_value)
    for t in reversed(range(T)):
        delta = r[t] + gamma * nv - v[t]
        last = delta + gl * last
        adv[t] = last
        nv = v[t]
        if start is not None:
            nv = torch.where(start[t], 0.0, nv)
            last = torch.where(start[t], 0.0, last)
    return adv.reshape(T * apt, B), (adv + v).reshape(T * apt, B)


def advantages(env, rollout: Rollout, next_value: torch.Tensor, gamma: float, lam: float,
               dones: torch.Tensor | None = None):
    """(advantages, returns) fp32 [T*apt, B] of ``rollout`` with the bootstrap ``next_value`` [apt, B], from one
    ``ctf_gae`` launch on the current stream, or one ``ctf_gae_dones`` launch when ``dones`` [T*apt, B] is given (a
    rollout that crosses episode boundaries); bit for bit ``reference_advantages``."""
    rew, val = rollout.rewards, rollout.values
    if next_value.dim() != 2 or next_value.shape[1] != rew.shape[1] or rew.shape[0] % next_value.shape[0]:
        raise ValueError(f"next_value must be [apt, B] with B = {rew.shape[1]} and apt dividing {rew.shape[0]}")
    if dones is not None and dones.shape != rew.shape:
        raise ValueError(f"dones must have the rewards' shape {tuple(rew.shape)}")
    for name, x in (("rewards", rew), ("values", val), ("next_value", next_value), ("dones", dones)):
        if x is not None and (x.dtype != torch.float32 or x.device != env.device):
            raise ValueError(f"{name} must be a float32 tensor on {env.device}")
    rew, val, nv = rew.contiguous(), val.contiguous(), next_value.contiguous()
    adv, ret = torch.empty_like(rew), torch.empty_like(rew)
    apt, B = nv.shape
    ptr = lambda x: C.c_void_p(x.data_ptr())
    sizes = (rew.shape[0] // apt, apt, B, float(gamma), float(gamma * lam),
             C.c_void_p(torch.cuda.current_stream(env.device).cuda_stream))
    if dones is None:
        rc = env._lib.ctf_gae(env._handle, ptr(rew), ptr(val), ptr(nv), ptr(adv), ptr(ret), *sizes)
    else:
        d = dones.contiguous()
        rc = env._lib.ctf_gae_dones(env._handle, ptr(rew), ptr(val), ptr(d), ptr(nv), ptr(adv), ptr(ret), *sizes)
    _native.check(rc)
    return adv, ret


# ---------------------------------------------------------------------------------------------------- loss
def ppo_loss(new_logprob, entropy, new_value, old_logprob, old_value, adv, ret, args, adv_stats=None):
    """The clipped PPO loss (CleanRL's, whose names the reference's arguments follow) as the mean over the samples
    given: ``pg_loss - ent_coef * entropy + vf_coef * v_loss``.

    With ``args.norm_adv`` the advantages are normalised by ``adv_stats`` = (mean, std) when given (a chunk of a
    minibatch uses the whole minibatch's), else by their own mean and std; ``std`` is torch's unbiased one, + 1e-8.
    With ``args.clip_vloss`` the value loss is the larger of the unclipped and the clipped squared error.
    Returns (loss, stats): stats holds the detached means ``pg_loss``, ``v_loss``, ``entropy``, ``approx_kl``
    ((ratio - 1) - log ratio) and ``clipfrac`` (|ratio - 1| > clip_coef) as 0-d tensors."""
    clip = args.clip_coef
    logratio = new_logprob - old_logprob
    ratio = logratio.exp()
    if args.norm_adv:
        mean, std = adv_stats if adv_stats is not None else (adv.mean(), adv.std())
        adv = (adv - mean) / (std + 1e-8)
    pg_loss = torch.max(-adv * ratio, -adv * torch.clamp(ratio, 1 - clip, 1 + clip)).mean()
    new_value = new_value.reshape(-1)
    if args.clip_vloss:
        v_unclipped = (new_value - ret) ** 2
        v_clipped = old_value + torch.clamp(new_value - old_value, -clip, clip)
        v_loss = 0.5 * torch.max(v_unclipped, (v_clipped - ret) ** 2).mean()
    else:
        v_loss = 0.5 * ((new_value - ret) ** 2).mean()
    ent = entropy.mean()
    loss = pg_loss - args.ent_coef * ent + args.vf_coef * v_loss
    with torch.no_grad():
        stats = dict(pg_loss=pg_loss.detach(), v_loss=v_loss.detach(), entropy=ent.detach(),
                     approx_kl=((ratio - 1) - logratio).mean(), clipfrac=((ratio - 1).abs() > clip).float().mean())
    return loss, stats


def minibatches(perm: torch.Tensor, num_minibatches: int):
    """The minibatches of one epoch: consecutive slices of ``perm`` of ``len(perm) // num_minibatches`` samples (at
    least one), the last one shorter when that size does not divide the batch.  Every sample is in exactly one."""
    n = perm.numel()
    size = max(n // num_minibatches, 1)
    return [perm[s : s + size] for s in range(0, n, size)]


# ---------------------------------------------------------------------------------------------------- trainer
class PackedPPO:
    """PPO for one ``CtfPolicy`` on a packed-observation env: ``update(opponent)`` = ``collect`` -> ``advantages``
    -> ``optimise`` (see the module docstring).

    ``env`` must be created with ``packed_obs=True`` and ``reverse_team1_actions=True``; a packed-only env
    (``dense_obs=False``) saves its dense observation writes.  ``agent`` is a ``CtfPolicy`` (load a reference ``Agent``
    into one with ``load_state_dict``); ``self.fused`` is its ``FusedPolicy``, which collects the rollouts and computes
    the training forward and backward.  ``chunk`` bounds the samples of one forward / backward: each holds about
    2 x stride bf16 values between them (15.6 KB at 8_arena).

    ``rollout_steps=None`` collects one fresh episode of every env per update.  An int T in 1..GAME_STEPS selects
    continuing mode: every ``collect`` runs T steps, the first one from ``env.reset()`` and every later one from where
    the env is (``collect_rollout(reset=False)``), resetting the env when its episodes end; GAE then stops at each
    episode boundary.  The opponent may change between updates; ``train_team1`` may change only between episodes
    (ValueError while one is in progress).  The env belongs to the trainer in this mode: stepping or resetting it
    elsewhere breaks the episodes the trainer continues."""

    def __init__(self, env, agent, args, optimizer=None, chunk=262144, rollout_steps=None):
        if env.obs_bits is None:
            raise ValueError("PackedPPO trains from packed observations: create the env with packed_obs=True")
        if not env.ce.cfg.reverse_team1_actions:
            raise ValueError("create the env with reverse_team1_actions=True: team-1 policies act in the flipped frame")
        if not isinstance(agent, CtfPolicy):
            raise ValueError("agent must be a CtfPolicy (load a reference Agent into one with load_state_dict)")
        if not getattr(args, "gae", True):
            raise ValueError("PackedPPO estimates advantages with GAE only: args.gae must be True")
        if int(chunk) < 1:
            raise ValueError("chunk must be >= 1")
        if rollout_steps is not None and not 1 <= int(rollout_steps) <= env.GAME_STEPS:
            raise ValueError(f"rollout_steps must be None or in 1..GAME_STEPS ({env.GAME_STEPS})")
        self.rollout_steps = None if rollout_steps is None else int(rollout_steps)
        self.env, self.agent, self.args, self.chunk = env, agent, args, int(chunk)
        self.fused = FusedPolicy(env, agent)
        self.optimizer = optimizer if optimizer is not None else torch.optim.Adam(
            agent.parameters(), lr=args.learning_rate, eps=1e-5)
        self.rollout = None
        self._train_team1 = None     # continuing mode: the team of the episode in progress (None before the first collect)
        self._running_return = None  # continuing mode: fp32 [apt, B] return of every trained (agent, env) so far

    def collect(self, opponent, train_team1=True, num_env_steps=None) -> Rollout:
        """One packed rollout of every env (``collect_rollout``) with the trained agent's ``FusedPolicy`` against
        ``opponent`` (a ``FusedPolicy``, or a ``CtfPolicy`` run through one), and its bootstrap ``next_value`` [apt, B]:
        0 when the rollout reached ``GAME_STEPS`` (every env ended), else the trained agents' V(s_T) from
        ``forward_from_env``.  The previous rollout is released first, so one rollout is alive at a time (as long as
        the caller keeps no reference to the old one).

        In continuing mode ``num_env_steps`` defaults to ``rollout_steps``, the rollout continues the env's episodes
        (its ``dones`` mark where new ones start), the bootstrap is 0 exactly where the last step ended the episode,
        and ``rollout.episode_stats`` holds the device tensors that ``optimise`` reports (see there)."""
        env = self.env
        continuing = self.rollout_steps is not None
        T = (self.rollout_steps if continuing else env.GAME_STEPS) if num_env_steps is None else int(num_env_steps)
        if not 1 <= T <= env.GAME_STEPS:
            raise ValueError(f"num_env_steps must be in 1..GAME_STEPS ({env.GAME_STEPS})"
                             + ("" if continuing else ": envs may not end inside a rollout"))
        train_team1 = bool(train_team1)
        if continuing and self._train_team1 is not None and train_team1 != self._train_team1:
            step = int(env.step_counts()[0])
            if 0 < step < env.GAME_STEPS:
                raise ValueError(f"train_team1 may change only between episodes: the envs are at step {step} of "
                                 f"{env.GAME_STEPS}")
        if not isinstance(opponent, FusedPolicy):
            opponent = FusedPolicy(env, opponent)
        self.rollout = None
        if continuing and self._train_team1 is None:
            # the first episode starts here; collecting with reset=False records its end wherever it falls, even on
            # the last step of this rollout
            env.reset()
            self._running_return = None
        ro = collect_rollout(env, self.fused, opponent, train_team1=train_team1, num_env_steps=T,
                             obs_storage_dtype="packed", reset=not continuing)
        mine = _team_indices(env, 0 if train_team1 else 1)
        apt, B = len(mine), env.num_envs
        if continuing:
            v, _ = self.fused.forward_from_env(mine)          # env-major samples b*apt + j
            ro.next_value = torch.where(ro.next_done.bool().unsqueeze(0), 0.0, v.reshape(B, apt).t()).contiguous()
            ro.episode_stats = self._episode_stats(ro, train_team1)
            self._train_team1 = train_team1
        elif T == env.GAME_STEPS:
            ro.next_value = torch.zeros((apt, B), device=env.device)
        else:
            v, _ = self.fused.forward_from_env(mine)          # env-major samples b*apt + j
            ro.next_value = v.reshape(B, apt).t().contiguous()
        self.rollout = ro
        return ro

    def _episode_stats(self, ro: Rollout, train_team1: bool) -> dict:
        """Device tensors of the episodes that ended in ``ro``, with the return of every trained (agent, env) carried
        from rollout to rollout in ``self._running_return`` (an episode spans several rollouts)."""
        apt, B = ro.next_value.shape
        r = ro.rewards.reshape(-1, apt, B)
        run = self._running_return
        if run is None or run.shape != (apt, B):   # the first rollout, or a team switch at an episode boundary
            run = torch.zeros((apt, B), device=r.device)
        me = 0 if train_team1 else 1
        returns, outcomes, t0 = [], [], 0
        for t, caps in ro.episode_ends:
            returns.append(run + r[t0 : t + 1].sum(0))
            outcomes.append(torch.sign(caps[:, me] - caps[:, 1 - me]))
            run, t0 = torch.zeros_like(run), t + 1
        self._running_return = run + r[t0:].sum(0)
        nan = torch.tensor(float("nan"), device=r.device)
        res = torch.stack(outcomes) if outcomes else None
        return dict(episodes_completed=apt * B * len(returns),
                    episode_return=torch.stack(returns).mean() if returns else nan,
                    win_fraction=(res == 1).float().mean() if outcomes else nan,
                    draw_fraction=(res == 0).float().mean() if outcomes else nan)

    def advantages(self, rollout: Rollout):
        """(advantages, returns) fp32 [T*apt, B] of a rollout from ``collect``, with ``args.gamma`` / ``gae_lambda``:
        ``ctf_gae``, or in continuing mode ``ctf_gae_dones`` with the rollout's ``dones``."""
        dones = rollout.dones if self.rollout_steps is not None else None
        return advantages(self.env, rollout, rollout.next_value, self.args.gamma, self.args.gae_lambda, dones)

    def optimise(self, rollout: Rollout, adv: torch.Tensor, ret: torch.Tensor, generator=None) -> dict:
        """``update_epochs`` epochs over the rollout's T*apt*B samples, each a ``torch.randperm`` (drawn with
        ``generator`` when given) cut into ``minibatches``.  Per minibatch: normalise the advantages by the whole
        minibatch's mean and std (``norm_adv``), run it in chunks of ``chunk`` samples through
        ``FusedPolicy.evaluate_actions`` and ``ppo_loss``, each chunk's loss scaled by its share of the minibatch and
        back-propagated so the gradients accumulate, then ``clip_grad_norm_(max_grad_norm)`` and one optimiser step.
        Training stops after an epoch whose last minibatch's ``approx_kl`` exceeds ``target_kl`` (when not None).
        ``FusedPolicy.refresh()`` runs once at the end, so the next rollout sees the new weights.

        Returns floats: ``v_loss``, ``pg_loss``, ``entropy`` and ``approx_kl`` of the last minibatch, ``clipfrac``
        averaged over every minibatch, ``epochs_run``, and ``first_approx_kl`` / ``first_clipfrac`` of the first
        minibatch, taken before any step (the rollout's log-probs come from the bf16 inference head, the update's from
        the fp32 heads of ``train_head``, so these are not exactly 0).  A rollout collected in continuing mode adds
        ``episodes_completed`` (episodes ended inside it, counted per trained (agent, env)), ``episode_return`` (the
        mean return of those episodes, including the rewards of earlier rollouts) and ``win_fraction`` /
        ``draw_fraction`` of the trained team over those episodes' envs (from ``env.flag_captures()`` at the last
        step); the last three are NaN when no episode ended."""
        args, env, fp = self.args, self.env, self.fused
        dev = env.device
        bits = rollout.grid_states.reshape(-1, env.bits_words_per_agent)
        meta = rollout.metadata_states.reshape(-1, env.meta_size)
        act = rollout.actions.reshape(-1).long()
        mask, old_lp, old_v = (x.reshape(-1) for x in (rollout.use_action_mask, rollout.logprobs, rollout.values))
        adv, ret = adv.reshape(-1), ret.reshape(-1)
        n = bits.shape[0]
        params = list(self.agent.parameters())
        clipfracs, first, out = [], None, {}
        epochs_run = 0
        for _ in range(args.update_epochs):
            perm = torch.randperm(n, device=dev, generator=generator)
            for idx in minibatches(perm, args.num_minibatches):
                m = idx.numel()
                adv_stats = (adv[idx].mean(), adv[idx].std()) if args.norm_adv else None
                self.optimizer.zero_grad()
                acc = None
                for c0 in range(0, m, self.chunk):
                    ci = idx[c0 : c0 + self.chunk]
                    share = ci.numel() / m
                    lp, ent, v = fp.evaluate_actions(bits[ci], meta[ci], mask[ci], act[ci])
                    loss, st = ppo_loss(lp, ent, v, old_lp[ci], old_v[ci], adv[ci], ret[ci], args, adv_stats)
                    (loss * share).backward()
                    acc = {k: x * share for k, x in st.items()} if acc is None else \
                        {k: acc[k] + x * share for k, x in st.items()}
                torch.nn.utils.clip_grad_norm_(params, args.max_grad_norm)
                self.optimizer.step()
                out = {k: float(x) for k, x in acc.items()}
                clipfracs.append(out["clipfrac"])
                if first is None:
                    first = out
            epochs_run += 1
            if args.target_kl is not None and out["approx_kl"] > args.target_kl:
                break
        fp.refresh()
        res = dict(v_loss=out["v_loss"], pg_loss=out["pg_loss"], entropy=out["entropy"], approx_kl=out["approx_kl"],
                   clipfrac=sum(clipfracs) / len(clipfracs), epochs_run=epochs_run,
                   first_approx_kl=first["approx_kl"], first_clipfrac=first["clipfrac"])
        stats = getattr(rollout, "episode_stats", None)
        if stats is not None:
            res.update({k: x if isinstance(x, int) else float(x) for k, x in stats.items()})
        return res

    def update(self, opponent, train_team1=True) -> dict:
        """One PPO update: ``collect`` (one episode of every env, or ``rollout_steps`` steps in continuing mode) ->
        ``advantages`` -> ``optimise``."""
        ro = self.collect(opponent, train_team1)
        adv, ret = self.advantages(ro)
        return self.optimise(ro, adv, ret)
