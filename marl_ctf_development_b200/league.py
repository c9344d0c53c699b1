"""Duel batches for league evaluation on GPU envs (SURVEY.md §8f row N3).

The reference evaluates a league by submitting ``number_of_duels`` Ray tasks per (agent, opponent) pair, each a
full ``utils.duel`` on a pickled env copy (league_training.py:368-459, 573-648).  Here every duel is one env of a
batch: pair p owns the envs [p*D, (p+1)*D) and all pairs advance with one step-kernel launch per step.  By default the
policy forwards are per pair; with ``grouped=True`` one ``PolicyPool`` runs every policy of every pair per step (one
grouped trunk launch and one batched head, whatever the number of pairs).  Results come back in the reference's formats:

* ``winrate_matrix_symmetric / non_symmetric``  ==  ``LeagueTrainer.calculate_winrate_matrix_*`` (:368-400, :427-455)
* ``generate_metrics_symmetric / non_symmetric`` ==  ``LeagueTrainer.generate_metrics_*`` (:573-648): every duel's
  ``env.metrics`` dict goes to ``MetricsLogger.harvest_metrics`` (metrics_logger.py:137-159) in the reference's
  order, with the reference's labels and scaling factors — pass the reference's own ``MetricsLogger``.
"""
from __future__ import annotations

from collections import defaultdict

import torch

from .env import GridworldCtfGPU, metrics_dict
from .fused_policy import FusedPolicy, PolicyPool
from .policy import CtfPolicy
from .rollout import batched_action


def pool_segments(pairs, duels_per_pair: int, team_ids):
    """(policies, segments) of a ``PolicyPool`` that plays ``pairs`` as ``duel_pairs`` lays them out: the distinct
    ``CtfPolicy`` modules (a ``FusedPolicy`` stands for its ``policy``, so a module and its views count once) by
    identity, in order of first appearance, and one segment (policy index, envs of the pair, team ids) per (pair, team)
    with agents, pair p owning the envs [p*D, (p+1)*D)."""
    D = int(duels_per_pair)
    uniq, index = [], {}

    def module(pol):
        return pol.policy if isinstance(pol, FusedPolicy) else pol

    for pair in pairs:
        for pol in pair:
            m = module(pol)
            if id(m) not in index:
                index[id(m)] = len(uniq)
                uniq.append(m)
    segments = [(index[id(module(pol))], slice(p * D, (p + 1) * D), tuple(ids))
                for p, pair in enumerate(pairs) for ids, pol in zip(team_ids, pair) if ids]
    return uniq, segments


@torch.no_grad()
def duel_pairs(env_config: dict, pairs, duels_per_pair: int, max_steps: int = 256, device=None, seed: int = 0,
               env_id_base: int = 0, collect_metrics: bool = False, per_duel_metrics: bool = False,
               grouped: bool = False):
    """Plays ``duels_per_pair`` duels (utils.py:500-573) for every (agent, opponent) in ``pairs`` at once.

    Returns (results [P, D] int64 of +1/0/-1 from team 0's view, metrics).  metrics is None unless collect_metrics;
    then a list of P ``env.metrics``-style dicts summed over the pair's duels, or with per_duel_metrics a list of P
    lists of D dicts — one per duel, what ``utils.duel(return_result=False)`` returns (utils.py:571).

    ``fused_policy.FusedPolicy`` policies read the env's packed observations in place; when every policy is one, the
    env is created packed-only and never writes dense observations.

    ``grouped=True``: every policy must be a ``FusedPolicy`` or a ``CtfPolicy``; the distinct modules go into
    one ``fused_policy.PolicyPool`` on a packed-only env, with one plan segment per (pair, team), and each step is
    ``pool.act`` followed by ``env.step``.  The results and metrics have the same structure as the per-pair path's;
    the draws differ (one ``Categorical`` over all rows consumes torch's random stream differently).
    """
    P, D = len(pairs), int(duels_per_pair)
    if grouped:
        if any(not isinstance(pol, (FusedPolicy, CtfPolicy)) for pair in pairs for pol in pair):
            raise ValueError("grouped=True needs every policy to be a FusedPolicy or a CtfPolicy")
        packed_kw = dict(packed_obs=True, dense_obs=False)
    else:
        fused = [isinstance(pol, FusedPolicy) for pair in pairs for pol in pair]
        packed_kw = {} if not any(fused) else dict(packed_obs=True, dense_obs=not all(fused))
    env = GridworldCtfGPU(**env_config, num_envs=P * D, device=device, seed=seed, env_id_base=env_id_base,
                          reverse_team1_actions=True, stats="counters" if collect_metrics else "none", **packed_kw)
    B, N, dev = env.num_envs, env.N_AGENTS, env.device
    C, G, M = env.n_channels, env.GRID_SIZE, env.meta_size
    team_ids = [[i for i in range(N) if env.AGENT_TEAMS[i] == t] for t in (0, 1)]
    teams = [torch.tensor(ids, device=dev) for ids in team_ids]
    if grouped:
        uniq, segments = pool_segments(pairs, D, team_ids)
        pool = PolicyPool(env, uniq)
        plan = pool.plan(segments)
    obs, meta, _ = env.reset()
    actions = torch.empty((B, N), dtype=torch.uint8, device=dev)
    step_count = 0
    while True:
        step_count += 1
        if grouped:
            pool.act(plan, actions)
        else:
            for p, pair in enumerate(pairs):
                sl = slice(p * D, (p + 1) * D)
                for idx, ids, pol in zip(teams, team_ids, pair):
                    k = idx.numel()
                    if k == 0:
                        continue
                    flags = env.use_action_mask[idx].unsqueeze(0).expand(D, k).reshape(D * k)
                    if isinstance(pol, FusedPolicy):
                        a = pol.get_action_and_value(flags, agent_ids=ids, env=env, envs=sl)[0]
                    else:
                        a = batched_action(pol, obs[sl][:, idx].reshape(D * k, C, G, G).float(),
                                           meta[sl][:, idx].reshape(D * k, M), flags)
                    actions[sl, idx] = a.reshape(D, k).to(torch.uint8)
        obs, meta, _, _, _ = env.step(actions)
        if step_count > max_steps or step_count >= env.GAME_STEPS:
            break
    caps = env.flag_captures()
    results = torch.sign(caps[:, 0] - caps[:, 1]).reshape(P, D)
    metrics = None
    if collect_metrics:
        c = env.counters()
        per_env = c.reshape(P, D, *c.shape[1:]).cpu().numpy()
        if per_duel_metrics:
            metrics = [[metrics_dict(env.ce, per_env[p, d]) for d in range(D)] for p in range(P)]
        else:
            metrics = [metrics_dict(env.ce, per_env[p].sum(0)) for p in range(P)]
    env.close()
    return results, metrics


def _matrices(results, labels, number_of_duels):
    winrate, draw = defaultdict(int), defaultdict(int)
    res = results.cpu()
    for p, (a_label, o_label) in enumerate(labels):
        for d in range(number_of_duels):
            r = int(res[p, d])
            winrate[(a_label, o_label)] += (r == 1) / number_of_duels   # league_training.py:391-392 / :446-447
            draw[(a_label, o_label)] += (r == 0) / number_of_duels
    for a_label, o_label in list(winrate.keys()):                        # :395-397 / :450-452
        winrate[(o_label, a_label)] = 1 - winrate[(a_label, o_label)] - draw[(a_label, o_label)]
    return winrate, draw


def winrate_matrix_non_symmetric(env_config, agents_t1, agents_t2, number_of_duels, **kw):
    """league_training.py:427-455: every team-1 agent against every team-2 agent; keys ('0_i', '1_j') and inverses."""
    pairs, labels = [], []
    for i, agent in enumerate(agents_t1):
        for j, opponent in enumerate(agents_t2):
            pairs.append((agent, opponent))
            labels.append((f"0_{i}", f"1_{j}"))
    results, _ = duel_pairs(env_config, pairs, number_of_duels, **kw)
    return _matrices(results, labels, number_of_duels)[0]


def winrate_matrix_symmetric(env_config, agents, number_of_duels, **kw):
    """league_training.py:368-400: pairs with agent_idx > opponent_idx; keys ('0_i', '0_j') and inverses."""
    pairs, labels = [], []
    for i, agent in enumerate(agents):
        for j, opponent in enumerate(agents):
            if i > j:
                pairs.append((agent, opponent))
                labels.append((f"0_{i}", f"0_{j}"))
    if not pairs:
        return defaultdict(int)
    results, _ = duel_pairs(env_config, pairs, number_of_duels, **kw)
    return _matrices(results, labels, number_of_duels)[0]


def _league_labels(prefix, n_main, n_coaching, n_league, n_historical=None):
    labels = [f"{prefix}m{i}" for i in range(n_main)] + [f"{prefix}c{i}" for i in range(n_coaching)] \
        + [f"{prefix}l{i}" for i in range(n_league)]
    if n_historical is not None:
        labels += [f"{prefix}h{i}" for i in range(n_historical)]
    return labels


def generate_metrics_symmetric(metlog, env_config, all_agents_t1, n_historical_t1, number_of_duels, iteration,
                               n_main_agents, n_coaching_agents, n_league_agents, **kw):
    """``LeagueTrainer.generate_metrics_symmetric`` (league_training.py:573-603) on one env batch.

    all_agents_t1 = main + coaching + league + historical agents (:405-408); the historical tail is not evaluated
    (:581).  Every duel's metrics are harvested under the agent's label 'm0', 'c0', 'l0', … with the reference's
    scaling factor 1 / (len(all_agents_t1) - 1 + number_of_duels) (:582), in the reference's task order.
    Returns the number of duels played (the reference prints it, :602).
    """
    labels = _league_labels("", n_main_agents, n_coaching_agents, n_league_agents)
    keep = len(all_agents_t1) - n_historical_t1
    scale = 1 / (len(all_agents_t1) - 1 + number_of_duels)
    agents = list(all_agents_t1[:keep])
    pairs = [(a, o) for a in agents for o in agents]
    _, metrics = duel_pairs(env_config, pairs, number_of_duels, collect_metrics=True, per_duel_metrics=True, **kw)
    p = 0
    for agent_idx in range(len(agents)):
        for _opponent_idx in range(len(agents)):
            for d in range(number_of_duels):
                metlog.harvest_metrics(metrics[p][d], labels[agent_idx], iteration, scale)
            p += 1
    return len(pairs) * number_of_duels


def generate_metrics_non_symmetric(metlog, env_config, all_agents_t1, all_agents_t2, n_historical_t1, n_historical_t2,
                                   number_of_duels, iteration, n_main_agents, n_coaching_agents, n_league_agents, **kw):
    """``LeagueTrainer.generate_metrics_non_symmetric`` (league_training.py:605-648) on one env batch.

    Each duel is harvested twice: for the team-0 agent's label ('t0_m0', …) with team_idx=0 and scaling factor
    1 / (len(all_agents_t2) - 1 + number_of_duels), and for the team-1 agent's label with team_idx=1 and
    1 / (len(all_agents_t1) - 1 + number_of_duels) (:621-622, :643-646).  The reference sizes BOTH label lists'
    historical part by ``historical_agents_t1`` (:613, :618) — kept.
    """
    labels_t1 = _league_labels("t0_", n_main_agents, n_coaching_agents, n_league_agents, n_historical_t1)
    labels_t2 = _league_labels("t1_", n_main_agents, n_coaching_agents, n_league_agents, n_historical_t1)
    keep_t1 = len(all_agents_t1) - n_historical_t1
    keep_t2 = len(all_agents_t2) - n_historical_t2
    scale_t1 = 1 / (len(all_agents_t2) - 1 + number_of_duels)
    scale_t2 = 1 / (len(all_agents_t1) - 1 + number_of_duels)
    t1, t2 = list(all_agents_t1[:keep_t1]), list(all_agents_t2[:keep_t2])
    pairs = [(a, o) for a in t1 for o in t2]
    _, metrics = duel_pairs(env_config, pairs, number_of_duels, collect_metrics=True, per_duel_metrics=True, **kw)
    p = 0
    for agent_idx in range(len(t1)):
        for opponent_idx in range(len(t2)):
            for d in range(number_of_duels):
                metlog.harvest_metrics(metrics[p][d], labels_t1[agent_idx], iteration, scale_t1, team_idx=0)
                metlog.harvest_metrics(metrics[p][d], labels_t2[opponent_idx], iteration, scale_t2, team_idx=1)
            p += 1
    return len(pairs) * number_of_duels
