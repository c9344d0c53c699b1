#!/usr/bin/env python
"""Seeded action sampling (ctf_sample_actions) against torch's sampling glue.

    python tools/policy_sample_bench.py [--envs 65536] [--reps 50] [--steps 20] [--rounds 3] [--out FILE]

Setup: 8_arena, B = --envs envs, one team's 4 agents per policy call (S = 4 B rows; 262 144 at B = 65 536), random
CtfPolicy weights.  Three measurements, each alternating its two paths --rounds times in this one process, with CUDA
events, median over rounds reported:
  sample    the sampling of one team's head output [S, 10] (computed once): torch path = ``CtfPolicy.masked_logits`` +
            ``Categorical`` sample / ``log_prob`` / ``entropy`` + ``index_copy_`` into the env's action buffer; seeded
            path = the mask flags (``use_action_mask == 1``) + one ``ctf_sample_actions``.  ms per call, --reps calls;
  selfplay  the fused self-play step of ``rollout.batched_duel``: both teams' ``FusedPolicy.get_action_and_value``
            (trunk + head + sampling) + the action scatter + ``env.step``, unseeded against ``policy_seed``; ms per
            step over --steps steps from a fresh reset;
  league    the per-pair league step of ``league.duel_pairs`` at L = 8 policies, D = 32 duels per pair (64 pairs,
            2 048 envs, 128 policy calls per step, host-bound), unseeded against ``policy_seed``; ms per step.
The card's name, power limit and max SM clock are read with nvidia-smi in the same run.  Prints text lines (also
written to --out) and one final JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402
from torch.distributions.categorical import Categorical  # noqa: E402

from marl_ctf_development_b200 import GridworldCtfGPU, experiment_env_config  # noqa: E402
from marl_ctf_development_b200.fused_policy import FusedPolicy, sample_actions  # noqa: E402
from marl_ctf_development_b200.policy import CtfPolicy  # noqa: E402

DEV = "cuda:0"
SEED = 12345


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else f"nvidia-smi failed: {q.stderr.strip()}"


def timed(fn, n):
    """ms per call of fn over n calls, CUDA events around them."""
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(n):
        fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) / n


def make_env(ec, B):
    return GridworldCtfGPU(**ec, num_envs=B, device=DEV, seed=3, reverse_team1_actions=True, packed_obs=True,
                           dense_obs=False)


def policy(env, seed):
    torch.manual_seed(seed)
    return CtfPolicy(9, env.n_channels, env.GRID_SIZE, env.meta_size).to(DEV).eval()


def teams(env):
    return [[i for i in range(env.N_AGENTS) if env.AGENT_TEAMS[i] == t] for t in (0, 1)]


def bench_sample(ec, B, reps, rounds):
    env = make_env(ec, B)
    pol = policy(env, 1)
    fp = FusedPolicy(env, pol)
    ids = teams(env)[0]
    k = len(ids)
    flags = env.use_action_mask[ids].repeat(B)
    with torch.no_grad():
        out = fp._head_out(fp.trunk_from_env(ids))
        logits = out[:, 1:]
    flat = fp._flat_index(ids, env, None)
    actions = torch.zeros((B, env.N_AGENTS), dtype=torch.uint8, device=DEV)

    @torch.no_grad()
    def torch_path():
        probs = Categorical(logits=pol.masked_logits(logits, flags), validate_args=False)
        a = probs.sample()
        probs.log_prob(a), probs.entropy()
        actions.view(-1).index_copy_(0, flat, a.to(torch.uint8))

    def seeded_path():
        sample_actions(env, out, (flags == 1).to(torch.uint8), flat, SEED, actions)

    res = {"torch": [], "seeded": []}
    for fn in (torch_path, seeded_path):
        timed(fn, 5)
    for _ in range(rounds):
        res["torch"].append(timed(torch_path, reps))
        res["seeded"].append(timed(seeded_path, reps))
    return res, B * k


def bench_selfplay(ec, B, steps, rounds):
    env = make_env(ec, B)
    fps = [FusedPolicy(env, policy(env, 1)), FusedPolicy(env, policy(env, 2))]
    tids = teams(env)
    idx = [torch.tensor(t, device=DEV) for t in tids]
    flags = [env.use_action_mask[t].repeat(B) for t in tids]
    actions = torch.zeros((B, env.N_AGENTS), dtype=torch.uint8, device=DEV)

    def step(seed):
        for fp, ids, ix, f in zip(fps, tids, idx, flags):
            if seed is None:        # batched_duel's unseeded body
                a = fp.get_action_and_value(f, agent_ids=ids, env=env)[0]
                actions[:, ix] = a.reshape(B, len(ids)).to(torch.uint8)
            else:
                fp.get_action_and_value(f, agent_ids=ids, env=env, seed=seed, actions=actions)
        env.step(actions)

    res = {"torch": [], "seeded": []}
    for _ in range(rounds + 1):   # the first round warms both paths up
        for name, seed in (("torch", None), ("seeded", SEED)):
            env.reset()
            step(seed)
            ms = timed(lambda: step(seed), steps)
            res[name].append(ms)
    return {k: v[1:] for k, v in res.items()}


def bench_league(ec, L, D, steps, rounds):
    probe = make_env(ec, 1)
    fps = [FusedPolicy(probe, policy(probe, 10 + i)) for i in range(L)]
    pairs = [(a, o) for a in fps for o in fps]
    env = make_env(ec, len(pairs) * D)
    tids = teams(env)
    idx = [torch.tensor(t, device=DEV) for t in tids]
    flags = [env.use_action_mask[t].repeat(D) for t in tids]
    actions = torch.zeros((env.num_envs, env.N_AGENTS), dtype=torch.uint8, device=DEV)

    def step(seed):   # duel_pairs' per-pair step body
        for p, pair in enumerate(pairs):
            sl = slice(p * D, (p + 1) * D)
            for ids, ix, f, pol in zip(tids, idx, flags, pair):
                if seed is None:
                    a = pol.get_action_and_value(f, agent_ids=ids, env=env, envs=sl)[0]
                    actions[sl, ix] = a.reshape(D, len(ids)).to(torch.uint8)
                else:
                    pol.get_action_and_value(f, agent_ids=ids, env=env, envs=sl, seed=seed, actions=actions)
        env.step(actions)

    res = {"torch": [], "seeded": []}
    for _ in range(rounds + 1):
        for name, seed in (("torch", None), ("seeded", SEED)):
            env.reset()
            step(seed)
            res[name].append(timed(lambda: step(seed), steps))
    return {k: v[1:] for k, v in res.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("policy_sample_bench needs a CUDA device")
    ec = experiment_env_config("8_arena")
    lines = [f"gpu: {gpu_info()}", f"torch {torch.__version__}, 8_arena, B = {args.envs}"]
    result = {"gpu": gpu_info(), "envs": args.envs}

    def report(name, res, unit):
        med = {k: statistics.median(v) for k, v in res.items()}
        spread = {k: (min(v), max(v)) for k, v in res.items()}
        result[name] = {"median_ms": med, "all_ms": res}
        lines.append(f"{name}: torch {med['torch']:.4f} {unit} (range {spread['torch'][0]:.4f}-{spread['torch'][1]:.4f}), "
                     f"seeded {med['seeded']:.4f} {unit} (range {spread['seeded'][0]:.4f}-{spread['seeded'][1]:.4f}), "
                     f"seeded/torch {med['seeded'] / med['torch']:.3f}")
        print(lines[-1], flush=True)

    for line in lines:
        print(line, flush=True)
    res, S = bench_sample(ec, args.envs, args.reps, args.rounds)
    lines.append(f"sample: S = {S} rows per call")
    report("sample", res, "ms/call")
    report("selfplay", bench_selfplay(ec, args.envs, args.steps, args.rounds), "ms/step")
    report("league_per_pair_L8_D32", bench_league(ec, 8, 32, args.steps, args.rounds), "ms/step")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n" + json.dumps(result) + "\n")
    print(json.dumps(result))


if __name__ == "__main__":
    main()
