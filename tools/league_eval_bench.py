#!/usr/bin/env python
"""League evaluation cost: grouped PolicyPool inference against per-pair policy calls.

    python tools/league_eval_bench.py [--agents 4 8] [--duels 32 1024] [--steps 20] [--rounds 2] [--out FILE]

Setup: 8_arena, L policies with random CtfPolicy weights, the symmetric all-pairs evaluation of
``league.generate_metrics_symmetric`` (L^2 pairs, D duels each, L^2 * D envs).  Three paths:
  grouped   ``duel_pairs(grouped=True)``: one PolicyPool, per step one grouped trunk launch + one batched head;
  fused     ``duel_pairs`` with a FusedPolicy per agent: two policy calls per pair per step;
  stock     ``duel_pairs`` with the CtfPolicy modules on a dense env (fp32 cuDNN), at D <= 32 only.
ms per step: CUDA events around --steps steps of each path's own step body (its policy calls + env.step) after a
warm-up, the paths alternated --rounds times, median reported.  Wall seconds per evaluation: one whole ``duel_pairs``
call (257 steps, env creation and teardown included, host clock around a device synchronise) per path and round,
alternated.  Then one grouped trunk launch against the sum of the per-pair trunk launches
(``FusedPolicy.trunk_from_env`` per (pair, team)), CUDA events over 20 repetitions.  The card's name and power limit
are read with nvidia-smi in the same run.  Prints text lines (also written to --out) and one final JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

from marl_ctf_development_b200 import GridworldCtfGPU, experiment_env_config  # noqa: E402
from marl_ctf_development_b200 import league  # noqa: E402
from marl_ctf_development_b200.fused_policy import FusedPolicy, PolicyPool  # noqa: E402
from marl_ctf_development_b200.policy import CtfPolicy  # noqa: E402
from marl_ctf_development_b200.rollout import batched_action  # noqa: E402

DEV = "cuda:0"
STOCK_MAX_D = 32


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else f"nvidia-smi failed: {q.stderr.strip()}"


class Stepper:
    """One path's duel step on its own env: the policy calls of duel_pairs' step body, then env.step."""

    def __init__(self, path, ec, mods, D, seed=0):
        self.path = path
        L = len(mods)
        pols = [FusedPolicy(self._probe(ec), m) for m in mods] if path == "fused" else mods
        self.pairs = [(a, o) for a in pols for o in pols]
        kw = dict(packed_obs=True, dense_obs=False) if path != "stock" else {}
        self.env = GridworldCtfGPU(**ec, num_envs=L * L * D, device=DEV, seed=seed, reverse_team1_actions=True, **kw)
        env, self.D = self.env, D
        N = env.N_AGENTS
        self.team_ids = [[i for i in range(N) if env.AGENT_TEAMS[i] == t] for t in (0, 1)]
        self.teams = [torch.tensor(ids, device=DEV) for ids in self.team_ids]
        self.actions = torch.empty((env.num_envs, N), dtype=torch.uint8, device=DEV)
        if path == "grouped":
            uniq, segs = league.pool_segments(self.pairs, D, self.team_ids)
            self.pool = PolicyPool(env, uniq)
            self.plan = self.pool.plan(segs)
        env.reset()

    _probes = {}

    @classmethod
    def _probe(cls, ec):
        if "p" not in cls._probes:
            cls._probes["p"] = GridworldCtfGPU(**ec, num_envs=1, device=DEV, packed_obs=True, dense_obs=False)
        return cls._probes["p"]

    def policies(self):
        env, D, actions = self.env, self.D, self.actions
        if self.path == "grouped":
            self.pool.act(self.plan, actions)
            return
        Cn, G, M = env.n_channels, env.GRID_SIZE, env.meta_size
        for p, pair in enumerate(self.pairs):
            sl = slice(p * D, (p + 1) * D)
            for idx, ids, pol in zip(self.teams, self.team_ids, pair):
                k = len(ids)
                flags = env.use_action_mask[idx].unsqueeze(0).expand(D, k).reshape(D * k)
                if self.path == "fused":
                    a = pol.get_action_and_value(flags, agent_ids=ids, env=env, envs=sl)[0]
                else:
                    a = batched_action(pol, env.obs[sl][:, idx].reshape(D * k, Cn, G, G).float(),
                                       env.meta[sl][:, idx].reshape(D * k, M), flags)
                actions[sl, idx] = a.reshape(D, k).to(torch.uint8)

    @torch.no_grad()
    def step(self):
        self.policies()
        self.env.step(self.actions)

    def ms_per_step(self, steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            self.step()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    def close(self):
        self.env.close()


def events_ms(fn, iters):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def wall_eval(path, ec, mods, D):
    pols = mods if path != "fused" else [FusedPolicy(Stepper._probe(ec), m) for m in mods]
    pairs = [(a, o) for a in pols for o in pols]
    torch.cuda.synchronize()
    t = time.perf_counter()
    league.duel_pairs(ec, pairs, D, device=DEV, seed=1, grouped=path == "grouped")
    torch.cuda.synchronize()
    return time.perf_counter() - t


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--agents", type=int, nargs="+", default=[4, 8])
    ap.add_argument("--duels", type=int, nargs="+", default=[32, 1024])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("league_eval_bench measures the GPU: no CUDA device")
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    ec = experiment_env_config("8_arena")
    say(f"gpu: {gpu_info()}")
    say(f"8_arena, symmetric all-pairs evaluation (L^2 pairs x D duels), {args.steps} timed steps per path, "
        f"{args.rounds} alternated rounds, medians")
    results = []
    for L in args.agents:
        torch.manual_seed(L)
        probe = Stepper._probe(ec)
        mods = [CtfPolicy(9, probe.n_channels, probe.GRID_SIZE, probe.meta_size).to(DEV).eval() for _ in range(L)]
        for D in args.duels:
            paths = ["grouped", "fused"] + (["stock"] if D <= STOCK_MAX_D else [])
            steppers = {p: Stepper(p, ec, mods, D) for p in paths}
            for s in steppers.values():          # warm-up: cuBLAS / cuDNN handles, feature buffers
                for _ in range(3):
                    s.step()
            torch.cuda.synchronize()
            ms = {p: [] for p in paths}
            for _ in range(args.rounds):
                for p in paths:
                    ms[p].append(steppers[p].ms_per_step(args.steps))
            # trunk only: one grouped launch vs the per-pair launches of the fused path
            g, f = steppers["grouped"], steppers["fused"]
            trunk_grouped = events_ms(lambda: g.pool.trunk(g.plan), 20)

            def per_pair_trunks():
                n_launch = n_rows = 0
                for p, pair in enumerate(f.pairs):
                    for ids, pol in zip(f.team_ids, pair):
                        n_rows += pol.trunk_from_env(ids, env=f.env, envs=slice(p * D, (p + 1) * D)).shape[0]
                        n_launch += 1
                return n_launch, n_rows

            n_launch, n_rows = per_pair_trunks()
            # the per-pair launches cover exactly the grouped launch's samples
            assert n_launch == 2 * L * L and n_rows == g.plan.n_outputs == L * L * D * probe.N_AGENTS, (n_launch, n_rows)
            trunk_pairs = events_ms(per_pair_trunks, 20)
            for s in steppers.values():
                s.close()
            del steppers, g, f
            torch.cuda.empty_cache()
            wall = {p: [] for p in paths}
            for _ in range(args.rounds):
                for p in paths:
                    wall[p].append(wall_eval(p, ec, mods, D))
            row = dict(L=L, D=D, envs=L * L * D, samples_per_step=L * L * D * probe.N_AGENTS,
                       ms_per_step={p: statistics.median(v) for p, v in ms.items()},
                       ms_per_step_all={p: v for p, v in ms.items()},
                       s_per_eval={p: statistics.median(v) for p, v in wall.items()},
                       s_per_eval_all={p: v for p, v in wall.items()},
                       trunk_ms={"grouped_one_launch": trunk_grouped, "per_pair_sum": trunk_pairs})
            results.append(row)
            say(f"L={L} D={D} envs={row['envs']}: ms/step " +
                ", ".join(f"{p} {v:.3f}" for p, v in row["ms_per_step"].items()) +
                " | s/eval " + ", ".join(f"{p} {v:.2f}" for p, v in row["s_per_eval"].items()) +
                f" | trunk ms: grouped {trunk_grouped:.3f}, per-pair sum {trunk_pairs:.3f}" +
                f" | fused/grouped per step {row['ms_per_step']['fused'] / row['ms_per_step']['grouped']:.2f}x")
    summary = json.dumps(dict(gpu=gpu_info(), results=results))
    lines.append(summary)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")
    print(summary)


if __name__ == "__main__":
    main()
