#!/usr/bin/env python
"""Whole PPO updates with PackedPPO at BASELINE size, timed phase by phase.

    python tools/ppo_update_bench.py [--envs 65536] [--updates 2] [--rollout-steps none,125] [--gae-reps 20] [--out FILE]

Workload: 8_arena, packed-only env, B envs, 4 trained agents, 4 epochs x 4 minibatches, chunks of 262 144 samples,
Adam(2.5e-4, eps=1e-5), the reference's PPO hyper-parameters.  Each --rollout-steps entry is one trainer with its own
env and policies (same initial weights): "none" collects one fresh episode (T = GAME_STEPS = 500) per update, an int T
continues the episodes across updates of T steps (PackedPPO(rollout_steps=T)).  The trainers' updates alternate,
--updates times each (the first of each includes every allocation).  Per update:
  rollout   PackedPPO.collect (FusedPolicy on both sides) by host clock around a device synchronise;
  gae       PackedPPO.advantages (one ctf_gae or ctf_gae_dones launch), host clock with synchronise;
  optimise  PackedPPO.optimise, host clock with synchronise;
then the total, samples/s over the T * 4 * B samples of the update, the first-minibatch approx_kl / clipfrac (bf16
inference log-probs against the fp32 heads of the update), and two peaks of allocated memory:
  max_memory_allocated  torch.cuda.max_memory_allocated since the update began, which includes the persistent buffers
                        of every trainer of the run (FusedPolicy's feature buffers are about 2 GB per policy at
                        B = 65 536);
  own_peak              what this trainer alone would peak at: the memory it has kept allocated so far (its env,
                        policies and optimiser, and the buffers its earlier updates left allocated) plus the peak this
                        update adds above everything allocated when it began.  Allocations are attributed to the
                        trainer that was running when they were made.
Then ctf_gae and ctf_gae_dones run on the same seeded 500 x 4 x B inputs (dones: episode starts on rows 125, 250 and
375), alternated, timed with CUDA events (median of --gae-reps runs each) and compared with torch.equal against
ppo.reference_advantages; ctf_gae moves 16 B per element (rewards and values read, advantages and returns written),
ctf_gae_dones 20 B (dones read too).  The inputs (2.6 GB) are far larger than L2.  The card's name, power limit and max
SM clock are read with nvidia-smi in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

from marl_ctf_development_b200 import GridworldCtfGPU, PackedPPO, experiment_env_config  # noqa: E402
from marl_ctf_development_b200.fused_policy import FusedPolicy  # noqa: E402
from marl_ctf_development_b200.policy import CtfPolicy  # noqa: E402
from marl_ctf_development_b200.ppo import advantages, reference_advantages  # noqa: E402

DEV = "cuda:0"
COPY_PEAK_GBS = 6549.0   # measured device-to-device copy rate of one B200 (DESIGN §4)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else f"nvidia-smi failed: {q.stderr.strip()}"


def median_ms(fn, reps):
    out = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        out.append(e0.elapsed_time(e1))
    return statistics.median(out)


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--updates", type=int, default=2)
    ap.add_argument("--rollout-steps", default="none",
                    help="comma-separated trainers: none (one episode per update) or T (continuing rollouts of T steps)")
    ap.add_argument("--gae-reps", type=int, default=20)
    ap.add_argument("--chunk", type=int, default=262144)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    modes = [None if x.strip().lower() == "none" else int(x) for x in a.rollout_steps.split(",")]
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    gpu = gpu_info()
    say(f"gpu: {gpu}")
    ec = experiment_env_config("8_arena")
    args = types.SimpleNamespace(num_minibatches=4, update_epochs=4, gamma=0.99, gae_lambda=0.95, norm_adv=True,
                                 clip_coef=0.2, clip_vloss=True, ent_coef=0.01, vf_coef=0.5, max_grad_norm=0.5,
                                 target_kl=None, learning_rate=2.5e-4, gae=True)
    trainers, own = {}, {}    # own[m]: bytes trainer m keeps allocated between its updates
    for m in modes:
        torch.cuda.synchronize()
        before = torch.cuda.memory_allocated()
        env = GridworldCtfGPU(**ec, num_envs=a.envs, device=DEV, seed=1, reverse_team1_actions=True, dense_obs=False,
                              packed_obs=True)
        torch.manual_seed(0)
        mk = lambda: CtfPolicy(9, env.n_channels, env.GRID_SIZE, env.meta_size).to(DEV)
        agent, opp = mk(), mk()
        trainers[m] = (PackedPPO(env, agent, args, chunk=a.chunk, rollout_steps=m), FusedPolicy(env, opp))
        torch.cuda.synchronize()
        own[m] = torch.cuda.memory_allocated() - before
    apt, GS = 4, env.GAME_STEPS
    say(f"workload: 8_arena, B = {a.envs}, apt = {apt}, rollout_steps {['none' if m is None else m for m in modes]} "
        f"alternated, {args.update_epochs} epochs x {args.num_minibatches} minibatches, chunks of {a.chunk}")
    results = []
    for u in range(a.updates):
        for m in modes:
            tr, opponent = trainers[m]
            T = GS if m is None else m
            n = T * apt * a.envs
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats()
            base = torch.cuda.memory_allocated()
            ro, t_roll = timed(lambda: tr.collect(opponent))
            (adv, ret), t_gae = timed(lambda: tr.advantages(ro))
            out, t_opt = timed(lambda: tr.optimise(ro, adv, ret))
            total = t_roll + t_gae + t_opt
            peak_b = torch.cuda.max_memory_allocated()
            peak, own_peak = peak_b / 1e9, (own[m] + peak_b - base) / 1e9
            r = dict(rollout_steps=m, T=T, samples=n, rollout_s=t_roll, gae_s=t_gae, optimise_s=t_opt, total_s=total,
                     samples_per_s=n / total, optimise_us_per_sample=1e6 * t_opt / n, max_memory_allocated_gb=peak,
                     own_peak_gb=own_peak,
                     **out)
            results.append(r)
            tag = f"update {u}, rollout_steps {'none' if m is None else m} (T = {T}, {n} samples)"
            say(f"{tag}: rollout {t_roll:.2f} s, gae {t_gae * 1e3:.1f} ms, optimise {t_opt:.2f} s "
                f"({1e6 * t_opt / n:.4f} us/sample), total {total:.2f} s, {n / total:.3e} samples/s, "
                f"max_memory_allocated {peak:.1f} GB, own_peak {own_peak:.1f} GB")
            say(f"{tag}: first minibatch before any step: approx_kl {out['first_approx_kl']:.3e}, "
                f"clipfrac {out['first_clipfrac']:.3e}; last: v_loss {out['v_loss']:.4g}, pg_loss {out['pg_loss']:.4g}, "
                f"entropy {out['entropy']:.4g}, approx_kl {out['approx_kl']:.3e}, clipfrac {out['clipfrac']:.3e}"
                + (f"; episodes_completed {out['episodes_completed']}, episode_return {out['episode_return']:.4g}, "
                   f"win {out['win_fraction']:.3f}, draw {out['draw_fraction']:.3f}" if m is not None else ""))
            ro = adv = ret = tr.rollout = None    # nothing of this update stays allocated during the next one
            torch.cuda.synchronize()
            own[m] += torch.cuda.memory_allocated() - base
    del ro, adv, ret
    # ctf_gae against ctf_gae_dones on one 500-step shape
    T, B = GS, a.envs
    n = T * apt * B
    g = torch.Generator(device=DEV).manual_seed(0)
    rew, val = (torch.randn((T * apt, B), generator=g, device=DEV) for _ in range(2))
    nv = torch.randn((apt, B), generator=g, device=DEV)
    dones = torch.zeros_like(rew)
    for t in (125, 250, 375):
        dones[t * apt : (t + 1) * apt] = 1
    ro = types.SimpleNamespace(rewards=rew, values=val)
    env = trainers[modes[0]][0].env
    run = {"ctf_gae": lambda: advantages(env, ro, nv, args.gamma, args.gae_lambda),
           "ctf_gae_dones": lambda: advantages(env, ro, nv, args.gamma, args.gae_lambda, dones=dones)}
    equal = {}
    for name, d in (("ctf_gae", None), ("ctf_gae_dones", dones)):
        kern = run[name]()
        ref = reference_advantages(rew, val, nv, args.gamma, args.gae_lambda, dones=d)
        equal[name] = torch.equal(kern[0], ref[0]) and torch.equal(kern[1], ref[1])
        assert equal[name], f"{name} differs from reference_advantages"
        del kern, ref
    times = {k: [] for k in run}
    for _ in range(a.gae_reps):
        for k, fn in run.items():
            times[k].append(median_ms(fn, 1))
    ms = {k: statistics.median(v) for k, v in times.items()}
    gbs = {"ctf_gae": 16 * n / (ms["ctf_gae"] * 1e-3) / 1e9, "ctf_gae_dones": 20 * n / (ms["ctf_gae_dones"] * 1e-3) / 1e9}
    for k in run:
        say(f"{k}: {ms[k]:.3f} ms (median of {a.gae_reps}, alternated), {gbs[k]:.0f} GB/s at "
            f"{16 if k == 'ctf_gae' else 20} B per element = {100 * gbs[k] / COPY_PEAK_GBS:.1f} % of the "
            f"{COPY_PEAK_GBS:.0f} GB/s copy peak; torch.equal with reference_advantages: {equal[k]}")
    say(f"ctf_gae_dones / ctf_gae: {ms['ctf_gae_dones'] / ms['ctf_gae']:.3f}")
    res = dict(gpu=gpu, envs=a.envs, agents_per_step=apt, chunk=a.chunk, updates=results, gae_ms=ms["ctf_gae"],
               gae_dones_ms=ms["ctf_gae_dones"], gae_gbytes_per_s=gbs["ctf_gae"],
               gae_dones_gbytes_per_s=gbs["ctf_gae_dones"], gae_bit_equal=equal["ctf_gae"],
               gae_dones_bit_equal=equal["ctf_gae_dones"])
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n" + json.dumps(res) + "\n")


if __name__ == "__main__":
    main()
