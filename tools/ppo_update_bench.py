#!/usr/bin/env python
"""One whole PPO update with PackedPPO at BASELINE size, timed phase by phase.

    python tools/ppo_update_bench.py [--envs 65536] [--updates 2] [--gae-reps 20] [--out FILE]

Workload: 8_arena, packed-only env, B envs, one episode (T = GAME_STEPS = 500) per rollout, 4 trained agents, 4 epochs x
4 minibatches, chunks of 262 144 samples, Adam(2.5e-4, eps=1e-5), the reference's PPO hyper-parameters.  The update runs
--updates times (the first one includes every allocation).  Per update:
  rollout   PackedPPO.collect (FusedPolicy on both sides) by host clock around a device synchronise;
  gae       PackedPPO.advantages (one ctf_gae launch), host clock with synchronise;
  optimise  PackedPPO.optimise, host clock with synchronise;
then the total, samples/s over the T * 4 * B samples of the update, torch.cuda.max_memory_allocated and the
first-minibatch approx_kl / clipfrac (bf16 inference log-probs against the fp32 heads of the update).
On the last rollout, ctf_gae and ppo.reference_advantages are timed with CUDA events (median of --gae-reps runs
each) and compared with torch.equal; the kernel's rate counts 16 B per element (rewards and values read, advantages
and returns written).  The card's name, power limit and max SM clock are read with nvidia-smi in the same run.
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
PROJECTED_OPTIMISE_S = 46.0   # the per-chunk projection this run replaces (profiles/r04_policy_train.log)


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
    ap.add_argument("--gae-reps", type=int, default=20)
    ap.add_argument("--chunk", type=int, default=262144)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    gpu = gpu_info()
    say(f"gpu: {gpu}")
    ec = experiment_env_config("8_arena")
    env = GridworldCtfGPU(**ec, num_envs=a.envs, device=DEV, seed=1, reverse_team1_actions=True, dense_obs=False,
                          packed_obs=True)
    torch.manual_seed(0)
    mk = lambda: CtfPolicy(9, env.n_channels, env.GRID_SIZE, env.meta_size).to(DEV)
    agent, opp = mk(), mk()
    args = types.SimpleNamespace(num_minibatches=4, update_epochs=4, gamma=0.99, gae_lambda=0.95, norm_adv=True,
                                 clip_coef=0.2, clip_vloss=True, ent_coef=0.01, vf_coef=0.5, max_grad_norm=0.5,
                                 target_kl=None, learning_rate=2.5e-4, gae=True)
    tr = PackedPPO(env, agent, args, chunk=a.chunk)
    opponent = FusedPolicy(env, opp)
    T, apt = env.GAME_STEPS, 4
    n = T * apt * a.envs
    say(f"workload: 8_arena, B = {a.envs}, T = {T}, apt = {apt}: {n} samples per update, "
        f"{args.update_epochs} epochs x {args.num_minibatches} minibatches, chunks of {a.chunk}")
    results = []
    for u in range(a.updates):
        ro = None    # with the trainer's own reference gone too, one rollout is alive at a time
        torch.cuda.reset_peak_memory_stats()
        ro, t_roll = timed(lambda: tr.collect(opponent))
        (adv, ret), t_gae = timed(lambda: tr.advantages(ro))
        out, t_opt = timed(lambda: tr.optimise(ro, adv, ret))
        total = t_roll + t_gae + t_opt
        peak = torch.cuda.max_memory_allocated() / 1e9
        r = dict(rollout_s=t_roll, gae_s=t_gae, optimise_s=t_opt, total_s=total, samples_per_s=n / total,
                 max_memory_allocated_gb=peak, **out)
        results.append(r)
        say(f"update {u}: rollout {t_roll:.2f} s, gae {t_gae * 1e3:.1f} ms, optimise {t_opt:.2f} s, total {total:.2f} s, "
            f"{n / total:.3e} samples/s, max_memory_allocated {peak:.1f} GB")
        say(f"update {u}: first minibatch before any step: approx_kl {out['first_approx_kl']:.3e}, "
            f"clipfrac {out['first_clipfrac']:.3e}; last: v_loss {out['v_loss']:.4g}, pg_loss {out['pg_loss']:.4g}, "
            f"entropy {out['entropy']:.4g}, approx_kl {out['approx_kl']:.3e}, clipfrac {out['clipfrac']:.3e}")
        del adv, ret
    # the advantage kernel against its torch statement on the last rollout
    nv = torch.randn_like(ro.next_value)    # a non-zero bootstrap, so the first row does real work too
    kern = advantages(env, ro, nv, args.gamma, args.gae_lambda)
    ref = reference_advantages(ro.rewards, ro.values, nv, args.gamma, args.gae_lambda)
    equal = torch.equal(kern[0], ref[0]) and torch.equal(kern[1], ref[1])
    assert equal, "ctf_gae differs from reference_advantages"
    del kern, ref
    ms_k = median_ms(lambda: advantages(env, ro, nv, args.gamma, args.gae_lambda), a.gae_reps)
    ms_r = median_ms(lambda: reference_advantages(ro.rewards, ro.values, nv, args.gamma, args.gae_lambda), a.gae_reps)
    gbs = 16 * n / (ms_k * 1e-3) / 1e9
    say(f"ctf_gae: {ms_k:.3f} ms (median of {a.gae_reps}), {gbs:.0f} GB/s at 16 B per element = "
        f"{100 * gbs / COPY_PEAK_GBS:.1f} % of the {COPY_PEAK_GBS:.0f} GB/s copy peak; reference_advantages (eager torch, "
        f"{T} steps): {ms_r:.3f} ms ({ms_r / ms_k:.1f}x); torch.equal: {equal}")
    last = results[-1]
    say(f"optimise {last['optimise_s']:.1f} s measured against the {PROJECTED_OPTIMISE_S:.0f} s projection from the "
        f"per-chunk time")
    res = dict(gpu=gpu, envs=a.envs, steps=T, agents_per_step=apt, samples=n, chunk=a.chunk, updates=results,
               gae_ms=ms_k, gae_gbytes_per_s=gbs, gae_share_of_copy_peak=gbs / COPY_PEAK_GBS,
               reference_advantages_ms=ms_r, gae_bit_equal=equal, projected_optimise_s=PROJECTED_OPTIMISE_S)
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n" + json.dumps(res) + "\n")


if __name__ == "__main__":
    main()
