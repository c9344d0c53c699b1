#!/usr/bin/env python
"""PPO-update cost per chunk: FusedPolicy training (packed observations) against stock CtfPolicy on unpacked ones.

    python tools/policy_train_bench.py [--envs 65536] [--steps 4] [--iters 5] [--rounds 3]

Collects a real packed 8_arena rollout (B envs, FusedPolicy on both sides, packed-only env), then times forward + PPO
clipped loss + backward over chunks of one team's samples of one step (B * 4 = 262 144 at B = 65 536), drawn at
random from the rollout, three ways:
  fused     FusedPolicy.evaluate_actions on the packed rows (trunk kernels, bf16 fc1/fc2 on cuBLAS, fp32 heads);
  fp32      env.unpack_obs to float32, then CtfPolicy (cuDNN / cuBLAS, fp32);
  autocast  the same under torch.autocast(bfloat16).
CUDA events, a warm-up of every path, then the paths alternated --rounds times; the median per path is reported with
samples/s.  Then the fused stages are timed one by one (trunk forward, FusedPolicy.train_head forward + loss +
backward, trunk backward), the backward's two kernels are split with torch.profiler in a separate pass, and the trunk
backward's achieved FLOP/s and bytes/s are computed from the shapes.  The projection of one BASELINE update (5.2e8 sample passes: 8_arena,
B = 65 536, T = 500, 4 trained agents, 4 epochs) multiplies the measured fused time per sample.  The card's name and
power limit are read with nvidia-smi in the same run.  Prints text lines and one final JSON line.
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

from marl_ctf_development_b200 import GridworldCtfGPU, experiment_env_config  # noqa: E402
from marl_ctf_development_b200.fused_policy import FusedPolicy, _PackedTrunk  # noqa: E402
from marl_ctf_development_b200.policy import CtfPolicy  # noqa: E402
from marl_ctf_development_b200.rollout import collect_rollout  # noqa: E402

DEV = "cuda:0"
BASELINE_SAMPLE_PASSES = 65536 * 500 * 4 * 4   # one BASELINE update: 4 epochs over B * T * 4 samples


def ppo_loss(logprob, entropy, value, old_logprob, adv, ret, clip=0.2):
    ratio = torch.exp(logprob - old_logprob)
    pg = torch.max(-adv * ratio, -adv * torch.clamp(ratio, 1 - clip, 1 + clip)).mean()
    return pg + 0.5 * ((value.reshape(-1) - ret) ** 2).mean() - 0.01 * entropy.mean()


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else f"nvidia-smi failed: {q.stderr.strip()}"


def time_ms(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=4, help="rollout steps to draw chunks from")
    ap.add_argument("--iters", type=int, default=5, help="chunks per timed window")
    ap.add_argument("--rounds", type=int, default=3, help="times the three paths are alternated")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("policy_train_bench needs a CUDA device")
    print("gpu:", gpu_info(), flush=True)

    B = args.envs
    env = GridworldCtfGPU(**experiment_env_config("8_arena"), num_envs=B, device=DEV, seed=0, reverse_team1_actions=True,
                          dense_obs=False, packed_obs=True)
    Cn, G, M, wpa = env.n_channels, env.GRID_SIZE, env.meta_size, env.bits_words_per_agent
    torch.manual_seed(0)
    pol = CtfPolicy(9, Cn, G, M).to(DEV)
    opp = CtfPolicy(9, Cn, G, M).to(DEV)
    agent = FusedPolicy(env, pol)
    ro = collect_rollout(env, agent, FusedPolicy(env, opp), num_env_steps=args.steps, obs_storage_dtype="packed")
    bits_all = ro.grid_states.reshape(-1, wpa)
    meta_all = ro.metadata_states.reshape(-1, M)
    act_all, mask_all, lp_all = ro.actions.reshape(-1).long(), ro.use_action_mask.reshape(-1), ro.logprobs.reshape(-1)
    adv_all = ro.rewards.reshape(-1) - ro.values.reshape(-1)
    adv_all = (adv_all - adv_all.mean()) / (adv_all.std() + 1e-8)
    ret_all = ro.rewards.reshape(-1)
    n_all = bits_all.shape[0]
    S = n_all // args.steps                           # one step of the trained team: B * 4 at 8_arena
    print(f"rollout: {n_all} packed samples ({args.steps} steps x {n_all // args.steps}); chunk {S} samples", flush=True)

    g = torch.Generator(device=DEV).manual_seed(1)
    idx = torch.randperm(n_all, generator=g, device=DEV)[:S]
    bits, meta = bits_all[idx].contiguous(), meta_all[idx].contiguous()
    act, mask, old, adv, ret = act_all[idx], mask_all[idx], lp_all[idx], adv_all[idx], ret_all[idx]

    def fused():
        pol.zero_grad(set_to_none=True)
        lp, ent, v = agent.evaluate_actions(bits, meta, mask, act)
        ppo_loss(lp, ent, v, old, adv, ret).backward()

    def stock(amp):
        def run():
            pol.zero_grad(set_to_none=True)
            dense = env.unpack_obs(bits)                     # float32 [S, C, G, G]
            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
                _, lp, ent, v = pol.get_action_and_value(dense, meta, mask, act)
            ppo_loss(lp.float(), ent.float(), v.float(), old, adv, ret).backward()
        return run

    paths = {"fused": fused, "fp32": stock(False), "autocast_bf16": stock(True)}
    for fn in paths.values():        # warm-up: cuDNN / cuBLAS algorithm choice, allocator
        fn(); fn()
    torch.cuda.synchronize()
    times = {k: [] for k in paths}
    for r in range(args.rounds):
        for k, fn in paths.items():
            times[k].append(time_ms(fn, args.iters))
        print(f"round {r}: " + ", ".join(f"{k} {times[k][-1]:.2f} ms" for k in paths), flush=True)
    med = {k: statistics.median(v) for k, v in times.items()}
    for k in paths:
        print(f"{k:14s} {med[k]:8.2f} ms/chunk  {S / med[k] * 1e3:.3e} samples/s  (rounds: "
              + ", ".join(f"{x:.2f}" for x in times[k]) + ")", flush=True)

    # fused stages
    p = pol
    conv = [p.conv1.weight, p.conv1.bias, p.conv2.weight, p.conv2.bias]
    rows = _PackedTrunk.apply(bits, *conv, agent, meta)
    rows_d = rows.detach().requires_grad_(True)
    grad_rows = torch.empty_like(rows_d)

    def trunk_fwd():
        agent._train_forward(bits, meta, *[t.detach() for t in conv])

    def head():
        rows_d.grad = None
        value, logits = agent.train_head(rows_d)          # the code evaluate_actions runs after the trunk
        probs = torch.distributions.Categorical(logits=p.masked_logits(logits, mask), validate_args=False)
        ppo_loss(probs.log_prob(act), probs.entropy(), value, old, adv, ret).backward()
        grad_rows.copy_(rows_d.grad)

    def trunk_bwd():
        agent._train_backward(bits, rows.detach(), grad_rows, *[t.detach() for t in conv])

    for fn in (trunk_fwd, head, trunk_bwd):
        fn()
    torch.cuda.synchronize()
    st = {"trunk_forward": time_ms(trunk_fwd, args.iters), "head_fwd_bwd": time_ms(head, args.iters),
          "trunk_backward": time_ms(trunk_bwd, args.iters)}
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        trunk_bwd()
        torch.cuda.synchronize()
    kern = {}
    for ev in prof.key_averages():
        for name in ("k_policy_trunk_backward", "k_policy_grad_reduce"):
            if name in ev.key:
                kern[name] = ev.device_time_total / 1e3 if hasattr(ev, "device_time_total") else ev.cuda_time_total / 1e3
    st.update({f"{k}_kernel": v for k, v in kern.items()})
    S1, S2 = G - 2, G - 4
    flops = S * (2 * 32 * 144 * S2 * S2 + 2 * S1 * S1 * 16 * 288)            # dW2 GEMM + dh1 implicit GEMM
    nbytes = S * (wpa * 4 + 2 * 2 * 32 * S2 * S2)                             # packed bits, saved rows, dRows (conv part)
    kb = kern.get("k_policy_trunk_backward", st["trunk_backward"])
    st["trunk_backward_tflops"] = flops / (kb * 1e-3) / 1e12
    st["trunk_backward_gbytes_per_s"] = nbytes / (kb * 1e-3) / 1e9
    for k, v in st.items():
        print(f"fused stage {k}: {v:.3f}" + (" ms" if not k.endswith(("tflops", "per_s")) else ""), flush=True)
    per_sample = med["fused"] * 1e-3 / S
    proj = {k: med[k] * 1e-3 / S * BASELINE_SAMPLE_PASSES for k in med}
    for k, v in proj.items():
        print(f"projected BASELINE update (5.2e8 sample passes), {k}: {v:.1f} s", flush=True)
    print(json.dumps({
        "gpu": gpu_info(), "chunk_samples": S, "iters": args.iters, "rounds": args.rounds, "ms_per_chunk": med,
        "ms_per_chunk_rounds": times, "samples_per_s": {k: S / v * 1e3 for k, v in med.items()},
        "fused_speedup": {"vs_fp32": med["fp32"] / med["fused"], "vs_autocast_bf16": med["autocast_bf16"] / med["fused"]},
        "fused_stages_ms": st, "fused_s_per_sample": per_sample, "projected_baseline_update_s": proj,
    }), flush=True)


if __name__ == "__main__":
    main()
