#!/usr/bin/env python
"""BASELINE config 5: self-play rollout on 8_arena with the GPU env feeding the agent_network-style policy.

    python bench_rollout.py [--envs B] [--steps K] [--warmup W] [--policy-dtype bf16|fp32] [--chunk S] [--fused]
    torchrun --nproc-per-node N bench_rollout.py ...      (env sharding, one rank per GPU)

Reports, as one JSON line from rank 0, agent-steps/s of the whole loop — policy forward for both teams on the
observation buffers the step kernel wrote, action sampling, env.step, and the packed (1 bit per element) copy of the
trained team's observations stored into a rollout ring buffer — next to the env-only and the policy-only figures.
With --graph the whole loop body (both policy forwards + step + store) is captured in ONE CUDA graph and replayed.
This is a functional integration of SURVEY §8f row N1: the policy is stock torch/cuDNN (≈3.9 MFLOP per agent-step)
and dominates the time.  With --fused the env is created packed-only and both teams run through FusedPolicy
(k_policy_trunk from the packed observations, then fc1 .. heads in bf16 on cuBLAS), one forward per team.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536, help="envs per GPU (BASELINE.json config 5: 65536)")
    ap.add_argument("--graph", action="store_true", help="capture policy forwards + step + rollout store in one CUDA graph")
    ap.add_argument("--store-steps", type=int, default=16, help="depth of the packed rollout ring buffer (env steps)")
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--policy-dtype", choices=["bf16", "fp32"], default="bf16")
    ap.add_argument("--chunk", type=int, default=32768, help="policy samples per forward")
    ap.add_argument("--channels-last", action="store_true", help="run the convolutions in NHWC (stock torch option)")
    ap.add_argument("--obs-dtype", choices=["float32", "bfloat16"], default=None,
                    help="env observation buffer type (default: bfloat16 when the policy runs in bf16)")
    ap.add_argument("--fused", action="store_true",
                    help="packed-only env, both teams through FusedPolicy (bf16; --chunk, --channels-last, --obs-dtype "
                         "and --policy-dtype do not apply)")
    return ap.parse_args(argv)


def measure(args):
    """Runs the loop on this rank's GPU (torch.distributed already initialised when WORLD_SIZE > 1).
    Returns the result dict on rank 0, None elsewhere.  bench.py calls this for its config-5 side figure."""
    import torch
    import torch.distributed as dist

    from marl_ctf_development_b200 import GridworldCtfGPU, experiment_env_config
    from marl_ctf_development_b200.policy import CtfPolicy

    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    B = args.envs
    obs_dtype = args.obs_dtype or ("bfloat16" if args.policy_dtype == "bf16" else "float32")
    torch.backends.cudnn.benchmark = True
    if args.fused:
        from marl_ctf_development_b200.fused_policy import FusedPolicy

        obs_dtype = "packed-only"
        env = GridworldCtfGPU(**experiment_env_config("8_arena"), num_envs=B, device=dev, seed=0, env_id_base=rank * B,
                              reverse_team1_actions=True, stats="counters", dense_obs=False, packed_obs=True)
    else:
        env = GridworldCtfGPU(**experiment_env_config("8_arena"), num_envs=B, device=dev, seed=0, env_id_base=rank * B,
                              reverse_team1_actions=True, stats="counters", obs_dtype=getattr(torch, obs_dtype),
                              packed_obs=True)
    N, C, G, M = env.N_AGENTS, env.n_channels, env.GRID_SIZE, env.meta_size
    torch.manual_seed(rank)
    pols = [CtfPolicy(9, C, G, M).to(dev).eval() for _ in range(2)]
    if args.channels_last:
        pols = [p.to(memory_format=torch.channels_last) for p in pols]
    teams = [torch.tensor([i for i in range(N) if env.AGENT_TEAMS[i] == t], device=dev) for t in (0, 1)]
    team_ids = [[i for i in range(N) if env.AGENT_TEAMS[i] == t] for t in (0, 1)]   # host lists: capturable
    fused = [FusedPolicy(env, p) for p in pols] if args.fused else None
    actions = torch.empty((B, N), dtype=torch.uint8, device=dev)
    amp = torch.autocast("cuda", dtype=torch.bfloat16, enabled=args.policy_dtype == "bf16")

    @torch.no_grad()
    def policy_step(obs, meta):
        if fused is not None:
            for idx, ids, fp in zip(teams, team_ids, fused):
                k = len(ids)
                f = env.use_action_mask[idx].unsqueeze(0).expand(B, k).reshape(B * k)
                actions[:, idx] = fp.get_action(f, agent_ids=ids).reshape(B, k).to(torch.uint8)
            return
        for idx, pol in zip(teams, pols):
            k = idx.numel()
            g = obs[:, idx].reshape(B * k, C, G, G)
            if args.channels_last:
                g = g.contiguous(memory_format=torch.channels_last)
            m = meta[:, idx].reshape(B * k, M)
            f = env.use_action_mask[idx].unsqueeze(0).expand(B, k).reshape(B * k)
            outs = []
            for s in range(0, B * k, args.chunk):
                with amp:
                    outs.append(pol.get_action(g[s : s + args.chunk], m[s : s + args.chunk], f[s : s + args.chunk]))
            actions[:, idx] = torch.cat(outs).reshape(B, k).to(torch.uint8)

    # packed rollout storage of the trained team (team 0): [store_steps, apt, B, words_per_agent] int32, 32x smaller than
    # float32 (a float32 [500*4, 65536, 14, 15, 15] rollout would be 1.6 PB, SURVEY §7); unpacked per minibatch at update time
    apt = int(teams[0].numel())
    ring = torch.zeros((args.store_steps, apt, B, env.bits_words_per_agent), dtype=torch.int32, device=dev)
    ring_meta = torch.zeros((args.store_steps, apt, B, M), dtype=torch.float32, device=dev)
    slot = [0]

    def body(with_policy=True, with_env=True):
        if with_policy:
            policy_step(env.obs, env.meta)
        if with_env:
            k = slot[0] % args.store_steps
            ring[k].copy_(env.obs_bits[:, teams[0]].transpose(0, 1))
            ring_meta[k].copy_(env.meta[:, teams[0]].transpose(0, 1))
            slot[0] += 1
            env.step(actions)

    graphs = {}

    def run(k_steps, with_policy, with_env=True):
        key = (with_policy, with_env)
        if args.graph and key not in graphs:
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                body(with_policy, with_env)           # warm-up outside the capture (cuDNN autotune, allocator)
            torch.cuda.current_stream(dev).wait_stream(side)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                body(with_policy, with_env)
            graphs[key] = g
        for _ in range(k_steps):
            if args.graph:
                graphs[key].replay()
            else:
                body(with_policy, with_env)

    def timed(k_steps, with_policy, with_env=True):
        run(1, with_policy, with_env)                 # graph capture / first call outside the timed region
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run(k_steps, with_policy, with_env)
        e1.record()
        torch.cuda.synchronize(dev)
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    env.reset()
    actions.fill_(4)
    run(args.warmup, True)
    ms_full = timed(args.steps, True)
    ms_env = timed(args.steps, False)
    ms_pol = timed(args.steps, True, False)
    result = None
    if rank == 0:
        total = world * B * N * args.steps
        result = ({
            "metric": "rollout_agent_steps_per_sec", "value": total / (ms_full * 1e-3), "unit": "agent-steps/s",
            "env_only_value": total / (ms_env * 1e-3), "policy_only_value": total / (ms_pol * 1e-3),
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_full / args.steps, "env_ms_per_step": ms_env / args.steps, "policy_ms_per_step": ms_pol / args.steps,
            "cuda_graph": bool(args.graph),
            "policy_path": "fused" if args.fused else "cudnn",
            "rollout_storage": f"packed observations of the trained team, ring of {args.store_steps} steps: "
                               f"{ring.numel() * 4 / 1e6:.0f} MB (float32 would be {ring.numel() * 4 * 32 / 1e9:.1f} GB)",
            "config": {"workload": f"8_arena self-play rollout, B={B} envs/GPU, CtfPolicy (agent_network.py architecture) "
                                   f"for both teams, "
                                   + ("FusedPolicy (k_policy_trunk + bf16 cuBLAS heads), packed-only env" if args.fused else
                                      f"policy dtype {args.policy_dtype}, {obs_dtype} observations"
                                      f"{', channels_last' if args.channels_last else ''}")
                                   + "; env-only = step + packed rollout store",
                       "envs_per_gpu": B},
            "data": "synthetic (random-init policies)",
        })
    env.close()
    del env, ring, ring_meta, pols, graphs, fused
    torch.cuda.empty_cache()
    return result


def main():
    import torch
    import torch.distributed as dist

    args = parse_args()
    world, local = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    result = measure(args)
    if result is not None:
        print(json.dumps(result), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
