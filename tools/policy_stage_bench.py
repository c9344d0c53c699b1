#!/usr/bin/env python
"""Stage breakdown of policy inference at rollout scale (8_arena, B envs, both teams).

    python tools/policy_stage_bench.py [--envs 65536] [--iters 20]                 # FusedPolicy stages, CUDA events
    python tools/policy_stage_bench.py --profile-cudnn OUT.txt [--envs 65536]      # torch.profiler of the cuDNN path

The first form prints one JSON line: per team the trunk kernel (ctf_policy_features) ms, the head (fc1 -> tanh -> fc2
-> tanh -> heads) ms, fc1 alone (over the padded row as FusedPolicy runs it, and over the K1-column view for comparison),
and the achieved rates: trunk tensor-core TFLOP/s (conv2 MACs from the shapes; the
sparse conv1 FMAs are not counted), fc1 TFLOP/s, and trunk bytes/s (packed bits + metadata in, bf16 feature rows out).
The second runs today's path of bench_rollout.py (bf16 autocast, channels_last, bf16 observations) eagerly under
torch.profiler and writes the per-kernel CUDA time table, so the cuDNN policy time can be attributed to layers.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from marl_ctf_development_b200 import GridworldCtfGPU, experiment_env_config  # noqa: E402
from marl_ctf_development_b200.fused_policy import FusedPolicy  # noqa: E402
from marl_ctf_development_b200.policy import CtfPolicy  # noqa: E402


def _time(fn, iters):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def _env(B, dense):
    kw = dict(obs_dtype=torch.bfloat16, packed_obs=True) if dense else dict(dense_obs=False, packed_obs=True)
    env = GridworldCtfGPU(**experiment_env_config("8_arena"), num_envs=B, device="cuda:0", seed=0,
                          reverse_team1_actions=True, **kw)
    g = torch.Generator(device="cuda:0").manual_seed(0)
    for _ in range(5):
        env.step(torch.randint(0, 9, (B, env.N_AGENTS), generator=g, device="cuda:0").to(torch.uint8))
    return env


def stages(args):
    B = args.envs
    env = _env(B, dense=False)
    N, M, wpa = env.N_AGENTS, env.meta_size, env.bits_words_per_agent
    side = env.GRID_SIZE - 4
    out = {"device": torch.cuda.get_device_name(0), "envs": B, "iters": args.iters, "teams": []}
    total = 0.0
    for t in (0, 1):
        ids = [i for i in range(N) if env.AGENT_TEAMS[i] == t]
        S = B * len(ids)
        torch.manual_seed(t)
        fp = FusedPolicy(env, CtfPolicy(9, env.n_channels, env.GRID_SIZE, M).cuda().eval())
        feat = fp.trunk_from_env(ids)
        flags = env.use_action_mask[ids].unsqueeze(0).expand(B, len(ids)).reshape(-1)
        with torch.no_grad():
            ms_trunk = _time(lambda: fp.trunk_from_env(ids), args.iters)
            ms_head = _time(lambda: fp._head(feat), args.iters)
            ms_fc1 = _time(lambda: F.linear(feat, fp._fc1w, fp._fc1b), args.iters)
            w_k1 = fp._fc1w[:, : fp.k1].contiguous()
            ms_fc1_k1 = _time(lambda: F.linear(feat[:, : fp.k1], w_k1, fp._fc1b), args.iters)
            ms_all = _time(lambda: fp.get_action(flags, agent_ids=ids), args.iters)
        conv2_flop = 2.0 * S * 32 * 144 * side * side
        fc1_flop = 2.0 * S * fp.k1 * 256
        trunk_bytes = S * (wpa * 4 + M * 4) + S * fp.stride * 2
        out["teams"].append({
            "team": t, "samples": S, "trunk_ms": ms_trunk, "head_ms": ms_head, "fc1_ms": ms_fc1,
            "forward_and_sample_ms": ms_all,
            "trunk_tensor_core_tflops": conv2_flop / (ms_trunk * 1e-3) / 1e12,
            "trunk_gb_per_s": trunk_bytes / (ms_trunk * 1e-3) / 1e9, "trunk_gb": trunk_bytes / 1e9,
            "fc1_tflops": fc1_flop / (ms_fc1 * 1e-3) / 1e12,
            "fc1_on_k1_view_ms": ms_fc1_k1, "fc1_on_k1_view_tflops": fc1_flop / (ms_fc1_k1 * 1e-3) / 1e12,
        })
        total += ms_all
    out["policy_ms_per_step_both_teams"] = total
    print(json.dumps(out), flush=True)


def profile_cudnn(args):
    from torch.profiler import ProfilerActivity, profile

    B = args.envs
    env = _env(B, dense=True)
    N, C, G, M = env.N_AGENTS, env.n_channels, env.GRID_SIZE, env.meta_size
    torch.backends.cudnn.benchmark = True
    pols = []
    for t in (0, 1):
        torch.manual_seed(t)
        pols.append(CtfPolicy(9, C, G, M).cuda().eval().to(memory_format=torch.channels_last))
    teams = [torch.tensor([i for i in range(N) if env.AGENT_TEAMS[i] == t], device="cuda:0") for t in (0, 1)]

    @torch.no_grad()
    def step():
        for idx, pol in zip(teams, pols):
            k = idx.numel()
            g = env.obs[:, idx].reshape(B * k, C, G, G).contiguous(memory_format=torch.channels_last)
            m = env.meta[:, idx].reshape(B * k, M)
            f = env.use_action_mask[idx].unsqueeze(0).expand(B, k).reshape(B * k)
            for s in range(0, B * k, args.chunk):
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    pol.get_action(g[s : s + args.chunk], m[s : s + args.chunk], f[s : s + args.chunk])

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(args.iters):
            step()
        torch.cuda.synchronize()
    table = prof.key_averages().table(sort_by="cuda_time_total", row_limit=40)
    text = (f"# cuDNN policy path of bench_rollout.py (bf16 autocast, channels_last, chunk {args.chunk}), "
            f"8_arena B={B}, both teams, {args.iters} steps, {torch.cuda.get_device_name(0)}\n{table}\n")
    os.makedirs(os.path.dirname(os.path.abspath(args.profile_cudnn)), exist_ok=True)
    with open(args.profile_cudnn, "w") as fh:
        fh.write(text)
    print(text, flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--chunk", type=int, default=32768, help="cuDNN path: samples per forward (bench_rollout default)")
    ap.add_argument("--profile-cudnn", default=None, metavar="OUT", help="write the torch.profiler table of the cuDNN path")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    if args.profile_cudnn:
        profile_cudnn(args)
    else:
        stages(args)


if __name__ == "__main__":
    main()
