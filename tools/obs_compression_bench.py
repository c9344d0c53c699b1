"""Does compressible memory make the dense-observation step faster?  (DESIGN §4, profiles/r05_obs_compression.log)

Prints, in this order:
  1. the device name, power limit and max SM clock (nvidia-smi query only; nothing is set);
  2. CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED;
  3. whether the compressible buffer's allocation was granted CU_MEM_ALLOCATION_COMP_GENERIC;
  4. the step time of the real env at the headline shape (8_arena, B = 65536, float32, stats counters) on a plain
     buffer (obs_out=torch.empty) and on a compressible one, alternating, --blocks blocks of --steps steps each;
  5. torch.equal of the two envs' outputs after the same seeded steps;
  6. torch fill_(0) of both buffers, and a copy of incompressible data (torch.rand bytes) into both: the worst case.

    python tools/obs_compression_bench.py [--envs 65536] [--blocks 6] [--steps 200] [--out FILE]
"""
from __future__ import annotations

import argparse
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--experiment", default="8_arena")
    ap.add_argument("--obs-dtype", default="float32", choices=["float32", "uint8", "float16", "bfloat16"])
    ap.add_argument("--blocks", type=int, default=6)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--out", default=None, help="also write the report to this file")
    args = ap.parse_args()

    import torch

    from marl_ctf_development_b200 import GridworldCtfGPU, experiment_env_config
    from marl_ctf_development_b200.compressible import compressible_empty, compression_supported, is_compressed

    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                       capture_output=True, text=True)
    say("1. device: " + " | ".join(q.stdout.strip().splitlines()) if q.returncode == 0 else f"1. nvidia-smi failed: {q.stderr.strip()}")
    dev = torch.device("cuda", 0)
    say(f"   torch: {torch.cuda.get_device_name(dev)}")
    supported = compression_supported(dev)
    say(f"2. CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED = {int(supported)}")

    ec = experiment_env_config(args.experiment)
    dt = getattr(torch, args.obs_dtype)
    B = args.envs
    kw = dict(num_envs=B, device=dev, seed=0, stats="counters", obs_dtype=dt)
    probe = GridworldCtfGPU(**ec, num_envs=1, device=dev)
    shape = (B, probe.N_AGENTS, probe.n_channels, probe.GRID_SIZE, probe.GRID_SIZE)
    probe.close()
    comp_buf = compressible_empty(shape, dt, dev)
    granted = is_compressed(comp_buf)
    say(f"3. compressible buffer {tuple(shape)} {args.obs_dtype}, {comp_buf.numel() * comp_buf.element_size() / 1e9:.3f} GB: "
        f"allocation granted COMP_GENERIC = {int(granted)}")
    plain_buf = torch.empty(shape, dtype=dt, device=dev)
    envs = {
        "plain": GridworldCtfGPU(**ec, **kw, obs_out=plain_buf),
        "compressible": GridworldCtfGPU(**ec, **kw, obs_out=comp_buf),
    }
    say(f"   env.obs_compressed: plain {envs['plain'].obs_compressed}, compressible {envs['compressible'].obs_compressed}")

    N = envs["plain"].N_AGENTS
    gen = torch.Generator(device=dev).manual_seed(1234)
    actions = torch.randint(0, 9, (8, B, N), dtype=torch.uint8, device=dev, generator=gen)
    counters = {k: 0 for k in envs}

    def run(name, steps):
        env = envs[name]
        for _ in range(steps):
            k = counters[name]
            env.step(actions[k % 8])
            counters[name] = k + 1
            if (k + 1) % env.GAME_STEPS == 0:
                env.reset()

    for name in envs:   # warm-up: modules loaded, clocks up
        run(name, 100)
    torch.cuda.synchronize(dev)
    times = {k: [] for k in envs}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.blocks):
        for name in envs:
            e0.record()
            run(name, args.steps)
            e1.record()
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1) / args.steps)
    obs_bytes = comp_buf.numel() * comp_buf.element_size()
    say(f"4. step time, {args.experiment} {args.obs_dtype} B = {B}, {args.blocks} blocks x {args.steps} steps, alternating "
        f"(ms/step; GB/s of dense observations)")
    for name, t in times.items():
        say(f"   {name:13s} median {statistics.median(t):.4f}  min {min(t):.4f}  max {max(t):.4f}  "
            f"({obs_bytes / statistics.median(t) / 1e6:.0f} GB/s)  blocks: " + " ".join(f"{x:.4f}" for x in t))
    p, c = times["plain"], times["compressible"]
    say(f"   compressible / plain (medians) = {statistics.median(c) / statistics.median(p):.3f}; ranges "
        f"{'do not overlap' if max(c) < min(p) or min(c) > max(p) else 'overlap'}")

    a, b = envs["plain"], envs["compressible"]
    assert counters["plain"] == counters["compressible"]
    same = {n: bool(torch.equal(getattr(a, n), getattr(b, n))) for n in ("obs", "meta", "rewards", "dones")}
    same["state"] = all(bool(torch.equal(x, y)) for x, y in zip((a._grid, a._agents, a._envs), (b._grid, b._agents, b._envs)))
    say(f"5. after {counters['plain']} identical seeded steps: torch.equal " + ", ".join(f"{k} {v}" for k, v in same.items()))
    for env in envs.values():
        env.close()

    def rate(fn, reps=20):
        fn()
        torch.cuda.synchronize(dev)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        e1.synchronize()
        ms = e0.elapsed_time(e1) / reps
        return ms, obs_bytes / ms / 1e6

    noise = torch.rand(obs_bytes // 4, device=dev).view(torch.uint8)   # random mantissas: incompressible
    plain_u8, comp_u8 = plain_buf.view(-1).view(torch.uint8), comp_buf.view(-1).view(torch.uint8)
    say(f"6. bulk writes of the {obs_bytes / 1e9:.3f} GB buffer (ms; GB/s written)")
    for label, fn_p, fn_c in (
        ("fill_(0)", lambda: plain_buf.fill_(0), lambda: comp_buf.fill_(0)),
        ("copy of torch.rand bytes", lambda: plain_u8.copy_(noise), lambda: comp_u8.copy_(noise)),
    ):
        res = {}
        for rep in range(3):   # alternate, keep the best of three for each
            for name, fn in (("plain", fn_p), ("compressible", fn_c)):
                ms, gbs = rate(fn)
                if name not in res or ms < res[name][0]:
                    res[name] = (ms, gbs)
        say(f"   {label:25s} plain {res['plain'][0]:.4f} ms ({res['plain'][1]:.0f} GB/s)   compressible "
            f"{res['compressible'][0]:.4f} ms ({res['compressible'][1]:.0f} GB/s)   ratio {res['compressible'][0] / res['plain'][0]:.3f}")
    assert torch.equal(plain_u8, comp_u8), "the copies differ"
    say("   the two copies read back equal")

    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
