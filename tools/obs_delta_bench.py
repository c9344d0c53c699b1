"""Delta observation writes (the env's own buffer with its record) against full writes (a caller-bound buffer).

    python tools/obs_delta_bench.py [--out profiles/r10_obs_delta.log] [--cap-lib 5=path/libctf_b200.so ...]

1. the card (nvidia-smi query);
2. per shape, blocks of steps of the delta env and of the full-write env, alternated, in ms per step;
3. the share of 32-byte sectors of the dense buffer that change from one step to the next (torch, on the device);
4. with --cap-lib, the residency sweep of delta steps: one library per k_step delta cap (built with
   -DCTF_DELTA_CTAS_PER_SM=cap), on compressed and on plain memory, each in its own process;
5. torch.equal of the two envs' outputs after the run.
Both envs use stats="counters", uniform random actions from a seeded generator, and reset every GAME_STEPS steps.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = [("8_arena", "float32", 65536), ("8_arena", "bfloat16", 65536), ("8_arena", "uint8", 65536),
          ("7_gridlocked", "float32", 65536), ("8_arena", "float32", 16384)]
ORACLE_SECTOR_SHARE = "CPU oracle, 256 envs, steps 1-200: 1.2-1.4 % (8_arena), 1.3 % (7_gridlocked)"


def _envs(exp, dtype, B, plain=False):
    import torch

    from marl_ctf_development_b200 import GridworldCtfGPU, _native, experiment_env_config
    from marl_ctf_development_b200.compressible import compressible_empty

    ec = experiment_env_config(exp)
    kw = dict(num_envs=B, device="cuda:0", seed=0, stats="counters", obs_dtype=getattr(torch, dtype))
    if plain:
        _native.load().ctf_compressible_set_enabled(0)
    delta = GridworldCtfGPU(**ec, **kw)   # uint8: no record, so both envs write in full
    full = GridworldCtfGPU(**ec, **kw, obs_out=compressible_empty(tuple(delta.obs.shape), getattr(torch, dtype), "cuda:0"))
    if plain:
        _native.load().ctf_compressible_set_enabled(1)
    return delta, full


def _block(env, acts, state, steps):
    import torch

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        env.step(acts[state["k"] % len(acts)])
        state["k"] += 1
        if state["k"] % env.GAME_STEPS == 0:
            env.reset()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def _acts(env, n=8):
    import torch

    g = torch.Generator(device="cuda:0").manual_seed(1234)
    return [torch.randint(0, 9, (env.num_envs, env.N_AGENTS), dtype=torch.uint8, device="cuda:0", generator=g) for _ in range(n)]


def _stats(xs):
    xs = sorted(xs)
    return {"median": xs[len(xs) // 2], "min": xs[0], "max": xs[-1]}


def measure_shape(exp, dtype, B, rounds, steps, plain=False, full_too=True):
    """Alternated blocks of the delta env and the full-write env; ms per step of every block."""
    import torch

    delta, full = _envs(exp, dtype, B, plain)
    acts = _acts(delta)
    sd, sf = {"k": 0}, {"k": 0}
    _block(delta, acts, sd, 150)
    if full_too:
        _block(full, acts, sf, 150)
    td, tf = [], []
    for _ in range(rounds):
        td.append(_block(delta, acts, sd, steps))
        if full_too:
            tf.append(_block(full, acts, sf, steps))
    out = {"shape": f"{exp}/{dtype}/{B}", "memory": "plain" if plain else "compressed" if delta.obs_compressed else "plain",
           "delta_ms": _stats(td), "delta_blocks": td}
    if full_too:
        out.update(full_ms=_stats(tf), full_blocks=tf)
        # both envs took the same number of steps from the same seed and actions: their outputs must agree
        out["torch_equal"] = all(torch.equal(getattr(delta, k).view(torch.uint8), getattr(full, k).view(torch.uint8))
                                 for k in ("obs", "meta", "rewards", "dones"))
    delta.close()
    full.close()
    del delta, full
    torch.cuda.empty_cache()
    return out


def sector_share(exp, dtype, B, samples=(1, 2, 5, 20, 50, 100, 200)):
    """Share of the dense buffer's 32-byte sectors that differ between consecutive steps' outputs."""
    import torch

    delta, _ = _envs(exp, dtype, B)
    acts = _acts(delta)
    out, k = [], 0
    for t in range(1, max(samples) + 1):
        prev = delta.obs.clone() if t in samples else None
        delta.step(acts[k % len(acts)])
        k += 1
        if prev is not None:
            a, b = prev.reshape(-1).view(torch.int64).view(-1, 4), delta.obs.reshape(-1).view(torch.int64).view(-1, 4)
            out.append((t, float((a != b).any(dim=1).float().mean())))
            del prev, a, b
    delta.close()
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_obs_delta.log"))
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--cap-lib", action="append", default=[], metavar="CAP=PATH",
                    help="library built with -DCTF_DELTA_CTAS_PER_SM=CAP, for the residency sweep")
    ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)   # the sweep points of one library
    args = ap.parse_args()
    if args.worker:
        for exp, dtype, B in SHAPES:
            for mem in ("compressed", "plain"):
                print(json.dumps(measure_shape(exp, dtype, B, 3, args.steps, mem == "plain", full_too=False)), flush=True)
        return

    lines = []

    def log(s=""):
        print(s, flush=True)
        lines.append(s)

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    log("# k_step delta writes (env-owned obs with its record) vs full writes (obs_out= buffer), tools/obs_delta_bench.py")
    log(f"# card: {smi}")
    log(f"# stats=counters, seed 0, uniform random actions, reset every GAME_STEPS; {args.rounds} alternated blocks of "
        f"{args.steps} steps per env, CUDA events, ms per step")
    log("\n## alternated blocks, delta vs full")
    for exp, dtype, B in SHAPES:
        r = measure_shape(exp, dtype, B, args.rounds, args.steps)
        d, f = r["delta_ms"], r["full_ms"]
        log(f"{r['shape']:<26} {r['memory']:<10} delta {d['median']:.4f} [{d['min']:.4f}-{d['max']:.4f}]  "
            f"full {f['median']:.4f} [{f['min']:.4f}-{f['max']:.4f}]  x{f['median'] / d['median']:.2f}  "
            f"torch.equal after the run: {r['torch_equal']}")
        log("  blocks " + json.dumps({"delta": r["delta_blocks"], "full": r["full_blocks"]}))
    log("\n## changed 32-byte sectors between consecutive steps (device, torch)")
    log(f"# {ORACLE_SECTOR_SHARE}")
    for exp, dtype in (("8_arena", "float32"), ("7_gridlocked", "float32"), ("8_arena", "bfloat16")):
        share = sector_share(exp, dtype, 65536)
        log(f"{exp}/{dtype}/65536 " + "  ".join(f"step {t}: {100 * s:.2f} %" for t, s in share))
    if args.cap_lib:
        log("\n## residency sweep of delta steps: CTAs per SM (one library each), 3 blocks per point, ms per step")
        caps = sorted((int(c.split("=")[0]), c.split("=", 1)[1]) for c in args.cap_lib)
        rows = {}
        for cap, lib in caps:
            env = dict(os.environ, CTF_B200_LIB=os.path.abspath(lib))
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", "--steps", str(args.steps)],
                               capture_output=True, text=True, env=env)
            if p.returncode != 0:
                log(f"cap {cap}: failed: {p.stderr.strip()[-500:]}")
            for line in p.stdout.strip().splitlines():
                r = json.loads(line)
                d = r["delta_ms"]
                rows.setdefault((r["shape"], r["memory"]), []).append(f"cap{cap} {d['median']:.4f} [{d['min']:.4f}-{d['max']:.4f}]")
        for (shape, mem), row in rows.items():
            log(f"{shape:<26} {mem:<10} " + "  ".join(row))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
