#!/usr/bin/env python
"""Throughput of the GridworldCtf step path: agent-steps/s for 8_arena at B envs per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--envs B] [--impl ours|reference]

One "step" is one pass of the hot path over one batch: env.step(actions) for B envs — the fused
kernel advances all N agents of every env and writes their float32 observations + metadata into the
policy input buffers — so a step is B*N agent-steps.  Under torchrun (N > 1) every rank owns B envs
with global ids rank*B .. rank*B+B-1 (weak scaling, no collective inside the step); the episode
statistics are summed on the device and all-reduced over NCCL once per episode and once at the end of
the timed region.  Rank 0 prints ONE JSON line.

--dump-outputs DIR writes what the last of the K timed steps returned to the caller as DIR/<name>.npy.  The
inputs (env seed, pre-generated actions) depend on the arguments only, so two builds run with the same arguments
can be compared output for output.

--impl reference times the reference's own CPU implementation on all host cores: the unmodified Python
``GridworldCtf`` (one env per process; /root/reference, or its byte-compiled copy oracle/_ref on the GPU box),
falling back to the C port of the oracle only where neither exists.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

EXPERIMENT = "8_arena"  # BASELINE.json headline; --experiment selects another config for side measurements
METRIC = "agent_steps_per_sec"
UNIT = "agent-steps/s"
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md, used only when MEASURED_PEAKS.json is absent
OBS_ELEM_BYTES = {"float32": 4, "uint8": 1, "float16": 2, "bfloat16": 2}
DTYPE_TAG = {"float32": "f32", "uint8": "u8", "float16": "f16", "bfloat16": "bf16"}
KERNEL_T = {"float32": "float", "uint8": "uint8_t", "float16": "__half", "bfloat16": "__nv_bfloat16"}
REF_ENV_STEPS_PER_PASS = 100  # --impl reference: env steps every process advances per bench "step"
DUMP_BYTES = 60_000_000  # --dump-outputs stays below 64 MB: larger batches are written for a fixed, seeded sample of envs


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def algorithmic_bytes_per_agent_step(G: int, N: int, C: int, obs_elem_bytes: int = 4) -> float:
    """SURVEY.md §8(d): obs + metadata + reward + (state read+write + actions + done + mask) / N."""
    M = 6 + 2 * N
    state_rw = 2 * (G * G + 2 * N + 2 * N + N + 2 * N + 8)
    return C * G * G * obs_elem_bytes + M * 4 + 4 + (state_rw + N + 1 + N) / N


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU through NVML while the timed region runs.

    ``sample()`` can also be called from the main thread (one sample right before and right after the region), so
    even a 20 ms region carries clock evidence."""

    def __init__(self, index: int, period_s: float = 0.005):
        super().__init__(daemon=True)
        self.index, self.period = index, period_s
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self._lock = threading.Lock()
        self.error = None
        self._nv = self._h = self._names = self._get_reasons = None
        try:
            import pynvml as nv

            nv.nvmlInit()
            self._nv, self._h = nv, nv.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self._h, nv.NVML_CLOCK_SM)
            self._names = {
                getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
                getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake_slowdown",
            }
            self._get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        except Exception as exc:  # NVML missing: report it instead of inventing numbers
            self.error = repr(exc)

    def sample(self):
        if self._nv is None:
            return
        try:
            mhz = self._nv.nvmlDeviceGetClockInfo(self._h, self._nv.NVML_CLOCK_SM)
            mask = self._get_reasons(self._h)
            with self._lock:
                self.samples.append(mhz)
                for bit, name in self._names.items():
                    if mask & bit:
                        self.reasons.add(name)
        except Exception as exc:
            self.error = repr(exc)

    def run(self):
        while not self._stop_evt.is_set():
            self.sample()
            time.sleep(self.period)

    def stop(self) -> dict:
        self._stop_evt.set()
        self.join(timeout=2)
        out = {
            "sm_mhz": statistics.median(self.samples) if self.samples else None,
            "sm_max_mhz": self.max_mhz,
            "reasons": sorted(self.reasons),
            "samples": len(self.samples),
        }
        if self.error:
            out["error"] = self.error
        return out


def measured_hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs: read+write copy)"
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def ncu_traffic_per_launch():
    """dram bytes per step-kernel launch from the committed ncu capture (profiles/traffic.json), or None."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f)
    return None


# -----------------------------------------------------------------------------------------------------
# CPU legs: the one place outside tests/ where oracle/ is executed, as a reported baseline
# -----------------------------------------------------------------------------------------------------
def reference_python_leg(seconds=None, max_steps=None, warm_note="") -> dict | None:
    """The UNMODIFIED Python reference on all host cores (one env per process), in a subprocess (no CUDA there)."""
    script = os.path.join(ROOT, "oracle", "ref_cpu_baseline.py")
    cmd = [sys.executable, script, "--experiment", EXPERIMENT]
    cmd += ["--seconds", str(seconds if seconds is not None else 36000)]
    if max_steps:
        cmd += ["--max-steps", str(max_steps)]
    try:
        proc = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
        if proc.returncode != 0:
            return {"error": proc.stderr.strip().splitlines()[-1] if proc.stderr.strip() else f"exit {proc.returncode}"}
        line = [ln for ln in proc.stdout.splitlines() if ln.startswith("{")][-1]
        return json.loads(line)
    except Exception as exc:
        return {"error": repr(exc)}


def port_leg(envs_per_thread: int, warm_steps: int):
    from marl_ctf_development_b200 import compile_config, experiment_env_config
    from oracle.ctf_oracle import OracleBatch

    threads = host_threads()
    ce = compile_config(**experiment_env_config(EXPERIMENT))
    n_envs = envs_per_thread * threads
    batch = OracleBatch(ce, n_envs, seed=1)
    batch.run(warm_steps, 1, 1, threads)
    return batch, ce, threads, n_envs


def port_sample(n_agents: int, seconds: float, mode: int) -> tuple[float, str]:
    batch, ce, threads, n_envs = port_leg(envs_per_thread=64, warm_steps=5)
    steps, chunk = 0, 10
    t1 = time.perf_counter()
    while time.perf_counter() - t1 < seconds:
        batch.run(chunk, 7 + steps, mode, threads)
        steps += chunk
    dt = time.perf_counter() - t1
    return n_envs * n_agents * steps / dt, f"{n_envs} envs x {steps} steps in {dt:.1f} s on {threads} threads"


def cpu_baseline_sample(n_agents: int) -> dict:
    """Bounded samples of the same workload on the host cores: the unmodified reference (~12 s, the reported baseline)
    and, for context, the C port of its algorithm (oracle/ctf_oracle.c, ~5 s; and with a tuned observation writer)."""
    threads = host_threads()
    port, port_note = port_sample(n_agents, 5.0, 1)
    tuned, tuned_note = port_sample(n_agents, 4.0, 2)
    extra = {
        "port_value": port, "port_sample": "oracle/ctf_oracle.c (line-by-line C port of gridworld_ctf.py), per step obs+meta for all agents then step(): " + port_note,
        "tuned_port_value": tuned, "tuned_port_sample": "same port with a scatter-style observation writer (not the reference's algorithm): " + tuned_note,
    }
    ref = reference_python_leg(seconds=12.0)
    if ref and "error" not in ref:
        return dict({
            "value": ref["agent_steps_per_s"], "unit": UNIT, "cores": ref["processes"], "kind": "reference",
            "sample": f"unmodified gridworld_ctf.GridworldCtf ({ref['reference']}), one env per process x {ref['processes']} processes, "
                      f"{EXPERIMENT}, per step standardise_state + get_env_metadata for all agents then step(): "
                      f"{ref['agent_steps']} agent-steps in {ref['seconds']:.1f} s",
        }, **extra)
    return dict({
        "value": port, "unit": UNIT, "cores": threads, "kind": "port", "sample": extra["port_sample"],
        "reference_unavailable": (ref or {}).get("error", "oracle/_ref not built"),
    }, **extra)


def run_reference_arm(args) -> dict:
    """One 'step' = every host process advances its env by REF_ENV_STEPS_PER_PASS env steps (observations + metadata for
    all agents, then step) — the reference has no batch axis, its parallelism is one env per process (Ray tasks)."""
    from marl_ctf_development_b200 import compile_config, experiment_env_config

    ce = compile_config(**experiment_env_config(EXPERIMENT))
    n = ce.N_AGENTS
    ref = reference_python_leg(max_steps=args.steps * REF_ENV_STEPS_PER_PASS)
    if ref and "error" not in ref:
        value, dt, procs = ref["agent_steps_per_s"], ref["seconds"], ref["processes"]
        kind = "reference"
        sample = (f"unmodified gridworld_ctf.GridworldCtf ({ref['reference']}): {procs} processes x 1 env x "
                  f"{args.steps} passes of {REF_ENV_STEPS_PER_PASS} env steps of {EXPERIMENT} (25 warm-up steps per process), "
                  f"obs+meta for all agents then step()")
        n_envs = procs
    else:
        batch, ce, procs, n_envs = port_leg(envs_per_thread=256, warm_steps=2)
        for w in range(args.warmup):
            batch.run(1, 2 + w, 1, procs)
        t0 = time.perf_counter()
        for k in range(args.steps):
            batch.run(1, 100 + k, 1, procs)
        dt = time.perf_counter() - t0
        value = n_envs * n * args.steps / dt
        kind = "port"
        sample = (f"oracle/ctf_oracle.c (C port; the reference is not importable here: {(ref or {}).get('error')}): {n_envs} envs "
                  f"({procs} threads x 256) x {args.steps} steps of {EXPERIMENT}, obs+meta for all agents then step()")
    cfg = workload_config(args, n_envs, 1)
    cfg["workload"] = cfg["workload"].replace(f"B={n_envs} envs/GPU", f"{n_envs} envs on the host cores (no GPU)")
    return {
        "impl": "reference",
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / max(1, args.steps), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8" if kind == "reference" else "f32", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": procs, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }


def workload_config(args, envs_per_gpu: int, n_gpus: int, experiment: str | None = None) -> dict:
    from marl_ctf_development_b200 import compile_config, experiment_env_config

    exp = experiment or EXPERIMENT
    ce = compile_config(**experiment_env_config(exp))
    G, N, C = ce.GRID_SIZE, ce.N_AGENTS, ce.n_channels
    eb = OBS_ELEM_BYTES[args.obs_dtype]
    dense = not args.no_dense
    out_mb = envs_per_gpu * N * ((C * G * G * eb if dense else 0) + (6 + 2 * N) * 4) / 1e6
    obs_desc = f"{args.obs_dtype} observations [B,{N},{C},{G},{G}]" if dense else "no dense observations"
    if args.packed or args.no_dense:
        obs_desc += f" + packed 1-bit observations [B,{N},{(C * G * G + 31) // 32}] int32"
    return {
        "workload": f"{exp} ({ce.SCENARIO_NAME}, {G}x{G}, {N} agents), B={envs_per_gpu} envs/GPU, "
                    f"uniform random actions 0..8, {obs_desc} + metadata [B,{N},{6 + 2 * N}]",
        "envs_per_gpu": envs_per_gpu,
        "n_agents": N,
        "obs_dtype": args.obs_dtype,
        "parallelism": f"env-sharded x{n_gpus} (no collective in step; NCCL all-reduce of episode stats per episode and at the end of the timed region)",
        "l2": f"per-step output is {out_mb:.0f} MB " + ("(exceeds the 126 MB L2, no explicit flush)" if out_mb > 126 else
              "(fits the 126 MB L2 and is NOT flushed between steps: L2-resident, launch/latency-bound side measurement)"),
    }


# -----------------------------------------------------------------------------------------------------
def dump_env_index(env, torch):
    """Envs whose step outputs --dump-outputs writes: every env when they fit DUMP_BYTES, else a sample drawn with a
    fixed seed, so that two builds run with the same arguments write the same envs."""
    import numpy as np

    per_env = 8 + env.rewards[0].numel() * 4 + 4 + env.meta[0].numel() * 4
    if env.obs is not None:
        per_env += env.obs[0].numel() * 4
    if env.obs_bits is not None:
        per_env += env.obs_bits[0].numel() * 8
    n = min(env.num_envs, DUMP_BYTES // per_env)
    idx = np.sort(np.random.default_rng(0).choice(env.num_envs, n, replace=False))
    return torch.from_numpy(idx).to(env.device)


def take_outputs(env, idx) -> dict:
    """What env.step returned in the step just launched (observations, metadata, rewards, dones and the packed
    observations if enabled), gathered on the device at the envs `idx`."""
    outs = {"obs": env.obs, "meta": env.meta, "rewards": env.rewards, "dones": env.dones, "obs_bits": env.obs_bits}
    return {name: t.index_select(0, idx) for name, t in outs.items() if t is not None}


def write_outputs(path, idx, outs, torch) -> list:
    """DIR/<name>.npy per array: integer arrays as float64 (exact), everything else as float32 (exact for the
    float32, float16, bfloat16 and uint8 buffers).  env_index.npy names the env of every row."""
    import numpy as np

    os.makedirs(path, exist_ok=True)
    names = []
    for name, t in dict(outs, env_index=idx).items():
        t = t.double() if t.dtype in (torch.int32, torch.int64) else t.float()
        np.save(os.path.join(path, name + ".npy"), t.cpu().numpy())
        names.append(name)
    return sorted(names)


def time_steps(env, actions, steps, dev, torch):
    """ms per step of `steps` back-to-back step launches (CUDA events on the launching stream)."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e0.record()
    for i in range(steps):
        env.step(actions[i % actions.shape[0]])
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / steps


def side_config(args, experiment, B, dev, torch, peak, steps=50, graph=False) -> dict:
    """BASELINE.json configs[1] / configs[2] next to the headline: same kernel, other scenario and batch size."""
    from marl_ctf_development_b200 import GridworldCtfGPU, experiment_env_config

    env = GridworldCtfGPU(**experiment_env_config(experiment), num_envs=B, device=dev, seed=args.seed,
                          stats="none" if args.no_stats else "counters", obs_dtype=getattr(torch, args.obs_dtype))
    N, G, C = env.N_AGENTS, env.GRID_SIZE, env.n_channels
    gen = torch.Generator(device=dev).manual_seed(99)
    actions = torch.randint(0, 9, (8, B, N), dtype=torch.uint8, device=dev, generator=gen)
    time_steps(env, actions, 30, dev, torch)
    ms = time_steps(env, actions, steps, dev, torch)
    per = algorithmic_bytes_per_agent_step(G, N, C, OBS_ELEM_BYTES[args.obs_dtype])
    out = {
        "config": workload_config(args, B, 1, experiment)["workload"], "steps": steps, "ms_per_step": ms,
        "value": B * N / ms * 1e3, "unit": UNIT,
        "roofline": {"achieved": per * B * N / ms / 1e6, "peak": peak, "unit": "GB/s", "frac": per * B * N / ms / 1e6 / peak,
                     "algorithmic_bytes_per_agent_step": per},
        "l2": workload_config(args, B, 1, experiment)["l2"],
    }
    if graph:
        g = env.make_step_graph(actions[0], steps_per_replay=10)
        for _ in range(3):
            g.replay()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        e0.record()
        for _ in range(10):
            g.replay()
        e1.record()
        torch.cuda.synchronize(dev)
        out["cuda_graph_ms_per_step"] = e0.elapsed_time(e1) / 100
        out["cuda_graph_value"] = B * N / out["cuda_graph_ms_per_step"] * 1e3
    env.close()
    del env, actions
    torch.cuda.empty_cache()
    return out


def run_ours(args) -> dict | None:
    import torch
    import torch.distributed as dist

    from marl_ctf_development_b200 import GridworldCtfGPU, experiment_env_config

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    B, K, W = args.envs, args.steps, args.warmup
    ec = experiment_env_config(EXPERIMENT)
    env = GridworldCtfGPU(**ec, num_envs=B, device=dev, seed=args.seed, env_id_base=rank * B,
                          stats="none" if args.no_stats else "counters",
                          obs_dtype=getattr(torch, args.obs_dtype), packed_obs=args.packed or args.no_dense,
                          dense_obs=not args.no_dense)
    N, G, C = env.N_AGENTS, env.GRID_SIZE, env.n_channels
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    n_act = 8  # distinct pre-generated action tensors, resident in HBM before the timed region
    actions = torch.randint(0, 9, (n_act, B, N), dtype=torch.uint8, device=dev, generator=gen)
    stats_total = torch.zeros((13, N), dtype=torch.int64, device=dev)
    dump_idx = dump_env_index(env, torch) if args.dump_outputs and rank == 0 else None
    last_outputs = None

    launches = 0

    def reduce_stats():
        nonlocal launches
        if not args.no_stats:
            stats_total.add_(env.stats_sum(all_reduce=world > 1))   # k_stats_sum + (N > 1) one NCCL all-reduce of 13*N int64
            launches += 1

    def one_step(k, keep_outputs=False):
        nonlocal launches, last_outputs
        env.step(actions[k % n_act])
        launches += 1
        if (k + 1) % env.GAME_STEPS == 0:  # episode over: reduce its statistics, start the next one
            if keep_outputs:   # the reset below overwrites the output buffers: gather them first, inside the timed region
                last_outputs = take_outputs(env, dump_idx)
            reduce_stats()
            env.reset()
            launches += 1

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- untimed pre-warm: >= 0.6 s of steps so that clocks, HBM and the allocator are at their steady state even
    # when the driver asks for only a handful of warm-up steps; then the W warm-up steps of the contract
    step_idx = 0
    t_warm = time.perf_counter()
    while time.perf_counter() - t_warm < args.prewarm_s:
        for _ in range(20):
            env.step(actions[step_idx % n_act])
            step_idx += 1
        torch.cuda.synchronize(dev)
    if world > 1 and not args.no_stats:
        env.stats_sum(all_reduce=True)          # NCCL communicator warm-up outside the timed region
    prewarm_steps = step_idx
    env.reset()
    step_idx = 0
    for _ in range(W):
        one_step(step_idx)
        step_idx += 1
    if dump_idx is not None:
        take_outputs(env, dump_idx)   # loads the gather kernels and caches their buffers before the timed region
    graph = None
    if args.graph_steps > 0:
        graph = env.make_step_graph(actions[0], steps_per_replay=args.graph_steps)
    # ---- timed region: K steps, CUDA events on the launching stream, barrier + synchronize on both sides; the
    # statistics of the steps so far are reduced (device sum + NCCL all-reduce over ranks) inside it, after step K
    sampler = ClockSampler(local_rank)   # NVML initialisation BEFORE the barrier: it takes milliseconds and differs per rank,
    sampler.sample()                     # and a late starter would make every other rank wait at the all-reduce below
    barrier()
    sampler.start()
    launches = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    if graph is None:
        for i in range(K):
            one_step(step_idx, keep_outputs=dump_idx is not None and i == K - 1)
            step_idx += 1
    else:
        for _ in range(K // args.graph_steps):
            graph.replay()
        for _ in range(K % args.graph_steps):   # the same step as the captured one, so that exactly K steps are timed
            env.step(actions[0])
        launches = K
    if step_idx % env.GAME_STEPS != 0:
        reduce_stats()
    e1.record()
    if dump_idx is not None and last_outputs is None:
        last_outputs = take_outputs(env, dump_idx)   # nothing has touched the output buffers since the last step
    barrier()
    sampler.sample()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    gpu_launches = launches
    dumped = write_outputs(args.dump_outputs, dump_idx, last_outputs, torch) if dump_idx is not None else None

    # ---- e2e: the same steps through the host-buffer entry point (ctf_step_host): H2D actions from pinned
    # memory and D2H rewards + dones inside the timed region; observations stay in the policy's device buffer
    a_host = [actions[i].cpu().pin_memory() for i in range(n_act)]
    r_host = torch.empty((B, N), dtype=torch.float32).pin_memory()
    d_host = torch.empty((B,), dtype=torch.uint8).pin_memory()
    Ke = max(1, min(K, 200))
    for i in range(3):
        env.step_host(a_host[i % n_act], r_host, d_host)
    barrier()
    t0 = time.perf_counter()
    for i in range(Ke):
        env.step_host(a_host[i % n_act], r_host, d_host)
        if bool(d_host[0]):
            env.reset()
    torch.cuda.synchronize(dev)
    e2e_s = time.perf_counter() - t0

    times = torch.tensor([ms, e2e_s * 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    ms, e2e_ms = float(times[0]), float(times[1])

    result = None
    if rank == 0:
        eb = OBS_ELEM_BYTES[args.obs_dtype]
        agent_steps = world * B * N * K
        value = agent_steps / (ms * 1e-3)
        per_agent_step = algorithmic_bytes_per_agent_step(G, N, C, eb)
        if args.no_dense:
            per_agent_step -= C * G * G * eb
        if args.packed or args.no_dense:
            per_agent_step += env.bits_words_per_agent * 4
        launch_s = ms * 1e-3 / K
        achieved = per_agent_step * B * N / launch_s / 1e9
        peak, peak_src = measured_hbm_peak()
        traffic = ncu_traffic_per_launch()
        kernel = "k_step%s<%s,%s>" % ("_ws" if env.uses_persistent_kernel else "", KERNEL_T[args.obs_dtype], "false" if args.no_stats else "true")
        result = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": DTYPE_TAG[args.obs_dtype], "data": "synthetic",
            "config": dict(workload_config(args, B, world),
                           observation_outputs=("packed only" if args.no_dense else "dense + packed" if args.packed else "dense"),
                           prewarm=f"{prewarm_steps} untimed steps ({args.prewarm_s} s) before the {W} warm-up steps"),
            "clocks": clocks,
            "e2e": {
                "value": world * B * N * Ke / (e2e_ms * 1e-3), "unit": UNIT,
                "h2d_bytes_per_step": B * N, "d2h_bytes_per_step": B * N * 4 + B,
                "steps": Ke, "api": "GridworldCtfGPU.step_host -> ctf_step_host (pinned host actions in, rewards+dones out, moved over PCIe by the step kernel itself; obs/meta stay in HBM: they are the policy's input buffer)",
            },
            "gpu_launches": gpu_launches,
            "roofline": {
                "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic["bytes_per_launch"] if traffic and traffic.get("envs_per_gpu") == B and traffic.get("kernel") == kernel else None,
                "kernel": kernel,
                "algorithmic_bytes_per_agent_step": per_agent_step,
                "bytes_per_launch": per_agent_step * B * N,
                "launch_ms": launch_s * 1e3,
                "peak_source": peak_src,
            },
            "episode_stats_checksum": int(stats_total.sum().item()),
        }
        if dumped is not None:
            result["dump_outputs"] = {"dir": args.dump_outputs, "arrays": dumped, "envs": int(dump_idx.numel()),
                                      "step": "last timed step"}
        if world == 1 and not args.no_side:
            # the write-only ceiling of this GPU, measured now: torch.fill_ of the observation buffer
            if env.obs is not None:
                for _ in range(3):
                    env.obs.fill_(0)
                f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize(dev)
                f0.record()
                for _ in range(10):
                    env.obs.fill_(0)
                f1.record()
                torch.cuda.synchronize(dev)
                fill_gbs = env.obs.numel() * env.obs.element_size() * 10 / f0.elapsed_time(f1) / 1e6
                result["roofline"]["write_only_peak"] = fill_gbs
                result["roofline"]["frac_of_write_only_peak"] = achieved / fill_gbs
                result["roofline"]["write_only_peak_source"] = "torch.fill_ of the observation buffer, measured in this run (the kernel is 99 % writes)"
            # e2e with the observations copied to the host as well (not what a GPU policy does; for completeness)
            if env.obs is not None:
                o_host = torch.empty(env.obs.shape, dtype=env.obs.dtype).pin_memory()
                m_host = torch.empty(env.meta.shape, dtype=env.meta.dtype).pin_memory()
                t0 = time.perf_counter()
                for i in range(3):
                    env.step_host(a_host[i % n_act], r_host, d_host)
                    o_host.copy_(env.obs, non_blocking=True)
                    m_host.copy_(env.meta, non_blocking=True)
                    torch.cuda.synchronize(dev)
                dt = (time.perf_counter() - t0) / 3
                result["e2e_with_obs_d2h"] = {"value": B * N / dt, "unit": UNIT, "d2h_bytes_per_step": int(o_host.numel() * o_host.element_size() + m_host.numel() * 4 + B * N * 4 + B),
                                              "note": "observations + metadata also copied to pinned host memory every step (PCIe-bound)"}
                del o_host, m_host
    env.close()
    del env, actions
    torch.cuda.empty_cache()
    if rank == 0 and world == 1 and not args.no_side and EXPERIMENT == "8_arena":
        peak, _ = measured_hbm_peak()
        result["side_configs"] = [
            side_config(args, "0_the_split", 4096, dev, torch, peak, steps=50, graph=True),     # BASELINE.json configs[1]
            side_config(args, "7_gridlocked", 16384, dev, torch, peak, steps=50),               # BASELINE.json configs[2]
        ]
    if not args.no_side and EXPERIMENT == "8_arena":
        # BASELINE.json configs[4]: self-play rollout with the agent_network-style policy fed from the env's buffers, at the
        # headline B on every rank (stock cuDNN policy inference is ~98 % of this loop; it is outside the hot path)
        import bench_rollout

        ra = bench_rollout.parse_args(["--envs", str(B), "--steps", "3", "--warmup", "1", "--graph", "--channels-last"])
        ro = bench_rollout.measure(ra)
        if rank == 0:
            result["config5_rollout"] = ro
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        result["cpu_baseline"] = cpu_baseline_sample(N)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return result


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--envs", type=int, default=65536, help="envs per GPU (BASELINE.json: 65536)")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--no-stats", action="store_true", help="skip the episode-statistics counters")
    ap.add_argument("--packed", action="store_true", help="side measurement: also write the packed (1 bit/element) observation copy")
    ap.add_argument("--no-dense", action="store_true", help="side measurement: packed observations only (implies --packed)")
    ap.add_argument("--graph-steps", type=int, default=0,
                    help="side measurement: replay a CUDA graph of this many captured steps (launch-bound small batches)")
    ap.add_argument("--experiment", default="8_arena", help="experiment config (side measurements; the headline is 8_arena)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-side", action="store_true", help="skip the side configs / write-only calibration / obs-D2H figure")
    ap.add_argument("--prewarm-s", type=float, default=0.6, help="seconds of untimed steps before the warm-up steps")
    ap.add_argument("--obs-dtype", choices=["float32", "uint8", "float16", "bfloat16"], default="float32",
                    help="float32 is the drop-in default and the headline; the narrower buffers are reported separately")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (obs, meta, rewards, dones; packed obs with --packed) as "
                         "DIR/<name>.npy, for all envs or a fixed seeded sample of them (< 64 MB in all); rank 0 only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU step path (--impl ours)")
    args.warmup = max(3, args.warmup)
    global EXPERIMENT
    EXPERIMENT = args.experiment

    if args.impl == "reference":
        if int(os.environ.get("RANK", "0")) != 0:
            return  # under torchrun only rank 0 runs the CPU arm
        print(json.dumps(run_reference_arm(args)), flush=True)
        return
    result = run_ours(args)
    if result is not None:
        print(json.dumps(result), flush=True)


if __name__ == "__main__":
    main()
