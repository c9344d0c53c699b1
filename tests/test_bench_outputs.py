"""bench.py --dump-outputs writes what the last timed step returned, and --steps is the number of timed steps: the dump
is replayed on the CPU oracle from the bench's seeds (env seed 0, actions from a CUDA generator seeded 1234)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import bits, compiled
from oracle.ctf_oracle import OracleBatch

pytestmark = pytest.mark.gpu
ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def _packed(obs_u8):
    """Bit e of an agent's C*G*G block -> bit e % 32 of word e // 32 (the obs_bits layout)."""
    flat = obs_u8.reshape(obs_u8.shape[:2] + (-1,))
    pad = -flat.shape[-1] % 32
    flat = np.concatenate([flat, np.zeros(flat.shape[:2] + (pad,), dtype=np.uint8)], axis=-1)
    return np.packbits(flat, axis=-1, bitorder="little").view("<u4").astype(np.int64)


# 8_arena episodes last 500 steps: with 3 warm-up steps, the 497th timed step ends an episode and a reset follows it
CASES = {"sampled": (1024, 7, 0, False), "graph-remainder": (64, 7, 3, False), "packed": (64, 7, 0, True),
         "episode-end": (64, 497, 0, False)}


@pytest.mark.parametrize("envs,steps,graph_steps,packed", list(CASES.values()), ids=list(CASES))
def test_dump_outputs_are_the_last_timed_step(envs, steps, graph_steps, packed, tmp_path):
    out = tmp_path / "dump"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--envs", str(envs), "--steps", str(steps), "--warmup", "3",
           "--graph-steps", str(graph_steps), "--no-side", "--no-cpu-baseline", "--dump-outputs", str(out)]
    cmd += ["--packed"] if packed else []
    proc = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=tmp_path)
    assert proc.returncode == 0, proc.stderr[-2000:]
    lines = [ln for ln in proc.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["steps"] == steps

    files = sorted(os.listdir(out))
    assert files == sorted(["dones.npy", "env_index.npy", "meta.npy", "obs.npy", "rewards.npy"] + ["obs_bits.npy"] * packed)
    assert sum(os.path.getsize(out / f) for f in files) < 64 * 10**6
    got = {f[:-4]: np.load(out / f) for f in files}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    idx = got["env_index"].astype(np.int64)
    assert np.array_equal(idx, np.unique(idx)) and idx[-1] < envs
    assert (len(idx) < envs) == (envs == 1024)          # 1024 envs of 8_arena exceed the budget and are sampled
    assert d["dump_outputs"]["envs"] == len(idx)

    # the bench's inputs: constructor reset, untimed pre-warm, reset (episode 1), 3 warm-up steps, `steps` timed steps
    ce = compiled("8_arena")
    gen = torch.Generator(device="cuda:0").manual_seed(1234)
    actions = torch.randint(0, 9, (8, envs, ce.N_AGENTS), dtype=torch.uint8, device="cuda:0", generator=gen).cpu().numpy()
    seq = list(range(3)) + (list(range(3, 3 + steps)) if graph_steps == 0 else [0] * steps)
    orc = OracleBatch(ce, envs, seed=0)
    orc.reset()
    for k in seq:
        r_ref, d_ref = orc.step(actions[k % 8])
    o_ref, m_ref = orc.observe()
    assert np.array_equal(got["obs"], o_ref[idx])
    assert np.array_equal(bits(got["meta"]), bits(m_ref[idx]))
    assert np.array_equal(bits(got["rewards"]), bits(r_ref[idx]))
    assert np.array_equal(got["dones"], d_ref[idx].astype(np.float32))
    assert (d_ref.min() == 1) == (3 + steps == ce.GAME_STEPS)
    if packed:
        assert np.array_equal(got["obs_bits"].astype(np.int64) & 0xFFFFFFFF, _packed(o_ref[idx].astype(np.uint8)))
