"""Delta writes into the env's own observation buffer (DESIGN §4, the observation record).

A step into the buffer the env allocated itself stores only the sectors that changed since the env last wrote it.
Every test runs an env on its own buffer (delta writes) next to a same-seed env bound to a buffer of its caller
(``obs_out=``, always written in full) and requires bit-equal outputs, through every path that writes or may write
the buffer: steps, resets, ``observe``, ``step_host``, graph replays, state restores, torch writes to the buffer, and
writes torch cannot see followed by ``invalidate_obs()``.  The oracle checks the delta env at a few steps.
"""
import copy
import ctypes as C
import pickle

import numpy as np
import pytest
import torch

from marl_ctf_development_b200 import GridworldCtfGPU, _native, compile_config, experiment_env_config
from marl_ctf_development_b200.compressible import compressible_empty
from oracle.ctf_oracle import OracleBatch

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
DTYPES = [torch.float32, torch.bfloat16, torch.float16, torch.uint8]
B = 203   # not a multiple of 4: the last CTA has three envs


def _config(exp, game=None):
    ec = experiment_env_config(exp)
    if game is not None:
        ec["GAME_STEPS"] = game
    return ec


def _pair(exp="8_arena", dtype=torch.float32, packed=False, game=None, seed=3, n=B):
    ec = _config(exp, game)
    kw = dict(num_envs=n, device=DEV, seed=seed, stats="counters", obs_dtype=dtype, packed_obs=packed)
    delta = GridworldCtfGPU(**ec, **kw)
    full = GridworldCtfGPU(**ec, **kw, obs_out=compressible_empty(tuple(delta.obs.shape), dtype, DEV))
    assert (delta._obs_record is not None) == (dtype != torch.uint8) and full._obs_record is None   # uint8: full writes
    return delta, full


def _raw(t):
    return t if t.dtype == torch.uint8 else t.view(torch.uint8)


def _differs(a, b):
    names = ["obs", "meta", "rewards", "dones"] + (["obs_bits"] if a.obs_bits is not None else [])
    return [k for k in names if not torch.equal(_raw(getattr(a, k)), _raw(getattr(b, k)))]


def _same(a, b, where):
    bad = _differs(a, b)
    assert not bad, f"{where}: {bad} differ"


def _actions(g, n_agents, n=B):
    return torch.randint(0, 9, (n, n_agents), dtype=torch.uint8, device=DEV, generator=g)


def _step_both(a, b, g, k=1, where=""):
    for i in range(k):
        act = _actions(g, a.N_AGENTS, a.num_envs)
        a.step(act)
        b.step(act)
        _same(a, b, f"{where} step {i}")


@pytest.mark.parametrize("packed", [False, True], ids=["dense", "packed"])
@pytest.mark.parametrize("dtype", DTYPES, ids=lambda d: str(d).split(".")[-1])
@pytest.mark.parametrize("exp", ["8_arena", "7_gridlocked", "0_the_split"])
def test_two_episodes_equal_full_writes_and_the_oracle(exp, dtype, packed):
    game = 40
    delta, full = _pair(exp, dtype, packed, game=game)
    orc = OracleBatch(compile_config(**_config(exp, game)), B, seed=3)
    _same(delta, full, "after construction")
    g = torch.Generator(device=DEV).manual_seed(1)
    for t in range(2 * game):
        act = _actions(g, delta.N_AGENTS)
        delta.step(act)
        full.step(act)
        r_ref, d_ref = orc.step(act.cpu().numpy())
        _same(delta, full, f"step {t}")
        if t in (0, 1, game - 1, game + 7, 2 * game - 1):
            o_ref, m_ref = orc.observe()
            assert np.array_equal(delta.obs.float().cpu().numpy(), o_ref), f"obs differs from the oracle at step {t}"
            assert np.array_equal(delta.meta.cpu().numpy().view(np.uint32), m_ref.view(np.uint32))
            assert np.array_equal(delta.rewards.cpu().numpy().view(np.uint32), r_ref.view(np.uint32))
        if (t + 1) % game == 0:
            delta.reset()
            full.reset()
            orc.reset()
            _same(delta, full, f"reset after step {t}")


WRITES = {
    "fill": lambda o: o.fill_(1),
    "slice": lambda o: o.__setitem__(5, 1),
    "view_zero": lambda o: o[:, 0].zero_(),
    "copy_random": lambda o: _raw(o).copy_(torch.randint(0, 256, _raw(o).shape, dtype=torch.uint8, device=DEV)),
}


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["float32", "bfloat16"])
@pytest.mark.parametrize("write", sorted(WRITES))
def test_torch_write_to_obs_makes_the_next_step_write_in_full(write, dtype):
    delta, full = _pair(dtype=dtype)
    g = torch.Generator(device=DEV).manual_seed(2)
    _step_both(delta, full, g, 3)
    WRITES[write](delta.obs)
    assert _differs(delta, full) == ["obs"]
    _step_both(delta, full, g, 2, write)


def test_write_torch_cannot_see_needs_invalidate_obs():
    delta, full = _pair()
    g = torch.Generator(device=DEV).manual_seed(3)
    _step_both(delta, full, g, 2)
    delta.obs.data.fill_(1)          # .data has its own version counter: the env cannot notice this write
    delta.invalidate_obs()
    _step_both(delta, full, g, 2, "after invalidate_obs")
    delta.obs.data.fill_(1)
    act = _actions(g, delta.N_AGENTS)
    delta.step(act)
    full.step(act)
    assert _differs(delta, full) == ["obs"], "without invalidate_obs the foreign bytes stay (the documented contract)"
    delta.invalidate_obs()
    _step_both(delta, full, g, 1, "after the late invalidate_obs")


def test_bind_outputs_drops_the_record():
    delta, full = _pair()
    g = torch.Generator(device=DEV).manual_seed(4)
    _step_both(delta, full, g, 2)
    own = delta.obs
    delta.bind_outputs(obs=torch.zeros_like(own))
    assert delta._obs_record is None
    _step_both(delta, full, g, 2, "new buffer")
    own.fill_(1)
    delta.bind_outputs(obs=own)
    assert delta._obs_record is None
    _step_both(delta, full, g, 2, "original buffer again")


def test_observe_then_step():
    delta, full = _pair()
    g = torch.Generator(device=DEV).manual_seed(5)
    _step_both(delta, full, g, 2)
    flags = [1, 0, 1, 1, 0, 0, 1, 0][: delta.N_AGENTS]
    delta.observe(reverse_flags=flags)
    full.observe(reverse_flags=flags)
    _same(delta, full, "observe(reverse_flags)")
    _step_both(delta, full, g, 2, "after observe(reverse_flags)")
    o_new, _ = delta.observe(reverse_flags=flags, into_new=True)
    assert o_new.data_ptr() != delta.obs.data_ptr()
    _step_both(delta, full, g, 2, "after observe(into_new)")


def test_set_state_copy_and_pickle():
    delta, full = _pair()
    other, _ = _pair(seed=9)
    g = torch.Generator(device=DEV).manual_seed(6)
    _step_both(delta, full, g, 3)
    for _ in range(5):
        other.step(_actions(g, other.N_AGENTS))
    st = other.get_state()
    args = (st["grid"], st["pos"], st["hp_q"], st["has_flag"], st["inventory"], st["step"], st["episode"], st["captures"])
    delta.set_state(*args)
    full.set_state(*args)
    _step_both(delta, full, g, 2, "after set_state")
    for clone in (copy.deepcopy(delta), pickle.loads(pickle.dumps(delta))):
        assert clone._obs_record is not None
        act = _actions(g, delta.N_AGENTS)
        clone.step(act)
        ref = copy.deepcopy(full)   # owns its buffer too: compare with a full write of the same state instead
        ref.bind_outputs(obs=compressible_empty(tuple(full.obs.shape), full.obs_dtype, DEV))
        ref.step(act)
        _same(clone, ref, "restored copy")


def test_reset_mid_episode_and_step_host():
    delta, full = _pair()
    g = torch.Generator(device=DEV).manual_seed(7)
    _step_both(delta, full, g, 10)
    delta.reset()
    full.reset()
    _same(delta, full, "reset")
    _step_both(delta, full, g, 2, "after reset")
    r = [torch.empty((B, delta.N_AGENTS), dtype=torch.float32).pin_memory() for _ in range(2)]
    d = [torch.empty((B,), dtype=torch.uint8).pin_memory() for _ in range(2)]
    for i in range(3):
        a = _actions(g, delta.N_AGENTS).cpu().pin_memory()
        delta.step_host(a, r[0], d[0])
        full.step_host(a, r[1], d[1])
        assert _differs(delta, full) in ([], ["rewards", "dones"])   # rewards / dones went to the host buffers
        assert torch.equal(r[0].view(torch.int32), r[1].view(torch.int32)) and torch.equal(d[0], d[1]), f"step_host {i}"
    _step_both(delta, full, g, 2, "after step_host")


def test_step_graph_replays():
    delta, full = _pair()
    g = torch.Generator(device=DEV).manual_seed(8)
    _step_both(delta, full, g, 2)
    act = _actions(g, delta.N_AGENTS)
    gd, gf = delta.make_step_graph(act), full.make_step_graph(act)
    for i in range(3):
        act.copy_(_actions(g, delta.N_AGENTS))
        gd.replay()
        gf.replay()
        _same(delta, full, f"replay {i}")
    delta.obs.fill_(1)               # a torch write between replays
    gd.replay()
    gf.replay()
    _same(delta, full, "replay after a torch write")
    _step_both(delta, full, g, 1, "eager after replays")


def test_graph_capturing_an_in_place_op_and_a_step():
    delta, full = _pair()
    g = torch.Generator(device=DEV).manual_seed(9)
    _step_both(delta, full, g, 2)
    act = _actions(g, delta.N_AGENTS)
    graphs = []
    for env in (delta, full):
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            env.obs.add_(0)
            env.step(act)
        graphs.append(graph)
    for i in range(3):
        act.copy_(_actions(g, delta.N_AGENTS))
        for graph in graphs:
            graph.replay()
        _same(delta, full, f"replay {i}")
    _step_both(delta, full, g, 2, "eager after replays")


def test_poisoned_record_with_a_new_epoch_still_writes_exactly():
    delta, full = _pair()
    g = torch.Generator(device=DEV).manual_seed(10)
    _step_both(delta, full, g, 3)
    delta._obs_record.copy_(torch.randint(-2**31, 2**31 - 1, delta._obs_record.shape, dtype=torch.int32, device=DEV))
    delta.invalidate_obs()
    _step_both(delta, full, g, 3, "after poisoning")


def test_bind_obs_record_rejects_bad_arguments():
    delta, _ = _pair(n=8)
    lib, h = delta._lib, delta._handle
    rec, rep, ep = delta._obs_record, delta._obs_record_epoch, delta._obs_epoch
    p = lambda t, off=0: C.c_void_p(t.data_ptr() + off)   # noqa: E731
    obs = p(delta.obs)
    assert lib.ctf_bind_obs_record(h, obs, None, p(rep), p(ep)) == -1
    assert lib.ctf_bind_obs_record(h, obs, p(rec), p(rep), None) == -1
    assert lib.ctf_bind_obs_record(h, obs, p(rec, 4), p(rep), p(ep)) == -1
    assert lib.ctf_bind_obs_record(h, obs, p(rec), p(rep, 2), p(ep)) == -1
    assert lib.ctf_bind_obs_record(h, obs, p(delta.obs, 64), p(rep), p(ep)) == -1
    assert lib.ctf_bind_obs_record(h, obs, p(rec), p(rec, 16), p(ep)) == -1
    assert b"overlap" in lib.ctf_last_error()
    n = C.c_size_t(0)
    _native.check(lib.ctf_obs_record_size(h, C.byref(n)))
    assert n.value == rec.numel() * 4 and n.value % (8 * 64) == 0
    _native.check(lib.ctf_bind_obs_record(h, obs, p(rec), p(rep), p(ep)))
