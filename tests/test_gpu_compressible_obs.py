"""The dense observation buffer in compressible device memory (DESIGN §4).

Compression happens between L2 and DRAM and must be invisible: every output of an env on a compressible buffer is
bit-equal to that of a same-seed env on a plain ``torch.empty`` buffer, through steps, resets, graph replays,
``observe``, pickling and caller-bound buffers; torch owns the buffers' lifetime; and the non-compressed path of the
same allocator gives the same results.
"""
import ctypes as C
import gc
import pickle

import pytest
import torch

from marl_ctf_development_b200 import _native, experiment_env_config
from marl_ctf_development_b200.compressible import allocator, compressible_empty, compression_supported, is_compressed

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
DTYPES = [torch.float32, torch.uint8, torch.float16, torch.bfloat16]
OUTPUTS = ("obs", "meta", "rewards", "dones")


def _env(exp, B, plain=False, **kw):
    from marl_ctf_development_b200 import GridworldCtfGPU

    ec = experiment_env_config(exp)
    ec.update(kw.pop("env_overrides", {}))
    env = GridworldCtfGPU(**ec, num_envs=B, device=DEV, stats="counters", **kw)
    if plain:   # rebuild with the caller-bound plain buffer
        shape, dtype = tuple(env.obs.shape), env.obs.dtype
        env.close()
        env = GridworldCtfGPU(**ec, num_envs=B, device=DEV, stats="counters", obs_out=torch.empty(shape, dtype=dtype, device=DEV), **kw)
    return env


def _assert_same(a, b, where):
    for name in OUTPUTS:
        x, y = getattr(a, name), getattr(b, name)
        assert torch.equal(x.view(torch.uint8) if x.dtype != torch.uint8 else x, y.view(torch.uint8) if y.dtype != torch.uint8 else y), \
            f"{where}: {name} differs"


@pytest.fixture
def supported():
    return compression_supported(DEV)


def test_env_buffer_is_compressed_where_the_device_supports_it(supported):
    env = _env("8_arena", 64)
    assert env.obs_compressed == supported
    assert not _env("8_arena", 64, plain=True).obs_compressed


@pytest.mark.parametrize("dtype", DTYPES, ids=lambda d: str(d).split(".")[-1])
@pytest.mark.parametrize("exp", ["0_the_split", "7_gridlocked", "8_arena"])
def test_compressible_buffer_gives_identical_outputs(exp, dtype, supported):
    B, steps, game = 300, 320, 100     # 300 envs: a ragged last CTA; three resets inside the run
    kw = dict(seed=11, obs_dtype=dtype, env_overrides={"GAME_STEPS": game})
    comp, plain = _env(exp, B, **kw), _env(exp, B, plain=True, **kw)
    assert comp.obs_compressed == supported and not plain.obs_compressed
    _assert_same(comp, plain, "after construction")
    g = torch.Generator(device=DEV).manual_seed(5)
    n_dones = 0
    for t in range(steps):
        a = torch.randint(0, 9, (B, comp.N_AGENTS), dtype=torch.uint8, device=DEV, generator=g)
        comp.step(a)
        plain.step(a)
        _assert_same(comp, plain, f"step {t}")
        n_dones += int(comp.dones.sum())
        if (t + 1) % game == 0:
            comp.reset()
            plain.reset()
            _assert_same(comp, plain, f"reset after step {t}")
    assert n_dones > 0


def test_step_graph_replay_and_observe_into_new():
    B = 2048
    comp, plain = _env("8_arena", B, seed=3), _env("8_arena", B, seed=3, plain=True)
    acts = torch.zeros((B, comp.N_AGENTS), dtype=torch.uint8, device=DEV)
    graphs = [comp.make_step_graph(acts, steps_per_replay=2), plain.make_step_graph(acts, steps_per_replay=2)]
    g = torch.Generator(device=DEV).manual_seed(9)
    for r in range(20):
        acts.copy_(torch.randint(0, 9, acts.shape, dtype=torch.uint8, device=DEV, generator=g))
        for gr in graphs:
            gr.replay()
        torch.cuda.synchronize()
        _assert_same(comp, plain, f"replay {r}")
    for flags in (None, [1] * comp.N_AGENTS, [i % 2 for i in range(comp.N_AGENTS)]):
        (oc, mc), (op, mp) = comp.observe(reverse_flags=flags, into_new=True), plain.observe(reverse_flags=flags, into_new=True)
        assert torch.equal(oc, op) and torch.equal(mc, mp)
    comp.observe()
    plain.observe()
    _assert_same(comp, plain, "observe in place")


def test_pickling_round_trip_keeps_a_compressible_buffer(supported):
    B = 512
    env, plain = _env("8_arena", B, seed=4), _env("8_arena", B, seed=4, plain=True)
    g = torch.Generator(device=DEV).manual_seed(2)
    for _ in range(30):
        a = torch.randint(0, 9, (B, env.N_AGENTS), dtype=torch.uint8, device=DEV, generator=g)
        env.step(a)
        plain.step(a)
    copy = pickle.loads(pickle.dumps(env))
    assert copy.obs_compressed == supported
    assert torch.equal(copy.obs, env.obs) and torch.equal(copy.meta, env.meta)
    for t in range(30):
        a = torch.randint(0, 9, (B, env.N_AGENTS), dtype=torch.uint8, device=DEV, generator=g)
        copy.step(a)
        plain.step(a)
        _assert_same(copy, plain, f"step {t} after unpickling")


def test_bind_outputs_with_a_compressible_empty_buffer(supported):
    B = 1024
    env, plain = _env("7_gridlocked", B, seed=6, plain=True), _env("7_gridlocked", B, seed=6, plain=True)
    buf = compressible_empty(tuple(env.obs.shape), env.obs.dtype, DEV)
    assert is_compressed(buf) == supported
    env.bind_outputs(obs=buf)
    assert env.obs is buf and env.obs_compressed == supported
    g = torch.Generator(device=DEV).manual_seed(8)
    for t in range(40):
        a = torch.randint(0, 9, (B, env.N_AGENTS), dtype=torch.uint8, device=DEV, generator=g)
        env.step(a)
        plain.step(a)
        _assert_same(env, plain, f"step {t}")


def test_returned_tensors_stay_valid_after_close():
    B = 4096
    env = _env("8_arena", B, seed=1)
    obs, meta, *_ = env.step(torch.ones((B, env.N_AGENTS), dtype=torch.uint8, device=DEV))
    want_obs, want_meta = obs.clone(), meta.clone()
    env.close()
    del env
    gc.collect()
    torch.cuda.empty_cache()
    junk = compressible_empty(tuple(obs.shape), obs.dtype, DEV).fill_(7)   # would land on freed memory
    assert torch.equal(obs, want_obs) and torch.equal(meta, want_meta)
    del junk


def test_no_device_memory_growth_over_create_close_cycles():
    def cycle():
        env = _env("8_arena", 8192, seed=2)
        for _ in range(5):
            env.step(torch.ones((8192, env.N_AGENTS), dtype=torch.uint8, device=DEV))
        torch.cuda.synchronize()
        env.close()
        del env
        gc.collect()
        torch.cuda.empty_cache()
        return torch.cuda.memory_reserved(DEV), torch.cuda.memory_allocated(DEV)

    first = cycle()
    for i in range(5):
        now = cycle()
        assert now[0] <= first[0] and now[1] <= first[1], f"cycle {i + 2}: reserved/allocated {now} > {first}"


def test_non_compressed_path_of_the_same_allocator_gives_identical_outputs():
    lib = _native.load()
    B = 300
    ref = _env("8_arena", B, seed=12, env_overrides={"GAME_STEPS": 60})
    prev = lib.ctf_compressible_set_enabled(0)
    try:
        pool = torch.cuda.MemPool(allocator())   # a fresh pool: no cached segment of the module's pool is reused
        with torch.cuda.use_mem_pool(pool, torch.device(DEV)):
            buf = torch.empty(tuple(ref.obs.shape), dtype=ref.obs.dtype, device=DEV)
    finally:
        lib.ctf_compressible_set_enabled(prev)
    assert not is_compressed(buf)
    assert sum(seg["total_size"] for seg in pool.snapshot()) >= buf.numel() * buf.element_size()
    env = _env("8_arena", B, seed=12, env_overrides={"GAME_STEPS": 60}, obs_out=buf)
    assert not env.obs_compressed
    _assert_same(env, ref, "after construction")
    g = torch.Generator(device=DEV).manual_seed(3)
    for t in range(130):
        a = torch.randint(0, 9, (B, env.N_AGENTS), dtype=torch.uint8, device=DEV, generator=g)
        env.step(a)
        ref.step(a)
        _assert_same(env, ref, f"step {t}")
        if (t + 1) % 60 == 0:
            env.reset()
            ref.reset()
    env.close()
    del env, buf
    torch.cuda.synchronize()
    del pool
    gc.collect()


def test_native_allocator_entry_points(supported):
    lib = _native.load()
    v = C.c_int(-1)
    _native.check(lib.ctf_compression_supported(0, C.byref(v)))
    assert bool(v.value) == supported
    assert lib.ctf_compression_supported(10_000, C.byref(v)) != 0
    p = lib.ctf_compressible_alloc(1, 0, None)
    assert p
    try:
        _native.check(lib.ctf_mem_is_compressed(C.c_void_p(p), C.byref(v)))
        assert bool(v.value) == supported
        _native.check(lib.ctf_mem_is_compressed(C.c_void_p(p + 100), C.byref(v)))   # any address inside the mapping
        assert bool(v.value) == supported
    finally:
        lib.ctf_compressible_free(C.c_void_p(p), 1, 0, None)
    plain = torch.empty(1024, device=DEV)
    _native.check(lib.ctf_mem_is_compressed(C.c_void_p(plain.data_ptr()), C.byref(v)))
    assert v.value == 0
    _native.check(lib.ctf_mem_is_compressed(None, C.byref(v)))
    assert v.value == 0
    assert lib.ctf_compressible_alloc(-1, 0, None) is None
