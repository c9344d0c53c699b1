"""Parity of the CUDA step path (through the C ABI) against the reference's golden traces and the CPU oracle.

Bar: bit-exact grid / positions / HP / flags / inventory / dones / observations / masks / statistics;
rewards and metadata exact in fp32 (compared as bit patterns).
"""
import numpy as np
import pytest
import torch

import traces
from helpers import STATE_KEYS, bits, compiled, golden_ids, golden_traces
from marl_ctf_development_b200 import experiment_env_config
from oracle.ctf_oracle import OracleBatch
from kwarg_cases import CASE_IDS, KWARG_CASES

pytestmark = pytest.mark.gpu


def _env(exp, B, **kw):
    from marl_ctf_development_b200 import GridworldCtfGPU

    ec = experiment_env_config(exp)
    ec.update(kw.pop("env_overrides", {}))
    return GridworldCtfGPU(**ec, num_envs=B, device="cuda:0", **kw)


def _assert_batch_state(env, orc, where, keys=STATE_KEYS + ("step", "episode")):
    st, so = env.get_state(), orc.state()
    if env.hp_float:   # HP lives in doubles, compared bit for bit; the fixed-point field is unused
        keys = tuple(k for k in keys if k != "hp_q")
        assert np.array_equal(st["hp"].view(np.uint64), so["hp"].view(np.uint64)), f"{where}: float HP differs\n got={st['hp']}\nwant={so['hp']}"
    for k in keys:
        got, want = np.asarray(st[k]).astype(np.int64), np.asarray(so[k]).astype(np.int64)
        if not np.array_equal(got, want):
            bad = np.argwhere(got.reshape(got.shape[0], -1) != want.reshape(want.shape[0], -1))[0][0]
            raise AssertionError(f"{where}: {k} differs in env {bad}\n got={got[bad]}\nwant={want[bad]}")


def _assert_obs(env, orc, where, u8=False):
    o_ref, m_ref = orc.observe(u8=u8)
    got = env.obs if env.obs.dtype in (torch.float32, torch.uint8) else env.obs.float()  # {0,1} are exact in fp16/bf16
    assert np.array_equal(got.cpu().numpy(), o_ref), where + ": observations differ"
    assert np.array_equal(bits(env.meta.cpu().numpy()), bits(m_ref)), where + ": metadata differs"


# ---------------------------------------------------------------------------------------------------
# 1. the reference's own traces (tests/golden, generated from the unmodified reference)
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("exp,kind,path", golden_traces(), ids=golden_ids())
def test_cuda_replays_reference_trace(exp, kind, path):
    tr = np.load(path)
    B, slot = 37, 5  # the golden env sits at batch index 5; ragged last CTA on purpose
    env = _env(exp, B, seed=int(tr["seed"]), env_id_base=int(tr["env_id"]) - slot, stats="full")
    rng = np.random.default_rng(1)
    t, oi = 0, 0
    for episode, steps in enumerate(tr["episode_lengths"]):
        if episode:
            env.reset()
        assert tr["obs_steps"][oi] == t
        assert np.array_equal(env.obs[slot].cpu().numpy(), tr["obs"][oi].astype(np.float32)), f"reset obs ep{episode}"
        assert np.array_equal(bits(env.meta[slot].cpu().numpy()), bits(tr["meta"][oi]))
        oi += 1
        for _ in range(int(steps)):
            a = rng.integers(0, 9, (B, env.N_AGENTS)).astype(np.uint8)
            a[slot] = tr["actions"][t]
            obs, meta, rew, done, mask = env.step(torch.from_numpy(a).cuda())
            st = env.get_state()
            for k in STATE_KEYS:
                assert np.array_equal(st[k][slot].astype(np.int64), tr[k][t].astype(np.int64)), f"{exp}/{kind} t={t} {k}"
            assert np.array_equal(bits(rew[slot].cpu().numpy()), bits(tr["rewards"][t])), f"t={t} rewards"
            assert bool(done[slot].item()) == bool(tr["done"][t])
            assert int(st["episode"][slot]) == episode
            t += 1
            if traces.snap_after_step(t, int(st["step"][slot]), env.GAME_STEPS):
                assert tr["obs_steps"][oi] == t
                assert np.array_equal(obs[slot].cpu().numpy(), tr["obs"][oi].astype(np.float32)), f"t={t} obs"
                assert np.array_equal(bits(meta[slot].cpu().numpy()), bits(tr["meta"][oi])), f"t={t} meta"
                oi += 1
        st = env.get_state()
        assert np.array_equal(st["stats"][slot], tr["stats"][episode]), f"stats ep{episode}"
        assert np.array_equal(st["visits"][slot], tr["visits"][episode]), f"visits ep{episode}"
    assert oi == len(tr["obs_steps"])


# ---------------------------------------------------------------------------------------------------
# 2. BASELINE.json configs against the oracle on seeded traces
# ---------------------------------------------------------------------------------------------------
def _run_against_oracle(exp, B, steps, policy, seed, obs_every, stats="counters", obs_dtype=torch.float32, **kw):
    env = _env(exp, B, seed=seed, env_id_base=1000, stats=stats, obs_dtype=obs_dtype, **kw)
    orc = OracleBatch(env.ce, B, seed=seed, env_id_base=1000)
    u8 = obs_dtype == torch.uint8
    _assert_obs(env, orc, "reset", u8)
    rng = np.random.default_rng(seed)
    pol = traces.make_policy(policy, env.ce) if policy != "uniform" else None
    for t in range(steps):
        if pol is None:
            a = rng.integers(0, 9, (B, env.N_AGENTS)).astype(np.uint8)
        else:
            st = orc.state()
            a = np.stack([pol(rng, st["pos"][b], st["has_flag"][b]) for b in range(B)])
        _, _, rew, done, _ = env.step(torch.from_numpy(a).cuda())
        r_ref, d_ref = orc.step(a)
        assert np.array_equal(bits(rew.cpu().numpy()), bits(r_ref)), f"{exp} t={t}: rewards differ"
        assert np.array_equal(done.cpu().numpy(), d_ref), f"{exp} t={t}: dones differ"
        if t % obs_every == 0 or t == steps - 1:
            _assert_batch_state(env, orc, f"{exp} t={t}")
            _assert_obs(env, orc, f"{exp} t={t}", u8)
    st, so = env.get_state(), orc.state()
    if stats != "none":
        assert np.array_equal(st["stats"], so["stats"]), "statistics differ"
        assert np.array_equal(env.stats_sum(all_reduce=False).cpu().numpy(), so["stats"].sum(0)), "stats_sum differs"
    if stats == "full":
        assert np.array_equal(st["visits"], so["visits"])
    return env, orc


def test_config2_the_split_4096_envs_full_episode():
    """BASELINE configs[1]: 0_the_split, B=4096, bit-exact over a whole 500-step episode + 2 steps past done."""
    _run_against_oracle("0_the_split", 4096, 502, "uniform", seed=11, obs_every=125)


def test_config2_the_split_seek_policy_captures():
    env, orc = _run_against_oracle("0_the_split", 256, 500, "seek", seed=12, obs_every=50)
    assert orc.state()["captures"].sum() > 50  # the capture / adjusted / terminal reward paths fired


def test_config3_gridlocked_builder_paths():
    """BASELINE configs[2] semantics: miners (2->3->0, place) and vaulters (wall-jump, HP gate) on 7_gridlocked."""
    env, orc = _run_against_oracle("7_gridlocked", 512, 500, "builder", seed=13, obs_every=50, stats="full")
    s = orc.state()["stats"].sum(0).sum(1)
    assert s[5] > 0 and s[6] > 0 and s[1] > 0 and s[3] > 0  # laid, mined, respawns, captures


def test_config3_gridlocked_16384_envs_uniform():
    _run_against_oracle("7_gridlocked", 16384, 120, "uniform", seed=14, obs_every=119)


def test_config4_arena_seek_and_uniform():
    _run_against_oracle("8_arena", 512, 500, "seek", seed=15, obs_every=50, stats="full")
    _run_against_oracle("8_arena", 2048, 150, "uniform", seed=16, obs_every=75)


def test_uint8_observations_all_alignments():
    # 7_gridlocked: E = 13182 bytes per env -> every 16-byte phase occurs across envs
    _run_against_oracle("7_gridlocked", 67, 60, "builder", seed=17, obs_every=10, obs_dtype=torch.uint8)
    _run_against_oracle("8_arena", 33, 60, "seek", seed=18, obs_every=10, obs_dtype=torch.uint8)


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_half_precision_observation_buffers(dtype):
    """fp16 / bf16 policy input buffers: same {0,1} planes, 8 elements per 128-bit store, every alignment phase."""
    _run_against_oracle("7_gridlocked", 67, 40, "builder", seed=24, obs_every=8, obs_dtype=dtype)
    _run_against_oracle("8_arena", 130, 40, "seek", seed=25, obs_every=8, obs_dtype=dtype)
    _run_against_oracle("0_the_split", 9, 40, "seek", seed=26, obs_every=8, obs_dtype=dtype, stats="full")


@pytest.mark.parametrize("exp", ["1_fence", "2_jailbreak", "3_one_way_out", "4_keyhole", "5_skittles", "6_the_wall"])
def test_other_experiments_against_oracle(exp):
    _run_against_oracle(exp, 128, 260, "builder", seed=19, obs_every=20, stats="full")


@pytest.mark.parametrize("exp", ["alt_exp/1_fence_ii", "alt_exp/2_jailbreak_ii", "alt_exp/3_one_way_out_ii", "alt_exp/4_keyhole_ii",
                                 "alt_exp/5_skittles_ii", "alt_exp/6_the_wall_ii", "alt_exp/8_arena", "alt_exp/8_arena_ii"])
def test_alternative_experiments_against_oracle(exp):
    """The reference's alt_exp/*.py configs (other maps of scenarios.py); the oracle is pinned to the reference on them in
    test_oracle_vs_reference.py::test_alternative_experiment_configs_also_match."""
    _run_against_oracle(exp, 96, 150, "builder", seed=23, obs_every=25, stats="full")


@pytest.mark.parametrize("name,exp,overrides,kind", KWARG_CASES, ids=CASE_IDS)
def test_constructor_keyword_variations(name, exp, overrides, kind):
    """The ctor keywords / team layouts pinned against the reference in test_oracle_vs_reference.py, on the GPU."""
    steps = min(experiment_env_config(exp)["GAME_STEPS"] if "GAME_STEPS" not in overrides else overrides["GAME_STEPS"], 240) + 2
    _run_against_oracle(exp, 96, steps, kind, seed=23, obs_every=15, stats="full", env_overrides=dict(overrides))


@pytest.mark.parametrize("seed", list(range(24)) + list(range(100, 108)))
def test_random_scenarios_and_configs(seed):
    """The random maps / team layouts / HP tables pinned against the reference in test_oracle_vs_reference.py."""
    from marl_ctf_development_b200 import GridworldCtfGPU
    from random_scenarios import random_env_config

    ec = random_env_config(seed)
    B = 33
    dtype = [torch.float32, torch.uint8, torch.bfloat16][seed % 3]
    env = GridworldCtfGPU(**ec, num_envs=B, device="cuda:0", seed=77, env_id_base=seed, stats="full", obs_dtype=dtype)
    orc = OracleBatch(env.ce, B, seed=77, env_id_base=seed)
    pol = traces.make_policy("builder", env.ce)
    rng = np.random.default_rng(seed)
    u8 = dtype == torch.uint8
    _assert_obs(env, orc, f"seed {seed} reset", u8)
    for t in range(ec["GAME_STEPS"] + 2):
        st = orc.state()
        a = np.stack([pol(rng, st["pos"][b], st["has_flag"][b]) for b in range(B)])
        _, _, rew, done, _ = env.step(torch.from_numpy(a).cuda())
        r_ref, d_ref = orc.step(a)
        assert np.array_equal(bits(rew.cpu().numpy()), bits(r_ref)), f"seed {seed} t={t}: rewards differ"
        assert np.array_equal(done.cpu().numpy(), d_ref)
        if t % 10 == 0 or t >= ec["GAME_STEPS"] - 1:
            _assert_batch_state(env, orc, f"seed {seed} t={t}")
            _assert_obs(env, orc, f"seed {seed} t={t}", u8)
    st, so = env.get_state(), orc.state()
    assert np.array_equal(st["stats"], so["stats"]) and np.array_equal(st["visits"], so["visits"])


def test_no_stats_variant_matches():
    _run_against_oracle("8_arena", 130, 80, "seek", seed=20, obs_every=20, stats="none")


# ---------------------------------------------------------------------------------------------------
# 3. full BASELINE size: size-independent properties + a checked subset
# ---------------------------------------------------------------------------------------------------
def test_config4_full_size_properties_and_subset():
    B, steps, seed = 65536, 40, 21
    env = _env("8_arena", B, seed=seed, stats="counters")
    N, G = env.N_AGENTS, env.GRID_SIZE
    sub = np.sort(np.random.default_rng(0).choice(B, 256, replace=False))
    # oracle envs for the subset only (global env id = batch index)
    orcs = [OracleBatch(env.ce, 1, seed=seed, env_id_base=int(b)) for b in sub]
    gen = torch.Generator(device="cuda").manual_seed(5)
    for t in range(steps):
        a = torch.randint(0, 9, (B, N), dtype=torch.uint8, device="cuda", generator=gen)
        _, _, rew, done, _ = env.step(a)
        a_sub = a[torch.from_numpy(sub).cuda()].cpu().numpy()
        for i, o in enumerate(orcs):
            r_ref, _ = o.step(a_sub[i : i + 1])
            assert np.array_equal(bits(rew[int(sub[i])].cpu().numpy()), bits(r_ref[0]))
    st = env.get_state()
    for i, o in enumerate(orcs):
        so = o.state()
        for k in STATE_KEYS:
            assert np.array_equal(st[k][sub[i]].astype(np.int64), so[k][0].astype(np.int64)), (k, int(sub[i]))
    o_ref = np.concatenate([o.observe()[0] for o in orcs])
    assert np.array_equal(env.obs[torch.from_numpy(sub).cuda()].cpu().numpy(), o_ref)
    # properties over all 65536 envs
    grid, pos = torch.from_numpy(st["grid"]).long(), torch.from_numpy(st["pos"]).long()
    tiles = torch.tensor([env.AGENT_TILE_MAP[i] for i in range(N)])
    at_pos = grid[torch.arange(B)[:, None], pos[..., 0], pos[..., 1]]
    assert bool((at_pos == tiles[None]).all()), "every agent's tile sits at its recorded position"
    for tile in range(4, 12):
        assert bool(((grid == tile).sum((1, 2)) == (tiles == tile).sum()).all()), "agent tiles are conserved"
    hp = torch.from_numpy(st["hp_q"])
    mx = torch.tensor([env.ce.cfg.hp_max_q[env.AGENT_TYPES[i]] for i in range(N)])
    assert bool(((hp > 0) & (hp <= mx[None])).all())
    flag = torch.from_numpy(st["has_flag"]).long()
    for team in (0, 1):
        fr, fc = env.FLAG_POSITIONS[team]
        home = grid[:, fr, fc] == 12 + team
        carried = flag[:, [i for i in range(N) if env.AGENT_TEAMS[i] != team]].sum(1)
        assert bool((home == (carried == 0)).all()) and bool((carried <= 1).all()), "a flag is home xor carried by one opponent"
    obs = env.obs
    assert bool((obs[:, :, 0].sum((2, 3)) == 1).all()), "self plane is one-hot"
    nonopen = torch.from_numpy((st["grid"] != 0).sum((1, 2))).cuda().float()
    assert bool((obs[:, :, 1:].sum((2, 3, 4)) == nonopen[:, None]).all()), "8_arena: every non-open cell is in exactly one channel"
    assert bool(((obs == 0) | (obs == 1)).all())
    assert int(st["step"].min()) == steps and int(st["step"].max()) == steps


def test_results_do_not_depend_on_sharding_or_batch_order():
    """Env b of a 1024-env batch equals env b - 512 of a shard created with env_id_base=512 (multi-GPU partition rule)."""
    seed, steps = 22, 60
    full = _env("8_arena", 1024, seed=seed)
    shard = _env("8_arena", 512, seed=seed, env_id_base=512)
    gen = torch.Generator(device="cuda").manual_seed(6)
    for _ in range(steps):
        a = torch.randint(0, 9, (1024, full.N_AGENTS), dtype=torch.uint8, device="cuda", generator=gen)
        full.step(a)
        shard.step(a[512:].contiguous())
    assert torch.equal(full.obs[512:], shard.obs) and torch.equal(full.meta[512:], shard.meta)
    assert torch.equal(full.rewards[512:], shard.rewards)
    sf, ss = full.get_state(), shard.get_state()
    for k in STATE_KEYS:
        assert np.array_equal(sf[k][512:], ss[k])


def test_determinism_and_seed_sensitivity():
    outs = []
    for seed in (30, 30, 31):
        env = _env("8_arena", 300, seed=seed)
        gen = torch.Generator(device="cuda").manual_seed(7)
        for _ in range(50):
            env.step(torch.randint(0, 9, (300, env.N_AGENTS), dtype=torch.uint8, device="cuda", generator=gen))
        outs.append(env.get_state())
    assert all(np.array_equal(outs[0][k], outs[1][k]) for k in STATE_KEYS)
    assert any(not np.array_equal(outs[0][k], outs[2][k]) for k in STATE_KEYS)


# ---------------------------------------------------------------------------------------------------
# 4. edge cases of the boundary
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [1, 3, 4, 5])
def test_tiny_and_ragged_batches(B):
    _run_against_oracle("8_arena", B, 30, "seek", seed=40 + B, obs_every=5, stats="full")


def test_step_from_injected_states_round_trip():
    """set_state -> step equals the oracle stepped from the same injected state (flag carried next to home, low HP)."""
    B = 64
    env = _env("8_arena", B, seed=50, stats="none")
    orc = OracleBatch(env.ce, B, seed=50)
    rng = np.random.default_rng(3)
    for t in range(25):
        a = rng.integers(0, 9, (B, env.N_AGENTS)).astype(np.uint8)
        orc.step(a)
    so = orc.state()
    so["hp_q"] = np.maximum(1, so["hp_q"] - rng.integers(0, 30, so["hp_q"].shape)).astype(np.int32)  # many agents near death
    so["step"][:] = 497  # three steps before the terminal step
    args = (so["grid"], so["pos"], so["hp_q"], so["has_flag"], so["inventory"], so["step"], so["episode"], so["captures"])
    orc.set_state(*args)
    env.set_state(*args)
    for t in range(6):
        a = rng.integers(0, 9, (B, env.N_AGENTS)).astype(np.uint8)
        _, _, rew, done, _ = env.step(torch.from_numpy(a).cuda())
        r_ref, d_ref = orc.step(a)
        assert np.array_equal(bits(rew.cpu().numpy()), bits(r_ref))
        assert np.array_equal(done.cpu().numpy(), d_ref)
        _assert_batch_state(env, orc, f"injected t={t}")
        _assert_obs(env, orc, f"injected t={t}")
    assert done.all()


def test_out_of_range_action_faults_like_keyerror():
    env = _env("0_the_split", 8, seed=1, validate_actions=True)
    a = torch.full((8, env.N_AGENTS), 4, dtype=torch.uint8, device="cuda")
    env.step(a)
    a[3, 1] = 9
    with pytest.raises(KeyError):
        env.step(a)
    for bad in (-1, 300):          # wider integer inputs: out-of-range values must not be folded into valid actions
        b = torch.full((8, env.N_AGENTS), 4, dtype=torch.int64, device="cuda")
        b[0, 0] = bad
        with pytest.raises(KeyError):
            env.step(b)


def test_observe_with_explicit_reverse_flags_and_symmetry():
    env = _env("8_arena", 16, seed=2)
    orc = OracleBatch(env.ce, 16, seed=2)
    rng = np.random.default_rng(4)
    for _ in range(30):
        a = rng.integers(0, 9, (16, env.N_AGENTS)).astype(np.uint8)
        env.step(torch.from_numpy(a).cuda())
        orc.step(a)
    for flags in ([0] * 8, [1] * 8, [1, 0, 0, 1, 1, 0, 1, 0]):
        obs, meta = env.observe(reverse_flags=flags, into_new=True)
        o_ref, m_ref = orc.observe(reverse_flags=flags)
        assert np.array_equal(obs.cpu().numpy(), o_ref)
        assert np.array_equal(bits(meta.cpu().numpy()), bits(m_ref))


def test_reverse_team1_actions_folded_into_step():
    B = 32
    plain = _env("0_the_split", B, seed=3)
    folded = _env("0_the_split", B, seed=3, reverse_team1_actions=True)
    lut = plain.reversed_action_lut()
    team1 = torch.tensor([plain.AGENT_TEAMS[i] == 1 for i in range(plain.N_AGENTS)], device="cuda")
    gen = torch.Generator(device="cuda").manual_seed(8)
    for _ in range(40):
        a = torch.randint(0, 9, (B, plain.N_AGENTS), device="cuda", generator=gen)
        plain.step(torch.where(team1[None], lut[a], a).to(torch.uint8))  # what ppo.py:84-93 / utils.py:549 do on the host
        folded.step(a.to(torch.uint8))
    assert torch.equal(plain.obs, folded.obs) and torch.equal(plain.rewards, folded.rewards)


def test_step_host_matches_device_step():
    B = 48
    dev = _env("8_arena", B, seed=4)
    host = _env("8_arena", B, seed=4)
    a_h = torch.empty((B, dev.N_AGENTS), dtype=torch.uint8).pin_memory()
    r_h = torch.empty((B, dev.N_AGENTS), dtype=torch.float32).pin_memory()
    d_h = torch.empty((B,), dtype=torch.uint8).pin_memory()
    rng = np.random.default_rng(9)
    for _ in range(20):
        a_h.copy_(torch.from_numpy(rng.integers(0, 9, (B, dev.N_AGENTS)).astype(np.uint8)))
        dev.step(a_h.cuda())
        host.step_host(a_h, r_h, d_h)
        assert torch.equal(dev.rewards.cpu(), r_h) and torch.equal(dev.dones.cpu(), d_h)
    assert torch.equal(dev.obs, host.obs)
    # pageable host buffers take the staged-copy path and give the same results
    pa, pr, pd = torch.empty((B, dev.N_AGENTS), dtype=torch.uint8), torch.empty((B, dev.N_AGENTS)), torch.empty((B,), dtype=torch.uint8)
    for _ in range(5):
        pa.copy_(torch.from_numpy(rng.integers(0, 9, (B, dev.N_AGENTS)).astype(np.uint8)))
        dev.step(pa.cuda())
        host.step_host(pa, pr, pd)
        assert torch.equal(dev.rewards.cpu(), pr) and torch.equal(dev.dones.cpu(), pd)
    assert torch.equal(dev.obs, host.obs)


def test_outputs_written_into_caller_buffers():
    B = 20
    env = _env("0_the_split", B, seed=5)
    N, C, G, M = env.N_AGENTS, env.n_channels, env.GRID_SIZE, env.meta_size
    big = torch.zeros((3, B, N, C, G, G), device="cuda")
    env.bind_outputs(obs=big[1])
    env.step(torch.full((B, N), 4, dtype=torch.uint8, device="cuda"))
    assert float(big[1].sum()) > 0 and float(big[0].sum()) == 0 and float(big[2].sum()) == 0


def test_action_mask_and_dims():
    env = _env("8_arena", 4, seed=6)
    assert tuple(env.action_mask.shape) == (4, 8, 9)
    want = [[1] * 5 + [0] * 4 if env.AGENT_TYPES[i] in (0, 1) else [1] * 9 for i in range(8)]
    assert env.action_mask[2].cpu().tolist() == want
    assert env.get_env_dims() == ((14, 15, 15), (13, 15, 15), (22,), (115,))


def test_half_rounding_on_device_matches_numpy():
    """metadata[0:2] go through float16 (gridworld_ctf.py:1044): check every step fraction and many capture ratios."""
    env = _env("8_arena", 1, seed=7)
    st = env.get_state()
    for step, c0, c1 in [(s, (s * 7) % 61, (s * 13) % 59) for s in range(0, 1001, 3)]:
        st["step"][:] = step
        st["captures"][:] = (c0, c1)
        env.set_state(st["grid"], st["pos"], st["hp_q"], st["has_flag"], st["inventory"], st["step"], st["episode"], st["captures"])
        _, meta = env.observe(into_new=True)
        m = meta[0].cpu().numpy()
        assert m[0, 0] == np.float32(np.float16(step / 500))
        assert m[0, 1] == np.float32(np.float16((c0 + 1) / (c1 + 1)))
        assert m[1, 1] == np.float32(np.float16((c1 + 1) / (c0 + 1)))


def test_step_is_cuda_graph_capturable():
    """A captured step replays bit-identically to eager steps (one warm-up step is taken by make_step_graph)."""
    B = 512
    eager = _env("0_the_split", B, seed=8, stats="counters")
    graphed = _env("0_the_split", B, seed=8, stats="counters")
    acts = torch.zeros((B, eager.N_AGENTS), dtype=torch.uint8, device="cuda")
    gen = torch.Generator(device="cuda").manual_seed(9)
    acts.copy_(torch.randint(0, 9, acts.shape, dtype=torch.uint8, device="cuda", generator=gen))
    graph = graphed.make_step_graph(acts)       # leaves the env state untouched
    assert int(graphed.step_counts().max()) == 0
    for _ in range(50):
        acts.copy_(torch.randint(0, 9, acts.shape, dtype=torch.uint8, device="cuda", generator=gen))
        eager.step(acts)
        graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(eager.obs, graphed.obs) and torch.equal(eager.rewards, graphed.rewards)
    se, sg = eager.get_state(), graphed.get_state()
    for k in STATE_KEYS + ("step", "stats"):
        assert np.array_equal(se[k], sg[k]), k


def _pack_reference(obs_u8, wpa):
    """numpy restatement of the packed layout: bit e of an agent's C*G*G block -> bit e % 32 of word e // 32."""
    lead = obs_u8.shape[:-3]
    flat = obs_u8.reshape(lead + (-1,))
    pad = wpa * 32 - flat.shape[-1]
    flat = np.concatenate([flat, np.zeros(lead + (pad,), dtype=np.uint8)], axis=-1)
    return np.packbits(flat, axis=-1, bitorder="little").view("<u4").astype(np.int64)


@pytest.mark.parametrize("exp", ["8_arena", "7_gridlocked", "0_the_split"])
def test_packed_observations_and_unpack_round_trip(exp):
    """obs_bits == packbits(standardise_state) per agent, and ctf_unpack_obs gives the dense tensors back in every dtype."""
    B = 70
    env = _env(exp, B, seed=31, packed_obs=True)
    orc = OracleBatch(env.ce, B, seed=31)
    rng = np.random.default_rng(5)
    pol = traces.make_policy("builder", env.ce)
    for t in range(45):
        st = orc.state()
        a = np.stack([pol(rng, st["pos"][b], st["has_flag"][b]) for b in range(B)])
        env.step(torch.from_numpy(a).cuda())
        orc.step(a)
        if t % 11 == 0:
            o_ref, _ = orc.observe(u8=True)
            want = _pack_reference(o_ref, env.bits_words_per_agent)
            got = env.obs_bits.cpu().numpy().astype(np.int64) & 0xFFFFFFFF
            assert np.array_equal(got, want), f"{exp} t={t}: packed observations differ"
            assert np.array_equal(env.obs.cpu().numpy(), o_ref.astype(np.float32))
    for dtype in (torch.float32, torch.uint8, torch.float16, torch.bfloat16):
        dense = env.unpack_obs(env.obs_bits, dtype=dtype)
        assert tuple(dense.shape) == tuple(env.obs.shape) and dense.dtype == dtype
        assert torch.equal(dense.float(), env.obs)
    # a gathered minibatch with an odd number of blocks and an unaligned output slice
    idx = torch.tensor([3, 17, 4, 60, 9], device="cuda")
    mb = env.obs_bits[idx][:, 1:]
    big = torch.zeros((mb.shape[0] * mb.shape[1] * env.n_channels * env.GRID_SIZE**2 + 3,), device="cuda")
    view = big[3:].view(mb.shape[0], mb.shape[1], env.n_channels, env.GRID_SIZE, env.GRID_SIZE)
    env.unpack_obs(mb, out=view)
    assert torch.equal(view, env.obs[idx][:, 1:]) and float(big[:3].abs().sum()) == 0.0


def test_packed_only_env_skips_the_dense_buffer():
    B = 40
    dense = _env("8_arena", B, seed=32)
    packed = _env("8_arena", B, seed=32, packed_obs=True, dense_obs=False)
    assert packed.obs is None
    gen = torch.Generator(device="cuda").manual_seed(3)
    for _ in range(30):
        a = torch.randint(0, 9, (B, 8), dtype=torch.uint8, device="cuda", generator=gen)
        dense.step(a)
        packed.step(a)
    assert torch.equal(packed.unpack_obs(packed.obs_bits), dense.obs)
    assert torch.equal(packed.meta, dense.meta) and torch.equal(packed.rewards, dense.rewards)


def _case_overrides(name):
    return dict([c for c in KWARG_CASES if c[0] == name][0][2])


@pytest.mark.parametrize("exp,B,case", [("8_arena", 2048, None), ("7_gridlocked", 2048, None), ("0_the_split", 4096, None),
                                        ("8_arena", 2048, "one_hit_kills_arena"), ("7_gridlocked", 1024, "glass_cannons_gridlocked")])
def test_soak_three_episodes_with_resets(exp, B, case):
    """Long differential run: 3 episodes x 500 steps with resets in between, flag-seeking/builder actions, every reward
    and done compared each step, full state + observations + statistics at checkpoints.  Rare paths must have fired."""
    seed = 33
    env = _env(exp, B, seed=seed, stats="counters", env_overrides=_case_overrides(case) if case else {})
    orc = OracleBatch(env.ce, B, seed=seed)
    rng = np.random.default_rng(seed)
    totals = np.zeros((13,), dtype=np.int64)
    for episode in range(3):
        if episode:
            env.reset()
            orc.reset()
        for t in range(500):
            st = orc.state() if t % 1 == 0 else st
            a = traces.seek_actions_batch(rng, env.ce, st["pos"], st["has_flag"], eps=0.3 + 0.1 * episode, second_p=0.3 + 0.15 * episode)
            _, _, rew, done, _ = env.step(torch.from_numpy(a).cuda())
            r_ref, d_ref = orc.step(a)
            if t % 5 == 0 or t >= 497:
                assert np.array_equal(bits(rew.cpu().numpy()), bits(r_ref)), f"{exp} ep{episode} t={t}: rewards differ"
                assert np.array_equal(done.cpu().numpy(), d_ref)
            if t % 100 == 99:
                _assert_batch_state(env, orc, f"{exp} ep{episode} t={t}")
                _assert_obs(env, orc, f"{exp} ep{episode} t={t}")
        so = orc.state()
        assert np.array_equal(env.get_state()["stats"], so["stats"]), f"{exp} ep{episode}: statistics differ"
        totals += so["stats"].sum(0).sum(1)
    # tag, respawn, pickup, capture, dispossession fired in every scenario; mining / placing where miners exist
    assert (totals[:5] > 0).all(), totals
    if 3 in env.AGENT_TYPES.values():
        assert totals[5] > 0 and totals[6] > 0, totals


def test_terminal_reward_is_not_fused_multiply_add():
    """Regression found by the soak test: a punished agent of the winning team at the terminal step gets
    -0.5 + margin * 0.1 with two roundings (exactly 0.0 for margin 5), never an FMA (2.8e-17)."""
    B = 8
    env = _env("8_arena", B, seed=1, stats="none")
    orc = OracleBatch(env.ce, B, seed=1)
    so = orc.state()
    grid, pos, flag = so["grid"].copy(), so["pos"].copy(), so["has_flag"].copy()
    # agent 7 (team 1 scout) stands two cells above its own flag (12, 7) carrying team 0's flag
    for b in range(B):
        r, c = pos[b, 7]
        grid[b, r, c] = 0
        pos[b, 7] = (10, 7)
        grid[b, 10, 7] = 8          # team-1 scout tile
        grid[b, 2, 7] = 1           # team 0's flag cell holds a block tile while the flag is carried (:587)
        flag[b, 7] = 1
    so["step"][:] = 499
    caps = np.tile(np.array([[6, 0]]), (B, 1))
    caps[1] = (3, 0)
    caps[2] = (8, 0)
    args = (grid, pos, so["hp_q"], flag, so["inventory"], so["step"], so["episode"], caps)
    orc.set_state(*args)
    env.set_state(*args)
    a = np.full((B, 8), 4, dtype=np.uint8)
    a[:, 7] = 1                     # D: (10,7) -> (11,7), within 1 of the own flag -> capture
    _, _, rew, done, _ = env.step(torch.from_numpy(a).cuda())
    r_ref, d_ref = orc.step(a)
    assert orc.state()["captures"][0].tolist() == [6, 1] and bool(d_ref.all())
    assert r_ref[0, 0] == 0.0 and r_ref[0, 7] == 1.0       # -0.5 + 5 * 0.1 == 0.0 exactly in the reference
    assert np.array_equal(bits(rew.cpu().numpy()), bits(r_ref)), (rew.cpu().numpy(), r_ref)


def test_visitation_maps_wrap_and_non_default_stream():
    """uint8 visitation maps wrap at 256 (standing still for 300 steps); the same run on a side stream gives the same state."""
    B = 33
    a = torch.full((B, 4), 4, dtype=torch.uint8, device="cuda")
    env0 = _env("0_the_split", B, seed=3, stats="full")
    orc = OracleBatch(env0.ce, B, seed=3)
    side = torch.cuda.Stream()
    env1 = _env("0_the_split", B, seed=3, stats="full")
    for t in range(300):
        env0.step(a)
        orc.step(a.cpu().numpy())
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for t in range(300):
            env1.step(a)
    side.synchronize()
    torch.cuda.synchronize()
    s0, s1, so = env0.get_state(), env1.get_state(), orc.state()
    assert np.array_equal(s0["visits"], so["visits"]) and int(s0["visits"].max()) == 301 % 256
    for k in STATE_KEYS + ("stats", "visits", "step"):
        assert np.array_equal(s0[k], s1[k]), k
    assert torch.equal(env0.obs, env1.obs)


def test_closed_env_fails_loudly():
    from marl_ctf_development_b200._native import NativeError

    env = _env("0_the_split", 4, seed=1)
    env.close()
    with pytest.raises(NativeError):
        env.step(torch.zeros((4, 4), dtype=torch.uint8, device="cuda"))


@pytest.mark.parametrize("exp", ["0_the_split", "1_fence", "2_jailbreak", "3_one_way_out", "4_keyhole", "5_skittles", "6_the_wall", "7_gridlocked", "8_arena"])
def test_soak_every_experiment_full_episode_with_visits(exp):
    """Every experiment script's config: 1 024 envs, one full episode + 2 steps past done, statistics and visitation maps."""
    B, seed = 1024, 44
    env = _env(exp, B, seed=seed, stats="full", obs_dtype=torch.uint8)
    orc = OracleBatch(env.ce, B, seed=seed)
    rng = np.random.default_rng(seed)
    for t in range(env.GAME_STEPS + 2):
        st = orc.state()
        a = traces.seek_actions_batch(rng, env.ce, st["pos"], st["has_flag"], eps=0.35, second_p=0.5)
        _, _, rew, done, _ = env.step(torch.from_numpy(a).cuda())
        r_ref, d_ref = orc.step(a)
        if t % 4 == 0 or t >= env.GAME_STEPS - 2:
            assert np.array_equal(bits(rew.cpu().numpy()), bits(r_ref)), f"{exp} t={t}: rewards differ"
            assert np.array_equal(done.cpu().numpy(), d_ref)
        if t % 125 == 124 or t >= env.GAME_STEPS - 1:
            _assert_batch_state(env, orc, f"{exp} t={t}")
            _assert_obs(env, orc, f"{exp} t={t}", u8=True)
    st, so = env.get_state(), orc.state()
    assert np.array_equal(st["stats"], so["stats"]) and np.array_equal(st["visits"], so["visits"])


def test_step_graph_replay_with_dense_and_packed_outputs():
    """Captured steps writing dense + packed observations replay like eager steps; the packed copy unpacks to the dense one."""
    B = 2000
    eager = _env("8_arena", B, seed=8, stats="counters", packed_obs=True)
    graphed = _env("8_arena", B, seed=8, stats="counters", packed_obs=True, validate_actions=True)
    acts = torch.zeros((B, 8), dtype=torch.uint8, device="cuda")
    gen = torch.Generator(device="cuda").manual_seed(9)
    graph = graphed.make_step_graph(acts, steps_per_replay=1)   # validate_actions is suspended inside the capture
    for _ in range(25):
        acts.copy_(torch.randint(0, 9, acts.shape, dtype=torch.uint8, device="cuda", generator=gen))
        eager.step(acts)
        graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(eager.obs, graphed.obs) and torch.equal(eager.obs_bits, graphed.obs_bits)
    assert torch.equal(eager.unpack_obs(eager.obs_bits), eager.obs)
    se, sg = eager.get_state(), graphed.get_state()
    for k in STATE_KEYS + ("step", "stats"):
        assert np.array_equal(se[k], sg[k]), k


# ---------------------------------------------------------------------------------------------------
# defined behaviour where the reference raises: a lethal tag with a full spawn window (gridworld_ctf.py:771)
# ---------------------------------------------------------------------------------------------------
def test_respawn_into_a_full_spawn_window_sets_the_fault_bit():
    from marl_ctf_development_b200 import _native

    B = 6
    env = _env("0_the_split", B, seed=3, env_id_base=50, env_overrides={"AGENT_TYPE_DAMAGE": {0: 100, 1: 100, 2: 100, 3: 100}, "TAG_PROBABILITY": 1.0})
    ce = env.ce
    orc = OracleBatch(ce, B, seed=3, env_id_base=50)
    st = orc.state()
    G = ce.GRID_SIZE
    grid = st["grid"].copy()
    pos = st["pos"].copy()
    # wall in team 1's spawn window completely, and put agents 0 (team 0) and 1 (team 1) next to each other elsewhere
    sx, sy = ce.SPAWN_POSITIONS[1]
    for b in range(B):
        for i in range(ce.N_AGENTS):
            grid[b, pos[b, i, 0], pos[b, i, 1]] = 0
        grid[b, max(sx - 1, 0):sx + 2, max(sy - 1, 0):sy + 2] = 1
        free = [(r, c) for r in range(G) for c in range(G - 1) if grid[b, r, c] == 0 and grid[b, r, c + 1] == 0]
        cells = [free[0], (free[0][0], free[0][1] + 1)] + [f for f in free[4:] if f[0] != free[0][0]][: ce.N_AGENTS - 2]
        for i, (r, c) in enumerate(cells):
            pos[b, i] = (r, c)
            grid[b, r, c] = ce.AGENT_TILE_MAP[i]
    args = dict(grid=grid, pos=pos, hp_q=st["hp_q"], has_flag=st["has_flag"], inventory=st["inventory"], step=st["step"],
                episode=st["episode"], captures=st["captures"])
    orc.set_state(**args)
    env.set_state(**args)
    a = np.full((B, ce.N_AGENTS), 4, dtype=np.uint8)
    _, _, rew, done, _ = env.step(torch.from_numpy(a).cuda())
    r_ref, _ = orc.step(a)
    assert np.array_equal(bits(rew.cpu().numpy()), bits(r_ref))
    _assert_batch_state(env, orc, "blocked respawn")
    assert (orc.state()["hp_q"] <= 0).any()                      # a victim was left in place with HP <= 0
    assert orc.take_faults() & _native.FAULT_RESPAWN_BLOCKED
    assert env.take_faults() == _native.FAULT_RESPAWN_BLOCKED and env.take_faults() == 0
    # later steps keep agreeing with the oracle, fault word included
    for _ in range(3):
        env.step(torch.from_numpy(a).cuda())
        orc.step(a)
        assert env.take_faults() == orc.take_faults()
    _assert_batch_state(env, orc, "after blocked respawns")
    # validate_actions=True turns the bit into the reference's exception type
    strict = _env("0_the_split", B, seed=3, env_id_base=50, validate_actions=True,
                  env_overrides={"AGENT_TYPE_DAMAGE": {0: 100, 1: 100, 2: 100, 3: 100}, "TAG_PROBABILITY": 1.0})
    strict.set_state(**args)
    with pytest.raises(ValueError):
        strict.step(torch.from_numpy(a).cuda())


def test_get_state_of_selected_envs_and_current_device_is_preserved():
    env = _env("7_gridlocked", 300, seed=4)
    a = torch.randint(0, 9, (300, env.N_AGENTS), dtype=torch.uint8, device="cuda")
    for _ in range(5):
        env.step(a)
    full = env.get_state()
    one = env.get_state(env_index=17)
    some = env.get_state(env_index=slice(10, 20))
    for k in full:
        assert np.array_equal(one[k], full[k][17:18]) and np.array_equal(some[k], full[k][10:20]), k
    assert np.array_equal(env.get_state(env_index=-1)["grid"], full["grid"][-1:])
    with pytest.raises(IndexError):
        env.get_state(env_index=300)
    if torch.cuda.device_count() > 1:   # entry points run on the env's device and restore the caller's (ADVICE r1)
        with torch.cuda.device(1):
            env.step(a)
            assert torch.cuda.current_device() == 1
            assert torch.empty(1, device="cuda").device.index == 1
    assert torch.cuda.current_device() == 0


# ---------------------------------------------------------------------------------------------------
# pickling / deepcopy: Ray ships pickled env copies to its workers (league_training.py:686-687)
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("overrides", [{}, {"AGENT_HP_HEALING_PER_STEP": 0.1, "AGENT_TYPE_DAMAGE": {0: 0.3, 1: 0.7, 2: 0.9, 3: 0.35}}],
                         ids=["fixed_point_hp", "float_hp"])
def test_env_pickles_mid_episode_and_the_copy_continues_identically(overrides):
    import copy
    import pickle

    env = _env("7_gridlocked", 40, seed=9, env_id_base=300, stats="full", packed_obs=True, env_overrides=overrides)
    gen = torch.Generator(device="cuda").manual_seed(4)
    acts = torch.randint(0, 9, (60, 40, env.N_AGENTS), dtype=torch.uint8, device="cuda", generator=gen)
    for t in range(25):
        env.step(acts[t])
    clone = pickle.loads(pickle.dumps(env))
    assert clone._handle.value != env._handle.value and clone.obs.data_ptr() != env.obs.data_ptr()
    assert torch.equal(clone.obs, env.obs) and torch.equal(clone.meta, env.meta) and torch.equal(clone.obs_bits, env.obs_bits)
    twin = copy.deepcopy(clone)
    for t in range(25, 60):
        a, b, c = env.step(acts[t]), clone.step(acts[t]), twin.step(acts[t])
        for x, y, z in zip(a[:4], b[:4], c[:4]):
            assert torch.equal(x, y) and torch.equal(x, z), t
    s0, s1 = env.get_state(), twin.get_state()
    for k in s0:
        assert np.array_equal(s0[k], s1[k]), k


def test_single_env_view_deepcopies_like_the_reference_env():
    import copy

    from marl_ctf_development_b200 import GridworldCtf

    env = GridworldCtf(**experiment_env_config("8_arena"), seed=2, env_id=5)
    rng = np.random.default_rng(0)
    for _ in range(12):
        env.step(rng.integers(0, 9, 8).tolist())
    other = copy.deepcopy(env)
    assert other.env_step_count == 12 and other.agent_positions == env.agent_positions
    for _ in range(20):
        a = rng.integers(0, 9, 8).tolist()
        g0, r0, d0 = env.step(a)
        g1, r1, d1 = other.step(a)
        assert np.array_equal(g0, g1) and r0 == r1 and d0 == d1
    assert np.array_equal(env.standardise_state(3, reverse_grid=True), other.standardise_state(3, reverse_grid=True))
    assert env.metrics["agent_tag_count"] == other.metrics["agent_tag_count"]
