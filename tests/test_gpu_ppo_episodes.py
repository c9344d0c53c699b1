"""PPO across episode boundaries on the GPU: ctf_gae_dones (k_gae<true>) bit for bit against reference_advantages with
dones, its rejections and graph replay; collect_rollout(reset=False) continuing episodes bit for bit like one long
rollout and like a manual replay across step GAME_STEPS; and PackedPPO(rollout_steps=...) over several updates."""
import ctypes as C
import math

import pytest
import torch

from test_gpu_fused_policy import DEV, _policy, _team
from test_gpu_ppo import _args, _env, _gae_inputs, _ro
from marl_ctf_development_b200 import PackedPPO
from marl_ctf_development_b200.fused_policy import FusedPolicy
from marl_ctf_development_b200.ppo import advantages, reference_advantages
from marl_ctf_development_b200.rollout import collect_rollout
from oracle import ref_shim as rs
from test_ppo_episodes_spec import _cleanrl64

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def small_env():
    return _env(2)


# ---------------------------------------------------------------------------------------------------- 1. bit equality
def _dones(kind, T, apt, B, seed):
    """fp32 [T*apt, B]: boundaries on one row, on every row, or on random (agent, env) entries with random nonzero
    values; -0.0 stands in for some of the zeros (it is not a boundary)."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    d = torch.zeros((T, apt, B), device=DEV)
    if kind == "every":
        d[:] = 1
    elif kind == "random":
        val = torch.rand((T, apt, B), generator=g, device=DEV) * 4 - 2
        d = torch.where(torch.rand((T, apt, B), generator=g, device=DEV) < 0.1, val, torch.full_like(val, -0.0))
    else:
        d[{"row0": 0, "row1": min(1, T - 1), "last": T - 1}[kind]] = 1
    return d.reshape(T * apt, B)


@pytest.mark.parametrize("kind", ["row0", "row1", "last", "every", "random"])
@pytest.mark.parametrize("shape", [(1, 1, 1), (7, 3, 33), (32, 4, 4101), (500, 4, 65536)])
def test_gae_dones_is_bit_equal_to_the_reference(small_env, shape, kind):
    T, apt, B = shape
    r, v, nv = _gae_inputs(T, apt, B, T * 5 + B, False)
    d = _dones(kind, T, apt, B, T + B)
    adv, ret = advantages(small_env, _ro(r, v), nv, 0.99, 0.95, dones=d)
    want_adv, want_ret = reference_advantages(r, v, nv, 0.99, 0.95, dones=d)
    assert torch.equal(adv, want_adv)
    assert torch.equal(ret, want_ret)


@pytest.mark.parametrize("gamma,lam", [(0.99, 0.95), (1.0, 1.0), (0.9, 0.0)])
@pytest.mark.parametrize("shape", [(1, 1, 1), (9, 2, 257), (500, 4, 65536)])
def test_zero_dones_are_bit_equal_to_ctf_gae(small_env, shape, gamma, lam):
    T, apt, B = shape
    r, v, nv = _gae_inputs(T, apt, B, T + B, True)
    got = advantages(small_env, _ro(r, v), nv, gamma, lam, dones=torch.zeros_like(r))
    want = advantages(small_env, _ro(r, v), nv, gamma, lam)
    assert torch.equal(got[0].view(torch.int32), want[0].view(torch.int32))
    assert torch.equal(got[1].view(torch.int32), want[1].view(torch.int32))


# ---------------------------------------------------------------------------------------------------- 2. graph replay
def test_gae_dones_graph_replay(small_env):
    T, apt, B = 40, 4, 1000
    r, v, nv = _gae_inputs(T, apt, B, 5, False)
    d = _dones("random", T, apt, B, 5)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        advantages(small_env, _ro(r, v), nv, 0.99, 0.95, dones=d)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        adv, ret = advantages(small_env, _ro(r, v), nv, 0.99, 0.95, dones=d)
    for seed in (6, 7):
        r2, v2, nv2 = _gae_inputs(T, apt, B, seed, False)
        r.copy_(r2), v.copy_(v2), nv.copy_(nv2), d.copy_(_dones("random", T, apt, B, seed))
        graph.replay()
        torch.cuda.synchronize()
        want_adv, want_ret = reference_advantages(r, v, nv, 0.99, 0.95, dones=d)
        assert torch.equal(adv, want_adv) and torch.equal(ret, want_ret)


# ---------------------------------------------------------------------------------------------------- 3. rejections
def test_gae_dones_rejections(small_env):
    lib, h = small_env._lib, small_env._handle
    T, apt, B = 3, 2, 5
    n = T * apt * B
    buf = torch.zeros(6 * n + 2 * apt * B + 8, device=DEV)
    base = buf.data_ptr()
    # byte addresses: rewards, values, dones, next_value, advantages and returns, apart and 16-byte aligned
    r, v, d, nv = base, base + 4 * n, base + 8 * n, base + 12 * n
    adv, ret = nv + 4 * apt * B + 64, nv + 4 * n + 4 * apt * B + 128
    ok = dict(r=r, v=v, d=d, nv=nv, adv=adv, ret=ret, T=T, apt=apt, B=B, g=0.99, gl=0.95)

    def call(**kw):
        a = dict(ok, **kw)
        return lib.ctf_gae_dones(h, C.c_void_p(a["r"]), C.c_void_p(a["v"]), C.c_void_p(a["d"]), C.c_void_p(a["nv"]),
                                 C.c_void_p(a["adv"]), C.c_void_p(a["ret"]), a["T"], a["apt"], a["B"], a["g"], a["gl"],
                                 None)

    assert call() == 0
    torch.cuda.synchronize()
    bad = [dict(r=None), dict(v=None), dict(d=None), dict(nv=None), dict(adv=None), dict(ret=None),
           dict(T=0), dict(T=-1), dict(apt=0), dict(apt=9), dict(B=0), dict(B=-3),
           dict(g=math.nan), dict(g=math.inf), dict(g=-0.1), dict(g=1.5),
           dict(gl=math.nan), dict(gl=-math.inf), dict(gl=-1e-3), dict(gl=1.01),
           dict(adv=r), dict(adv=r + 4 * (n - 1)), dict(ret=v + 4), dict(adv=v - 4 * (n - 1)), dict(ret=nv + 4),
           dict(adv=nv - 4 * n + 4), dict(ret=adv), dict(ret=adv + 4 * (n - 1)), dict(adv=adv + 2),
           dict(d=d + 2), dict(adv=d), dict(ret=d + 4 * (n - 1)), dict(adv=d - 4 * (n - 1))]
    for kw in bad:
        lib.ctf_get_sizes(None, None)   # leaves a message that does not start with ctf_gae_dones
        rc = call(**kw)
        assert rc == -1, kw
        assert lib.ctf_last_error().startswith(b"ctf_gae_dones: "), (kw, lib.ctf_last_error())
    with pytest.raises(ValueError):
        advantages(small_env, _ro(*_gae_inputs(3, 2, 5, 1, False)[:2]), torch.zeros((2, 5), device=DEV), 0.99, 0.95,
                   dones=torch.zeros((6, 4), device=DEV))


# ---------------------------------------------------------------------------------------------------- 4. continuing
FIELDS = ("grid_states", "metadata_states", "actions", "use_action_mask", "logprobs", "values", "rewards")


def test_four_continuing_collects_are_one_rollout():
    """PackedPPO(rollout_steps=125): four collects from a fresh trainer are, under the same torch seed, bit for bit the
    one 500-step rollout of an identical env; no row starts an episode, and only the last bootstrap is 0."""
    B = 16
    env, env2 = _env(B), _env(B)
    pol, opp = _policy(env, 61), _policy(env, 62)
    tr = PackedPPO(env, pol, _args(), rollout_steps=125)
    opponent = FusedPolicy(env, opp)
    mine = _team(env, 0)
    apt = len(mine)
    torch.manual_seed(123)
    parts = []
    for k in range(4):
        ro = tr.collect(opponent)
        assert ro.rewards.shape == (125 * apt, B)
        assert not bool(ro.dones.any())
        v, _ = FusedPolicy(env, pol).forward_from_env(mine)
        want_nv = torch.zeros((apt, B), device=DEV) if k == 3 else v.reshape(B, apt).t()
        assert torch.equal(ro.next_value, want_nv)
        assert torch.equal(ro.next_done, torch.full((B,), float(k == 3), device=DEV))
        assert [t for t, _ in ro.episode_ends] == ([124] if k == 3 else [])
        parts.append({f: getattr(ro, f).clone() for f in FIELDS})
    torch.manual_seed(123)
    ref = collect_rollout(env2, FusedPolicy(env2, pol), FusedPolicy(env2, opp), num_env_steps=500,
                          obs_storage_dtype="packed")
    for f in FIELDS:
        assert torch.equal(torch.cat([p[f] for p in parts]), getattr(ref, f)), f


def _set_captures(env, caps):
    st = env.get_state()
    env.set_state(st["grid"], st["pos"], st["hp_q"], st["has_flag"], st["inventory"], st["step"], st["episode"],
                  torch.tensor(caps).expand(env.num_envs, 2).numpy(), hp=st.get("hp"))


def test_continuing_rollouts_cross_the_episode_end():
    """Four 150-step rollouts run 600 steps: the episode ends at step 500 (t = 49 of the fourth rollout) and a new one
    starts on its row t = 50.  Two flag captures are credited to team 0 at step 450, so step 500 pays a terminal
    reward.  The env's step and reset calls are recorded and replayed on an identical env: every observation,
    metadata row and reward of the rollouts is the replay's, bit for bit."""
    B = 8
    env, rep = _env(B), _env(B)
    pol, opp = _policy(env, 71), _policy(env, 72)
    tr = PackedPPO(env, pol, _args(), rollout_steps=150)
    opponent = FusedPolicy(env, opp)
    mine = _team(env, 0)
    apt, GS = len(mine), env.GAME_STEPS
    assert GS == 500
    events = []
    step, reset = env.step, env.reset
    env.step = lambda a: (events.append(a.clone()), step(a))[1]
    env.reset = lambda: (events.append("reset"), reset())[1]
    ros = []
    for k in range(4):
        if k == 3:
            _set_captures(env, (2, 0))
            events.append("captures")
            episode = env.get_state()["episode"].copy()
        ro = tr.collect(opponent)
        v, _ = FusedPolicy(env, pol).forward_from_env(mine)
        assert torch.equal(ro.next_value, v.reshape(B, apt).t()), k   # no rollout ends on step 500
        ros.append(ro)
    assert (env.get_state()["episode"] == episode + 1).all()
    assert events.count("reset") == 2
    assert [len(ro.episode_ends) for ro in ros] == [0, 0, 0, 1] and ros[3].episode_ends[0][0] == 49

    # replay: the recorded actions on an identical env, with its reset at step 500
    bits, meta, rew, caps_at_end = [], [], [], None
    mine_t = torch.tensor(mine, device=DEV)
    for e in events:
        if isinstance(e, str):
            if e == "reset":
                if caps_at_end is None and len(rew) == GS:
                    caps_at_end = rep.flag_captures().clone()
                rep.reset()
            else:
                _set_captures(rep, (2, 0))
            continue
        bits.append(rep.obs_bits[:, mine_t].transpose(0, 1).clone())
        meta.append(rep.meta[:, mine_t].transpose(0, 1).clone())
        rep.step(e)
        rew.append(rep.rewards[:, mine_t].t().clone())
    assert len(rew) == 600
    flat = lambda xs: torch.stack(xs).reshape((600 * apt,) + xs[0].shape[1:])
    got = {f: torch.cat([getattr(ro, f) for ro in ros]) for f in ("grid_states", "metadata_states", "rewards", "dones")}
    assert torch.equal(got["grid_states"], flat(bits))
    assert torch.equal(got["metadata_states"], flat(meta))
    assert torch.equal(got["rewards"], flat(rew))
    want_dones = torch.zeros_like(got["dones"])
    want_dones[GS * apt : (GS + 1) * apt] = 1
    assert torch.equal(got["dones"], want_dones)
    # the terminal row pays the margin of at least two captures to the winners, team 0
    term = got["rewards"][(GS - 1) * apt : GS * apt]
    others = torch.cat((got["rewards"][(GS - 51) * apt : (GS - 1) * apt], got["rewards"][GS * apt :]))
    assert float(term.mean()) - float(others.mean()) > 0.1
    assert torch.equal(ros[3].episode_ends[0][1], caps_at_end)
    stats = ros[3].episode_stats
    assert stats["episodes_completed"] == apt * B
    want_win = (caps_at_end[:, 0] > caps_at_end[:, 1]).float().mean()
    assert float(stats["win_fraction"]) == float(want_win) and float(stats["draw_fraction"]) == 0.0
    whole = got["rewards"][: GS * apt].reshape(GS, apt, B).sum(0)
    assert math.isclose(float(stats["episode_return"]), float(whole.mean()), rel_tol=1e-5, abs_tol=1e-6)
    # GAE of the fourth rollout stops at the boundary, and the trainer passes the rollout's dones
    adv, ret = tr.advantages(ros[3])
    want_adv, want_ret = reference_advantages(ros[3].rewards, ros[3].values, ros[3].next_value, 0.99, 0.95,
                                              dones=ros[3].dones)
    assert torch.equal(adv, want_adv) and torch.equal(ret, want_ret)


def test_collect_rollout_refuses_envs_out_of_lock_step():
    env = _env(4)
    pol = FusedPolicy(env, _policy(env, 81))
    env.reset()
    st = env.get_state()
    steps = st["step"].copy()
    steps[1] = 3
    env.set_state(st["grid"], st["pos"], st["hp_q"], st["has_flag"], st["inventory"], steps, st["episode"],
                  st["captures"], hp=st.get("hp"))
    with pytest.raises(ValueError, match="lock-step"):
        collect_rollout(env, pol, pol, num_env_steps=2, obs_storage_dtype="packed", reset=False)


def test_an_env_at_its_end_is_reset_first():
    env = _env(4, game_steps=12)
    pol = FusedPolicy(env, _policy(env, 82))
    apt = len(_team(env, 0))
    ro = collect_rollout(env, pol, pol, num_env_steps=12, obs_storage_dtype="packed", reset=False)
    assert not bool(ro.dones.any()) and bool((ro.next_done == 1).all())   # a never-reset env starts fresh
    ro = collect_rollout(env, pol, pol, num_env_steps=5, obs_storage_dtype="packed", reset=False)
    assert bool((ro.dones[:apt] == 1).all()) and not bool(ro.dones[apt:].any())
    assert bool((env.step_counts() == 5).all()) and not bool(ro.next_done.any())


# ---------------------------------------------------------------------------------------------------- 5. trainer
@torch.no_grad()
def _value_loss(tr, ro, ret):
    bits = ro.grid_states.reshape(-1, tr.env.bits_words_per_agent)
    meta = ro.metadata_states.reshape(-1, tr.env.meta_size)
    value, _ = tr.fused.train_head(tr.fused.trunk_packed(bits, meta).clone())
    return float(0.5 * ((value.reshape(-1) - ret.reshape(-1)) ** 2).mean())


def test_continuing_trainer_learns_and_counts_episodes():
    """Five 125-step updates of PackedPPO(rollout_steps=125) on 64 envs.  A random policy's GAE returns leave its value
    loss nowhere to go (see test_gpu_ppo), so every update gets the fixed value target 1, about 0.5 away in value loss;
    at lr 2.5e-5 the 40 Adam steps move the value well short of it, and the value loss of the first rollout falls.
    Each update reports its episodes: apt * B in the fourth, whose rollout ends on step 500, and 0 in the others."""
    env = _env(64)
    pol, opp = _policy(env, 91), _policy(env, 92)
    tr = PackedPPO(env, pol, _args(update_epochs=2, clip_vloss=False, learning_rate=2.5e-5), rollout_steps=125)
    opponent = FusedPolicy(env, opp)
    apt, B = len(_team(env, 0)), env.num_envs
    first = None
    for u in range(5):
        ro = tr.collect(opponent)
        adv, _ = tr.advantages(ro)
        target = torch.ones_like(ro.values)
        if first is None:
            first = (ro, target, _value_loss(tr, ro, target))
        out = tr.optimise(ro, adv, target)
        assert all(math.isfinite(out[k]) for k in ("v_loss", "pg_loss", "entropy", "approx_kl", "clipfrac"))
        assert out["episodes_completed"] == (apt * B if u == 3 else 0), (u, out)
        if u == 3:
            assert math.isfinite(out["episode_return"]) and 0 <= out["win_fraction"] + out["draw_fraction"] <= 1
        else:
            assert math.isnan(out["episode_return"]) and math.isnan(out["win_fraction"])
    ro0, target0, before = first
    assert _value_loss(tr, ro0, target0) < 0.9 * before


def test_team_switch_only_between_episodes():
    env = _env(16)
    pol, opp = _policy(env, 93), _policy(env, 94)
    tr = PackedPPO(env, pol, _args(update_epochs=1), rollout_steps=250)
    opponent = FusedPolicy(env, opp)
    out = tr.update(opponent)
    assert out["episodes_completed"] == 0
    with pytest.raises(ValueError, match="between episodes"):
        tr.update(opponent, train_team1=False)
    out = tr.update(opponent)                   # the episode ends on step 500
    assert out["episodes_completed"] == len(_team(env, 0)) * 16
    out = tr.update(opponent, train_team1=False)
    assert out["episodes_completed"] == 0
    assert bool((tr.rollout.dones[: len(_team(env, 1))] == 1).all())
    with pytest.raises(ValueError):
        PackedPPO(env, pol, _args(), rollout_steps=501)
    with pytest.raises(ValueError):
        PackedPPO(env, pol, _args(), rollout_steps=0)


@pytest.mark.parametrize("rollout_steps,first_steps", [(12, None), (5, 12)])
def test_rollouts_of_a_whole_episode_count_every_episode(rollout_steps, first_steps):
    """Rollouts that end exactly on GAME_STEPS (rollout_steps == GAME_STEPS, or a first collect given
    num_env_steps=GAME_STEPS) report apt * B episodes each, the first one included, with the return of that rollout
    alone: nothing carries over into the next episode."""
    env = _env(8, game_steps=12)
    pol, opp = _policy(env, 95), _policy(env, 96)
    tr = PackedPPO(env, pol, _args(update_epochs=1), rollout_steps=rollout_steps)
    opponent = FusedPolicy(env, opp)
    apt, B = len(_team(env, 0)), env.num_envs
    for k in range(3):
        ro = tr.collect(opponent, num_env_steps=first_steps if k == 0 else 12)
        assert [t for t, _ in ro.episode_ends] == [11]
        assert bool((ro.dones[:apt] == float(k > 0)).all()) and not bool(ro.dones[apt:].any())
        assert torch.equal(ro.next_value, torch.zeros((apt, B), device=DEV))
        st = ro.episode_stats
        assert st["episodes_completed"] == apt * B
        want = float(ro.rewards.reshape(12, apt, B).sum(0).mean())
        assert math.isclose(float(st["episode_return"]), want, rel_tol=1e-5, abs_tol=1e-6), (k, st, want)
        caps = ro.episode_ends[0][1]
        assert float(st["win_fraction"]) == float((caps[:, 0] > caps[:, 1]).float().mean())
        assert float(st["draw_fraction"]) == float((caps[:, 0] == caps[:, 1]).float().mean())
    out = tr.optimise(ro, *tr.advantages(ro))
    assert out["episodes_completed"] == apt * B and math.isfinite(out["episode_return"])


# ---------------------------------------------------------------------------------------------------- 6. the reference
@pytest.mark.skipif(not rs.available(), reason="reference neither under /root/reference nor in oracle/_ref")
def test_reference_calculate_advantages_reads_dones_as_cleanrl():
    """The reference's own PPOTrainer.calculate_advantages (ppo.py:133-172), unmodified, on rollouts with nonzero dones.
    With one trained agent per step its rows are the steps, as in ctf_gae_dones.  Its result is CleanRL's recurrence
    (nextnonterminal = 1 - dones[t + 1], 1 - next_done on the last row), which is the dones convention of
    collect_rollout(reset=False) and ctf_gae_dones, and which depends on dones: the reference reads them."""
    import types

    from helpers import compiled
    from marl_ctf_development_b200.config import env_dims

    mods = rs.caller_modules()
    Agent, PPOTrainer = mods["agent_network"].Agent, mods["ppo"].PPOTrainer
    ce = compiled("8_arena")
    dims = env_dims(ce)
    torch.manual_seed(3)
    agent = Agent(9, ce.n_channels, ce.GRID_SIZE, dims[2][0], "cpu")
    grid = torch.rand((1,) + dims[0]).round()
    meta = torch.rand((1,) + dims[2])
    B = 6

    def run(T, r, v, d, next_done, gamma, lam):
        args = types.SimpleNamespace(device="cpu", num_steps=T, num_envs=B, gae=True, gamma=gamma, gae_lambda=lam)
        tr = PPOTrainer(args, dims[0], dims[2])
        tr.device, tr.num_steps = "cpu", T
        with torch.no_grad():
            adv, ret = tr.calculate_advantages(agent, grid, meta, r, torch.tensor([float(next_done)]), d, v)
        return adv.float(), ret.float()

    # the agent's bootstrap V, read through the reference itself: one zero row with gamma = 1 gives advantages = V
    z = torch.zeros((1, B))
    nv, _ = run(1, z, z, z, 0, 1.0, 0.95)
    T = 9
    g = torch.Generator().manual_seed(4)
    r, v = torch.randn((T, B), generator=g), torch.randn((T, B), generator=g)
    d = (torch.rand((T, B), generator=g) < 0.3).float()
    d[3] = 1
    for next_done in (0, 1):
        boot = nv * (1 - next_done)
        for gamma, lam in ((0.99, 0.95), (1.0, 1.0), (0.9, 0.0)):
            adv, ret = run(T, r, v, d, next_done, gamma, lam)
            want = _cleanrl64(r, v, boot, d, gamma, lam)
            tol = 4 * T * 2.0 ** -24 * (float(want.abs().max()) + float(v.abs().max()) + 1)
            assert float((adv.double() - want).abs().max()) <= tol, (next_done, gamma, lam)
            ours, _ = reference_advantages(r, v, boot, gamma, lam, dones=d)
            assert float((adv - ours).abs().max()) <= tol
            assert torch.allclose(ret, adv + v, atol=tol, rtol=0)
        no_dones, _ = run(T, r, v, torch.zeros_like(d), next_done, 0.99, 0.95)
        assert float((no_dones - run(T, r, v, d, next_done, 0.99, 0.95)[0]).abs().max()) > 1e-3
