"""CPU side of the caller parity (SURVEY §8f N1/N3/N4): the committed outputs of the reference's UNMODIFIED callers
(tests/golden/callers/) against (a) the same loops on the CPU oracle — pins the oracle-side loops — and, where the
reference is importable (this container, or oracle/_ref), (b) a fresh run of the unmodified callers — pins the
generator — plus the state_dict compatibility of CtfPolicy with the reference Agent."""
import os

import numpy as np
import pytest
import torch

import caller_cases as cc
from helpers import GOLDEN, bits, compiled
from oracle import ref_shim as rs

needs_reference = pytest.mark.skipif(not rs.available(), reason="reference neither under /root/reference nor in oracle/_ref")


@pytest.mark.parametrize("case", cc.CASES["rollouts"], ids=lambda c: c[0])
def test_oracle_rollout_loop_equals_unmodified_get_single_rollout(case):
    name, exp, overrides, T, env_id0, n_envs, train_team1 = case
    want = cc.load_rollout(name)
    agent, opponent = cc.policies(exp, overrides, (1, 2))
    got = cc.oracle_rollout(compiled(exp, **overrides), n_envs, cc.SEED, env_id0, agent, opponent, train_team1, T)
    for k in cc.ROLLOUT_FIELDS:
        assert got[k].shape == want[k].shape, k
        assert np.array_equal(bits(got[k]), bits(want[k])), k
    if "GAME_STEPS" in overrides:   # whole episode: done at the last step, terminal rewards paid
        assert want["next_done"].min() == 1.0
    assert float(np.abs(want["dones"]).sum()) == 0.0


@pytest.mark.parametrize("case", cc.CASES["duels"], ids=lambda c: c[0])
def test_oracle_duel_loop_equals_unmodified_utils_duel(case):
    name, exp, overrides, max_steps, env_id0, n = case
    want = cc.load_duel(name)
    agent, opponent = cc.policies(exp, overrides, (3, 4))
    res, counters, caps, steps = cc.oracle_duel(compiled(exp, **overrides), n, cc.SEED, env_id0, agent, opponent, max_steps)
    assert np.array_equal(res, want["results"])
    assert np.array_equal(counters, want["counters"])
    assert np.array_equal(caps, want["captures"]) and np.array_equal(steps, want["steps"])


def test_fixtures_exercise_captures_and_terminal_rewards():
    """The traces are not trivial: flags get captured, rewards are paid, duels are won and lost."""
    r = cc.load_rollout("rollout_8_arena_t1")
    assert float(np.abs(r["rewards"]).sum()) > 0
    results = np.concatenate([cc.load_duel(c[0])["results"] for c in cc.CASES["duels"]])
    assert (results == 1).any() and (results == -1).any() and (results == 0).any()
    caps = np.concatenate([cc.load_duel(c[0])["captures"] for c in cc.CASES["duels"]])
    assert caps.sum() > 0


# ------------------------------------------------------------------------------------------------------------------
@needs_reference
def test_fixture_generator_is_reproducible_with_the_unmodified_callers(tmp_path):
    import types

    mods = rs.caller_modules()
    name, exp, overrides, T, env_id0, n_envs, train_team1 = cc.CASES["rollouts"][2]
    want = cc.load_rollout(name)
    ec = rs.experiment_env_config(exp)
    ec.update(overrides)
    agent, opponent = cc.policies(exp, overrides, (1, 2))
    env = rs.make_injected_env(ec, seed=cc.SEED, env_id=env_id0 + 1)
    dims = env.get_env_dims()
    tr = mods["ppo"].PPOTrainer(types.SimpleNamespace(device="cpu", num_steps=T), dims[0], dims[2])
    tr.reverse_grid, tr.team_to_train, tr.device = (False, 0, "cpu") if train_team1 else (True, 1, "cpu")
    tr.num_agents_per_team = env.N_AGENTS // 2
    tr.num_steps = T * tr.num_agents_per_team
    tr.max_rewards = -np.inf
    out = tr.get_single_rollout(env, agent, opponent)                      # ppo.py:31-131, unmodified
    for k, v in zip(cc.ROLLOUT_FIELDS[:8], out[:8]):
        assert np.array_equal(bits(v.numpy()), bits(want[k][:, 1])), k
    name, exp, overrides, max_steps, env_id0, n = cc.CASES["duels"][0]
    wd = cc.load_duel(name)
    ec = rs.experiment_env_config(exp)
    agent, opponent = cc.policies(exp, overrides, (3, 4))
    env = rs.make_injected_env(ec, seed=cc.SEED, env_id=env_id0)
    _, _, result = mods["utils"].duel(env, agent, opponent, (0, 0), return_result=True, device="cpu", max_steps=max_steps)
    assert result == wd["results"][0]


@needs_reference
def test_ctf_policy_loads_the_reference_agent_state_dict_bit_for_bit():
    """policy.CtfPolicy claims state_dict compatibility with agent_network.Agent (agent_network.py:5-81)."""
    from marl_ctf_development_b200.policy import CtfPolicy

    Agent = rs.caller_modules()["agent_network"].Agent
    torch.manual_seed(3)
    ref = Agent(9, 14, 15, 22)
    ours = CtfPolicy(9, 14, 15, 22)
    missing = ours.load_state_dict(ref.state_dict(), strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    g = (torch.rand(37, 14, 15, 15) < 0.1).float()
    m = torch.rand(37, 22)
    flags = (torch.arange(37) % 2).float()
    v_ref, l_ref = ref(g, m)
    v, l = ours(g, m)
    assert torch.equal(v, v_ref) and torch.equal(l, l_ref)
    # masked sampling: same distribution parameters -> same samples under the same torch seed, for a batch ...
    torch.manual_seed(11)
    a_ref, lp_ref, ent_ref, val_ref = ref.get_action_and_value(g, m, flags)
    torch.manual_seed(11)
    a, lp, ent, val = ours.get_action_and_value(g, m, flags)
    assert torch.equal(a, a_ref) and torch.equal(lp, lp_ref) and torch.equal(ent, ent_ref) and torch.equal(val, val_ref)
    assert bool((a[flags == 1] <= 4).all())
    # ... and evaluated on given actions (the PPO update path, ppo.py:201)
    assert torch.equal(ours.get_action_and_value(g, m, flags, a_ref)[1], ref.get_action_and_value(g, m, flags, a_ref)[1])
    # Agent.get_action is scalar-only (action.item(), agent_network.py:58): the batched adapters go through
    # get_action_and_value instead, which the reference Agent supports unchanged
    with pytest.raises((RuntimeError, ValueError)):
        ref.get_action(g, m, flags)
    from marl_ctf_development_b200.rollout import batched_action

    torch.manual_seed(5)
    b_ref = batched_action(ref, g, m, flags)
    torch.manual_seed(5)
    assert torch.equal(b_ref, batched_action(ours, g, m, flags))


# ------------------------------------------------------------------------------------------------------------------
POLICY_RECORD = os.path.join(GOLDEN, "ctf_policy_outputs.npz")


def _policy_case():
    """A small network (9 actions, 4 channels, 6x6 grid, 10 metadata) with weights and inputs from a fixed numpy seed."""
    from marl_ctf_development_b200.policy import CtfPolicy

    rng = np.random.default_rng(3)
    shapes = {k: v.shape for k, v in CtfPolicy(9, 4, 6, 10).state_dict().items()}
    sd = {k: torch.from_numpy(rng.uniform(-0.3, 0.3, shape).astype(np.float32)) for k, shape in shapes.items()}
    g = torch.from_numpy((rng.random((37, 4, 6, 6)) < 0.2).astype(np.float32))
    m = torch.from_numpy(rng.random((37, 10)).astype(np.float32))
    flags = (torch.arange(37) % 2).float()
    actions = torch.from_numpy(np.where(flags.numpy() == 1, rng.integers(0, 5, 37), rng.integers(0, 9, 37)))
    return sd, g, m, flags, actions


def _policy_outputs(net, g, m, flags, actions) -> dict:
    with torch.no_grad():
        value, logits = net(g, m)
        _, log_prob, entropy, _ = net.get_action_and_value(g, m, flags, actions)
    return {"value": value.numpy(), "logits": logits.numpy(), "log_prob": log_prob.numpy(), "entropy": entropy.numpy()}


def test_ctf_policy_outputs_match_the_stored_agent_outputs():
    """CtfPolicy's values, logits, masked log-probs and entropies for fixed weights and inputs, against
    tests/golden/ctf_policy_outputs.npz.  The record was written from CtfPolicy (PYTHONPATH=.:tests python
    tests/test_callers_fixtures.py) at a commit where test_ctf_policy_loads_the_reference_agent_state_dict_bit_for_bit
    passed; where the reference is importable, agent_network.Agent with the same weights is checked against the
    record bit for bit as well."""
    from marl_ctf_development_b200.policy import CtfPolicy

    sd, g, m, flags, actions = _policy_case()
    ours = CtfPolicy(9, 4, 6, 10)
    ours.load_state_dict(sd, strict=True)
    got = _policy_outputs(ours, g, m, flags, actions)
    want = dict(np.load(POLICY_RECORD))
    assert sorted(got) == sorted(want)
    for k in want:   # float32 convolutions and matmuls: summation order may differ between CPU kernels
        np.testing.assert_allclose(got[k], want[k], rtol=1e-5, atol=1e-6, err_msg=k)
    masked = _policy_outputs(ours, g, m, flags, torch.full((37,), 6))["log_prob"]
    assert (masked[flags.numpy() == 1] < -1e6).all() and (masked[flags.numpy() == 0] > -1e6).all()   # only 0..4 when masked
    if rs.available():
        ref = rs.caller_modules()["agent_network"].Agent(9, 4, 6, 10)
        ref.load_state_dict(sd, strict=True)
        for k, v in _policy_outputs(ref, g, m, flags, actions).items():
            assert np.array_equal(bits(v), bits(want[k])), k


if __name__ == "__main__":
    from marl_ctf_development_b200.policy import CtfPolicy

    sd, g, m, flags, actions = _policy_case()
    net = CtfPolicy(9, 4, 6, 10)
    net.load_state_dict(sd, strict=True)
    np.savez_compressed(POLICY_RECORD, **_policy_outputs(net, g, m, flags, actions))
