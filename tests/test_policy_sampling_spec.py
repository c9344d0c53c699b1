"""Host statement of the seeded policy draw (draws.policy_words / sample_action), checked without a GPU."""
import numpy as np
import pytest

from marl_ctf_development_b200 import draws

# Random123 kat_vectors, philox4x32-10: the one whose counter policy_words can address (every site word has its top
# bit set), and the other two through philox4x32_10 itself
KAT_ONES = ([0xFFFFFFFF] * 4, [0xFFFFFFFF] * 2, [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD])
KAT_PI = ([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0],
          [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1])


def test_policy_words_known_answers():
    got = draws.policy_words(0xFFFFFFFFFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, 0x7FFFFFFF)
    assert [int(w) for w in got] == KAT_ONES[2]
    ctr, key, want = KAT_PI
    assert [int(w) for w in draws.philox4x32_10(np.array(ctr, np.uint32), np.array(key, np.uint32))] == want


def test_policy_words_counter_layout():
    seed = 0x0123456789ABCDEF
    env_id, episode, step, agent = np.array([0, 37, 70000]), np.array([0, 3, 9]), np.array([0, 499, 12]), np.array([0, 5, 7])
    got = draws.policy_words(seed, env_id, episode, step, agent)
    ctr = np.stack([env_id, episode, step, 0x80000000 | agent], -1).astype(np.uint32)
    want = draws.philox4x32_10(ctr, np.array([seed & 0xFFFFFFFF, seed >> 32], np.uint32))
    assert np.array_equal(got, want)
    # scalars broadcast against arrays
    assert np.array_equal(draws.policy_words(seed, 37, 3, 499, agent)[1], want[1])


def test_policy_sites_are_disjoint_from_env_sites():
    env_sites = set(range(draws.SITES_PER_STEP))
    policy_sites = {draws.POLICY_SITE | a for a in range(8)}
    assert not env_sites & policy_sites
    # same seed, env, episode and step: no policy word equals any env word of that step
    seed = 11
    env_words = draws.step_words(seed, 5, 2, 17)
    pol = draws.policy_words(seed, 5, 2, 17, np.arange(8))
    assert not {tuple(r) for r in env_words.tolist()} & {tuple(r) for r in pol.tolist()}


def test_policy_uniform_is_24_bit_and_below_one():
    w = np.array([[0, 0, 0, 0], [0xFFFFFFFF, 0, 0, 0], [0x00000100, 0, 0, 0], [0x000000FF, 0, 0, 0]], np.uint32)
    assert draws.policy_uniform(w).tolist() == [0.0, 1 - 2.0 ** -24, 2.0 ** -24, 0.0]


def _one(logits, masked, u):
    a, lp, ent = draws.sample_action(np.array(logits, np.float64), masked, u)
    return int(a), float(lp), float(ent)


def test_one_hot_distribution():
    for hot in range(9):
        x = [-1e4] * 9
        x[hot] = 3.0
        for u in (0.0, 0.5, 1 - 2.0 ** -24):
            a, lp, ent = _one(x, False, u)
            assert a == hot and lp == 0.0 and ent == 0.0


def test_all_mass_on_the_last_unmasked_action():
    x = [-1e4] * 9
    x[4] = 0.0
    x[8] = 50.0            # masked away: -1e9 + 50
    a, lp, ent = _one(x, True, 1 - 2.0 ** -24)
    assert (a, lp, ent) == (4, 0.0, 0.0)
    # unmasked, action 8 holds all but e^-50 of the mass
    assert _one(x, False, 0.5)[0] == 8


def test_u_just_below_and_above_a_cdf_boundary():
    # uniform over 4 actions: c = 1, 2, 3, 4 (times e = 1), Z = 4; boundaries at u = 1/4, 1/2, 3/4
    x = [0.0] * 4 + [-1e4] * 5
    for k in (1, 2, 3):
        b = k / 4
        assert _one(x, False, np.nextafter(b, 0))[0] == k - 1
        assert _one(x, False, b)[0] == k          # u*Z == c_{k-1} is not < c_{k-1}
        assert _one(x, False, np.nextafter(b, 1))[0] == k
    a, lp, ent = _one(x, False, 0.6)
    assert a == 2 and lp == pytest.approx(-np.log(4), abs=1e-15) and ent == pytest.approx(np.log(4), abs=1e-15)


def test_masked_row():
    x = [0.0, 1.0, 2.0, 0.5, -1.0, 9.0, 9.0, 9.0, 9.0]
    e = np.exp(np.array(x[:5]) - 2.0)
    c = np.cumsum(e)
    for u in np.linspace(0, 1 - 2.0 ** -24, 101):
        a, lp, ent = _one(x, True, u)
        assert a == int(np.argmax(u * c[-1] < c))
        p = e / c[-1]
        assert lp == pytest.approx(np.log(p[a]), abs=1e-12)
        assert ent == pytest.approx(-(p * np.log(p)).sum(), abs=1e-12)
    # unmasked, the 9.0 logits take almost all the mass
    assert _one(x, False, 0.5)[0] in (5, 6, 7, 8)


def test_non_finite_logits_give_a_valid_action():
    assert _one([np.nan] * 9, False, 0.5)[0] == draws.NO_OP_ACTION
    assert _one([np.inf] + [0.0] * 8, False, 0.5)[0] == draws.NO_OP_ACTION    # inf - inf: no positive mass
    assert _one([-np.inf] * 9, True, 0.5)[0] == draws.NO_OP_ACTION
    x = [0.0, 0.0, np.nan, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0]
    for u in (0.0, 0.9):                                   # Z is NaN, so no u*Z < c_i: the last action with mass
        assert _one(x, False, u)[0] == 8


def test_vectorised_rows_equal_single_rows():
    rng = np.random.default_rng(0)
    x = rng.normal(0, 3, (200, 9))
    masked = rng.random(200) < 0.5
    u = rng.random(200)
    a, lp, ent = draws.sample_action(x, masked, u)
    for i in range(200):
        assert (a[i], lp[i], ent[i]) == _one(x[i], masked[i], u[i])
        if masked[i]:
            assert a[i] < 5
