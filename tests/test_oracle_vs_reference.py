"""Pins the CPU oracle against the unmodified reference with injected draws.

Where the reference is importable (its source tree, or the byte-compiled oracle/_ref), every case runs it step by step
next to the oracle and compares states, rewards, dones, observations and counters.  Everywhere else the oracle is
compared with tests/golden/reference_digests.npz: per case, one 32-bit digest of every quantity the comparison covers,
in the order it is compared (the state, rewards and done of every step, the observations and metadata at the steps
where they are compared, the counters, the standardise_state outputs, dims and tile sets).  Where the reference runs,
the stored digests are checked against it too, so the record itself stays pinned to the reference.

The record was written from the oracle at a commit where this module's live comparison with the reference passed:

    CTF_RECORD_REFERENCE_DIGESTS=1 python -m pytest tests/test_oracle_vs_reference.py
"""
import hashlib
import json
import os

import numpy as np
import pytest

import traces
from helpers import GOLDEN, STATE_KEYS, assert_state_equal, bits
from marl_ctf_development_b200.config import compile_config, env_dims
from marl_ctf_development_b200.scenario_io import experiment_env_config as local_env_config
from marl_ctf_development_b200.scenario_io import experiment_names as local_experiment_names
from oracle import ref_shim as rs
from oracle.ctf_oracle import OracleEnv
from kwarg_cases import CASE_IDS, KWARG_CASES, build_env_config

pytestmark = pytest.mark.filterwarnings("ignore")

LIVE = rs.available()
RECORD = bool(os.environ.get("CTF_RECORD_REFERENCE_DIGESTS"))
RECORD_PATH = os.path.join(GOLDEN, "reference_digests.npz")
STORED = dict(np.load(RECORD_PATH)) if os.path.exists(RECORD_PATH) else {}
RECORDED = {}
needs_reference = pytest.mark.skipif(not LIVE, reason="needs the reference's own code, which is not part of the repository")


@pytest.fixture(scope="module", autouse=True)
def _write_record():
    yield
    if RECORD and RECORDED:
        np.savez_compressed(RECORD_PATH, **dict(STORED, **RECORDED))


def env_config(exp: str) -> dict:
    return rs.experiment_env_config(exp) if LIVE else local_env_config(exp)


def _digest(blob: bytes) -> int:
    return int.from_bytes(hashlib.blake2b(blob, digest_size=4).digest(), "little")


def _canonical(value) -> bytes:
    if isinstance(value, np.ndarray):
        return np.ascontiguousarray(value).tobytes()
    return json.dumps(value, sort_keys=True, default=lambda x: x.tolist() if hasattr(x, "tolist") else int(x)).encode()


class Pair:
    """The oracle next to the reference (live) or next to the stored digests of the reference's run of the same case."""

    def __init__(self, case: str, ec: dict, seed: int, env_id: int):
        self.case, self.ce = case, compile_config(**ec)
        self.float_hp = bool(self.ce.cfg.hp_float)
        self.orc = OracleEnv(self.ce, seed=seed, env_id=env_id)
        self.ref = rs.make_injected_env(ec, seed=seed, env_id=env_id) if LIVE else None
        if not LIVE and not RECORD and case not in STORED:
            pytest.fail(f"{case}: no stored record in {RECORD_PATH} and no reference to compare with")
        self.digests = []

    def _record(self, where: str, blob: bytes):
        d, i = _digest(blob), len(self.digests)
        self.digests.append(d)
        if not RECORD and self.case in STORED:
            want = STORED[self.case]
            assert i < len(want) and int(want[i]) == d, f"{self.case} {where}: differs from the stored reference record"

    def same(self, where: str, ours, theirs=None):
        """One quantity compared once; `theirs(ref)` gives the reference's value where the reference runs."""
        if self.ref is not None:
            want = theirs(self.ref)
            assert np.array_equal(ours, want) if isinstance(ours, np.ndarray) else ours == want, (where, ours, want)
        self._record(where, _canonical(ours))

    def step(self, a, where: str, observe: bool = False) -> dict:
        orr, od = self.orc.step(a)
        st = self.orc.state()
        keys = [k for k in STATE_KEYS if not (self.float_hp and k == "hp_q")]
        blob = b"".join(np.asarray(st[k]).astype(np.int64).tobytes() for k in keys)
        blob += np.asarray(st["hp"], dtype=np.float64).tobytes() + bits(orr).tobytes() + bytes([int(od)])
        if self.ref is not None:
            _, rr, rd = self.ref.step(a.tolist())
            assert_state_equal(st, rs.snapshot(self.ref, self.ce.cfg.hp_scale), where, float_hp=self.float_hp)
            assert rd == od, where
            assert np.array_equal(bits(np.array(rr, dtype=np.float32)), bits(orr)), (where, rr, orr)
        if observe:
            oo, om = self.orc.observe()
            if self.ref is not None:
                ro, rm = rs.observations(self.ref)
                assert np.array_equal(ro, oo), where
                assert np.array_equal(bits(rm), bits(om)), (where, rm, om)
            blob += np.ascontiguousarray(oo).tobytes() + bits(om).tobytes()
        self._record(where, blob)
        return st

    def reset(self):
        self.orc.reset()
        if self.ref is not None:
            self.ref.reset()

    def counters(self, where: str, visits: bool = True):
        """Agent-level counters (and visitation maps) against env.metrics of the reference."""
        st = self.orc.state()
        self.same(where + " counters", st["stats"], rs.agent_metrics)
        if visits:
            self.same(where + " visits", st["visits"],
                      lambda ref: np.stack([ref.metrics["agent_visitation_maps"][i] for i in range(self.ce.N_AGENTS)]))

    def dims(self, opponents: bool = False):
        self.same("env_dims", env_dims(self.ce), lambda ref: ref.get_env_dims())
        self.same("TILES_USED", [int(t) for t in self.ce.TILES_USED], lambda ref: [int(t) for t in ref.TILES_USED])
        if opponents:
            self.same("OPPONENTS", self.ce.OPPONENTS, lambda ref: ref.OPPONENTS)

    def close(self):
        if RECORD:
            RECORDED[self.case] = np.array(self.digests, dtype=np.uint32)
        elif self.case in STORED:
            assert len(self.digests) == len(STORED[self.case]), f"{self.case}: fewer comparisons than the stored record"


CASES = [
    ("0_the_split", "seek", 260),
    ("1_fence", "builder", 200),
    ("2_jailbreak", "seek", 260),
    ("3_one_way_out", "builder", 200),
    ("4_keyhole", "seek", 200),
    ("5_skittles", "builder", 200),
    ("6_the_wall", "seek", 200),
    ("7_gridlocked", "builder", 503),
    ("8_arena", "seek", 503),
    ("8_arena", "uniform", 200),
]


@pytest.mark.parametrize("exp,kind,steps", CASES, ids=[f"{e}-{k}" for e, k, _ in CASES])
def test_oracle_equals_reference_step_by_step(exp, kind, steps, request):
    ec = env_config(exp)
    p = Pair(request.node.name, ec, seed=99, env_id=1234)
    p.dims()
    pol = traces.make_policy(kind, p.ce)
    rng = np.random.default_rng(5)
    for episode in range(2):
        if episode:
            p.reset()
        for t in range(steps if episode == 0 else 30):
            s = p.orc.state()
            a = pol(rng, s["pos"], s["has_flag"])
            p.step(a, f"{exp}/{kind} ep{episode} t={t}", observe=t % 5 == 0)
        p.counters(f"ep{episode}")
    p.close()


def test_arbitrary_reverse_flags_and_symmetry_assert(request):
    """standardise_state(i, reverse_grid) for both flag values; the ctor's symmetry assert (gridworld_ctf.py:476-477)."""
    p = Pair(request.node.name, env_config("8_arena"), seed=1, env_id=1)
    assert np.array_equal(p.orc.standardise_state(0), p.orc.standardise_state(1, reverse_grid=True))
    rng = np.random.default_rng(0)
    for t in range(60):
        p.step(traces.uniform_actions(rng, p.ce.N_AGENTS), f"t={t}")
    for i in range(p.ce.N_AGENTS):
        for rev in (False, True):
            p.same(f"standardise_state({i}, {rev})", p.orc.standardise_state(i, reverse_grid=rev),
                   lambda ref: ref.standardise_state(i, reverse_grid=rev))
    p.close()


@pytest.mark.parametrize("exp,flip", [("0_the_split", 2), ("1_fence", 0), ("8_arena", None), ("7_gridlocked", 1)])
def test_all_flip_axes_are_covered(exp, flip, request):
    """FLIP_AXIS 2, 0 and None appear in shipped scenarios; 1 is forced onto a map to cover np.flip(axis=1)."""
    ec = env_config(exp)
    ec["SCENARIO"] = dict(ec["SCENARIO"], FLIP_AXIS=flip)
    ec["MAP_SYMMETRY_CHECK"] = False
    p = Pair(request.node.name, ec, seed=3, env_id=3)
    rng = np.random.default_rng(1)
    for t in range(25):
        p.step(traces.uniform_actions(rng, p.ce.N_AGENTS), f"t={t}")
    for i in range(p.ce.N_AGENTS):
        p.same(f"standardise_state({i}, True)", p.orc.standardise_state(i, reverse_grid=True),
               lambda ref: ref.standardise_state(i, reverse_grid=True))
    p.same("reversed actions", [int(p.ce.cfg.reversed_action[a]) for a in range(9)],
           lambda ref: [ref.get_reversed_action(a) for a in range(9)])
    p.close()


@pytest.mark.parametrize("name,exp,overrides,kind", KWARG_CASES, ids=CASE_IDS)
def test_constructor_keyword_variations(name, exp, overrides, kind, request):
    """Every ctor keyword the step path reads (gridworld_ctf.py:19-52), odd team layouts, other HP grids."""
    ec = build_env_config(env_config(exp), overrides)
    p = Pair(request.node.name, ec, seed=4242, env_id=17)
    p.dims(opponents=True)
    pol = traces.make_policy(kind, p.ce)
    rng = np.random.default_rng(11)
    steps = min(ec["GAME_STEPS"] + 2, 300)
    for t in range(steps):
        s = p.orc.state()
        a = pol(rng, s["pos"], s["has_flag"])
        p.step(a, f"{name} t={t}", observe=t % 7 == 0 or t == steps - 1)
    p.counters("end")
    p.close()


@pytest.mark.parametrize("seed", list(range(24)) + list(range(100, 108)))
def test_random_scenarios_and_configs(seed, request):
    """Random maps (grid 6..16, any FLIP_AXIS), team layouts, HP tables: reference == oracle step by step."""
    from random_scenarios import random_env_config

    ec = random_env_config(seed)
    p = Pair(request.node.name, ec, seed=77, env_id=seed)
    p.dims()
    pol = traces.make_policy("builder", p.ce)
    rng = np.random.default_rng(seed)
    for t in range(ec["GAME_STEPS"] + 2):
        s = p.orc.state()
        a = pol(rng, s["pos"], s["has_flag"])
        p.step(a, f"seed {seed} t={t}", observe=t % 5 == 0)
    p.counters("end", visits=False)
    p.close()


@pytest.mark.reference
@needs_reference
def test_metrics_dict_feeds_the_reference_metrics_logger():
    """env.metrics rebuilt from the agent-level counters (metrics_dict) is harvested by the reference's
    MetricsLogger (metrics_logger.py:137-159) exactly like the reference env's own dict."""
    import importlib

    from marl_ctf_development_b200.env import metrics_dict

    rs.reference_modules()
    ml = importlib.import_module("metrics_logger")
    ec = rs.experiment_env_config("8_arena")
    ce = compile_config(**ec)
    ref = rs.make_injected_env(ec, seed=5, env_id=5)
    orc = OracleEnv(ce, seed=5, env_id=5)
    pol = traces.make_policy("seek", ce)
    rng = np.random.default_rng(2)
    for t in range(300):
        s = rs.snapshot(ref, ce.cfg.hp_scale)
        a = pol(rng, s["pos"], s["has_flag"])
        ref.step(a.tolist())
        orc.step(a)
    ours = metrics_dict(ce, orc.state()["stats"], orc.state()["visits"])
    team_types = {t: sorted({ce.AGENT_TYPES[i] for i in range(ce.N_AGENTS) if ce.AGENT_TEAMS[i] == t}) for t in (0, 1)}
    loggers = []
    for metrics in (ref.metrics, ours):
        lg = ml.MetricsLogger(1, 0, 0, team_types, list(range(ce.N_AGENTS)), symmetric_teams=False)
        lg.harvest_metrics(metrics, "t0_m0", 0, 0.5, team_idx=0)
        lg.harvest_metrics(metrics, "t1_m0", 0, 0.25, team_idx=1)
        loggers.append(lg)
    a, b = loggers
    for label in ("t0_m0", "t1_m0"):
        for metric, val in a.metrics[label].items():
            if isinstance(val, list):
                assert val == b.metrics[label][metric], (label, metric)
            else:
                assert {k: v for k, v in val.items()} == {k: v for k, v in b.metrics[label][metric].items()}, (label, metric)
    assert a.metrics["t0_m0"]["team_steps_adj_teammate"][0] > 0  # something was actually harvested


def test_multi_lethal_turns_and_carrier_kills_match_the_reference(request):
    """One-hit-kill settings for 4 episodes: several lethal hits inside one actor's turn (chained respawns whose
    windows depend on each other) and killed flag carriers must have happened, and match step by step."""
    name, exp, overrides, kind = [c for c in KWARG_CASES if c[0] == "one_hit_kills_arena"][0]
    ec = build_env_config(env_config(exp), overrides)
    ec["GAME_STEPS"] = 400
    p = Pair(request.node.name, ec, seed=606, env_id=9)
    rng = np.random.default_rng(4)
    multi_lethal, carrier_kills = 0, 0
    for episode in range(4):
        if episode:
            p.reset()
        prev = np.zeros((13, p.ce.N_AGENTS), dtype=np.int64)
        for t in range(400):
            s = p.orc.state()
            a = traces.seek_actions_batch(rng, p.ce, s["pos"][None], s["has_flag"][None], eps=0.15)[0]
            st = p.step(a, f"ep{episode} t={t}", observe=t % 20 == 0)
            cur = st["stats"]
            multi_lethal += int(((cur[1] - prev[1]) >= 2).sum())
            carrier_kills += int((cur[4] - prev[4]).sum())
            prev = cur
        p.counters(f"ep{episode}", visits=False)
    p.close()
    assert multi_lethal >= 2 and carrier_kills >= 10, (multi_lethal, carrier_kills)


def test_visitation_maps_wrap_at_256_like_numpy_uint8(request):
    """Agents that stand still for 300 steps: the reference's uint8 visitation maps overflow and wrap (gridworld_ctf.py:469, :486)."""
    p = Pair(request.node.name, env_config("0_the_split"), seed=1, env_id=1)
    a = np.full(p.ce.N_AGENTS, 4, dtype=np.uint8)
    for t in range(300):
        p.step(a, f"t={t}")
    p.counters("end")
    p.close()
    assert p.orc.state()["visits"].max() == (301 % 256)  # 1 at reset + 300 steps, wrapped


@pytest.mark.parametrize("exp", rs.EXPERIMENTS)
def test_full_episode_with_the_aggressive_policy(exp, request):
    """Every experiment config for one whole episode (+2 steps past done) under the flag-seeking / second-action-heavy
    policy the GPU soak tests use: captures, terminal margins, mining, placing and respawns all occur."""
    ec = env_config(exp)
    p = Pair(request.node.name, ec, seed=808, env_id=3)
    rng = np.random.default_rng(8)
    for t in range(ec["GAME_STEPS"] + 2):
        s = p.orc.state()
        a = traces.seek_actions_batch(rng, p.ce, s["pos"][None], s["has_flag"][None], eps=0.35, second_p=0.5)[0]
        p.step(a, f"{exp} t={t}", observe=t % 25 == 0 or t >= ec["GAME_STEPS"] - 1)
    p.counters("end")
    p.close()


def alt_env_config(name: str) -> dict:
    """alt_exp/<x>: the reference's alt_exp/<x>.py where its source tree is here, the shipped copy of that config otherwise."""
    return rs.alt_experiment_env_config(name.split("/", 1)[1]) if rs.source_tree_available() else local_env_config(name)


@pytest.mark.parametrize("name", local_experiment_names(alternative=True), ids=lambda n: n.split("/", 1)[1])
def test_alternative_experiment_configs_also_match(name, request):
    """alt_exp/*.py (arena, arena_ii, jailbreak_ii, ... maps that the nine main scripts do not use): every scenario dict
    of scenarios.py that has a script goes through the config compiler and the oracle, step by step against the reference."""
    p = Pair(request.node.name, alt_env_config(name), seed=7, env_id=77)
    p.dims()
    pol = traces.make_policy("builder" if 3 in p.ce.AGENT_TYPES.values() else "seek", p.ce)
    rng = np.random.default_rng(11)
    for t in range(150):
        s = p.orc.state()
        a = pol(rng, s["pos"], s["has_flag"])
        p.step(a, f"{name} t={t}", observe=t % 10 == 0)
    p.counters("end", visits=False)
    p.close()
