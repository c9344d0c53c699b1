"""Host-side mirror of the reference's ``GridworldCtf`` over the CUDA step path.

``GridworldCtfGPU`` is the batched environment: same constructor keywords as the
reference (gridworld_ctf.py:19-52) plus ``num_envs / device / seed``; ``reset()``
and ``step(actions)`` return device tensors for all B envs.  ``GridworldCtf`` is
the single-env view with the reference's exact method surface
(``standardise_state``, ``get_env_metadata``, ``step(list) -> (grid, rewards,
done)``, ``metrics`` …) so that un-modified callers (ppo.py:31-131,
utils.py:500-573, league_training.py:63-65) run on it.

PyTorch is used for device memory and streams only; all compute is in
libctf_b200.so (csrc/ctf_kernels.cu) behind the C ABI of include/ctf_b200.h.
There is no CPU path: constructing an env without a CUDA device raises.
"""
from __future__ import annotations

import ctypes as C
from collections import defaultdict

import numpy as np
import torch

from . import _native
from .compressible import compressible_empty, is_compressed
from .config import METRIC_NAMES, N_METRICS, compile_config, env_dims
from .sharding import all_reduce_stats

_STATS_LEVELS = {"none": 0, "counters": 1, "full": 2}
_OBS_DTYPES = {torch.float32: 0, torch.uint8: 1, torch.float16: 2, torch.bfloat16: 3}
_GRID_ROW = 16


class GridworldCtfGPU:
    """B independent GridworldCtf environments resident in HBM, stepped by one kernel launch."""

    def __init__(
        self,
        AGENT_CONFIG=None,
        SCENARIO=None,
        GAME_STEPS=256,
        GRID_SIZE=10,
        ENABLE_OBSTACLES=False,
        DROP_FLAG_WHEN_NO_HP=False,
        HOME_FLAG_CAPTURE=False,
        USE_EASY_CAPTURE=True,
        USE_ADJUSTED_REWARDS=False,
        MAX_BLOCK_TILE_PCT=0.2,
        LOG_METRICS=True,
        MAP_SYMMETRY_CHECK=True,
        AGENT_TYPE_HP=None,
        AGENT_HP_HEALING_PER_STEP=0.25,
        AGENT_TYPE_DAMAGE=None,
        TAG_PROBABILITY=0.75,
        GUARDIAN_DAMAGE_MULTIPLIER=5.0,
        VAULT_HP_COST=0.5,
        VAULT_MIN_HP=2.5,
        *,
        num_envs=1,
        device=None,
        seed=0,
        env_id_base=0,
        stats="none",
        obs_dtype=torch.float32,
        reverse_team1_actions=False,
        validate_actions=False,
        obs_out=None,
        meta_out=None,
        packed_obs=False,
        dense_obs=True,
    ):
        self._handle = None
        self._lib = _native.load()  # raises when the extension is missing
        if not torch.cuda.is_available():
            raise _native.NativeError("GridworldCtfGPU needs a CUDA device (sm_100a); there is no CPU fallback")
        # what pickling / copy.deepcopy rebuild the env from (Ray ships pickled env copies: league_training.py:686-687)
        self._ctor = dict(
            AGENT_CONFIG=AGENT_CONFIG, SCENARIO=SCENARIO, GAME_STEPS=GAME_STEPS, GRID_SIZE=GRID_SIZE,
            ENABLE_OBSTACLES=ENABLE_OBSTACLES, DROP_FLAG_WHEN_NO_HP=DROP_FLAG_WHEN_NO_HP, HOME_FLAG_CAPTURE=HOME_FLAG_CAPTURE,
            USE_EASY_CAPTURE=USE_EASY_CAPTURE, USE_ADJUSTED_REWARDS=USE_ADJUSTED_REWARDS, MAX_BLOCK_TILE_PCT=MAX_BLOCK_TILE_PCT,
            LOG_METRICS=LOG_METRICS, MAP_SYMMETRY_CHECK=MAP_SYMMETRY_CHECK, AGENT_TYPE_HP=AGENT_TYPE_HP,
            AGENT_HP_HEALING_PER_STEP=AGENT_HP_HEALING_PER_STEP, AGENT_TYPE_DAMAGE=AGENT_TYPE_DAMAGE,
            TAG_PROBABILITY=TAG_PROBABILITY, GUARDIAN_DAMAGE_MULTIPLIER=GUARDIAN_DAMAGE_MULTIPLIER, VAULT_HP_COST=VAULT_HP_COST,
            VAULT_MIN_HP=VAULT_MIN_HP, num_envs=num_envs, device=None if device is None else str(device), seed=seed,
            env_id_base=env_id_base, stats=stats, obs_dtype=obs_dtype, reverse_team1_actions=reverse_team1_actions,
            validate_actions=validate_actions, packed_obs=packed_obs, dense_obs=dense_obs,
        )
        self.ce = compile_config(
            AGENT_CONFIG=AGENT_CONFIG, SCENARIO=SCENARIO, GAME_STEPS=GAME_STEPS, GRID_SIZE=GRID_SIZE,
            ENABLE_OBSTACLES=ENABLE_OBSTACLES, DROP_FLAG_WHEN_NO_HP=DROP_FLAG_WHEN_NO_HP,
            HOME_FLAG_CAPTURE=HOME_FLAG_CAPTURE, USE_EASY_CAPTURE=USE_EASY_CAPTURE,
            USE_ADJUSTED_REWARDS=USE_ADJUSTED_REWARDS, MAX_BLOCK_TILE_PCT=MAX_BLOCK_TILE_PCT,
            LOG_METRICS=LOG_METRICS, MAP_SYMMETRY_CHECK=MAP_SYMMETRY_CHECK, AGENT_TYPE_HP=AGENT_TYPE_HP,
            AGENT_HP_HEALING_PER_STEP=AGENT_HP_HEALING_PER_STEP, AGENT_TYPE_DAMAGE=AGENT_TYPE_DAMAGE,
            TAG_PROBABILITY=TAG_PROBABILITY, GUARDIAN_DAMAGE_MULTIPLIER=GUARDIAN_DAMAGE_MULTIPLIER,
            VAULT_HP_COST=VAULT_HP_COST, VAULT_MIN_HP=VAULT_MIN_HP, reverse_team1_actions=reverse_team1_actions,
        )
        ce = self.ce
        # the attribute surface the reference's callers read (SURVEY.md §8b)
        for name in (
            "N_AGENTS", "GRID_SIZE", "GAME_STEPS", "FLIP_AXIS", "AGENT_CONFIG", "SCENARIO", "AGENT_TEAMS", "AGENT_TYPES",
            "AGENT_TILE_MAP", "AGENT_TYPE_ACTION_MASK", "AGENT_TYPE_HP", "AGENT_TYPE_DAMAGE", "OPPONENTS", "TILES_USED",
            "FLAG_POSITIONS", "CAPTURE_POSITIONS", "SPAWN_POSITIONS", "AGENT_STARTING_POSITIONS", "SCENARIO_NAME",
            "MAP_SYMMETRY_CHECK", "USE_ADJUSTED_REWARDS", "REVERSED_ACTION_MAP",
        ):
            setattr(self, name, getattr(ce, name))
        self.ACTION_SPACE = 8
        self.n_channels = ce.n_channels
        self.meta_size = ce.meta_size
        self.hp_scale = int(ce.cfg.hp_scale)

        self.num_envs = int(num_envs)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.type != "cuda":
            raise _native.NativeError(f"device must be a CUDA device, got {self.device}")
        dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.device = torch.device("cuda", dev_index)
        if stats not in _STATS_LEVELS:
            raise ValueError(f"stats must be one of {list(_STATS_LEVELS)}")
        if obs_dtype not in _OBS_DTYPES:
            raise ValueError("obs_dtype must be torch.float32, torch.uint8, torch.float16 or torch.bfloat16")
        self.stats_level = _STATS_LEVELS[stats]
        self.obs_dtype = obs_dtype
        self.seed = int(seed)
        self.env_id_base = int(env_id_base)
        self.validate_actions = bool(validate_actions)

        h = C.c_void_p()
        _native.check(
            self._lib.ctf_create(
                C.byref(ce.cfg), self.num_envs, dev_index, self.seed, self.env_id_base, self.stats_level,
                _OBS_DTYPES[obs_dtype], C.byref(h),
            )
        )
        self._handle = h
        sizes = _native.CtfSizes()
        _native.check(self._lib.ctf_get_sizes(self._handle, C.byref(sizes)))
        self.sizes = sizes

        B, N, G, Cn, M = self.num_envs, ce.N_AGENTS, ce.GRID_SIZE, ce.n_channels, ce.meta_size
        dev = self.device
        # ---- state (SoA of field groups, env-major), resident in HBM
        self._grid = torch.zeros((B, _GRID_ROW, _GRID_ROW), dtype=torch.uint8, device=dev)
        self._agents = torch.zeros((B, N), dtype=torch.int64, device=dev)
        self._envs = torch.zeros((B, 4), dtype=torch.int32, device=dev)
        # HP as doubles for configurations whose HP quantities are not dyadic (cfg.hp_float); fixed point in `_agents` otherwise
        self.hp_float = bool(ce.cfg.hp_float)
        self._hp = torch.zeros((B, N), dtype=torch.float64, device=dev) if self.hp_float else None
        self._stats = torch.zeros((B, N_METRICS, N), dtype=torch.int32, device=dev) if self.stats_level > 0 else None
        self._visits = torch.zeros((B, N, G, G), dtype=torch.uint8, device=dev) if self.stats_level > 1 else None
        # ---- outputs (the policy's input buffers unless the caller binds its own)
        # dense_obs=False skips the [B,N,C,G,G] buffer (storage-only use: packed_obs=True + unpack_obs on demand).
        # The env's own buffer is compressible memory where the device has it: the observations are ~90 % zero
        # sectors, so the step's store stream, which bounds it, moves far fewer DRAM bytes (DESIGN §4).
        self.obs = None
        if dense_obs:
            self.obs = compressible_empty((B, N, Cn, G, G), obs_dtype, dev) if obs_out is None else obs_out
            self._check_out(self.obs, (B, N, Cn, G, G), obs_dtype, "obs_out")
        elif not packed_obs:
            raise ValueError("dense_obs=False needs packed_obs=True")
        # packed copy of the same observations, 1 bit per element, [B, N, ceil(C*G*G/32)] int32 (rollout storage)
        self.bits_words_per_agent = int(sizes.bits_words_per_agent)
        self.obs_bits = torch.zeros((B, N, self.bits_words_per_agent), dtype=torch.int32, device=dev) if packed_obs else None
        self.meta = torch.empty((B, N, M), dtype=torch.float32, device=dev) if meta_out is None else meta_out
        self._check_out(self.meta, (B, N, M), torch.float32, "meta_out")
        self.rewards = torch.zeros((B, N), dtype=torch.float32, device=dev)
        self.dones = torch.zeros((B,), dtype=torch.uint8, device=dev)
        mask_rows = [[1] * 5 + [0] * 4 if ce.AGENT_TYPE_ACTION_MASK[ce.AGENT_TYPES[i]] == 1 else [1] * 9 for i in range(N)]
        self._mask_row = torch.tensor(mask_rows, dtype=torch.uint8, device=dev)
        # per-agent scalar flag as the reference's callers pass it to the policy (ppo.py:68, utils.py:530-533)
        self.use_action_mask = torch.tensor(
            [ce.AGENT_TYPE_ACTION_MASK[ce.AGENT_TYPES[i]] for i in range(N)], dtype=torch.float32, device=dev
        )
        self._state_struct = _native.CtfState(
            self._grid.data_ptr(), self._agents.data_ptr(), self._envs.data_ptr(),
            self._stats.data_ptr() if self._stats is not None else None,
            self._visits.data_ptr() if self._visits is not None else None,
            self._hp.data_ptr() if self._hp is not None else None,
        )
        self._first = True
        self.reset()
        if self.MAP_SYMMETRY_CHECK:
            # gridworld_ctf.py:476-477: standardise_state(0) == standardise_state(1, reverse_grid=True)
            flags = [0] * N
            if N > 1:
                flags[1] = 1
            if self.obs is not None:
                obs, _ = self.observe(reverse_flags=flags, into_new=True)
                assert N < 2 or bool(torch.equal(obs[0, 0], obs[0, 1])), "map symmetry check failed (gridworld_ctf.py:477)"

    # ------------------------------------------------------------------ plumbing
    def _check_out(self, t, shape, dtype, name):
        if tuple(t.shape) != tuple(shape) or t.dtype != dtype or t.device != self.device or not t.is_contiguous():
            raise ValueError(f"{name} must be a contiguous {dtype} tensor of shape {shape} on {self.device}")

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _step_outputs(self):
        """ctf_outputs_t of the bound buffers, rebuilt only when a buffer was rebound."""
        key = (self.obs.data_ptr() if self.obs is not None else 0, self.meta.data_ptr())
        if getattr(self, "_out_key", None) != key:
            self._out_key = key
            self._out_struct = self._outputs()
        return self._out_struct

    def _outputs(self, obs=True, meta=True, rewards=True, dones=True, obs_t=None, meta_t=None, bits=True):
        o = self.obs if obs_t is None else obs_t
        m = self.meta if meta_t is None else meta_t
        return _native.CtfOutputs(
            o.data_ptr() if (obs and o is not None) else None,
            self.obs_bits.data_ptr() if (bits and self.obs_bits is not None) else None,
            m.data_ptr() if meta else None,
            self.rewards.data_ptr() if rewards else None, self.dones.data_ptr() if dones else None,
        )

    def bind_outputs(self, obs=None, meta=None):
        """Write observations / metadata of later steps straight into the caller's (policy input) buffers."""
        B, N, G, Cn, M = self.num_envs, self.N_AGENTS, self.GRID_SIZE, self.n_channels, self.meta_size
        if obs is not None:
            self._check_out(obs, (B, N, Cn, G, G), self.obs_dtype, "obs")
            self.obs = obs
        if meta is not None:
            self._check_out(meta, (B, N, M), torch.float32, "meta")
            self.meta = meta

    # ------------------------------------------------------------------ pickling (Ray object store, copy.deepcopy)
    def __getstate__(self):
        """Constructor arguments + the decoded device state; the copy owns a new handle and new buffers (caller-bound
        output buffers are not carried over).  Synchronises."""
        return {"ctor": dict(self._ctor), "state": self.get_state(), "first": self._first}

    def __setstate__(self, d):
        ctor = dict(d["ctor"])
        ctor["MAP_SYMMETRY_CHECK"] = False                       # already checked when the original was built
        self.__init__(**ctor)
        self._ctor["MAP_SYMMETRY_CHECK"] = d["ctor"]["MAP_SYMMETRY_CHECK"]
        self.MAP_SYMMETRY_CHECK = d["ctor"]["MAP_SYMMETRY_CHECK"]
        st = d["state"]
        self.set_state(st["grid"], st["pos"], st["hp_q"], st["has_flag"], st["inventory"], st["step"], st["episode"], st["captures"],
                       hp=st.get("hp"))
        if self._stats is not None:
            self._stats.copy_(torch.from_numpy(st["stats"].astype(np.int32)))
        if self._visits is not None:
            self._visits.copy_(torch.from_numpy(st["visits"]))
        self._first = d["first"]
        # observations / metadata of the restored state; rewards and dones are those of the next step
        out = self._outputs(rewards=False, dones=False)
        _native.check(self._lib.ctf_observe(self._handle, self._state_struct, None, out, self._stream()))
        self.dones.copy_((self._envs[:, 0] >= self.GAME_STEPS).to(torch.uint8))

    def close(self):
        if getattr(self, "_handle", None) is not None:
            self._lib.ctf_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ the step path
    @property
    def action_mask(self) -> torch.Tensor:
        """[B, N, 9] uint8, 1 = allowed (static per agent type, AGENT_TYPE_ACTION_MASK gridworld_ctf.py:218-223)."""
        return self._mask_row.unsqueeze(0).expand(self.num_envs, -1, -1)

    def reset(self):
        """All envs back to the scenario's initial state (gridworld_ctf.py:383-477). Returns (obs, meta, action_mask)."""
        _native.check(
            self._lib.ctf_reset(self._handle, self._state_struct, self._outputs(), int(self._first), self._stream())
        )
        self._first = False
        return self.obs, self.meta, self.action_mask

    def step(self, actions):
        """actions: [B, N] integer tensor on the device (uint8 preferred). Returns (obs, meta, rewards, dones, action_mask)."""
        a = self._as_actions(actions)
        rc = self._lib.ctf_step(self._handle, self._state_struct, a.data_ptr(), self._step_outputs(), self._stream())
        if rc:
            _native.check(rc)
        self._last_actions = a  # keep alive until the launch has consumed it
        if self.validate_actions:
            self.raise_on_faults()
        return self.obs, self.meta, self.rewards, self.dones, self.action_mask

    def make_step_graph(self, actions: torch.Tensor, steps_per_replay: int = 1):
        """Captures ``steps_per_replay`` step launches on static buffers into a CUDA graph (launch-bound small batches).

        ``actions`` is the static uint8 [B, N] device tensor the caller refills before each replay (with
        steps_per_replay > 1 the same actions are applied every step — useful for no-op/benchmark loops only).
        The env state is unchanged by this call (the warm-up launch runs on a snapshot); the output buffers
        (obs / meta / rewards / dones) are overwritten.
        Returns the ``torch.cuda.CUDAGraph``; call ``.replay()``.  ctf_step makes no allocation and no host
        synchronisation, so it is capturable as is; a policy forward can be captured in the same graph by the caller.
        """
        a = self._as_actions(actions)
        if a.data_ptr() != actions.data_ptr():
            raise ValueError("actions must already be a contiguous uint8 [B, N] tensor on the env's device")
        # warm-up launch outside the capture, on a snapshot so that the env does not advance
        state = [t for t in (self._grid, self._agents, self._envs, self._stats, self._visits, self._hp) if t is not None]
        saved = [t.clone() for t in state]
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):
            self.step(a)   # with validate_actions this also checks the actions once, outside the capture
            for t, s_ in zip(state, saved):
                t.copy_(s_)
        torch.cuda.current_stream(self.device).wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        validate, self.validate_actions = self.validate_actions, False   # ctf_take_faults synchronises: not capturable
        try:
            with torch.cuda.graph(graph):
                for _ in range(int(steps_per_replay)):
                    self.step(a)
        finally:
            self.validate_actions = validate
        return graph

    def step_host(self, actions_host: torch.Tensor, rewards_host: torch.Tensor, dones_host: torch.Tensor):
        """Host-buffer step: uint8 actions [B,N] (pinned) in, float32 rewards [B,N] / uint8 dones [B] out; obs/meta stay on the device."""
        B, N = self.num_envs, self.N_AGENTS
        if actions_host.dtype != torch.uint8 or tuple(actions_host.shape) != (B, N) or actions_host.is_cuda:
            raise ValueError("actions_host must be a host uint8 tensor of shape [B, N]")
        if rewards_host.dtype != torch.float32 or tuple(rewards_host.shape) != (B, N) or rewards_host.is_cuda:
            raise ValueError("rewards_host must be a host float32 tensor of shape [B, N]")
        if dones_host.dtype != torch.uint8 or tuple(dones_host.shape) != (B,) or dones_host.is_cuda:
            raise ValueError("dones_host must be a host uint8 tensor of shape [B]")
        _native.check(
            self._lib.ctf_step_host(
                self._handle, self._state_struct, C.c_void_p(actions_host.data_ptr()), self._outputs(),
                C.c_void_p(rewards_host.data_ptr()), C.c_void_p(dones_host.data_ptr()), self._stream(),
            )
        )
        return self.obs, self.meta, rewards_host, dones_host

    def observe(self, reverse_flags=None, into_new=False):
        """standardise_state / get_env_metadata of the current state for all agents; reverse_flags: per-agent reverse_grid."""
        if self.obs is None:
            raise RuntimeError("this env was created with dense_obs=False; use obs_bits / unpack_obs")
        obs_t = torch.empty_like(self.obs) if into_new else self.obs
        meta_t = torch.empty_like(self.meta) if into_new else self.meta
        rf = None
        if reverse_flags is not None:
            rf = (C.c_uint8 * self.N_AGENTS)(*[int(bool(x)) for x in reverse_flags])
        out = self._outputs(rewards=False, dones=False, obs_t=obs_t, meta_t=meta_t, bits=False)
        _native.check(self._lib.ctf_observe(self._handle, self._state_struct, rf, out, self._stream()))
        return obs_t, meta_t

    def unpack_obs(self, packed: torch.Tensor, dtype=torch.float32, out=None) -> torch.Tensor:
        """Expands packed observations [..., words_per_agent] int32 (any leading shape, e.g. a minibatch gathered from
        a rollout buffer of ``env.obs_bits`` snapshots) into [..., C, G, G] of ``dtype`` with the CUDA unpack kernel."""
        if dtype not in _OBS_DTYPES:
            raise ValueError("dtype must be torch.float32, torch.uint8, torch.float16 or torch.bfloat16")
        wpa, Cn, G = self.bits_words_per_agent, self.n_channels, self.GRID_SIZE
        if packed.dtype != torch.int32 or packed.shape[-1] != wpa or packed.device != self.device:
            raise ValueError(f"packed must be an int32 tensor [..., {wpa}] on {self.device}")
        packed = packed.contiguous()
        lead = tuple(packed.shape[:-1])
        n = int(packed.numel() // wpa)
        if out is None:
            out = torch.empty(lead + (Cn, G, G), dtype=dtype, device=self.device)
        elif tuple(out.shape) != lead + (Cn, G, G) or out.dtype != dtype or not out.is_contiguous() or out.device != self.device:
            raise ValueError("out has the wrong shape / dtype / layout")
        _native.check(
            self._lib.ctf_unpack_obs(self._handle, packed.data_ptr(), out.data_ptr(), _OBS_DTYPES[dtype], n, self._stream())
        )
        return out

    def _as_actions(self, actions) -> torch.Tensor:
        if (isinstance(actions, torch.Tensor) and actions.dtype == torch.uint8 and actions.device == self.device
                and actions.is_contiguous() and tuple(actions.shape) == (self.num_envs, self.N_AGENTS)):
            return actions  # the common case: no conversion, no copy
        if not isinstance(actions, torch.Tensor):
            actions = torch.as_tensor(np.asarray(actions))
        if tuple(actions.shape) != (self.num_envs, self.N_AGENTS):
            raise ValueError(f"actions must have shape {(self.num_envs, self.N_AGENTS)}, got {tuple(actions.shape)}")
        if actions.dtype != torch.uint8:
            # anything outside 0..8 (KeyError in the reference) becomes 255 so that the device fault bit fires
            actions = torch.where((actions < 0) | (actions > 8), torch.full_like(actions, 255), actions).to(torch.uint8)
        return actions.to(self.device, non_blocking=True).contiguous()

    def take_faults(self) -> int:
        """Reads and clears the device fault word (synchronises): bit 0 = action outside 0..8, bit 1 = a lethal tag
        found the victim's 3x3 spawn window full (the reference raises there, gridworld_ctf.py:771), bit 2 = a row of
        ``ctf_sample_actions`` named a flat index outside [0, B*N)."""
        f = C.c_uint32(0)
        _native.check(self._lib.ctf_take_faults(self._handle, self._stream(), C.byref(f)))
        return int(f.value)

    def raise_on_faults(self):
        f = self.take_faults()
        if f & _native.FAULT_BAD_ACTION:
            raise KeyError("an action outside 0..8 was passed to step() (KeyError in the reference's ACTION_DELTAS lookup)")
        if f & _native.FAULT_RESPAWN_BLOCKED:
            raise ValueError("respawn found no open cell in a 3x3 spawn window (np.random.randint(0) raises ValueError in "
                             "the reference, gridworld_ctf.py:771); the victim was left in place with HP <= 0")
        if f & _native.FAULT_BAD_INDEX:
            raise IndexError("ctf_sample_actions was given a flat index outside [0, B*N); that row wrote nothing")

    @property
    def obs_compressed(self) -> bool:
        """Whether the bound observation buffer lies in memory the driver compresses (see ``compressible_empty``)."""
        return self.obs is not None and is_compressed(self.obs)

    @property
    def uses_persistent_kernel(self) -> bool:
        """Always False: step() launches the warp-per-env kernel k_step; kept for callers that name the kernel by it."""
        return False

    # ------------------------------------------------------------------ reference API that does not touch the device
    def get_env_dims(self):
        return env_dims(self.ce)

    def get_reversed_action(self, action):
        """gridworld_ctf.py:968-973."""
        return self.REVERSED_ACTION_MAP[self.FLIP_AXIS][int(action)]

    def reversed_action_lut(self) -> torch.Tensor:
        return torch.tensor([self.get_reversed_action(a) for a in range(9)], dtype=torch.int64, device=self.device)

    # ------------------------------------------------------------------ state access (tests, snapshots)
    def get_state(self, env_index=None) -> dict:
        """Decoded device state as CPU numpy arrays (synchronises).  ``env_index`` (int or slice) copies only those
        envs off the device; every array keeps its leading env axis."""
        G = self.GRID_SIZE
        if env_index is None:
            sel = slice(None)
        elif isinstance(env_index, slice):
            sel = env_index
        else:
            i = int(env_index)
            if not -self.num_envs <= i < self.num_envs:
                raise IndexError(f"env_index {i} out of range for {self.num_envs} envs")
            i %= self.num_envs
            sel = slice(i, i + 1)
        rec = self._agents[sel].cpu().numpy().astype(np.uint64)
        envs = self._envs[sel].cpu().numpy().astype(np.int64) & 0xFFFFFFFF
        out = {
            "grid": self._grid[sel, :G, :G].cpu().numpy(),
            "pos": np.stack([(rec & 0xFF), ((rec >> 8) & 0xFF)], axis=-1).astype(np.uint8),
            "has_flag": ((rec >> 16) & 1).astype(np.uint8),
            "hp_q": ((rec >> 32) & 0xFFFF).astype(np.uint16).view(np.int16).astype(np.int32),
            "inventory": ((rec >> 48) & 0xFFFF).astype(np.int32),
            "step": envs[:, 0].copy(),
            "episode": envs[:, 1].copy(),
            "captures": envs[:, 2:4].copy(),
        }
        if self._hp is not None:
            out["hp"] = self._hp[sel].cpu().numpy()          # agent_hp as float64
            out["hp_q"] = np.zeros_like(out["hp_q"])          # the record's HP field is a don't-care in this mode
        if self._stats is not None:
            out["stats"] = self._stats[sel].cpu().numpy().astype(np.int64) & 0xFFFFFFFF
        if self._visits is not None:
            out["visits"] = self._visits[sel].cpu().numpy()
        return out

    def set_state(self, grid, pos, hp_q, has_flag, inventory, step, episode, captures, hp=None):
        """Inverse of get_state for the core fields (arrays with a leading B dimension); ``hp`` (float64) when hp_float."""
        B, N, G = self.num_envs, self.N_AGENTS, self.GRID_SIZE
        if self.hp_float:
            if hp is None:
                raise ValueError("this env keeps HP as doubles (non-dyadic HP configuration): pass hp=")
            self._hp.copy_(torch.from_numpy(np.asarray(hp, dtype=np.float64).reshape(B, N)))
            hp_q = np.zeros((B, N), dtype=np.int64)
        g = np.zeros((B, _GRID_ROW, _GRID_ROW), dtype=np.uint8)
        g[:, :G, :G] = np.asarray(grid, dtype=np.uint8).reshape(B, G, G)
        pos = np.asarray(pos).reshape(B, N, 2).astype(np.uint64)
        rec = (
            pos[..., 0]
            | (pos[..., 1] << np.uint64(8))
            | (np.asarray(has_flag).reshape(B, N).astype(np.uint64) << np.uint64(16))
            | ((np.asarray(hp_q).reshape(B, N).astype(np.int64) & 0xFFFF).astype(np.uint64) << np.uint64(32))
            | ((np.asarray(inventory).reshape(B, N).astype(np.int64) & 0xFFFF).astype(np.uint64) << np.uint64(48))
        )
        envs = np.zeros((B, 4), dtype=np.int64)
        envs[:, 0] = np.asarray(step).reshape(B)
        envs[:, 1] = np.asarray(episode).reshape(B)
        envs[:, 2:4] = np.asarray(captures).reshape(B, 2)
        self._grid.copy_(torch.from_numpy(g))
        self._agents.copy_(torch.from_numpy(rec.view(np.int64)))
        self._envs.copy_(torch.from_numpy(envs.astype(np.uint32).view(np.int32)))

    def flag_captures(self) -> torch.Tensor:
        """metrics['team_flag_captures'] of every env: int64 [B, 2] (device)."""
        return self._envs[:, 2:4].long()

    def step_counts(self) -> torch.Tensor:
        """env_step_count of every env: int64 [B] (device)."""
        return self._envs[:, 0].long()

    def counters(self) -> torch.Tensor:
        """Per-env agent-level statistics, int64 [B, 13, N] in ctf_metric order (needs stats != 'none')."""
        if self._stats is None:
            raise RuntimeError("create the env with stats='counters' or 'full'")
        return self._stats.long()

    # ------------------------------------------------------------------ episode statistics (env.metrics schema)
    def stats_sum(self, all_reduce=True) -> torch.Tensor:
        """int64 [13, N]: counters summed over this rank's envs, then over ranks (NCCL) when torch.distributed is up."""
        if self.stats_level == 0:
            raise RuntimeError("create the env with stats='counters' or 'full' to collect episode statistics")
        out = torch.empty((N_METRICS, self.N_AGENTS), dtype=torch.int64, device=self.device)
        _native.check(self._lib.ctf_stats_sum(self._handle, self._state_struct, C.c_void_p(out.data_ptr()), self._stream()))
        if all_reduce:
            all_reduce_stats(out)
        return out

    def metrics_from_counters(self, counters: np.ndarray, visits=None) -> dict:
        """Agent-level counters [13, N] -> the reference's ``env.metrics`` dict (gridworld_ctf.py:425-470)."""
        return metrics_dict(self.ce, counters, visits)

    def episode_stats(self, all_reduce=True) -> dict:
        return self.metrics_from_counters(self.stats_sum(all_reduce=all_reduce).cpu().numpy())


def metrics_dict(ce, counters, visits=None) -> dict:
    """Rebuilds team / agent-type / agent level families from the agent-level counters.

    Every increment in the reference bumps the three levels together with the acting agent's
    (team, type, id) (e.g. gridworld_ctf.py:589-591), so the agent level determines the others.
    """
    counters = np.asarray(counters)
    n = ce.N_AGENTS
    m = {"team_wins": {0: 0, 1: 0}}
    for k, name in enumerate(METRIC_NAMES):
        team = {0: 0, 1: 0}
        by_type = defaultdict(lambda: defaultdict(int))
        agent = defaultdict(int)
        for i in range(n):
            v = int(counters[k, i])
            team[ce.AGENT_TEAMS[i]] += v
            if v:
                by_type[ce.AGENT_TEAMS[i]][ce.AGENT_TYPES[i]] += v
                agent[i] += v
        m["team_" + name] = team
        m["agent_type_" + name] = by_type
        m["agent_" + name] = agent
    g = ce.GRID_SIZE
    vm = defaultdict(lambda: np.zeros((g, g), dtype=np.uint8))
    if visits is not None:
        for i in range(n):
            vm[i] = np.asarray(visits[i], dtype=np.uint8)
    m["agent_visitation_maps"] = vm
    return m


_VIEW_ATTRS = (
    "N_AGENTS", "GRID_SIZE", "GAME_STEPS", "FLIP_AXIS", "AGENT_CONFIG", "SCENARIO", "AGENT_TEAMS", "AGENT_TYPES",
    "AGENT_TILE_MAP", "AGENT_TYPE_ACTION_MASK", "AGENT_TYPE_HP", "AGENT_TYPE_DAMAGE", "OPPONENTS", "TILES_USED",
    "FLAG_POSITIONS", "CAPTURE_POSITIONS", "SPAWN_POSITIONS", "AGENT_STARTING_POSITIONS", "SCENARIO_NAME",
    "ACTION_SPACE", "REVERSED_ACTION_MAP",
)


class GridworldCtf:
    """Single-env view with the reference's exact surface (gridworld_ctf.py), backed by one GPU env.

    Every call synchronises with the device, so this is for drop-in compatibility of un-modified
    callers and for parity tests — throughput work uses ``GridworldCtfGPU`` directly.
    """

    def __init__(self, *args, device=None, seed=0, env_id=0, **kwargs):
        kwargs.setdefault("MAP_SYMMETRY_CHECK", True)
        self._gpu = GridworldCtfGPU(
            *args, num_envs=1, device=device, seed=seed, env_id_base=env_id, stats="full", obs_dtype=torch.uint8, **kwargs
        )
        g = self._gpu
        for name in _VIEW_ATTRS:
            setattr(self, name, getattr(g, name))
        self._cache = {}

    def __getstate__(self):
        return {"gpu": self._gpu}

    def __setstate__(self, d):
        self._gpu = d["gpu"]
        for name in _VIEW_ATTRS:
            setattr(self, name, getattr(self._gpu, name))
        self._cache = {}

    # -- reference methods
    def reset(self):
        self._gpu.reset()
        self._cache = {}

    def step(self, actions):
        a = np.asarray([int(x) for x in actions], dtype=np.int64)
        if a.shape != (self.N_AGENTS,):
            raise ValueError(f"expected {self.N_AGENTS} actions")
        if ((a < 0) | (a > 8)).any():
            raise KeyError(int(a[(a < 0) | (a > 8)][0]))  # ACTION_DELTAS lookup (gridworld_ctf.py:710)
        _, _, rewards, dones, _ = self._gpu.step(torch.from_numpy(a.astype(np.uint8)).unsqueeze(0))
        self._cache = {}
        r = rewards[0].cpu().tolist()
        return self.grid, r, bool(dones[0].item())

    def standardise_state(self, agent_idx, reverse_grid=False):
        i, rev = int(agent_idx), bool(reverse_grid)
        if rev == (self.AGENT_TEAMS[i] != 0):
            # the view every caller asks for (ppo.py:69/87, utils.py:535): already written by the last step / reset
            if "canonical" not in self._cache:
                self._cache["canonical"] = self._gpu.obs[0].cpu().numpy()
            return self._cache["canonical"][i][None].copy()
        key = ("obs", rev)
        if key not in self._cache:
            obs, _ = self._gpu.observe(reverse_flags=[int(rev)] * self.N_AGENTS, into_new=True)
            self._cache[key] = obs[0].cpu().numpy()
        return self._cache[key][i][None].copy()

    def get_env_metadata(self, agent_idx):
        if "meta" not in self._cache:
            self._cache["meta"] = self._gpu.meta[0].cpu().numpy()  # written by the last step / reset
        return self._cache["meta"][int(agent_idx)].astype(np.float16)[None]

    def get_env_dims(self):
        return self._gpu.get_env_dims()

    def get_reversed_action(self, action):
        return self._gpu.get_reversed_action(action)

    # -- reference attributes, read back from the device
    def _state(self):
        if "state" not in self._cache:
            self._cache["state"] = self._gpu.get_state()
        return self._cache["state"]

    @property
    def grid(self):
        return self._state()["grid"][0]

    @property
    def agent_positions(self):
        p = self._state()["pos"][0]
        return {i: (int(p[i, 0]), int(p[i, 1])) for i in range(self.N_AGENTS)}

    @property
    def has_flag(self):
        return self._state()["has_flag"][0]

    @property
    def agent_hp(self):
        st = self._state()
        if self._gpu.hp_float:
            return {i: float(st["hp"][0][i]) for i in range(self.N_AGENTS)}
        hp = st["hp_q"][0]
        return {i: float(hp[i]) / self._gpu.hp_scale for i in range(self.N_AGENTS)}

    @property
    def block_inventory(self):
        inv = self._state()["inventory"][0]
        return {i: int(inv[i]) for i in range(self.N_AGENTS)}

    @property
    def env_step_count(self):
        return int(self._state()["step"][0])

    @property
    def done(self):
        return self.env_step_count >= self.GAME_STEPS

    @property
    def metrics(self):
        st = self._state()
        m = metrics_dict(self._gpu.ce, st["stats"][0], st["visits"][0])
        # team_flag_captures is authoritative in the env record (also used by get_env_metadata)
        return m
