"""Policy inference from packed observations: the trunk of ``CtfPolicy`` as one CUDA kernel.

``FusedPolicy(env, policy)`` runs a ``CtfPolicy`` (or the reference ``Agent``'s weights loaded into one) for rollouts,
duels and league evaluation without dense observations.  ``ctf_policy_features`` (``k_policy_trunk`` in
csrc/ctf_kernels.cu) reads the env's packed 1-bit observations (``env.obs_bits``) and metadata in place and writes
one bf16 fc1 input row per sample: conv1 by sparse fp32 accumulation over the set bits, tanh, bf16, conv2 on tensor
cores with fp32 accumulation, tanh, bf16, then the metadata.  fc1 -> tanh -> fc2 -> tanh -> heads run in torch
(cuBLAS, bf16 weights, fp32 accumulation) on those rows: fc1 runs over the whole stride with fc1.weight zero-padded
to it (the pad columns of the rows are exact zeros), which keeps K a multiple of 8 for cuBLAS.  The env can then be created packed-only
(``dense_obs=False, packed_obs=True``) and never writes the dense observation tensor.

Precision: this is a bf16 path, like running ``CtfPolicy`` under ``torch.autocast(dtype=torch.bfloat16)``; it is not
bit-equal to fp32 ``CtfPolicy``.  ``reference_features`` states in torch exactly what the kernel computes.

Training: ``FusedPolicy.evaluate_actions`` is the differentiable counterpart of ``CtfPolicy.get_action_and_value`` with
a given action, for the PPO update on a packed minibatch.  Its trunk runs ``ctf_policy_features`` forward and
``ctf_policy_features_backward`` (``k_policy_trunk_backward``) for the conv1 / conv2 gradients; fc1 ... heads run in
bf16 through autograd.  ``reference_trunk_grads`` states in torch what the backward kernel computes.  Each sample keeps
2 x stride bf16 values alive between forward and backward (its rows and their gradient: 15.6 KB at 8_arena), so a
caller splits a large minibatch into chunks and lets the gradients accumulate.

Seeded sampling: with ``seed=`` (``FusedPolicy.get_action_and_value`` / ``get_action``, ``PolicyPool.act``) the head's
output rows go straight to ``ctf_sample_actions`` (``k_sample_actions``), one kernel that masks, samples and writes the
log-prob, the entropy and the env's action buffer.  Each draw is a Philox word keyed by (seed, global env id, episode,
step, agent), like the env's own draws (draws.py), so the actions do not depend on torch's random state or on how the
envs are batched.  ``seed=None`` keeps torch's ``Categorical``.

Several policies on one env batch: ``PolicyPool(env, policies)`` runs any number of (policy, env slice, agent ids)
segments with one ``ctf_policy_features_grouped`` launch (``k_policy_trunk_grouped``, the same per-sample code as
``k_policy_trunk``, so every row is bit-identical to ``FusedPolicy``'s) and one bf16 ``torch.baddbmm`` head chain over
all policies; league evaluation uses it (``league.duel_pairs(grouped=True)``).
"""
from __future__ import annotations

import ctypes as C

import torch
import torch.nn.functional as F
from torch.distributions.categorical import Categorical

from . import _native

N_ACTIONS = 9
MAX_IDS = 8


def trunk_dims(n_channels: int, grid_size: int, metadata_size: int):
    """(K1, feature_stride): fc1 input width 32*(G-4)^2 + M and the row stride of the kernel's output (multiple of 8)."""
    side = grid_size - 4
    k1 = 32 * side * side + metadata_size
    return k1, (k1 + 7) // 8 * 8


def conv2_kernel_layout_index(device=None) -> torch.Tensor:
    """Index into ``conv2.weight.reshape(-1)`` ([32][16][3][3]) that gives the kernel's bf16 layout
    [tap 9][n-tile 4][lane 32][4]: the two mma.sync m16n8k16 B registers of every lane.  Lane 4*g + t of n-tile j holds,
    for output channel 8*j + g, input channels (2t, 2t+1, 2t+8, 2t+9) of the tap (K = the 16 input channels of a tap)."""
    tap = torch.arange(9).view(9, 1, 1, 1)
    nt = torch.arange(4).view(1, 4, 1, 1)
    lane = torch.arange(32).view(1, 1, 32, 1)
    g, t = lane // 4, lane % 4
    ci = 2 * t + torch.tensor([0, 1, 8, 9]).view(1, 1, 1, 4)
    return ((8 * nt + g) * 144 + ci * 9 + tap).reshape(-1).to(device)


def conv2_transpose_layout_index(device=None) -> torch.Tensor:
    """Index into ``conv2.weight.reshape(-1)`` that gives the backward kernel's bf16 layout of conv2 transposed,
    [tap 9][k-half 2][n-tile 2][lane 32][4]: the mma.sync m16n8k16 B registers of dh1 = conv2^T(dz2), whose K is the
    32 output channels of a tap (two k-steps) and N the 16 input channels.  Lane 4*g + t of n-tile j in k-half h holds,
    for input channel 8*j + g, output channels 16*h + (2t, 2t+1, 2t+8, 2t+9) of the tap."""
    tap = torch.arange(9).view(9, 1, 1, 1, 1)
    kh = torch.arange(2).view(1, 2, 1, 1, 1)
    nt = torch.arange(2).view(1, 1, 2, 1, 1)
    lane = torch.arange(32).view(1, 1, 1, 32, 1)
    g, t = lane // 4, lane % 4
    co = 16 * kh + 2 * t + torch.tensor([0, 1, 8, 9]).view(1, 1, 1, 1, 4)
    return (co * 144 + (8 * nt + g) * 9 + tap).reshape(-1).to(device)


@torch.no_grad()
def reference_conv1(policy, dense_obs: torch.Tensor, round_bf16: bool = True) -> torch.Tensor:
    """conv1 -> tanh as ``k_policy_trunk`` computes it: [S, 16, G-2, G-2] float32.  Every output starts at its fp32 bias
    and adds ``x * W1[:, c, dy, dx]`` in the kernel's order (dy, dx, then c ascending), one fp32 rounding per term; for
    {0,1} inputs the products are exact and the sum is bit-for-bit the kernel's.  Then tanh, and bf16 if round_bf16."""
    x = dense_obs.float()
    S, Cn, G, _ = x.shape
    S1 = G - 2
    w1 = policy.conv1.weight.float()
    acc = policy.conv1.bias.float().view(1, 16, 1, 1).expand(S, 16, S1, S1).clone()
    for dy in range(3):
        for dx in range(3):
            for c in range(Cn):
                acc += x[:, c : c + 1, dy : dy + S1, dx : dx + S1] * w1[:, c, dy, dx].view(1, 16, 1, 1)
    h1 = torch.tanh(acc)
    return h1.bfloat16().float() if round_bf16 else h1


@torch.no_grad()
def reference_features(policy, dense_obs: torch.Tensor, meta: torch.Tensor, round_bf16: bool = True) -> torch.Tensor:
    """What ``k_policy_trunk`` computes, in torch: [S, K1] float32 (bf16 values when ``round_bf16``).

    conv1 summed in fp32 in the kernel's order (``reference_conv1``), tanh, bf16; conv2 of those bf16 activations with
    bf16 weights, summed exactly and rounded to fp32 (the kernel accumulates in fp32 on tensor cores, in an order of the
    hardware's), + fp32 bias, tanh, bf16; flattened in (c, y, x) order, then the metadata as bf16.  With
    round_bf16=False every rounding to bf16 is skipped, and the rows fed through fc1 ... heads reproduce
    ``CtfPolicy.forward`` in fp32.
    """
    bf = (lambda x: x.bfloat16().float()) if round_bf16 else (lambda x: x)
    h1 = reference_conv1(policy, dense_obs, round_bf16)
    w2 = bf(policy.conv2.weight.float()).double()
    h2 = F.conv2d(h1.double(), w2).float() + policy.conv2.bias.float().view(1, -1, 1, 1)
    h2 = bf(torch.tanh(h2))
    return torch.cat((h2.reshape(h2.shape[0], -1), bf(meta.float())), dim=1)


def reference_trunk_grads(policy, dense_obs: torch.Tensor, grad_rows: torch.Tensor, round_bf16: bool = True,
                          features: torch.Tensor | None = None):
    """What ``k_policy_trunk_backward`` computes, in torch: the gradients (conv1.weight, conv1.bias, conv2.weight,
    conv2.bias) of sum(rows[:, :32*(G-4)^2] * grad_rows[:, :32*(G-4)^2]), float32.

    h1 is ``reference_conv1`` (bf16 values); h2 is the conv2 part of ``features`` (the rows the forward kernel wrote)
    or, when None, of ``reference_features``; dz2 = bf16(dF * (1 - h2^2)) in fp32 operations; db2 and dW2 = dz2 (x) h1
    are summed exactly (float64) and rounded to fp32 once; dh1 = conv2^T(dz2) with bf16 weights, summed exactly and
    rounded to fp32; dz1 = dh1 * (1 - h1^2) in fp32; dW1 and db1 are exact sums of dz1 over the set input bits, rounded
    once.  The kernel's sums are fp32 (tensor cores for dW2, db2 and dh1, ordered adds for dW1 and db1), which is the
    whole difference.  With round_bf16=False nothing is rounded: everything runs in float64 from the float64
    parameters (``features`` is ignored) and the result, float64, is autograd of the ``CtfPolicy`` trunk.
    """
    from torch.nn.grad import conv2d_input, conv2d_weight

    S, Cn, G, _ = dense_obs.shape
    S2 = G - 4
    n2 = 32 * S2 * S2
    x = dense_obs.double()
    w1, b1 = policy.conv1.weight.detach(), policy.conv1.bias.detach()
    w2, b2 = policy.conv2.weight.detach(), policy.conv2.bias.detach()
    with torch.no_grad():
        if round_bf16:
            h1 = reference_conv1(policy, dense_obs)
            if features is None:
                h2 = F.conv2d(h1.double(), w2.float().bfloat16().double()).float() + b2.float().view(1, -1, 1, 1)
                h2 = torch.tanh(h2).bfloat16().float()
            else:
                h2 = features[:, :n2].float().reshape(S, 32, S2, S2)
            d = grad_rows[:, :n2].float().reshape(S, 32, S2, S2)
            dz2 = (d * (1 - h2 * h2)).bfloat16().float()
            dh1 = conv2d_input(h1.shape, w2.float().bfloat16().double(), dz2.double()).float()
            dz1 = dh1 * (1 - h1 * h1)
            out = (conv2d_weight(x, w1.shape, dz1.double()), dz1.double().sum((0, 2, 3)),
                   conv2d_weight(h1.double(), w2.shape, dz2.double()), dz2.double().sum((0, 2, 3)))
            return tuple(t.float() for t in out)
        w1, b1, w2, b2 = w1.double(), b1.double(), w2.double(), b2.double()
        h1 = torch.tanh(F.conv2d(x, w1, b1))
        h2 = torch.tanh(F.conv2d(h1, w2, b2))
        dz2 = grad_rows[:, :n2].double().reshape(S, 32, S2, S2) * (1 - h2 * h2)
        dz1 = conv2d_input(h1.shape, w2, dz2) * (1 - h1 * h1)
        return (conv2d_weight(x, w1.shape, dz1), dz1.sum((0, 2, 3)), conv2d_weight(h1, w2.shape, dz2),
                dz2.sum((0, 2, 3)))


def _check_policies(env, policies):
    """(K1, stride) of ``env``'s trunk (``trunk_dims``).  Raises ValueError unless the env has G >= 5 and every policy
    has the layer shapes of a CtfPolicy for ``env`` and lives on its device."""
    Cn, G, M = env.n_channels, env.GRID_SIZE, env.meta_size
    if G < 5:
        raise ValueError(f"the policy needs GRID_SIZE >= 5 (two valid 3x3 convolutions), env has {G}")
    k1, stride = trunk_dims(Cn, G, M)
    want = {
        "conv1.weight": (16, Cn, 3, 3), "conv2.weight": (32, 16, 3, 3), "fc1.weight": (256, k1),
        "fc2.weight": (128, 256), "action_head.weight": (N_ACTIONS, 128), "value_head.weight": (1, 128),
    }
    for policy in policies:
        for name, shape in want.items():
            mod, attr = name.split(".")
            got = tuple(getattr(getattr(policy, mod, None), attr, torch.empty(0)).shape)
            if got != shape:
                raise ValueError(f"policy {name} has shape {got}; this env (C={Cn}, G={G}, M={M}, {N_ACTIONS} actions) "
                                 f"needs {shape}")
        if policy.conv1.weight.device != env.device:
            raise ValueError(f"policy is on {policy.conv1.weight.device}, env on {env.device}")
    return k1, stride


def _check_agent_ids(agent_ids, n_per_env, where=""):
    """``agent_ids`` (a sequence or tensor) as a tuple of ints; raises ValueError (message prefixed by ``where``) unless
    it names 1..MAX_IDS agents, each in [0, n_per_env)."""
    ids = tuple(int(i) for i in (agent_ids.tolist() if isinstance(agent_ids, torch.Tensor) else agent_ids))
    if not 1 <= len(ids) <= MAX_IDS:
        raise ValueError(f"{where}agent ids must name 1..{MAX_IDS} agents, got {len(ids)}")
    if any(i < 0 or i >= n_per_env for i in ids):
        raise ValueError(f"{where}agent ids {ids} out of range for {n_per_env} agents per env")
    return ids


def _check_packed(env, bits, meta):
    """Raises ValueError unless ``bits`` is int32 [S, wpa] and ``meta`` float32 [S, M] on ``env``'s device."""
    wpa, M = env.bits_words_per_agent, env.meta_size
    if bits.dtype != torch.int32 or bits.dim() != 2 or bits.shape[1] != wpa or bits.device != env.device:
        raise ValueError(f"bits must be an int32 tensor [S, {wpa}] on {env.device}")
    if meta.dtype != torch.float32 or tuple(meta.shape) != (bits.shape[0], M) or meta.device != env.device:
        raise ValueError(f"meta must be a float32 tensor [{bits.shape[0]}, {M}] on {env.device}")


def _check_seed(seed) -> int:
    seed = int(seed)
    if not 0 <= seed < 1 << 64:
        raise ValueError(f"a policy seed must be in [0, 2**64), got {seed}")
    return seed


def sample_actions(env, head_out: torch.Tensor, masked, flat_index: torch.Tensor, seed: int, actions=None):
    """One ``ctf_sample_actions`` launch on the current stream: (action int64 [S], logprob [S], entropy [S]) of the rows
    of ``head_out`` (fp32 [S, 10], value then the 9 logits, unit column stride), drawn with ``seed`` for the agents
    ``flat_index`` (int64 [S], env * N + agent of ``env``) at the env's current episode and step.  ``masked``: uint8
    [S] (nonzero: ``CtfPolicy.masked_logits`` applies) or None.  ``actions`` (uint8 [B, N], contiguous) also receives
    every action at its flat index when given."""
    seed = _check_seed(seed)
    S, dev = head_out.shape[0], env.device
    a = torch.empty(S, dtype=torch.int64, device=dev)
    logp, ent = torch.empty(S, dtype=torch.float32, device=dev), torch.empty(S, dtype=torch.float32, device=dev)
    if S == 0:
        return a, logp, ent
    ptr = lambda t: C.c_void_p(None if t is None else t.data_ptr())
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    _native.check(env._lib.ctf_sample_actions(
        env._handle, env._state_struct, ptr(head_out), head_out.stride(0), ptr(masked), ptr(flat_index), S, seed,
        ptr(actions), ptr(a), ptr(logp), ptr(ent), stream))
    return a, logp, ent


def _check_actions(env, actions):
    if actions.dtype != torch.uint8 or tuple(actions.shape) != (env.num_envs, env.N_AGENTS) \
            or not actions.is_contiguous() or actions.device != env.device:
        raise ValueError(f"actions must be a contiguous uint8 tensor [{env.num_envs}, {env.N_AGENTS}] on {env.device}")


def _trunk_forward(env, weights, packed_ptr, meta_ptr, n_envs, agents_per_env, ids, k, out, stride):
    """Runs ``ctf_policy_features`` on the current stream with ``weights`` (``C.byref`` of a ``CtfPolicyWeights``) into
    ``out``, bf16 [n_envs * k, stride]; returns ``out``."""
    stream = C.c_void_p(torch.cuda.current_stream(env.device).cuda_stream)
    _native.check(env._lib.ctf_policy_features(
        env._handle, weights, C.c_void_p(packed_ptr), C.c_void_p(meta_ptr), n_envs, agents_per_env, ids, k,
        C.c_void_p(out.data_ptr()), stride, stream))
    return out


class _TrunkWeights:
    """The conv weights of L policies in the layouts the trunk kernels read, one slot per policy: conv1.weight and the
    biases fp32, conv2.weight bf16 gathered by ``conv2_kernel_layout_index`` and, with ``transposed`` (the backward),
    also by ``conv2_transpose_layout_index`` into ``c2wt``.  ``native`` is the ``CtfPolicyWeights`` array over the
    slots.  ``load`` copies into the buffers in place, so the pointers (and CUDA graphs captured around them) stay."""

    def __init__(self, L, n_channels, device, transposed=False):
        f32, bf = dict(dtype=torch.float32, device=device), dict(dtype=torch.bfloat16, device=device)
        self.c1w = torch.empty((L, 16, n_channels, 3, 3), **f32)
        self.c1b = torch.empty((L, 16), **f32)
        self.c2w = torch.empty((L, 9 * 4 * 32 * 4), **bf)
        self.c2b = torch.empty((L, 32), **f32)
        self._c2_index = conv2_kernel_layout_index(device)
        self.c2wt = torch.empty((L, 9 * 2 * 2 * 32 * 4), **bf) if transposed else None
        self._c2t_index = conv2_transpose_layout_index(device) if transposed else None
        self.native = (_native.CtfPolicyWeights * L)(*(
            _native.CtfPolicyWeights(self.c1w[p].data_ptr(), self.c1b[p].data_ptr(), self.c2w[p].data_ptr(),
                                     self.c2b[p].data_ptr()) for p in range(L)))

    @torch.no_grad()
    def load(self, slot, w1, b1, w2, b2):
        self.c1w[slot].copy_(w1)
        self.c1b[slot].copy_(b1)
        w2 = w2.reshape(-1)
        self.c2w[slot].copy_(w2[self._c2_index])
        if self.c2wt is not None:
            self.c2wt[slot].copy_(w2[self._c2t_index])
        self.c2b[slot].copy_(b2)


class _HeadWeights:
    """bf16 copies of the fc1, fc2 and value | action head layers of L policies, one slot per policy: fc1.weight in
    columns :K1 of [256, stride], zeros after (a K that is a multiple of 8 keeps cuBLAS on its aligned kernel; the pad
    columns of the feature rows are zeros too), fc2 [128, 256], the value and action heads stacked as [1 + 9, 128]."""

    def __init__(self, L, k1, stride, device):
        bf = dict(dtype=torch.bfloat16, device=device)
        self.k1 = k1
        self.fc1w, self.fc1b = torch.zeros((L, 256, stride), **bf), torch.empty((L, 256), **bf)
        self.fc2w, self.fc2b = torch.empty((L, 128, 256), **bf), torch.empty((L, 128), **bf)
        self.hw, self.hb = torch.empty((L, 1 + N_ACTIONS, 128), **bf), torch.empty((L, 1 + N_ACTIONS), **bf)

    @torch.no_grad()
    def load(self, slot, policy):
        self.fc1w[slot, :, : self.k1].copy_(policy.fc1.weight)
        self.fc1b[slot].copy_(policy.fc1.bias)
        self.fc2w[slot].copy_(policy.fc2.weight)
        self.fc2b[slot].copy_(policy.fc2.bias)
        self.hw[slot, :1].copy_(policy.value_head.weight)
        self.hw[slot, 1:].copy_(policy.action_head.weight)
        self.hb[slot, :1].copy_(policy.value_head.bias)
        self.hb[slot, 1:].copy_(policy.action_head.bias)


class _PackedTrunk(torch.autograd.Function):
    """rows = trunk(bits, meta; conv1, conv2) through ctf_policy_features, with ctf_policy_features_backward as its
    backward.  The rows are saved (a tensor of their own) and the backward re-reads the parameters it was given."""

    @staticmethod
    def forward(ctx, bits, w1, b1, w2, b2, fused, meta):
        rows = fused._train_forward(bits, meta, w1, b1, w2, b2)
        ctx.fused = fused
        ctx.save_for_backward(bits, rows, w1, b1, w2, b2)
        return rows

    @staticmethod
    def backward(ctx, grad_rows):
        bits, rows, w1, b1, w2, b2 = ctx.saved_tensors
        g = ctx.fused._train_backward(bits, rows, grad_rows, w1, b1, w2, b2)
        return (None, *g, None, None)


class FusedPolicy:
    """Inference-only view of a ``CtfPolicy`` that reads packed observations (see the module docstring).

    ``refresh()`` copies the module's current weights into persistent device buffers in place (called once here;
    call it again after every optimiser step): a CUDA graph captured around ``forward_*`` stays valid.
    """

    def __init__(self, env, policy):
        self.env, self.policy = env, policy
        self.k1, self.stride = _check_policies(env, [policy])
        self._trunk_w = _TrunkWeights(1, env.n_channels, env.device)
        self._weights = self._trunk_w.native[0]     # the CtfPolicyWeights of the one slot, what the trunk reads
        self._head_w = _HeadWeights(1, self.k1, self.stride, env.device)
        # the one slot's 2-D views, what _head passes to F.linear (value | logits heads stacked)
        hw = self._head_w
        self._fc1w, self._fc1b, self._fc2w, self._fc2b, self._hw, self._hb = (
            t[0] for t in (hw.fc1w, hw.fc1b, hw.fc2w, hw.fc2b, hw.hw, hw.hb))
        self._features = None   # bf16 [S_max, stride] rows, reused by every call (see features())
        self._ids = {}
        self._flat = {}         # (ids, e0, e1, N) -> int64 [S] device flat indices env * N + agent of the samples
        self._train = None      # training-only weight buffers and workspace, created by the first evaluate_actions
        self.refresh()

    def refresh(self):
        """Copies the policy's current weights into the persistent buffers, on the device (no host round trip)."""
        p = self.policy
        self._trunk_w.load(0, p.conv1.weight, p.conv1.bias, p.conv2.weight, p.conv2.bias)
        self._head_w.load(0, p)

    # ------------------------------------------------------------------ plumbing
    def _env_for(self, env):
        if env is None:
            return self.env
        mine = (self.env.n_channels, self.env.GRID_SIZE, self.env.meta_size, self.env.bits_words_per_agent)
        if (env.n_channels, env.GRID_SIZE, env.meta_size, env.bits_words_per_agent) != mine or env.device != self.env.device:
            raise ValueError("env does not have the shapes (C, G, M) or the device this FusedPolicy was built for")
        return env

    def _id_array(self, agent_ids, n_per_env):
        ids = _check_agent_ids(agent_ids, n_per_env)
        arr = self._ids.get(ids)
        if arr is None:
            arr = self._ids[ids] = (C.c_uint8 * len(ids))(*ids)
        return arr, len(ids)

    def features(self, n_samples: int) -> torch.Tensor:
        """bf16 [n_samples, stride] feature rows: the first rows of ONE buffer per FusedPolicy, sized for the largest
        sample count seen so far (8_arena, B = 65 536, one team: 2 GB).  A call with more samples than ever before
        replaces the buffer, so warm up with the largest forward before capturing a CUDA graph around this policy."""
        if self._features is None or self._features.shape[0] < n_samples:
            self._features = None   # release the old rows before allocating the larger ones
            self._features = torch.empty((n_samples, self.stride), dtype=torch.bfloat16, device=self.env.device)
        return self._features[:n_samples]

    def _head_out(self, feat):
        """fp32 [S, 10]: the value, then the 9 logits, of every feature row."""
        x = torch.tanh(F.linear(feat, self._fc1w, self._fc1b))
        x = torch.tanh(F.linear(x, self._fc2w, self._fc2b))
        return F.linear(x, self._hw, self._hb).float()

    def _head(self, feat):
        out = self._head_out(feat)
        return out[:, :1], out[:, 1:]

    def _flat_index(self, agent_ids, env, envs):
        """int64 [S] on the device: env * N + agent of every sample of ``trunk_from_env(agent_ids, env, envs)``."""
        N = env.N_AGENTS
        ids = _check_agent_ids(agent_ids, N)
        e0, e1, _ = (envs if envs is not None else slice(None)).indices(env.num_envs)
        key = (ids, e0, max(e1, e0), N)
        flat = self._flat.get(key)
        if flat is None:
            k = len(ids)
            s = torch.arange((key[2] - e0) * k)
            flat = self._flat[key] = ((e0 + s // k) * N + torch.tensor(ids)[s % k]).to(env.device)
        return flat

    def _seeded(self, use_action_mask, agent_ids, bits, env, envs, seed, actions):
        """(action, logprob, entropy, value) of ``get_action_and_value`` with ``seed``: one ``ctf_sample_actions``."""
        if agent_ids is None or bits is not None:
            raise ValueError("a seeded draw is keyed by (env, episode, step, agent): pass agent_ids (read the env in "
                             "place), not bits / meta")
        env = self._env_for(env)
        if actions is not None:
            _check_actions(env, actions)
        out = self._head_out(self.trunk_from_env(agent_ids, env, envs))
        masked = (use_action_mask.reshape(-1) == 1).to(torch.uint8) if self.policy.use_masking else None
        a, logp, ent = sample_actions(env, out, masked, self._flat_index(agent_ids, env, envs), seed, actions)
        return a, logp, ent, out[:, :1]

    # ------------------------------------------------------------------ trunk and forwards
    def trunk_from_env(self, agent_ids, env=None, envs=None) -> torch.Tensor:
        """bf16 feature rows [S, stride] (the fc1 input in columns :K1, zeros after) for the agents ``agent_ids`` of
        every env (or of ``envs``, a slice of env indices), read in place from ``env.obs_bits`` / ``env.meta``; sample
        s = e*k + j is agent agent_ids[j] of env e.  ``env`` defaults to the one given at construction (any env of the
        same shapes may be passed).  The rows live in a buffer that the next call overwrites (see ``features``)."""
        env = self._env_for(env)
        if env.obs_bits is None:
            raise ValueError("FusedPolicy reads env.obs_bits: create the env with packed_obs=True")
        N, wpa, M = env.N_AGENTS, env.bits_words_per_agent, env.meta_size
        e0, e1, step = (envs if envs is not None else slice(None)).indices(env.num_envs)
        if step != 1 or e1 < e0:
            raise ValueError("envs must be a contiguous slice of env indices")
        ids, k = self._id_array(agent_ids, N)
        return _trunk_forward(env, C.byref(self._weights), env.obs_bits.data_ptr() + e0 * N * wpa * 4,
                              env.meta.data_ptr() + e0 * N * M * 4, e1 - e0, N, ids, k, self.features((e1 - e0) * k),
                              self.stride)

    def trunk_packed(self, bits: torch.Tensor, meta: torch.Tensor) -> torch.Tensor:
        """Feature rows (as ``trunk_from_env``) for packed observations ``bits`` int32 [S, wpa] and ``meta`` [S, M]."""
        _check_packed(self.env, bits, meta)
        bits, meta = bits.contiguous(), meta.contiguous()
        ids, _ = self._id_array((0,), 1)
        return _trunk_forward(self.env, C.byref(self._weights), bits.data_ptr(), meta.data_ptr(), bits.shape[0], 1, ids,
                              1, self.features(bits.shape[0]), self.stride)

    @torch.no_grad()
    def forward_from_env(self, agent_ids, env=None, envs=None):
        """(value [S, 1], logits [S, 9]) fp32 for the samples of ``trunk_from_env``."""
        return self._head(self.trunk_from_env(agent_ids, env, envs))

    @torch.no_grad()
    def forward_packed(self, bits: torch.Tensor, meta: torch.Tensor):
        """(value [S, 1], logits [S, 9]) fp32 for packed observations ``bits`` int32 [S, wpa] and ``meta`` [S, M]."""
        return self._head(self.trunk_packed(bits, meta))

    def forward(self, agent_ids=None, bits=None, meta=None, env=None, envs=None):
        if agent_ids is not None:
            return self.forward_from_env(agent_ids, env=env, envs=envs)
        if bits is None or meta is None:
            raise ValueError("pass agent_ids (read the env in place) or bits and meta")
        return self.forward_packed(bits, meta)

    __call__ = forward

    @torch.no_grad()
    def get_action_and_value(self, use_action_mask, action=None, *, agent_ids=None, bits=None, meta=None, env=None,
                             envs=None, seed=None, actions=None):
        """``CtfPolicy.get_action_and_value``'s (action, log_prob, entropy, value) for the samples of ``forward``;
        use_action_mask is the per-sample flag in sample order.  Masking is ``CtfPolicy.masked_logits``.

        ``seed`` (an int in [0, 2**64)) samples with ``ctf_sample_actions`` instead of torch's generator: each action
        is a function of the logits, the mask flag and (seed, global env id, episode, step, agent), so it needs
        ``agent_ids`` (ValueError with ``bits`` / ``meta`` or a given ``action``).  ``actions`` (uint8 [B, N]) then
        also receives every action at its (env, agent), in the same launch."""
        if seed is not None:
            if action is not None:
                raise ValueError("seed draws the action: pass a seed or an action, not both")
            return self._seeded(use_action_mask, agent_ids, bits, env, envs, seed, actions)
        if actions is not None:
            raise ValueError("actions is written by the seeded draw only: pass a seed with it")
        value, logits = self.forward(agent_ids, bits, meta, env, envs)
        probs = Categorical(logits=self.policy.masked_logits(logits, use_action_mask), validate_args=False)
        if action is None:
            action = probs.sample()
        return action, probs.log_prob(action), probs.entropy(), value

    @torch.no_grad()
    def get_action(self, use_action_mask, *, agent_ids=None, bits=None, meta=None, env=None, envs=None, seed=None):
        """The action of ``get_action_and_value`` (with ``seed``, drawn by ``ctf_sample_actions``)."""
        if seed is not None:
            return self._seeded(use_action_mask, agent_ids, bits, env, envs, seed, None)[0]
        _, logits = self.forward(agent_ids, bits, meta, env, envs)
        return Categorical(logits=self.policy.masked_logits(logits, use_action_mask), validate_args=False).sample()

    # ------------------------------------------------------------------ training
    def evaluate_actions(self, bits: torch.Tensor, meta: torch.Tensor, use_action_mask, action):
        """(log_prob [S], entropy [S], value [S, 1]) of ``action`` for packed observations ``bits`` int32 [S, wpa] and
        ``meta`` [S, M], differentiable into every parameter of ``self.policy``: what ``CtfPolicy.get_action_and_value``
        with a given action gives the PPO loss, from packed observations.

        The trunk runs the CUDA kernels (``ctf_policy_features`` forward, ``ctf_policy_features_backward`` backward)
        with the live conv parameters, copied into training-only buffers: the inference buffers of ``refresh()`` (and
        CUDA graphs captured around them) do not change.  fc1 -> tanh -> fc2 -> tanh run in bf16 on cuBLAS from the
        fp32 parameters (fc1.weight zero-padded to the row stride as in inference); the small heads run in fp32
        (``train_head``).  Between forward and backward each sample holds 2 x stride bf16 values (rows and their
        gradient); split large minibatches into chunks and accumulate gradients over them."""
        _check_packed(self.env, bits, meta)
        p = self.policy
        rows = _PackedTrunk.apply(bits.contiguous(), p.conv1.weight, p.conv1.bias, p.conv2.weight, p.conv2.bias, self,
                                  meta.contiguous())
        value, logits = self.train_head(rows)
        probs = Categorical(logits=p.masked_logits(logits, use_action_mask), validate_args=False)
        return probs.log_prob(action), probs.entropy(), value

    def train_head(self, rows: torch.Tensor):
        """(value [S, 1], logits [S, 9]) fp32 from feature rows [S, stride], differentiable into fc1, fc2 and the heads:
        the part of ``evaluate_actions`` after the trunk.  fc1 -> tanh -> fc2 -> tanh in bf16 on cuBLAS, fc1.weight
        zero-padded to the stride.  The heads (128 -> 10, 0.1 % of the FLOPs) run in fp32, so value and logits enter
        the loss unrounded: a bf16 output adds a per-sample rounding that dominates the error of the value-head bias
        gradient."""
        p, bf = self.policy, torch.bfloat16
        x = torch.tanh(F.linear(rows, F.pad(p.fc1.weight, (0, self.stride - self.k1)).to(bf), p.fc1.bias.to(bf)))
        x = torch.tanh(F.linear(x, p.fc2.weight.to(bf), p.fc2.bias.to(bf)))
        hw = torch.cat((p.value_head.weight, p.action_head.weight))
        out = F.linear(x.float(), hw, torch.cat((p.value_head.bias, p.action_head.bias)))
        return out[:, :1], out[:, 1:]

    def _train_state(self):
        """The training-only buffers, created by the first call and separate from the inference buffers, which only
        ``refresh()`` changes: ``trunk``, a one-slot ``_TrunkWeights`` with the transposed conv2; ``weights`` and
        ``c2wt``, its slot's ``CtfPolicyWeights`` and transposed conv2 as the trunk kernels read them; ``workspace``,
        the backward's partial gradient sums."""
        if self._train is None:
            env = self.env
            n = C.c_size_t()
            _native.check(env._lib.ctf_policy_grad_workspace_size(env._handle, C.byref(n)))
            tw = _TrunkWeights(1, env.n_channels, env.device, transposed=True)
            self._train = dict(trunk=tw, weights=tw.native[0], c2wt=tw.c2wt[0],
                               workspace=torch.empty(max(n.value // 4, 4), dtype=torch.float32, device=env.device))
        return self._train

    def _train_forward(self, bits, meta, w1, b1, w2, b2):
        tr = self._train_state()
        tr["trunk"].load(0, w1, b1, w2, b2)
        rows = torch.empty((bits.shape[0], self.stride), dtype=torch.bfloat16, device=self.env.device)
        if bits.shape[0] == 0:
            return rows
        ids, _ = self._id_array((0,), 1)
        return _trunk_forward(self.env, C.byref(tr["weights"]), bits.data_ptr(), meta.data_ptr(), bits.shape[0], 1, ids,
                              1, rows, self.stride)

    def _train_backward(self, bits, rows, grad_rows, w1, b1, w2, b2):
        env = self.env
        tr = self._train_state()
        tr["trunk"].load(0, w1, b1, w2, b2)
        grad_rows = grad_rows.to(torch.bfloat16).contiguous()
        grads = [torch.empty_like(t, dtype=torch.float32) for t in (w1, b1, w2, b2)]
        gs = _native.CtfPolicyGrads(*(g.data_ptr() for g in grads))
        ids, _ = self._id_array((0,), 1)
        ws = tr["workspace"]
        # no samples: the kernel reads no input and writes zero gradients; empty tensors have no address, so the
        # workspace stands in for the three input pointers
        ptrs = [t.data_ptr() if bits.shape[0] else ws.data_ptr() for t in (bits, rows, grad_rows)]
        stream = C.c_void_p(torch.cuda.current_stream(env.device).cuda_stream)
        _native.check(env._lib.ctf_policy_features_backward(
            env._handle, C.byref(tr["weights"]), C.c_void_p(tr["c2wt"].data_ptr()), C.c_void_p(ptrs[0]),
            bits.shape[0], 1, ids, 1, C.c_void_p(ptrs[1]), C.c_void_p(ptrs[2]), self.stride,
            C.c_void_p(ws.data_ptr()), ws.numel() * 4, C.byref(gs), stream))
        return [g.to(t.dtype) for g, t in zip(grads, (w1, b1, w2, b2))]


# ---------------------------------------------------------------------------------------------------- policy pools
class PoolPlan:
    """The launch plan ``PolicyPool.plan`` builds once on the host for a fixed list of segments.

    Policy p owns the feature rows [p*s_max, p*s_max + n_samples[p]); s_max is the largest policy's sample count, and
    the rest of each block (the pad rows) stays zero and is never scattered.  The forward's outputs are in plan order:
    segment after segment as given, sample s = e*k + j of a segment (agent ids[j] of its e-th env).

    * ``seg_rows[i]``: (start, stop) of segment i in the outputs;
    * ``row_index`` [S]: the feature row of every output row; ``policy_of_row`` [S]: its policy;
    * ``flat_index`` [S]: env * N + agent of every output row (where ``act`` writes its action in ``actions[B, N]``);
    * ``mask_add`` [S, 9] float32: the additive action mask, ``(mask - 1) * 1e9`` of ``CtfPolicy.masked_logits`` for
      rows whose policy masks and whose agent type is masked, zeros elsewhere;
    * ``masked`` [S] uint8: 1 on exactly those rows (what ``ctf_sample_actions`` reads for a seeded ``act``);
    * ``features`` bf16 [L * s_max, stride]: the trunk's output buffer.
    """

    def __init__(self, segments, n_samples, s_max, seg_rows, row_index, flat_index, mask_add, features, tables):
        self.segments, self.n_samples, self.s_max, self.seg_rows = segments, n_samples, s_max, seg_rows
        self.row_index, self.flat_index, self.mask_add, self.features = row_index, flat_index, mask_add, features
        self.masked = (mask_add[:, 5:] != 0).any(1).to(torch.uint8)
        self.policy_of_row = row_index // s_max
        self.n_rows = features.shape[0]
        self._tables = tables   # [(ctypes segment array, count)], policy-major, at most GROUPED_MAX_SEGMENTS each

    @property
    def n_outputs(self) -> int:
        return int(self.row_index.numel())


class PolicyPool:
    """Inference for several policies on one env batch: one grouped trunk launch (``ctf_policy_features_grouped``,
    ``k_policy_trunk_grouped``) and one bf16 ``torch.baddbmm`` chain for the heads of all policies per forward.

    ``policies``: ``CtfPolicy`` modules or ``FusedPolicy`` views of them (their ``policy`` is used), each policy once,
    at most ``GROUPED_MAX_POLICIES`` (64).  Every weight lives in stacked persistent buffers: conv1 / conv2 in the
    kernel's layouts, fc1 bf16 [L, 256, stride] zero-padded as in ``FusedPolicy``, fc2 [L, 128, 256], the value | action
    heads [L, 10, 128].  ``refresh()`` copies the modules' current weights into them in place, so a CUDA graph captured
    around ``forward`` / ``act`` follows optimiser steps.

    Precision: each policy's rows are exactly what ``FusedPolicy.trunk_from_env`` writes for it (the kernels share the
    per-sample code); the heads are the same bf16 computation as ``FusedPolicy`` run as a batched GEMM, within the same
    contract against fp32 ``CtfPolicy``.
    """

    def __init__(self, env, policies):
        mods = [p.policy if isinstance(p, FusedPolicy) else p for p in policies]
        if not mods:
            raise ValueError("a PolicyPool needs at least one policy")
        if len(mods) > _native.GROUPED_MAX_POLICIES:
            raise ValueError(f"a PolicyPool holds at most {_native.GROUPED_MAX_POLICIES} policies, got {len(mods)}")
        if len({id(m) for m in mods}) != len(mods):
            raise ValueError("every policy may appear only once in a PolicyPool")
        self.k1, self.stride = _check_policies(env, mods)
        self.env, self.policies = env, mods
        self._trunk_w = _TrunkWeights(len(mods), env.n_channels, env.device)
        self._weights = self._trunk_w.native        # the grouped kernel's weight table, one entry per policy
        self._head_w = _HeadWeights(len(mods), self.k1, self.stride, env.device)
        self.refresh()

    def __len__(self):
        return len(self.policies)

    def refresh(self):
        """Copies every policy's current weights into the stacked buffers, on the device (no host round trip)."""
        for p, m in enumerate(self.policies):
            self._trunk_w.load(p, m.conv1.weight, m.conv1.bias, m.conv2.weight, m.conv2.bias)
            self._head_w.load(p, m)

    def _env_for(self, env):
        if env is None:
            return self.env
        mine = (self.env.n_channels, self.env.GRID_SIZE, self.env.meta_size, self.env.N_AGENTS, self.env.device)
        if (env.n_channels, env.GRID_SIZE, env.meta_size, env.N_AGENTS, env.device) != mine:
            raise ValueError("env does not have the shapes (C, G, M, N) or the device this PolicyPool was built for")
        return env

    # ------------------------------------------------------------------ plan
    def plan(self, segments) -> PoolPlan:
        """Builds the launch plan for ``segments``, a list of (policy index, env slice, agent ids): the agents ``ids``
        (1..8 of them) of the envs ``slice`` (contiguous, step 1) of the pool's env, run by policy ``index``.  Runs on
        the host once; ``forward`` and ``act`` with the plan are then a fixed sequence of launches."""
        env = self.env
        B, N, L = env.num_envs, env.N_AGENTS, len(self.policies)
        norm = []
        for i, seg in enumerate(segments):
            pol, sl, ids = seg
            pol = int(pol)
            if not 0 <= pol < L:
                raise ValueError(f"segment {i}: policy index {pol} out of range for {L} policies")
            if isinstance(sl, tuple):
                sl = slice(*sl)
            e0, e1, step = sl.indices(B)
            if step != 1 or e1 < e0:
                raise ValueError(f"segment {i}: envs must be a contiguous slice of env indices")
            norm.append((pol, e0, e1, _check_agent_ids(ids, N, f"segment {i}: ")))
        n_samples = [0] * L
        seg_first_row = []
        for pol, e0, e1, ids in norm:            # rows of a policy: its segments in the order given
            seg_first_row.append(n_samples[pol])
            n_samples[pol] += (e1 - e0) * len(ids)
        s_max = max(max(n_samples), 1)
        # per agent, the additive mask CtfPolicy.masked_logits applies: (mask_5 - 1) * 1e9 for masked agent types
        masked_type = env.use_action_mask.detach().cpu().reshape(N, 1) == 1
        mask5 = torch.tensor([0.0] * 5 + [-1e9] * (N_ACTIONS - 5))
        agent_mask = torch.where(masked_type, mask5, torch.zeros(N_ACTIONS))
        seg_rows, row_index, flat_index, mask_add = [], [], [], []
        out = 0
        for (pol, e0, e1, ids), first in zip(norm, seg_first_row):
            k = len(ids)
            n = (e1 - e0) * k
            seg_rows.append((out, out + n))
            out += n
            s = torch.arange(n)
            agent = torch.tensor(ids, dtype=torch.int64)[s % k]
            row_index.append(pol * s_max + first + s)
            flat_index.append((e0 + s // k) * N + agent)
            mask_add.append(agent_mask[agent] if self.policies[pol].use_masking else torch.zeros((n, N_ACTIONS)))
        dev = env.device
        # the kernel's tables, policy-major (a CTA restages weights only where the policy changes)
        order = sorted(range(len(norm)), key=lambda i: norm[i][0])
        tables = []
        for c in range(0, len(order), _native.GROUPED_MAX_SEGMENTS):
            chunk = order[c : c + _native.GROUPED_MAX_SEGMENTS]
            arr = (_native.CtfPolicySegment * len(chunk))()
            for slot, i in enumerate(chunk):
                pol, e0, e1, ids = norm[i]
                arr[slot].env_begin, arr[slot].n_envs = e0, e1 - e0
                arr[slot].out_row, arr[slot].policy, arr[slot].k = pol * s_max + seg_first_row[i], pol, len(ids)
                for j, a in enumerate(ids):
                    arr[slot].agent_ids[j] = a
            tables.append((arr, len(chunk)))
        def cat(ts, shape):
            return (torch.cat(ts) if ts else torch.zeros(shape)).to(dev)

        return PoolPlan(
            norm, n_samples, s_max, seg_rows,
            cat(row_index, (0,)).long(), cat(flat_index, (0,)).long(), cat(mask_add, (0, N_ACTIONS)).float(),
            torch.zeros((L * s_max, self.stride), dtype=torch.bfloat16, device=dev),
            tables,
        )

    # ------------------------------------------------------------------ launches
    def trunk(self, plan: PoolPlan, env=None) -> torch.Tensor:
        """Runs the grouped trunk for ``plan`` on ``env`` (default: the pool's env) and returns ``plan.features``:
        bf16 [L * s_max, stride], policy p's rows at [p*s_max, p*s_max + plan.n_samples[p]), pad rows untouched."""
        env = self._env_for(env)
        if env.obs_bits is None:
            raise ValueError("PolicyPool reads env.obs_bits: create the env with packed_obs=True")
        stream = C.c_void_p(torch.cuda.current_stream(env.device).cuda_stream)
        feat = plan.features
        for arr, n in plan._tables:
            _native.check(env._lib.ctf_policy_features_grouped(
                env._handle, self._weights, len(self.policies), arr, n, C.c_void_p(env.obs_bits.data_ptr()),
                C.c_void_p(env.meta.data_ptr()), env.num_envs, env.N_AGENTS, C.c_void_p(feat.data_ptr()), self.stride,
                feat.shape[0], stream))
        return feat

    def _head_out(self, plan: PoolPlan, feat: torch.Tensor | None = None):
        """fp32 [S, 10] in plan order: the value, then the 9 logits, of every row (see ``head``)."""
        L, w = len(self.policies), self._head_w
        x = (plan.features if feat is None else feat).view(L, plan.s_max, self.stride)
        x = torch.tanh(torch.baddbmm(w.fc1b.unsqueeze(1), x, w.fc1w.transpose(1, 2)))
        x = torch.tanh(torch.baddbmm(w.fc2b.unsqueeze(1), x, w.fc2w.transpose(1, 2)))
        out = torch.baddbmm(w.hb.unsqueeze(1), x, w.hw.transpose(1, 2)).view(L * plan.s_max, 1 + N_ACTIONS)
        return out.index_select(0, plan.row_index).float()

    def head(self, plan: PoolPlan, feat: torch.Tensor | None = None):
        """(value [S, 1], logits [S, 9]) fp32 in plan order from the feature rows: fc1 -> tanh -> fc2 -> tanh -> heads
        as one bf16 ``torch.baddbmm`` chain over [L, s_max, .], then the plan's rows gathered."""
        out = self._head_out(plan, feat)
        return out[:, :1], out[:, 1:]

    @torch.no_grad()
    def forward(self, plan: PoolPlan, env=None):
        """(value [S, 1], logits [S, 9]) fp32 of every sample of ``plan``, in plan order."""
        return self.head(plan, self.trunk(plan, env))

    __call__ = forward

    @torch.no_grad()
    def act(self, plan: PoolPlan, actions: torch.Tensor, env=None, seed=None) -> torch.Tensor:
        """Samples one action per row of ``plan`` (one ``Categorical`` over all rows, each masked by its own policy's
        ``use_masking`` as ``CtfPolicy.masked_logits`` does) and writes it into ``actions`` (uint8 [B, N], contiguous)
        at the row's (env, agent).  Returns the sampled actions [S] int64 in plan order.

        With ``seed`` one ``ctf_sample_actions`` launch draws and writes them instead: each row's action is keyed by
        (seed, global env id, episode, step, agent), as ``FusedPolicy.get_action_and_value(seed=...)`` draws it."""
        env = self._env_for(env)
        if actions.dtype != torch.uint8 or tuple(actions.shape) != (env.num_envs, env.N_AGENTS) \
                or not actions.is_contiguous():
            raise ValueError(f"actions must be a contiguous uint8 tensor [{env.num_envs}, {env.N_AGENTS}]")
        if seed is not None:
            out = self._head_out(plan, self.trunk(plan, env))
            return sample_actions(env, out, plan.masked, plan.flat_index, seed, actions)[0]
        _, logits = self.forward(plan, env)
        a = Categorical(logits=logits + plan.mask_add, validate_args=False).sample()
        actions.view(-1).index_copy_(0, plan.flat_index, a.to(torch.uint8))
        return a
