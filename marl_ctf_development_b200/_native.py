"""ctypes binding of libctf_b200.so (include/ctf_b200.h).  Fails loudly: no library, no env."""
from __future__ import annotations

import ctypes as C
import os

from .config import CtfConfig

_HERE = os.path.dirname(os.path.abspath(__file__))
# CTF_B200_LIB selects another build of the same extension (kernel A/B experiments); default is the in-tree one
LIB_PATH = os.environ.get("CTF_B200_LIB") or os.path.join(_HERE, "libctf_b200.so")

# every symbol include/ctf_b200.h declares
EXPORTS = (
    "ctf_last_error",
    "ctf_abi_version",
    "ctf_config_size",
    "ctf_create",
    "ctf_destroy",
    "ctf_get_sizes",
    "ctf_reset",
    "ctf_step",
    "ctf_observe",
    "ctf_unpack_obs",
    "ctf_stats_sum",
    "ctf_take_faults",
    "ctf_step_host",
    "ctf_policy_features",
    "ctf_policy_grad_workspace_size",
    "ctf_policy_features_backward",
    "ctf_policy_features_grouped",
    "ctf_policy_trunk_ctas",
    "ctf_gae",
    "ctf_gae_dones",
    "ctf_sample_actions",
    "ctf_compressible_alloc",
    "ctf_compressible_free",
    "ctf_compression_supported",
    "ctf_mem_is_compressed",
    "ctf_compressible_set_enabled",
)
ABI_VERSION = 12
FAULT_BAD_ACTION, FAULT_RESPAWN_BLOCKED, FAULT_BAD_INDEX = 1, 2, 4


class CtfState(C.Structure):
    _fields_ = [
        ("grid", C.c_void_p),
        ("agents", C.c_void_p),
        ("envs", C.c_void_p),
        ("stats", C.c_void_p),
        ("visits", C.c_void_p),
        ("hp", C.c_void_p),
    ]


class CtfOutputs(C.Structure):
    _fields_ = [("obs", C.c_void_p), ("obs_bits", C.c_void_p), ("meta", C.c_void_p), ("rewards", C.c_void_p), ("dones", C.c_void_p)]


class CtfSizes(C.Structure):
    _fields_ = [
        (name, C.c_size_t)
        for name in (
            "grid_stride",
            "grid_bytes",
            "agents_bytes",
            "envs_bytes",
            "stats_bytes",
            "visits_bytes",
            "obs_bytes",
            "meta_bytes",
            "rewards_bytes",
            "dones_bytes",
            "obs_elems_per_env",
            "meta_elems_per_env",
            "obs_bits_bytes",
            "bits_words_per_agent",
            "hp_bytes",
        )
    ]


class CtfPolicyWeights(C.Structure):
    _fields_ = [("conv1_w", C.c_void_p), ("conv1_b", C.c_void_p), ("conv2_w", C.c_void_p), ("conv2_b", C.c_void_p)]


GROUPED_MAX_POLICIES, GROUPED_MAX_SEGMENTS = 64, 512


class CtfPolicySegment(C.Structure):
    _fields_ = [("env_begin", C.c_int64), ("n_envs", C.c_int64), ("out_row", C.c_int64), ("policy", C.c_int32),
                ("k", C.c_int32), ("agent_ids", C.c_uint8 * 8)]


class CtfPolicyGrads(C.Structure):
    _fields_ = [("conv1_w", C.c_void_p), ("conv1_b", C.c_void_p), ("conv2_w", C.c_void_p), ("conv2_b", C.c_void_p)]


class NativeError(RuntimeError):
    pass


_lib = None


def load():
    """Loads the extension; raises if it is missing (build with ``python -m marl_ctf_development_b200.build``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.environ.get("CTF_B200_LIB"):
        # a fresh checkout has no .so (built artefacts are git-ignored): compile it in-tree with nvcc
        from .build import build_native

        try:
            build_native()
        except Exception as exc:
            if not os.path.exists(LIB_PATH):
                raise NativeError(
                    f"{LIB_PATH} is missing and could not be built ({exc}). "
                    "The step path is CUDA-only: there is no CPU fallback."
                ) from exc
    if not os.path.exists(LIB_PATH):
        raise NativeError(f"{LIB_PATH} not found. The step path is CUDA-only: there is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    for sym in EXPORTS:
        if not hasattr(L, sym):
            raise NativeError(f"{LIB_PATH} does not export {sym}")
    L.ctf_last_error.restype = C.c_char_p
    L.ctf_abi_version.restype = C.c_int
    L.ctf_config_size.restype = C.c_size_t
    L.ctf_create.argtypes = [C.POINTER(CtfConfig), C.c_int64, C.c_int, C.c_uint64, C.c_uint64, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
    L.ctf_destroy.argtypes = [C.c_void_p]
    L.ctf_get_sizes.argtypes = [C.c_void_p, C.POINTER(CtfSizes)]
    L.ctf_reset.argtypes = [C.c_void_p, CtfState, CtfOutputs, C.c_int, C.c_void_p]
    L.ctf_step.argtypes = [C.c_void_p, CtfState, C.c_void_p, CtfOutputs, C.c_void_p]
    L.ctf_observe.argtypes = [C.c_void_p, CtfState, C.c_void_p, CtfOutputs, C.c_void_p]
    L.ctf_unpack_obs.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_void_p]
    L.ctf_stats_sum.argtypes = [C.c_void_p, CtfState, C.c_void_p, C.c_void_p]
    L.ctf_take_faults.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_uint32)]
    L.ctf_step_host.argtypes = [C.c_void_p, CtfState, C.c_void_p, CtfOutputs, C.c_void_p, C.c_void_p, C.c_void_p]
    L.ctf_policy_features.argtypes = [C.c_void_p, C.POINTER(CtfPolicyWeights), C.c_void_p, C.c_void_p, C.c_int64, C.c_int,
                                      C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.c_void_p]
    L.ctf_policy_features_grouped.argtypes = [C.c_void_p, C.POINTER(CtfPolicyWeights), C.c_int, C.POINTER(CtfPolicySegment),
                                              C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int64,
                                              C.c_int64, C.c_void_p]
    L.ctf_policy_trunk_ctas.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.ctf_policy_grad_workspace_size.argtypes = [C.c_void_p, C.POINTER(C.c_size_t)]
    L.ctf_policy_features_backward.argtypes = [C.c_void_p, C.POINTER(CtfPolicyWeights), C.c_void_p, C.c_void_p, C.c_int64,
                                               C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int64,
                                               C.c_void_p, C.c_size_t, C.POINTER(CtfPolicyGrads), C.c_void_p]
    L.ctf_gae.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64,
                          C.c_int64, C.c_float, C.c_float, C.c_void_p]
    L.ctf_gae_dones.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_int64, C.c_int64, C.c_int64, C.c_float, C.c_float, C.c_void_p]
    L.ctf_sample_actions.argtypes = [C.c_void_p, CtfState, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64,
                                     C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.ctf_compressible_alloc.restype = C.c_void_p
    L.ctf_compressible_alloc.argtypes = [C.c_ssize_t, C.c_int, C.c_void_p]
    L.ctf_compressible_free.restype = None
    L.ctf_compressible_free.argtypes = [C.c_void_p, C.c_ssize_t, C.c_int, C.c_void_p]
    L.ctf_compression_supported.argtypes = [C.c_int, C.POINTER(C.c_int)]
    L.ctf_mem_is_compressed.argtypes = [C.c_void_p, C.POINTER(C.c_int)]
    L.ctf_compressible_set_enabled.argtypes = [C.c_int]
    if L.ctf_abi_version() != ABI_VERSION:
        raise NativeError(f"ABI version mismatch: library {L.ctf_abi_version()}, binding {ABI_VERSION}")
    if L.ctf_config_size() != C.sizeof(CtfConfig):
        raise NativeError(f"ctf_config_t layout mismatch: library {L.ctf_config_size()} B, binding {C.sizeof(CtfConfig)} B")
    _lib = L
    return L


def check(rc: int):
    if rc != 0:
        raise NativeError(f"ctf_b200 error {rc}: {load().ctf_last_error().decode()}")
