"""Device buffers in compressible memory (Compute Data Compression), for the dense observations.

On a device that reports compression support, memory from ``compressible_empty`` is compressed between L2 and DRAM.
Kernels and readers see the same bytes as in any other buffer, but the mostly-zero observation stream moves far fewer
DRAM bytes, which is what bounds the step (DESIGN §4).  The memory comes from ``ctf_compressible_alloc`` /
``ctf_compressible_free`` of libctf_b200.so through one ``torch.cuda.MemPool`` per device, so torch owns the buffers'
lifetime like that of any other tensor.  On a device without compression ``compressible_empty`` is ``torch.empty``.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _native

_pools: dict[int, torch.cuda.MemPool] = {}
_supported: dict[int, bool] = {}


def _device_index(device) -> int:
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    if dev.type != "cuda":
        raise ValueError(f"device must be a CUDA device, got {dev}")
    return dev.index if dev.index is not None else torch.cuda.current_device()


def compression_supported(device=None) -> bool:
    """Whether ``device`` reports CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED."""
    idx = _device_index(device)
    if idx not in _supported:
        v = C.c_int(0)
        _native.check(_native.load().ctf_compression_supported(idx, C.byref(v)))
        _supported[idx] = bool(v.value)
    return _supported[idx]


def is_compressed(t: torch.Tensor) -> bool:
    """Whether the tensor's memory was granted compression by the driver."""
    v = C.c_int(0)
    _native.check(_native.load().ctf_mem_is_compressed(C.c_void_p(t.data_ptr()), C.byref(v)))
    return bool(v.value)


def allocator():
    """A torch allocator over ctf_compressible_alloc / ctf_compressible_free."""
    _native.load()   # builds the library when it is missing
    return torch.cuda.memory.CUDAPluggableAllocator(
        _native.LIB_PATH, "ctf_compressible_alloc", "ctf_compressible_free"
    ).allocator()


def pool(device=None) -> torch.cuda.MemPool:
    """The module's compressible memory pool of ``device`` (created on first use, kept for the process)."""
    idx = _device_index(device)
    if idx not in _pools:
        with torch.cuda.device(idx):
            _pools[idx] = torch.cuda.MemPool(allocator())
    return _pools[idx]


def compressible_empty(shape, dtype, device=None) -> torch.Tensor:
    """``torch.empty(shape, dtype=dtype, device=device)`` in compressible memory when the device supports it.

    For callers that bind their own output buffers (``GridworldCtfGPU(obs_out=...)``, ``bind_outputs(obs=...)``)."""
    idx = _device_index(device)
    dev = torch.device("cuda", idx)
    if not compression_supported(idx):
        return torch.empty(shape, dtype=dtype, device=dev)
    with torch.cuda.use_mem_pool(pool(idx), dev):
        return torch.empty(shape, dtype=dtype, device=dev)
