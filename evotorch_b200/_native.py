"""ctypes binding of libevok.so (the C ABI declared in include/evok.h).

PyTorch only supplies device memory and the current CUDA stream here: every call passes raw pointers and sizes.
There is NO fallback: if the library is missing, `lib()` raises, so a CUDA problem can never silently run on
torch ops.
"""

from __future__ import annotations

import ctypes
import os
from ctypes import c_float, c_int, c_int64, c_size_t, c_uint64, c_void_p
from typing import Optional

import torch

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "lib", "libevok.so")

_P = c_void_p
_SIGNATURES = {
    # name: (restype, argtypes)
    "evok_abi_version": (c_int, []),
    "evok_launch_count": (c_uint64, []),
    "evok_error_string": (ctypes.c_char_p, [c_int]),
    "evok_sample_eval": (c_int, [c_int, _P, c_int64, _P, _P, c_int64, c_int64, c_int64, c_int, c_uint64, c_uint64, _P, _P, _P]),
    "evok_eval": (c_int, [c_int, _P, c_int64, c_int64, c_int64, _P, _P]),
    "evok_rank_workspace_bytes": (c_size_t, [c_int64]),
    "evok_rank": (c_int, [c_int, _P, c_int64, c_int, _P, _P, _P, c_size_t, _P]),
    "evok_argsort": (c_int, [_P, c_int64, c_int, _P, _P, c_size_t, _P]),
    "evok_sample_batched": (c_int, [_P, c_int64, c_int64, _P, c_int64, _P, c_int64, c_int64, c_int64, c_int64, c_int, c_uint64, c_uint64, _P]),
    "evok_rank_batched": (c_int, [c_int, _P, c_int64, c_int64, c_int, _P, _P, c_size_t, _P]),
    "evok_elite_mask_batched": (c_int, [_P, c_int64, c_int64, c_int64, _P, _P, c_size_t, _P]),
    "evok_weights_adjust_batched": (c_int, [_P, c_int64, c_int64, c_int, _P]),
    "evok_grad_batched_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64]),
    "evok_grad_batched": (c_int, [c_int, _P, c_int64, c_int64, _P, _P, c_int64, _P, c_int64, c_int64, c_int64, c_int64, c_float, c_float, _P, _P, _P,
                                  c_size_t, _P]),
    "evok_clipup_batched": (c_int, [_P, c_int64, c_int64, _P, _P, _P, _P, _P, _P]),
    "evok_sigma_update_batched": (c_int, [_P, _P, c_int64, c_int64, _P, c_int, _P, _P, _P, _P]),
    "evok_rank_table": (c_int, [_P, c_int64, c_int, _P, _P, _P, c_size_t, _P]),
    "evok_cholesky_workspace_bytes": (c_size_t, [c_int64]),
    "evok_cholesky": (c_int, [_P, c_int64, c_int64, _P, c_int64, _P, c_size_t, _P]),
    "evok_cmaes_row_weights": (c_int, [_P, _P, c_int64, c_int64, c_int64, c_int, _P, _P, _P]),
    "evok_cmaes_vector_update": (c_int, [_P, _P, c_int64, _P, _P, _P, _P, _P, c_int64, _P, c_int, _P, _P, _P]),
    "evok_weights_adjust": (c_int, [_P, c_int64, c_int, _P]),
    "evok_elite_mask": (c_int, [_P, c_int64, c_int64, _P, _P, c_size_t, _P]),
    "evok_grad_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "evok_grad": (c_int, [c_int, _P, c_int64, _P, _P, _P, c_int64, c_int64, c_float, c_float, _P, _P, _P, c_size_t, _P]),
    "evok_grad_regen": (c_int, [c_int, _P, _P, _P, c_int64, c_int64, c_int64, c_uint64, c_uint64, _P, c_float, c_float, _P, _P, _P,
                                c_size_t, _P]),
    "evok_clipup_step": (c_int, [_P, c_int64, _P, c_float, c_float, c_float, _P, _P, _P]),
    "evok_adam_step": (c_int, [_P, c_int64, _P, _P, c_int64, c_float, c_float, c_float, c_float, _P, _P, _P]),
    "evok_sgd_step": (c_int, [_P, c_int64, _P, c_int, c_float, c_float, _P, _P, _P]),
    "evok_axpy": (c_int, [_P, c_int64, c_float, _P, _P]),
    "evok_sigma_update": (c_int, [_P, _P, c_int64, c_float, c_int, _P, c_float, _P, c_float, _P, c_float, _P]),
    "evok_cem_finalize": (c_int, [_P, _P, _P, c_int64, c_int64, _P, _P, _P]),
    "evok_mlp_parameter_length": (c_int64, [c_int, _P]),
    "evok_mlp_forward": (c_int, [_P, c_int64, _P, c_int64, _P, c_int64, c_int64, c_int, _P, _P, _P]),
    "evok_mlp_forward_prep": (c_int, [_P, c_int64, _P, c_int64, _P, c_int64, c_int64, c_int, _P, _P, _P, _P, _P, c_float, c_float, c_float, _P, _P,
                                      c_size_t, _P]),
    "evok_mlp_forward_shared_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int, _P]),
    "evok_mlp_forward_shared": (c_int, [_P, c_int64, c_int64, _P, c_int64, c_int64, c_int, _P, _P, _P, _P, c_size_t, _P]),
    "evok_gemm_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64]),
    "evok_gemm_nt": (c_int, [_P, c_int64, _P, c_int64, c_int64, c_int64, c_int64, _P, c_int64, _P, c_int64, _P, _P, _P, c_size_t, _P]),
    "evok_gemm_nt_affine": (c_int, [_P, c_int64, _P, c_int64, c_int64, c_int64, c_int64, _P, c_int64, _P, _P, c_int64, _P, _P, c_size_t, _P]),
    "evok_transpose_pair": (c_int, [_P, c_int64, c_int64, c_int64, _P, _P, _P, c_int64, _P]),
    "evok_transpose_scale": (c_int, [_P, c_int64, c_int64, c_int64, _P, _P, c_int64, _P]),
    "evok_peer_alloc": (c_int, [c_size_t, _P, _P]),
    "evok_peer_open": (c_int, [_P, _P]),
    "evok_peer_close": (c_int, [_P]),
    "evok_peer_free": (c_int, [_P]),
    "evok_peer_push": (c_int, [_P, c_int64, c_int64, c_int, c_int, _P, _P, _P, _P]),
    "evok_peer_wait": (c_int, [_P, c_int, _P, _P, c_uint64, _P]),
    "evok_grad_push": (c_int, [c_int, _P, c_int64, _P, _P, _P, c_int64, c_int64, c_int64, c_uint64, c_uint64, _P, c_float, c_float, c_int, c_int,
                               _P, _P, _P, _P, _P, c_size_t, _P]),
    "evok_rank_sharded": (c_int, [c_int, _P, c_int64, c_int, c_int, c_int, _P, _P, _P, _P, _P, _P, _P, c_uint64, _P, _P, _P, c_size_t, _P]),
    "evok_peer_reduce": (c_int, [_P, c_int, c_int64, _P, _P, _P, _P, c_uint64, _P, _P]),
}

EXPORTED_SYMBOLS = tuple(sorted(_SIGNATURES))

_lib: Optional[ctypes.CDLL] = None


class EvokError(RuntimeError):
    pass


def lib() -> ctypes.CDLL:
    """Load libevok.so once; raise loudly if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise EvokError(
                f"{LIB_PATH} is missing: the sm_100a kernel library has not been built. "
                "Run `python -m evotorch_b200.build` (needs nvcc). There is no CPU/torch fallback for CUDA problems."
            )
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        if handle.evok_abi_version() != 1:
            raise EvokError("libevok.so ABI version mismatch; rebuild with `python -m evotorch_b200.build --force`")
        _lib = handle
    return _lib


def available() -> bool:
    return os.path.exists(LIB_PATH)


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().evok_error_string(rc).decode()
        if rc < 0:
            raise ValueError(f"{what}: {msg} (code {rc})")
        raise EvokError(f"{what}: CUDA error {rc}: {msg}")


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def stream_of(t: torch.Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


_workspaces: dict = {}


def workspace(device: torch.device, nbytes: int, tag: str = "ws") -> torch.Tensor:
    """A per-(device, stream, tag) scratch buffer that only grows, so pointers stay stable across generations.
    Keyed by the current stream: two searchers stepping on different streams never share scratch memory (a superseded
    buffer goes back to the caching allocator, which is stream-ordered, so kernels already enqueued on this stream stay
    valid).  A captured CUDA graph bakes the raw pointer in: captures run under `private_workspaces()` and own theirs."""
    dev = device.index if device.index is not None else torch.cuda.current_device()
    key = (dev, torch.cuda.current_stream(dev).cuda_stream, tag) if _private_depth == 0 else (dev, tag)
    buf = _workspaces.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
        _workspaces[key] = buf
    return buf


_private_depth = 0


class private_workspaces:
    """`with private_workspaces() as store:` -- every `workspace()` call inside allocates from (and is remembered in) a fresh
    `store` instead of the shared table.  Wrapped around a CUDA-graph capture: the graph then writes only to scratch buffers
    that it owns (keep `store` alive as long as the graph), so a later, larger request by anybody else -- which re-allocates
    the shared buffer -- can never pull memory from under a graph that still replays into it."""

    def __enter__(self) -> dict:
        global _workspaces, _private_depth
        self._saved = _workspaces
        _workspaces = self.store = {}
        _private_depth += 1
        # The cyclic garbage collector is held off for the duration of the capture: a collection that finalises an object owning
        # CUDA resources (a peer-exchange buffer with its IPC handles, an event) calls cudaFree / cudaIpcCloseMemHandle, which is
        # prohibited while a stream of the process is capturing and invalidates the capture ("operation failed due to a previous
        # error during capture" from the next launch -- seen once in the full GPU suite, never in the test alone).
        import gc

        self._gc_was_enabled = gc.isenabled()
        gc.collect()
        gc.disable()
        return self.store

    def __exit__(self, *exc):
        global _workspaces, _private_depth
        _workspaces = self._saved
        _private_depth -= 1
        if self._gc_was_enabled:
            import gc

            gc.enable()
        return False
