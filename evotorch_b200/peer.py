"""Peer exchange: the two collectives of the sharded generation done by libevok kernels over NVLink.

`torch.distributed` (NCCL) stays the control plane -- it carries the 64-byte IPC handles once, at set-up.  After that a
generation contains no library collective at all:

  K1+K2  sample_eval_kernel             writes this rank's fitness slice into its local copy of the fitness vector
         peer_push_kernel               copies the slice into EVERY peer's fitness vector and raises the flags
         peer_wait_kernel               one warp waits for all ranks' flags                         (was: all_gather)
  K3     rank (replicated, on the local copy of the full fitness vector)
  K4     grad_partial + grad_finalize_push_kernel   this rank's (grad_mu | grad_sigma) -> slot[rank] on every peer + flags
         peer_reduce_kernel             waits, then sums the slots in rank order                     (was: all_reduce)
  K5     update (replicated)

Everything is an ordinary kernel on the caller's stream, so the whole generation is CUDA-graph capturable without capturing
NCCL.  The reduction order is fixed (rank 0..R-1), so all GPUs compute bit-identical gradients.
Replaces the NCCL calls of `distributed.sharded_sample_and_gradients` (the reference's Ray round trip, core.py:2762-3073).
"""

from __future__ import annotations

import ctypes
import os
from typing import Optional

import torch
import torch.distributed as dist

from . import _native as nat

DEFAULT_TIMEOUT_NS = int(float(os.environ.get("EVOTORCH_B200_PEER_TIMEOUT_S", "20")) * 1e9)


class _RawCudaArray:
    """Minimal __cuda_array_interface__ carrier so that torch can view memory owned by libevok (zero copy)."""

    def __init__(self, ptr: int, shape: tuple, typestr: str):
        self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 2}


def _view(ptr: int, numel: int, typestr: str, device: torch.device) -> torch.Tensor:
    return torch.as_tensor(_RawCudaArray(ptr, (numel,), typestr), device=device)


def _align(n: int, a: int = 256) -> int:
    return (n + a - 1) // a * a


class PeerExchange:
    """The exchange buffer of this rank, mapped by all peers:
    [ f_all : N f32 | slots : R x 2D f32 | flags_f : R u64 | flags_g : R u64 | keys_all : N u32 | fsum : R f64 ]."""

    def __init__(self, popsize: int, solution_length: int, device: torch.device, *, timeout_ns: int = DEFAULT_TIMEOUT_NS):
        if not (dist.is_available() and dist.is_initialized()):
            raise RuntimeError("PeerExchange needs an initialised torch.distributed process group (it carries the IPC handles)")
        self.rank, self.world = dist.get_rank(), dist.get_world_size()
        if self.world > 16:
            raise ValueError("a peer exchange spans at most 16 GPUs (one NVLink domain)")
        self.device = torch.device(device)
        self.popsize, self.solution_length, self.timeout_ns = int(popsize), int(solution_length), int(timeout_ns)
        n, d, r = self.popsize, self.solution_length, self.world
        self._off_f = 0
        self._off_slots = _align(4 * n)
        self._off_flags_f = self._off_slots + _align(4 * r * 2 * d)
        self._off_flags_g = self._off_flags_f + _align(8 * r)
        self._off_keys = self._off_flags_g + _align(8 * r)      # sharded ranking: N sorted orderable keys (u32), shard by shard
        self._off_fsum = self._off_keys + _align(4 * n)         # ... and one local fitness sum (f64) per rank
        self.nbytes = self._off_fsum + _align(8 * r)

        lib = nat.lib()
        with torch.cuda.device(self.device):
            base, handle = ctypes.c_void_p(), ctypes.create_string_buffer(64)
            nat.check(lib.evok_peer_alloc(self.nbytes, ctypes.byref(base), handle), "evok_peer_alloc")
            self._base = int(base.value)
            handles = [None] * r
            dist.all_gather_object(handles, handle.raw)
            self._peer_bases = []
            for p in range(r):
                if p == self.rank:
                    self._peer_bases.append(self._base)
                    continue
                mapped = ctypes.c_void_p()
                nat.check(lib.evok_peer_open(ctypes.create_string_buffer(handles[p], 64), ctypes.byref(mapped)), "evok_peer_open")
                self._peer_bases.append(int(mapped.value))

        def table(offset: int):
            return (ctypes.c_void_p * r)(*[b + offset for b in self._peer_bases])

        self.peer_f, self.peer_slots = table(self._off_f), table(self._off_slots)
        self.peer_flags_f, self.peer_flags_g = table(self._off_flags_f), table(self._off_flags_g)
        self.peer_keys, self.peer_fsum = table(self._off_keys), table(self._off_fsum)
        # local views
        self.f_all = _view(self._base + self._off_f, n, "<f4", self.device)
        self.slots = _view(self._base + self._off_slots, r * 2 * d, "<f4", self.device)
        self._flags_f_ptr, self._flags_g_ptr = self._base + self._off_flags_f, self._base + self._off_flags_g
        # local (unshared) state: [epoch_f, epoch_g] u64, [done_f, done_g, done_r, err] u32 (done_f is unused: the fitness push
        # kernel raises the flags from its own per-peer CTA and needs no completion counter)
        self._epochs = torch.zeros(2, dtype=torch.int64, device=self.device)
        self._counters = torch.zeros(4, dtype=torch.int32, device=self.device)
        self._rank_counters = torch.zeros(4, dtype=torch.int32, device=self.device)  # sharded ranking: hist-scan / push / merge
        self._mean_eval = torch.zeros(1, dtype=torch.float32, device=self.device)
        self.reduced = torch.empty(2 * d, dtype=torch.float32, device=self.device)
        torch.cuda.synchronize(self.device)
        dist.barrier()  # nobody writes into a peer before that peer has zeroed and published its buffer

    # pointers of the local state
    @property
    def epoch_f(self) -> int:
        return self._epochs.data_ptr()

    @property
    def epoch_g(self) -> int:
        return self._epochs.data_ptr() + 8

    def _counter(self, i: int) -> int:
        return self._counters.data_ptr() + 4 * i

    def push_fitness(self, row0: int, n_local: int) -> None:
        """Copy this rank's fitness slice f_all[row0 : row0 + n_local] (already written locally by the sampler) into every peer's
        `f_all` and raise this rank's flag there (one CTA per peer).  Follow with `wait_fitness()`."""
        from . import ops

        with ops._timed("peer_push"):
            rc = nat.lib().evok_peer_push(self._base + self._off_f + 4 * row0, 4 * n_local, 4 * row0, self.world, self.rank, self.peer_f,
                                          self.peer_flags_f, self.epoch_f, nat.stream_of(self.f_all))
        nat.check(rc, "evok_peer_push")

    def wait_fitness(self) -> torch.Tensor:
        """Block the stream until every rank's fitness slice has landed in the local `f_all`."""
        from . import ops

        with ops._timed("peer_wait"):
            rc = nat.lib().evok_peer_wait(self._flags_f_ptr, self.world, self.epoch_f, self._counter(3), self.timeout_ns, nat.stream_of(self.f_all))
        nat.check(rc, "evok_peer_wait")
        return self.f_all

    def rank_sharded(self, f_local: torch.Tensor, method: str, higher_is_better: bool, row_offsets: list, w_local: torch.Tensor) -> tuple:
        """Sharded ranking (evok_rank_sharded): local sort -> sorted keys pushed to every peer -> global position of every LOCAL
        row by binary search over the peers' sorted shards.  Takes the place of `wait_fitness()` + the replicated global rank
        (it uses the same flag set / epoch as the fitness gather: a generation does one or the other).  Returns the utilities of
        the local rows (`w_local`, in local row order) and the global mean fitness (a 1-element device tensor)."""
        from . import ops

        lib = nat.lib()
        n_local = f_local.numel()
        offs = (ctypes.c_int64 * (self.world + 1))(*row_offsets)
        ws = nat.workspace(self.device, lib.evok_rank_workspace_bytes(max(n_local, 1)), "rank_sharded")
        with ops._timed("rank"):
            rc = lib.evok_rank_sharded(ops.RANK_IDS[method], f_local.data_ptr(), self.popsize, int(bool(higher_is_better)), self.world, self.rank,
                                       offs, self.peer_keys, self.peer_fsum, self.peer_flags_f, self.epoch_f, self._rank_counters.data_ptr(),
                                       self._counter(3), self.timeout_ns, w_local.data_ptr(), self._mean_eval.data_ptr(), ws.data_ptr(),
                                       ws.numel(), nat.stream_of(f_local))
        nat.check(rc, "evok_rank_sharded")
        return w_local, self._mean_eval

    def reduce_gradients(self) -> tuple:
        """Wait for every rank's slot, sum them in rank order -> (grad_mu, grad_sigma) views of `self.reduced`."""
        d = self.solution_length
        from . import ops

        with ops._timed("peer_reduce"):
            rc = nat.lib().evok_peer_reduce(self.slots.data_ptr(), self.world, 2 * d, self._flags_g_ptr, self.epoch_g, self._counter(2),
                                            self._counter(3), self.timeout_ns, self.reduced.data_ptr(), nat.stream_of(self.reduced))
        nat.check(rc, "evok_peer_reduce")
        return self.reduced[:d], self.reduced[d:]

    def timed_out(self) -> bool:
        """True if any wait gave up (a peer died or fell more than `timeout_ns` behind).  Synchronises."""
        return bool(self._counters[3].item())

    def close(self):
        lib = nat.lib()
        torch.cuda.synchronize(self.device)
        for p, b in enumerate(self._peer_bases):
            if p != self.rank:
                lib.evok_peer_close(b)
        dist.barrier()
        lib.evok_peer_free(self._base)
        self._peer_bases = []


def enable_peer_exchange(problem, popsize: int, *, timeout_ns: Optional[int] = None) -> PeerExchange:
    """Attach a PeerExchange to `problem`: from now on `sharded_sample_and_gradients` (hence distributed searchers) moves
    fitnesses and gradients between the GPUs from inside the producing kernels instead of calling NCCL."""
    px = PeerExchange(popsize, problem.solution_length, problem.device, timeout_ns=DEFAULT_TIMEOUT_NS if timeout_ns is None else timeout_ns)
    problem._peer_exchange = px
    problem.__dict__.pop("_grad_batches", None)
    return px
