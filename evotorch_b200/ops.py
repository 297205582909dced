"""Tensor-level entry points of the sm_100a kernels (CUDA, fp32 only).

Each function validates its tensors, pulls raw pointers + the current stream and calls the C ABI of
libevok.so (include/evok.h).  Callers in this package decide *whether* a tensor goes to these kernels
(`uses_kernels`); there is no silent fallback from here: a missing library raises.
"""

from __future__ import annotations

import math
from typing import Optional

import torch

from . import _native as nat
from .tools.readonlytensor import as_plain_tensor

OBJ_NONE, OBJ_SPHERE, OBJ_RASTRIGIN, OBJ_ACKLEY = 0, 1, 2, 3
OBJECTIVE_IDS = {"sphere": OBJ_SPHERE, "rastrigin": OBJ_RASTRIGIN, "ackley": OBJ_ACKLEY}
RANK_IDS = {"centered": 0, "linear": 1, "nes": 2, "normalized": 3, "raw": 4}
GRAD_SEPARABLE, GRAD_SYMMETRIC, GRAD_EXP, GRAD_MOMENTS = 0, 1, 2, 3
NAN = float("nan")


# ------------------------------------------------------------------------------------------------ device-side kernel timers
# bench.py turns these on to time each kernel group with CUDA events recorded on the launching stream (no host sync while
# the generations run; the elapsed times are read after the timed region).
_timers: Optional[dict] = None


def enable_timers() -> None:
    global _timers
    _timers = {}


def disable_timers() -> None:
    global _timers
    _timers = None


class _timed:
    __slots__ = ("name", "start")

    def __init__(self, name: str):
        self.name = name

    def __enter__(self):
        if _timers is not None:
            self.start = torch.cuda.Event(enable_timing=True)
            self.start.record()
        return self

    def __exit__(self, *exc):
        if _timers is not None:
            end = torch.cuda.Event(enable_timing=True)
            end.record()
            _timers.setdefault(self.name, []).append((self.start, end))
        return False


def timer_results() -> dict:
    """{kernel group: (launch count, mean milliseconds)}; call after torch.cuda.synchronize()."""
    out = {}
    for name, pairs in (_timers or {}).items():
        ms = [a.elapsed_time(b) for a, b in pairs]
        out[name] = (len(ms), sum(ms) / max(len(ms), 1))
    return out


_replayed_launches = 0


def count_replayed_launches(n: int) -> None:
    """CUDA-graph replays re-run captured kernels without passing through the library: the searchers report them here."""
    global _replayed_launches
    _replayed_launches += int(n)


def launch_count() -> int:
    """Kernels of libevok.so launched so far in this process: direct launches (counted inside the library) + graph replays."""
    return int(nat.lib().evok_launch_count()) + _replayed_launches


def uses_kernels(t: torch.Tensor) -> bool:
    """True for the tensors the hand-written kernels handle: CUDA + float32."""
    return t.is_cuda and t.dtype == torch.float32


def _vec(t: torch.Tensor, name: str, n: Optional[int] = None) -> torch.Tensor:
    if not (t.is_cuda and t.dtype == torch.float32 and t.ndim == 1 and t.is_contiguous()):
        raise ValueError(f"{name}: expected a contiguous 1-D float32 CUDA tensor, got {tuple(t.shape)} {t.dtype} {t.device}")
    if n is not None and t.numel() != n:
        raise ValueError(f"{name}: expected length {n}, got {t.numel()}")
    return as_plain_tensor(t)


def _mat(t: torch.Tensor, name: str) -> torch.Tensor:
    if not (t.is_cuda and t.dtype == torch.float32 and t.ndim == 2 and t.stride(1) == 1 and t.stride(0) >= t.shape[1]):
        raise ValueError(f"{name}: expected a row-major 2-D float32 CUDA tensor, got {tuple(t.shape)} strides {t.stride()} {t.dtype}")
    return as_plain_tensor(t)


# ------------------------------------------------------------------------------------------------ K1 / K2
def _offset_ptr(stream_offset: Optional[torch.Tensor]) -> Optional[int]:
    if stream_offset is None:
        return None
    if not (stream_offset.is_cuda and stream_offset.dtype == torch.int32 and stream_offset.numel() >= 1):
        raise ValueError("stream_offset: expected an int32 CUDA tensor with one element")
    return stream_offset.data_ptr()


def sample_eval(objective: int, X: Optional[torch.Tensor], mu: torch.Tensor, sigma: torch.Tensor, *, n_rows: int, symmetric: bool,
                seed: int, stream_id: int, row0: int = 0, f: Optional[torch.Tensor] = None,
                stream_offset: Optional[torch.Tensor] = None) -> None:
    D = mu.numel()
    _vec(mu, "mu"); _vec(sigma, "sigma", D)
    ldx = 0
    if X is not None:
        _mat(X, "X")
        if X.shape != (n_rows, D):
            raise ValueError(f"X: expected shape {(n_rows, D)}, got {tuple(X.shape)}")
        ldx = X.stride(0)
    if f is not None:
        _vec(f, "f", n_rows)
    if objective != OBJ_NONE and f is None:
        raise ValueError("f: a fitness buffer is required when an objective is fused into the sampler")
    if symmetric and (n_rows % 2 or row0 % 2):
        raise ValueError("symmetric sampling needs an even number of rows and an even first row")
    if n_rows == 0:
        return
    with _timed("sample_eval" if objective != OBJ_NONE else "sample"):
        rc = nat.lib().evok_sample_eval(objective, nat.ptr(X), ldx, mu.data_ptr(), sigma.data_ptr(), row0, n_rows, D, int(symmetric),
                                        seed & 0xFFFFFFFFFFFFFFFF, stream_id & 0xFFFFFFFFFFFFFFFF, _offset_ptr(stream_offset), nat.ptr(f),
                                        nat.stream_of(mu))
    nat.check(rc, "evok_sample_eval")


def grad_push(form: int, X: Optional[torch.Tensor], w: torch.Tensor, mu: torch.Tensor, sigma: torch.Tensor, *, scale_mu: float,
              scale_sigma: float, peer, seed: int = 0, stream_id: int = 0, row0: int = 0, stream_offset: Optional[torch.Tensor] = None) -> None:
    """K4 with the send half of the gradient all-reduce fused in (X = None: regenerate the rows from the Philox counters).
    Follow with `peer.reduce_gradients()`."""
    n, D = w.numel(), mu.numel()
    _vec(w, "weights"); _vec(mu, "mu"); _vec(sigma, "sigma", D)
    ldx = 0
    if X is not None:
        _mat(X, "X")
        if X.shape != (n, D):
            raise ValueError(f"X: expected shape {(n, D)}, got {tuple(X.shape)}")
        ldx = X.stride(0)
    ws = nat.workspace(mu.device, nat.lib().evok_grad_workspace_bytes(n, D), "grad")
    with _timed("grad" if X is not None else "grad_regen"):
        rc = nat.lib().evok_grad_push(form, nat.ptr(X), ldx, w.data_ptr(), mu.data_ptr(), sigma.data_ptr(), row0, n, D, seed & 0xFFFFFFFFFFFFFFFF,
                                      stream_id & 0xFFFFFFFFFFFFFFFF, _offset_ptr(stream_offset), scale_mu, scale_sigma, peer.world, peer.rank,
                                      peer.peer_slots, peer.peer_flags_g, peer.epoch_g, peer._counter(1), ws.data_ptr(), ws.numel(),
                                      nat.stream_of(mu))
    nat.check(rc, "evok_grad_push")


def evaluate(objective: int, X: torch.Tensor, f: Optional[torch.Tensor] = None) -> torch.Tensor:
    _mat(X, "X")
    n, D = X.shape
    if f is None:
        f = torch.empty(n, dtype=torch.float32, device=X.device)
    _vec(f, "f", n)
    with _timed("eval"):
        rc = nat.lib().evok_eval(objective, X.data_ptr(), X.stride(0), n, D, f.data_ptr(), nat.stream_of(X))
    nat.check(rc, "evok_eval")
    return f


# ------------------------------------------------------------------------------------------------ K3
def _rank_ws(device: torch.device, n: int) -> torch.Tensor:
    return nat.workspace(device, nat.lib().evok_rank_workspace_bytes(n), "rank")


def rank(f: torch.Tensor, method: str, higher_is_better: bool, out: Optional[torch.Tensor] = None,
         perm: Optional[torch.Tensor] = None) -> torch.Tensor:
    f = _vec(f, "fitnesses")
    n = f.numel()
    w = torch.empty_like(f) if out is None else _vec(out, "out", n)
    if perm is not None and not (perm.is_cuda and perm.dtype == torch.int64 and perm.is_contiguous() and perm.numel() == n):
        raise ValueError("perm: expected a contiguous int64 CUDA tensor of the same length")
    ws = _rank_ws(f.device, n)
    method_id = RANK_IDS[method]
    with _timed("rank"):
        rc = nat.lib().evok_rank(method_id, f.data_ptr(), n, int(bool(higher_is_better)), w.data_ptr(), nat.ptr(perm), ws.data_ptr(),
                                 ws.numel(), nat.stream_of(f))
    nat.check(rc, "evok_rank")
    return w


def argsort(keys: torch.Tensor, descending: bool) -> torch.Tensor:
    keys = _vec(keys, "keys")
    n = keys.numel()
    perm = torch.empty(n, dtype=torch.int64, device=keys.device)
    ws = _rank_ws(keys.device, n)
    nat.check(nat.lib().evok_argsort(keys.data_ptr(), n, int(bool(descending)), perm.data_ptr(), ws.data_ptr(), ws.numel(),
                                     nat.stream_of(keys)), "evok_argsort")
    return perm


def rank_table(keys: torch.Tensor, descending: bool, table: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out[i] = table[position of keys[i] in the stable sorted order] (position 0 = largest key if `descending`)."""
    keys = _vec(keys, "keys")
    n = keys.numel()
    _vec(table, "table", n)
    out = torch.empty_like(keys) if out is None else _vec(out, "out", n)
    ws = _rank_ws(keys.device, n)
    with _timed("rank"):
        rc = nat.lib().evok_rank_table(keys.data_ptr(), n, int(bool(descending)), table.data_ptr(), out.data_ptr(), ws.data_ptr(), ws.numel(),
                                       nat.stream_of(keys))
    nat.check(rc, "evok_rank_table")
    return out


def cmaes_row_weights(assigned: torch.Tensor, Z: torch.Tensor, active: bool, w_pos: torch.Tensor, w_act: torch.Tensor) -> None:
    """w_pos = max(assigned, 0); w_act = assigned > 0 ? assigned : D * assigned / ||z_i||^2 (or `assigned` when not `active`)."""
    _mat(Z, "Z")
    n, d = Z.shape
    _vec(assigned, "assigned", n); _vec(w_pos, "w_pos", n); _vec(w_act, "w_act", n)
    nat.check(nat.lib().evok_cmaes_row_weights(assigned.data_ptr(), Z.data_ptr(), Z.stride(0), n, d, int(bool(active)), w_pos.data_ptr(),
                                               w_act.data_ptr(), nat.stream_of(Z)), "evok_cmaes_row_weights")


def cmaes_vector_update(local_disp: torch.Tensor, shaped_disp: torch.Tensor, m: torch.Tensor, p_sigma: torch.Tensor, p_c: torch.Tensor,
                        sigma: torch.Tensor, consts, csa_squared: bool, k_out: torch.Tensor, *, steps: int = 0,
                        steps_dev: Optional[torch.Tensor] = None, h_sig_out: Optional[torch.Tensor] = None) -> None:
    """In place: m, p_sigma, sigma (1-element tensor), p_c; k_out (3 floats) = coefficients of the covariance update."""
    import ctypes

    d = m.numel()
    _vec(local_disp, "local_disp", d); _vec(shaped_disp, "shaped_disp", d); _vec(m, "m"); _vec(p_sigma, "p_sigma", d); _vec(p_c, "p_c", d)
    _vec(k_out, "k_out", 3)
    if not (sigma.is_cuda and sigma.dtype == torch.float32 and sigma.numel() == 1):
        raise ValueError("sigma: expected a 1-element float32 CUDA tensor")
    if steps_dev is not None and not (steps_dev.is_cuda and steps_dev.dtype == torch.int64 and steps_dev.numel() == 1):
        raise ValueError("steps_dev: expected a 1-element int64 CUDA tensor")
    carr = (ctypes.c_float * 10)(*[float(x) for x in consts])
    nat.check(nat.lib().evok_cmaes_vector_update(local_disp.data_ptr(), shaped_disp.data_ptr(), d, m.data_ptr(), p_sigma.data_ptr(), p_c.data_ptr(),
                                                 sigma.data_ptr(), nat.ptr(steps_dev), int(steps), carr, int(bool(csa_squared)), k_out.data_ptr(),
                                                 nat.ptr(h_sig_out), nat.stream_of(m)), "evok_cmaes_vector_update")


def weights_adjust_(w: torch.Tensor, mode: int) -> torch.Tensor:
    _vec(w, "weights")
    nat.check(nat.lib().evok_weights_adjust(w.data_ptr(), w.numel(), mode, nat.stream_of(w)), "evok_weights_adjust")
    return w


def elite_mask(w: torch.Tensor, num_elites: int) -> torch.Tensor:
    w = _vec(w, "weights")
    n = w.numel()
    mask = torch.empty_like(w)
    ws = _rank_ws(w.device, n)
    nat.check(nat.lib().evok_elite_mask(w.data_ptr(), n, num_elites, mask.data_ptr(), ws.data_ptr(), ws.numel(), nat.stream_of(w)),
              "evok_elite_mask")
    return mask


# ------------------------------------------------------------------------------------------------ K4
def grad(form: int, X: torch.Tensor, w: torch.Tensor, mu: torch.Tensor, sigma: torch.Tensor, scale_mu: float, scale_sigma: float,
         out_mu: Optional[torch.Tensor] = None, out_sigma: Optional[torch.Tensor] = None) -> tuple:
    _mat(X, "samples")
    n, D = X.shape
    _vec(w, "weights", n); _vec(mu, "mu", D); _vec(sigma, "sigma", D)
    out_mu = torch.empty_like(mu) if out_mu is None else _vec(out_mu, "out_mu", D)
    out_sigma = torch.empty_like(mu) if out_sigma is None else _vec(out_sigma, "out_sigma", D)
    ws = nat.workspace(X.device, nat.lib().evok_grad_workspace_bytes(n, D), "grad")
    with _timed("grad"):
        rc = nat.lib().evok_grad(form, X.data_ptr(), X.stride(0), w.data_ptr(), mu.data_ptr(), sigma.data_ptr(), n, D, scale_mu,
                                 scale_sigma, out_mu.data_ptr(), out_sigma.data_ptr(), ws.data_ptr(), ws.numel(), nat.stream_of(X))
    nat.check(rc, "evok_grad")
    return out_mu, out_sigma


def grad_regen(form: int, w: torch.Tensor, mu: torch.Tensor, sigma: torch.Tensor, *, seed: int, stream_id: int, row0: int,
               scale_mu: float, scale_sigma: float, out_mu: Optional[torch.Tensor] = None,
               out_sigma: Optional[torch.Tensor] = None, stream_offset: Optional[torch.Tensor] = None) -> tuple:
    n, D = w.numel(), mu.numel()
    _vec(w, "weights"); _vec(mu, "mu"); _vec(sigma, "sigma", D)
    out_mu = torch.empty_like(mu) if out_mu is None else _vec(out_mu, "out_mu", D)
    out_sigma = torch.empty_like(mu) if out_sigma is None else _vec(out_sigma, "out_sigma", D)
    ws = nat.workspace(mu.device, nat.lib().evok_grad_workspace_bytes(n, D), "grad")
    with _timed("grad_regen"):
        rc = nat.lib().evok_grad_regen(form, w.data_ptr(), mu.data_ptr(), sigma.data_ptr(), row0, n, D, seed & 0xFFFFFFFFFFFFFFFF,
                                       stream_id & 0xFFFFFFFFFFFFFFFF, _offset_ptr(stream_offset), scale_mu, scale_sigma, out_mu.data_ptr(),
                                       out_sigma.data_ptr(), ws.data_ptr(), ws.numel(), nat.stream_of(mu))
    nat.check(rc, "evok_grad_regen")
    return out_mu, out_sigma


# ------------------------------------------------------------------------------------------------ K5
def clipup_step(g: torch.Tensor, velocity: torch.Tensor, stepsize: float, momentum: float, max_speed: float,
                step_out: Optional[torch.Tensor] = None, mu: Optional[torch.Tensor] = None) -> None:
    D = g.numel()
    _vec(g, "g"); _vec(velocity, "velocity", D)
    with _timed("mu_step"):
        rc = nat.lib().evok_clipup_step(g.data_ptr(), D, velocity.data_ptr(), stepsize, momentum, max_speed, nat.ptr(step_out),
                                        nat.ptr(mu), nat.stream_of(g))
    nat.check(rc, "evok_clipup_step")


def adam_step(g: torch.Tensor, m: torch.Tensor, v: torch.Tensor, t: int, lr: float, beta1: float, beta2: float, eps: float,
              step_out: Optional[torch.Tensor] = None, mu: Optional[torch.Tensor] = None) -> None:
    D = g.numel()
    _vec(g, "g"); _vec(m, "m", D); _vec(v, "v", D)
    rc = nat.lib().evok_adam_step(g.data_ptr(), D, m.data_ptr(), v.data_ptr(), t, lr, beta1, beta2, eps, nat.ptr(step_out), nat.ptr(mu),
                                  nat.stream_of(g))
    nat.check(rc, "evok_adam_step")


def sgd_step(g: torch.Tensor, buf: Optional[torch.Tensor], first_step: bool, lr: float, momentum: float,
             step_out: Optional[torch.Tensor] = None, mu: Optional[torch.Tensor] = None) -> None:
    D = g.numel()
    _vec(g, "g")
    rc = nat.lib().evok_sgd_step(g.data_ptr(), D, nat.ptr(buf), int(first_step), lr, momentum, nat.ptr(step_out), nat.ptr(mu),
                                 nat.stream_of(g))
    nat.check(rc, "evok_sgd_step")


def axpy_(mu: torch.Tensor, g: torch.Tensor, lr: float) -> None:
    D = g.numel()
    _vec(g, "g"); _vec(mu, "mu", D)
    nat.check(nat.lib().evok_axpy(g.data_ptr(), D, lr, mu.data_ptr(), nat.stream_of(g)), "evok_axpy")


def _bound(x, D: int, device) -> tuple:
    """(vector pointer or None, scalar) for a None / scalar / vector bound."""
    if x is None:
        return None, NAN
    if isinstance(x, torch.Tensor) and x.ndim >= 1 and x.numel() > 1:
        v = x.to(device=device, dtype=torch.float32).contiguous()
        if v.numel() != D:
            raise IndexError(f"bound vector has length {v.numel()}, expected {D}")
        return v, NAN
    return None, float(x)


def sigma_update_(sigma: torch.Tensor, g: torch.Tensor, lr: float, exp_form: bool, lb=None, ub=None, max_change=None) -> None:
    D = sigma.numel()
    _vec(sigma, "sigma"); _vec(g, "g", D)
    lbv, lbs = _bound(lb, D, sigma.device)
    ubv, ubs = _bound(ub, D, sigma.device)
    mcv, mcs = _bound(max_change, D, sigma.device)
    with _timed("sigma_step"):
        rc = nat.lib().evok_sigma_update(sigma.data_ptr(), g.data_ptr(), D, lr, int(exp_form), nat.ptr(lbv), lbs, nat.ptr(ubv), ubs,
                                         nat.ptr(mcv), mcs, nat.stream_of(sigma))
    nat.check(rc, "evok_sigma_update")


def cem_finalize(s1: torch.Tensor, s2: torch.Tensor, sigma: torch.Tensor, num_elites: int) -> tuple:
    D = sigma.numel()
    gm, gs = torch.empty_like(sigma), torch.empty_like(sigma)
    nat.check(nat.lib().evok_cem_finalize(s1.data_ptr(), s2.data_ptr(), sigma.data_ptr(), D, num_elites, gm.data_ptr(), gs.data_ptr(),
                                          nat.stream_of(sigma)), "evok_cem_finalize")
    return gm, gs


# ------------------------------------------------------------------------------------------------ batched searches (functional API)
def _items(t: torch.Tensor, core_shape: tuple, name: str) -> tuple:
    """(tensor, n_items or None, item stride in elements) of an operand that is either shared (shape == core_shape, stride 0) or
    contiguous [items, *core_shape]."""
    if not (t.is_cuda and t.dtype == torch.float32):
        raise ValueError(f"{name}: expected a float32 CUDA tensor")
    t = as_plain_tensor(t)
    if tuple(t.shape) == tuple(core_shape):
        return t.contiguous(), None, 0
    if tuple(t.shape[1:]) != tuple(core_shape) or t.ndim != len(core_shape) + 1:
        raise ValueError(f"{name}: expected shape {core_shape} or (items, {', '.join(map(str, core_shape))}), got {tuple(t.shape)}")
    t = t.contiguous()
    return t, t.shape[0], int(t.stride(0))


def sample_batched(out: torch.Tensor, mu: torch.Tensor, sigma: torch.Tensor, *, symmetric: bool, seed: int, stream_id0: int = 0) -> torch.Tensor:
    """out[b] ~ N(mu[b], diag(sigma[b]^2)) for every batch item in one launch; item b uses Philox stream stream_id0 + b."""
    if not (out.is_cuda and out.dtype == torch.float32 and out.ndim == 3 and out.is_contiguous()):
        raise ValueError("out: expected a contiguous float32 CUDA tensor of shape (items, popsize, D)")
    B, n, d = out.shape
    mu, bm, sm = _items(mu, (d,), "mu")
    sigma, bs, ss = _items(sigma, (d,), "sigma")
    for cnt in (bm, bs):
        if cnt is not None and cnt != B:
            raise ValueError("mu / sigma: number of items differs from out")
    if symmetric and n % 2:
        raise ValueError(f"Symmetric sampling cannot be done if the number of solutions is odd: {n}")
    with _timed("sample"):
        rc = nat.lib().evok_sample_batched(out.data_ptr(), n * d, d, mu.data_ptr(), sm, sigma.data_ptr(), ss, B, n, d, int(symmetric),
                                           seed & 0xFFFFFFFFFFFFFFFF, stream_id0 & 0xFFFFFFFFFFFFFFFF, nat.stream_of(out))
    nat.check(rc, "evok_sample_batched")
    return out


def rank_batched(f: torch.Tensor, method: str, higher_is_better: bool) -> torch.Tensor:
    """Utilities of `items` independent fitness vectors, f: (items, N)."""
    if not (f.is_cuda and f.dtype == torch.float32 and f.ndim == 2):
        raise ValueError("f: expected a float32 CUDA tensor of shape (items, N)")
    f = as_plain_tensor(f).contiguous()
    B, n = f.shape
    w = torch.empty_like(f)
    lib = nat.lib()
    ws = nat.workspace(f.device, max(lib.evok_rank_workspace_bytes(n), 8 * B + 256), "rank")
    with _timed("rank"):
        rc = lib.evok_rank_batched(RANK_IDS[method], f.data_ptr(), n, B, int(bool(higher_is_better)), w.data_ptr(), ws.data_ptr(), ws.numel(),
                                   nat.stream_of(f))
    nat.check(rc, "evok_rank_batched")
    return w


def elite_mask_batched(w: torch.Tensor, num_elites: int) -> torch.Tensor:
    w = as_plain_tensor(w).contiguous()
    B, n = w.shape
    mask = torch.empty_like(w)
    ws = _rank_ws(w.device, n)
    nat.check(nat.lib().evok_elite_mask_batched(w.data_ptr(), n, B, num_elites, mask.data_ptr(), ws.data_ptr(), ws.numel(), nat.stream_of(w)),
              "evok_elite_mask_batched")
    return mask


def weights_adjust_batched_(w: torch.Tensor, mode: int) -> torch.Tensor:
    B, n = w.shape
    nat.check(nat.lib().evok_weights_adjust_batched(w.data_ptr(), n, B, mode, nat.stream_of(w)), "evok_weights_adjust_batched")
    return w


def grad_batched(form: int, X: torch.Tensor, w: torch.Tensor, mu: torch.Tensor, sigma: torch.Tensor, scale_mu: float, scale_sigma: float) -> tuple:
    """K4 for `items` independent searches in one launch chain.  X: (items, N, D), w: (items, N), mu / sigma: (D,) or (items, D)."""
    if not (X.is_cuda and X.dtype == torch.float32 and X.ndim == 3):
        raise ValueError("X: expected a float32 CUDA tensor of shape (items, N, D)")
    X = as_plain_tensor(X).contiguous()
    B, n, d = X.shape
    w = as_plain_tensor(w).contiguous()
    if tuple(w.shape) != (B, n):
        raise ValueError(f"w: expected shape {(B, n)}, got {tuple(w.shape)}")
    mu, bm, sm = _items(mu, (d,), "mu")
    sigma, bs, ss = _items(sigma, (d,), "sigma")
    out_mu = torch.empty(B, d, dtype=torch.float32, device=X.device)
    out_sigma = torch.empty_like(out_mu)
    lib = nat.lib()
    ws = nat.workspace(X.device, lib.evok_grad_batched_workspace_bytes(B, n, d), "grad_batched")
    with _timed("grad"):
        rc = lib.evok_grad_batched(form, X.data_ptr(), n * d, d, w.data_ptr(), mu.data_ptr(), sm, sigma.data_ptr(), ss, B, n, d, scale_mu, scale_sigma,
                                   out_mu.data_ptr(), out_sigma.data_ptr(), ws.data_ptr(), ws.numel(), nat.stream_of(X))
    nat.check(rc, "evok_grad_batched")
    return out_mu, out_sigma


def _host_floats(values, n: int):
    import ctypes

    vals = [float(v) for v in values]
    if len(vals) != n:
        raise ValueError(f"expected {n} per-item scalars, got {len(vals)}")
    return (ctypes.c_float * n)(*vals)


def clipup_batched_(g: torch.Tensor, velocity: torch.Tensor, center: torch.Tensor, stepsizes, momenta, max_speeds) -> None:
    """In place on contiguous (items, D) tensors: one CTA per item (per-item hyper-parameters are host scalars)."""
    B, d = center.shape
    for t, name in ((g, "g"), (velocity, "velocity"), (center, "center")):
        if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and tuple(t.shape) == (B, d)):
            raise ValueError(f"{name}: expected a contiguous float32 CUDA tensor of shape {(B, d)}")
    nat.check(nat.lib().evok_clipup_batched(g.data_ptr(), B, d, velocity.data_ptr(), center.data_ptr(), _host_floats(stepsizes, B),
                                            _host_floats(momenta, B), _host_floats(max_speeds, B), nat.stream_of(g)), "evok_clipup_batched")


def sigma_update_batched_(sigma: torch.Tensor, g: torch.Tensor, lrs, exp_form: bool, lb: Optional[torch.Tensor] = None,
                          ub: Optional[torch.Tensor] = None, max_change: Optional[torch.Tensor] = None) -> None:
    """In place on contiguous (items, D) tensors; lb / ub / max_change: (items, D) tensors or None."""
    B, d = sigma.shape
    for t, name in ((sigma, "sigma"), (g, "g"), (lb, "lb"), (ub, "ub"), (max_change, "max_change")):
        if t is not None and not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and tuple(t.shape) == (B, d)):
            raise ValueError(f"{name}: expected a contiguous float32 CUDA tensor of shape {(B, d)}")
    nat.check(nat.lib().evok_sigma_update_batched(sigma.data_ptr(), g.data_ptr(), B, d, _host_floats(lrs, B), int(bool(exp_form)), nat.ptr(lb),
                                                  nat.ptr(ub), nat.ptr(max_change), nat.stream_of(sigma)), "evok_sigma_update_batched")


# ------------------------------------------------------------------------------------------------ K8
ACT_IDS = {"none": 0, "identity": 0, "tanh": 1, "relu": 2, "sigmoid": 3}


def mlp_forward(params: torch.Tensor, obs: torch.Tensor, dims, acts, out: Optional[torch.Tensor] = None, *,
                obs_sum: Optional[torch.Tensor] = None, obs_sumsq: Optional[torch.Tensor] = None, obs_count: Optional[torch.Tensor] = None,
                min_variance: float = 1e-2, clip: Optional[tuple] = None, active: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Batched policy forward: row i of `params` (flat Linear-layer parameters) applied to row i of `obs`.
    With `obs_sum / obs_sumsq / obs_count` (the RunningNorm sums, all on the device) the observations are normalised and
    clipped while they are loaded; with `active` (bool / uint8, N) inactive policies are skipped and get zero actions."""
    import ctypes

    _mat(params, "parameters"); _mat(obs, "observations")
    n = params.shape[0]
    dims = [int(d) for d in dims]
    act_ids = [ACT_IDS[a] if isinstance(a, str) else int(a) for a in acts]
    if obs.shape != (n, dims[0]):
        raise ValueError(f"observations: expected shape {(n, dims[0])}, got {tuple(obs.shape)}")
    if out is None:
        out = torch.empty(n, dims[-1], dtype=torch.float32, device=params.device)
    _mat(out, "out")
    d_arr = (ctypes.c_int32 * len(dims))(*dims)
    a_arr = (ctypes.c_int32 * len(act_ids))(*act_ids)
    need = nat.lib().evok_mlp_parameter_length(len(act_ids), d_arr)
    if params.shape[1] != need:
        raise ValueError(f"parameters: expected {need} columns for layer widths {dims}, got {params.shape[1]}")
    if obs_sum is None and active is None:
        with _timed("mlp_forward"):
            rc = nat.lib().evok_mlp_forward(params.data_ptr(), params.stride(0), obs.data_ptr(), obs.stride(0), out.data_ptr(), out.stride(0), n,
                                            len(act_ids), d_arr, a_arr, nat.stream_of(params))
        nat.check(rc, "evok_mlp_forward")
        return out
    if obs_sum is not None:
        _vec(obs_sum, "obs_sum", dims[0]); _vec(obs_sumsq, "obs_sumsq", dims[0])
        if obs_count is None or obs_count.dtype != torch.int64 or obs_count.numel() != 1 or not obs_count.is_cuda:
            raise ValueError("obs_count: expected a 1-element int64 CUDA tensor")
    if active is not None:
        if active.dtype == torch.bool:
            active = active.view(torch.uint8)
        if active.dtype != torch.uint8 or active.numel() != n or not active.is_cuda or not active.is_contiguous():
            raise ValueError(f"active: expected {n} contiguous bool / uint8 flags on the GPU")
    ws = None if active is None else nat.workspace(params.device, 256, "mlp")
    lo, hi = (NAN, NAN) if clip is None else (NAN if clip[0] is None else float(clip[0]), NAN if clip[1] is None else float(clip[1]))
    with _timed("mlp_forward"):
        rc = nat.lib().evok_mlp_forward_prep(params.data_ptr(), params.stride(0), obs.data_ptr(), obs.stride(0), out.data_ptr(), out.stride(0), n,
                                             len(act_ids), d_arr, a_arr, nat.ptr(obs_sum), nat.ptr(obs_sumsq), nat.ptr(obs_count),
                                             float(min_variance), lo, hi, nat.ptr(active), nat.ptr(ws), 0 if ws is None else ws.numel(),
                                             nat.stream_of(params))
    nat.check(rc, "evok_mlp_forward_prep")
    return out


def mlp_forward_shared(params: torch.Tensor, x: torch.Tensor, dims, acts) -> torch.Tensor:
    """Row i of `params` (N x L flat feed-forward parameters) applied to the SHARED input batch `x` (B x in) -> N x B x out.
    First layer: one tensor-core product of the stacked weight rows of all N networks with the batch (weights read from HBM once,
    3xTF32 = fp32 accuracy); remaining layers: per-network fp32 kernel."""
    import ctypes

    _mat(params, "parameters"); _mat(x, "x")
    dims = [int(d) for d in dims]
    act_ids = [ACT_IDS[a] if isinstance(a, str) else int(a) for a in acts]
    n, B = params.shape[0], x.shape[0]
    if x.shape[1] != dims[0]:
        raise ValueError(f"x: expected {dims[0]} columns, got {x.shape[1]}")
    if len(act_ids) < 2 or max(dims[1:]) > 512:
        raise ValueError("mlp_forward_shared handles nets with >= 2 layers and widths <= 512")
    d_arr = (ctypes.c_int32 * len(dims))(*dims)
    a_arr = (ctypes.c_int32 * len(act_ids))(*act_ids)
    lib = nat.lib()
    if params.shape[1] != lib.evok_mlp_parameter_length(len(act_ids), d_arr):
        raise ValueError("parameters: wrong number of columns for these layer widths")
    if x.data_ptr() % 16 != 0 or x.stride(0) % 4 != 0:  # the batch is the TMA operand: 16-byte aligned rows
        padded = torch.zeros(B, (dims[0] + 3) // 4 * 4, dtype=torch.float32, device=x.device)
        padded[:, :dims[0]] = x
        x = padded[:, :dims[0]]
    out = torch.empty(n, B, dims[-1], dtype=torch.float32, device=params.device)
    ws = nat.workspace(params.device, lib.evok_mlp_forward_shared_workspace_bytes(n, B, len(act_ids), d_arr) + 512, "mlp_shared")
    with _timed("mlp_forward_shared"):
        rc = lib.evok_mlp_forward_shared(params.data_ptr(), params.stride(0), n, x.data_ptr(), x.stride(0), B, len(act_ids), d_arr, a_arr,
                                         out.data_ptr(), ws.data_ptr(), ws.numel(), nat.stream_of(params))
    nat.check(rc, "evok_mlp_forward_shared")
    return out


# ------------------------------------------------------------------------------------------------ K6 / K7
def gemm_nt(A: torch.Tensor, B: torch.Tensor, out: Optional[torch.Tensor] = None, *, out2: Optional[torch.Tensor] = None,
            alpha: Optional[torch.Tensor] = None, bias: Optional[torch.Tensor] = None) -> torch.Tensor:
    """C = A @ B.T on the tensor cores with fp32 accuracy (3xTF32); optionally also out2 = alpha * C + bias (broadcast over rows)."""
    _mat(A, "A"); _mat(B, "B")
    M, K = A.shape
    N, K2 = B.shape
    if K != K2:
        raise ValueError(f"inner dimensions differ: {K} vs {K2}")
    if out is None:
        out = torch.empty(M, N, dtype=torch.float32, device=A.device)
    _mat(out, "out")
    if out2 is not None:
        _mat(out2, "out2")
    if bias is not None:
        _vec(bias, "bias", N)
    nbytes = nat.lib().evok_gemm_workspace_bytes(M, N, K)
    ws = nat.workspace(A.device, nbytes, "gemm")
    with _timed("gemm"):
        rc = nat.lib().evok_gemm_nt(A.data_ptr(), A.stride(0), B.data_ptr(), B.stride(0), M, N, K, out.data_ptr(), out.stride(0), nat.ptr(out2),
                                    0 if out2 is None else out2.stride(0), nat.ptr(alpha), nat.ptr(bias), ws.data_ptr(), ws.numel(),
                                    nat.stream_of(A))
    nat.check(rc, "evok_gemm_nt")
    return out


def weighted_syrk_update(Y: torch.Tensor, w: torch.Tensor, k: torch.Tensor, C: torch.Tensor, u: Optional[torch.Tensor] = None,
                         out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out = k[0] * (Y^T diag(w) Y) + k[1] * C + k[2] * u u^T  -- the rank-mu + rank-1 covariance update of CMA-ES (cmaes.py:519-553)
    as one transposing pass over Y and one tensor-core GEMM whose epilogue (or split-K reduction) applies the update.
    `k`: 3 device floats.  `out` may be `C` (in place)."""
    _mat(Y, "Y"); _mat(C, "C")
    n, d = Y.shape
    _vec(w, "w", n); _vec(k, "k", 3)
    if C.shape != (d, d):
        raise ValueError(f"C: expected shape {(d, d)}, got {tuple(C.shape)}")
    if u is not None:
        _vec(u, "u", d)
    out = torch.empty_like(C) if out is None else _mat(out, "out")
    ldo = (n + 3) // 4 * 4
    lib = nat.lib()
    tws = nat.workspace(Y.device, 2 * d * ldo * 4 + 256, "syrk_operands")
    base = (tws.data_ptr() + 255) // 256 * 256
    a_w, a_p = base, base + d * ldo * 4
    nat.check(lib.evok_transpose_pair(Y.data_ptr(), Y.stride(0), n, d, w.data_ptr(), a_w, a_p, ldo, nat.stream_of(Y)), "evok_transpose_pair")
    ws = nat.workspace(Y.device, lib.evok_gemm_workspace_bytes(d, d, n), "gemm")
    with _timed("gemm"):
        rc = lib.evok_gemm_nt_affine(a_w, ldo, a_p, ldo, d, d, n, out.data_ptr(), out.stride(0), k.data_ptr(), C.data_ptr(), C.stride(0), nat.ptr(u),
                                     ws.data_ptr(), ws.numel(), nat.stream_of(Y))
    nat.check(rc, "evok_gemm_nt_affine")
    return out


def cholesky(A: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Lower Cholesky factor of a symmetric positive definite fp32 matrix (only the lower triangle of `A` is read); NaNs if `A` is not
    positive definite.  One persistent tile-dataflow kernel (csrc/evok_chol.cu)."""
    _mat(A, "A")
    n = A.shape[0]
    if A.shape[1] != n:
        raise ValueError(f"A: expected a square matrix, got {tuple(A.shape)}")
    out = torch.empty_like(A) if out is None else _mat(out, "out")
    if out.data_ptr() == A.data_ptr():
        raise ValueError("out must not alias A")
    lib = nat.lib()
    ws = nat.workspace(A.device, lib.evok_cholesky_workspace_bytes(n), "cholesky")
    with _timed("cholesky"):
        rc = lib.evok_cholesky(A.data_ptr(), A.stride(0), n, out.data_ptr(), out.stride(0), ws.data_ptr(), ws.numel(), nat.stream_of(A))
    nat.check(rc, "evok_cholesky")
    return out


def transpose_scale(X: torch.Tensor, w: Optional[torch.Tensor] = None) -> torch.Tensor:
    """(w[:, None] * X).T as a new row-major matrix."""
    _mat(X, "X")
    rows, cols = X.shape
    if w is not None:
        _vec(w, "w", rows)
    out = torch.empty(cols, rows, dtype=torch.float32, device=X.device)
    nat.check(nat.lib().evok_transpose_scale(X.data_ptr(), X.stride(0), rows, cols, nat.ptr(w), out.data_ptr(), out.stride(0),
                                             nat.stream_of(X)), "evok_transpose_scale")
    return out
