"""Exercise every kernel of libevok.so at small, ragged sizes -- meant to run under compute-sanitizer:

    compute-sanitizer --tool memcheck  python scripts/sanitize.py
    compute-sanitizer --tool racecheck python scripts/sanitize.py
    compute-sanitizer --tool synccheck python scripts/sanitize.py
"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from evotorch_b200 import Problem, ops  # noqa: E402
from evotorch_b200.algorithms import CEM, CMAES, PGPE, SNES  # noqa: E402
from evotorch_b200.objectives import rastrigin, sphere  # noqa: E402

dev = "cuda"
torch.manual_seed(0)
for sym in (True, False):
    for n, D in ((6, 1), (10, 7), (64, 16), (48, 130), (34, 1000), (4100, 1028)):
        mu, sg = torch.randn(D, device=dev), torch.rand(D, device=dev) + 0.1
        X, f = torch.empty(n, D, device=dev), torch.empty(n, device=dev)
        for obj in (0, 1, 2, 3):
            ops.sample_eval(obj, X, mu, sg, n_rows=n, symmetric=sym, seed=1, stream_id=2, f=f if obj else None)
        ops.sample_eval(2, None, mu, sg, n_rows=n, symmetric=sym, seed=1, stream_id=2, f=f)
        for obj in (1, 2, 3):
            ops.evaluate(obj, X)
        w = ops.rank(f, "centered", False)
        for method in ("linear", "nes", "normalized", "raw"):
            ops.rank(f, method, True, perm=torch.empty(n, dtype=torch.int64, device=dev))
        ops.argsort(f, True)
        ops.elite_mask(w, n // 3)
        ops.weights_adjust_(w.clone(), 1)
        ops.weights_adjust_(w.clone(), 2)
        for form in (ops.GRAD_SEPARABLE, ops.GRAD_EXP, ops.GRAD_MOMENTS) + ((ops.GRAD_SYMMETRIC,) if sym else ()):
            ops.grad(form, X, w, mu, sg, 1.0, 1.0)
            ops.grad_regen(form, w, mu, sg, seed=1, stream_id=2, row0=0, scale_mu=1.0, scale_sigma=1.0)
        g = torch.randn(D, device=dev)
        ops.clipup_step(g, torch.zeros(D, device=dev), 0.1, 0.9, 0.2, step_out=torch.empty(D, device=dev), mu=mu.clone())
        ops.adam_step(g, torch.zeros(D, device=dev), torch.zeros(D, device=dev), 1, 0.01, 0.9, 0.999, 1e-8, step_out=torch.empty(D, device=dev))
        ops.sgd_step(g, torch.zeros(D, device=dev), True, 0.1, 0.9, step_out=torch.empty(D, device=dev))
        ops.axpy_(mu.clone(), g, 0.1)
        ops.sigma_update_(sg.clone(), g, 0.1, False, lb=0.01, ub=2.0, max_change=0.2)
        ops.cem_finalize(g, g * g + 1, sg, 5)
# big-enough rank to use several tiles
ops.rank(torch.randn(10_000, device=dev), "centered", False)
# MLP: aligned and odd-length rows
for dims, acts, n in (([376, 256, 17], ["tanh", "none"], 9), ([5, 1], ["none"], 3), ([33, 70, 9, 4], ["relu", "sigmoid", "tanh"], 6)):
    L = sum(dims[i] * dims[i + 1] + dims[i + 1] for i in range(len(acts)))
    ops.mlp_forward(torch.randn(n, L, device=dev), torch.randn(n, dims[0], device=dev), dims, acts)
# GEMM: partial tiles, split-K, fused epilogue
for M, N_, K in ((128, 256, 32), (100, 70, 36), (129, 257, 40), (300, 520, 260)):
    A, B = torch.randn(M, K, device=dev), torch.randn(N_, K, device=dev)
    ops.gemm_nt(A, B)
    ops.gemm_nt(A, B, out2=torch.empty(M, N_, device=dev), alpha=torch.ones(1, device=dev), bias=torch.randn(N_, device=dev))
    ops.transpose_scale(A, torch.randn(M, device=dev))
# searchers end to end (eager and graph replay)
for make in (lambda p: PGPE(p, popsize=64, center_learning_rate=0.5, stdev_learning_rate=0.1, stdev_init=1.0),
             lambda p: SNES(p, popsize=50, stdev_init=1.0), lambda p: CEM(p, popsize=60, parenthood_ratio=0.3, stdev_init=1.0)):
    for graph in (False, True):
        s = make(Problem("min", rastrigin, initial_bounds=(-5, 5), solution_length=50, device=dev, seed=1))
        if graph:
            s.enable_cuda_graph()
        s.run(5)
CMAES(Problem("min", sphere, initial_bounds=(-3, 3), solution_length=40, device=dev, seed=1), stdev_init=1.0, popsize=64).run(3)
# rollout extras of the policy kernel: fused normalisation / clipping / active mask, masked running statistics
from evotorch_b200.neuroevolution import RunningNorm  # noqa: E402

for dims, acts, n in (([376, 256, 17], ["tanh", "none"], 9), ([33, 70, 9, 4], ["relu", "sigmoid", "tanh"], 6)):
    L = sum(dims[i] * dims[i + 1] + dims[i + 1] for i in range(len(acts)))
    obs = torch.randn(n, dims[0], device=dev)
    active = torch.rand(n, device=dev) < 0.6
    rn = RunningNorm(shape=dims[0], dtype="float32", device=dev, clip=(-3.0, 3.0))
    rn.update(obs, active)
    rn.update(obs)
    ops.mlp_forward(torch.randn(n, L, device=dev), obs, dims, acts, obs_sum=rn.sum, obs_sumsq=rn.sum_of_squares, obs_count=rn.count_tensor,
                    clip=(-3.0, 3.0), active=active)
# lazy population (X = NULL sampler + regenerating gradient) and the peer-exchange kernels (world size 1: same kernels, local "peers")
s = PGPE(Problem("min", rastrigin, initial_bounds=(-5, 5), solution_length=50, device=dev, seed=1, lazy_population=True), popsize=64,
         center_learning_rate=0.5, stdev_learning_rate=0.1, stdev_init=1.0)
s.run(4)
import tempfile  # noqa: E402

import torch.distributed as dist  # noqa: E402

from evotorch_b200.peer import PeerExchange  # noqa: E402

dist.init_process_group("gloo", init_method=f"file://{tempfile.mkdtemp()}/pg", rank=0, world_size=1)
n, D = 130, 70
px = PeerExchange(n, D, torch.device(dev), timeout_ns=2_000_000_000)
mu, sg = torch.randn(D, device=dev), torch.rand(D, device=dev) + 0.1
X = torch.empty(n, D, device=dev)
for gen in range(3):
    ops.sample_eval(2, X, mu, sg, n_rows=n, symmetric=True, seed=3, stream_id=gen, f=px.f_all[0:n])
    px.push_fitness(0, n)
    w = ops.rank(px.wait_fitness(), "centered", False)
    ops.grad_push(ops.GRAD_SYMMETRIC, X, w, mu, sg, scale_mu=1.0, scale_sigma=1.0, peer=px)
    px.reduce_gradients()
    ops.grad_push(ops.GRAD_SYMMETRIC, None, w, mu, sg, scale_mu=1.0, scale_sigma=1.0, peer=px, seed=3, stream_id=gen, row0=0)
    px.reduce_gradients()
assert not px.timed_out()
# ---- round-2 kernels
# shared-minibatch policy forward: persistent gather GEMM (16-byte path at every row alignment, 4-byte path, generic tail) + tail kernels
from evotorch_b200.neuroevolution import Policy  # noqa: E402

for dims, acts, nn_, B in (((376, 256, 17), ("tanh", "none"), 5, 70), ((8, 512, 2), ("none", "tanh"), 3, 300), ((6, 16, 3), ("relu", "none"), 9, 33),
                           ((33, 40, 24, 5), ("tanh", "sigmoid", "none"), 7, 31)):
    layers = []
    for l in range(len(acts)):
        layers.append(torch.nn.Linear(dims[l], dims[l + 1]))
        if acts[l] != "none":
            layers.append({"tanh": torch.nn.Tanh, "relu": torch.nn.ReLU, "sigmoid": torch.nn.Sigmoid}[acts[l]]())
    pol = Policy(torch.nn.Sequential(*layers).to(dev))
    for pad in (0, 1, 2, 3):
        P = torch.randn(nn_, pol.parameter_length + pad, device=dev)[:, :pol.parameter_length]
        pol.forward_shared(P, torch.randn(B, dims[0] + pad, device=dev)[:, :dims[0]])
# CMA-ES glue, SYRK with the fused covariance update, Cholesky, batched functional kernels
c = CMAES(Problem("min", sphere, initial_bounds=(-3, 3), solution_length=72, device=dev, seed=1), stdev_init=1.0, popsize=40)
c.run(3)
c.enable_cuda_graph()
c.run(3)
for nch in (1, 5, 64, 65, 200):
    Bm = torch.randn(nch, nch, device=dev)
    ops.cholesky((Bm @ Bm.T / nch + torch.eye(nch, device=dev)).contiguous())
from evotorch_b200.algorithms.functional import cem, cem_ask, cem_tell, pgpe, pgpe_ask, pgpe_tell  # noqa: E402

st = pgpe(center_init=torch.randn(3, 21, device=dev), center_learning_rate=0.3, stdev_learning_rate=0.1, objective_sense="min", stdev_init=1.0)
for _ in range(2):
    pop = pgpe_ask(st, popsize=10)
    st = pgpe_tell(st, pop, (pop * pop).sum(-1))
st = cem(center_init=torch.randn(3, 21, device=dev), parenthood_ratio=0.5, objective_sense="min", stdev_init=1.0)
for _ in range(2):
    pop = cem_ask(st, popsize=10)
    st = cem_tell(st, pop, (pop * pop).sum(-1))
torch.cuda.synchronize()
print("SANITIZE_RUN_COMPLETE")
