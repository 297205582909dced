"""Single GPU, world size 1: cost of the peer-exchange path of the producers (plain sampler + push kernel + wait, gradient push +
reduce) vs the plain kernels (same work, plus flag traffic)."""
import os
import sys
import tempfile

import torch
import torch.distributed as dist

sys.path.insert(0, ".")
from evotorch_b200 import ops  # noqa: E402
from evotorch_b200.peer import PeerExchange  # noqa: E402

dist.init_process_group("gloo", init_method=f"file://{tempfile.mkdtemp()}/pg", rank=0, world_size=1)
n, d = int(sys.argv[1]) if len(sys.argv) > 1 else 500_000, 10_000
dev = torch.device("cuda")
px = PeerExchange(n, d, dev)
mu = torch.zeros(d, device=dev)
sigma = torch.ones(d, device=dev)
X = torch.empty(n, d, device=dev)
f = torch.empty(n, device=dev)
w = torch.randn(n, device=dev)


def timeit(fn, reps=10):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def plain_sample():
    ops.sample_eval(ops.OBJ_RASTRIGIN, X, mu, sigma, n_rows=n, symmetric=True, seed=1, stream_id=5, f=f)


def push_sample():
    ops.sample_eval(ops.OBJ_RASTRIGIN, X, mu, sigma, n_rows=n, symmetric=True, seed=1, stream_id=5, f=px.f_all)
    px.push_fitness(0, n)
    px.wait_fitness()


def plain_grad():
    ops.grad(ops.GRAD_SYMMETRIC, X, w, mu, sigma, 1.0, 1.0)


def push_grad():
    ops.grad_push(ops.GRAD_SYMMETRIC, X, w, mu, sigma, scale_mu=1.0, scale_sigma=1.0, peer=px)
    px.reduce_gradients()


for _ in range(3):  # warm the chip up to its steady power state first
    timeit(plain_sample)
for _ in range(5):
    print(f"rows {n}: sample_eval plain {timeit(plain_sample):.4f} ms  push+wait {timeit(push_sample):.4f} ms | "
          f"grad plain {timeit(plain_grad):.4f} ms  push+reduce {timeit(push_grad):.4f} ms", flush=True)
assert not px.timed_out()
os._exit(0)
