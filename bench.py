#!/usr/bin/env python
"""bench.py -- PGPE generations/s on synthetic Rastrigin (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--popsize P] [--dim D] [--dump-outputs DIR]

Workload (config.workload): PGPE (symmetric sampling, ClipUp, centered ranking, stdev_max_change 0.2; the reference's
defaults), Rastrigin, popsize 1,000,000 x dim 10,000 fp32 -- the configuration BASELINE.json's metric is quoted on; the
40 GB population fits one B200.  With N > 1 (torchrun, one rank per GPU) the SAME population is row-sharded over the ranks
(strong scaling): per generation one all-gather of the fitness vector and one all-reduce of the stacked gradients.

One "step" = one generation through the public API (`searcher.step()`): rank -> weighted gradient reduction -> ClipUp /
sigma update -> fused Philox sampling + evaluation of a fresh population.

JSON line (rank 0): value = generations/s, device-timed (CUDA events, max over ranks) with the population resident in HBM;
e2e = the same generation driven through `Problem.sample_and_compute_gradients` with a HOST-resident distribution (mu, sigma in
pinned host memory are copied to the device every step, gradients and mean fitness are copied back; the reference's
`dist_on_cpu` actor protocol, core.py:2958); roofline = the dominant kernel (fused sample+evaluate) timed live with CUDA
events; cpu_baseline = the reference's torch-CPU op sequence (oracle/ref_cpu_path.py) on this box's host cores.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "PGPE generations/sec at popsize=1Mxdim=10k (Rastrigin, fp32)"
METRIC_BY_CONFIG = {"cfg2": "PGPE generations/sec at popsize=100kxdim=10k (Rastrigin, fp32)",
                    "cfg5": "PGPE generations/sec at popsize=1Mxdim=100k sharded (Rastrigin, fp32)"}
UNIT = "generations/s"
LR_MU, LR_SIGMA, STDEV_INIT, SEED = 0.5, 0.1, 1.0, 0


CONFIGS = {  # BASELINE.json configs that are bench workloads (the others are parity-test cases)
    "metric": dict(popsize=1_000_000, dim=10_000),  # the configuration the metric is quoted on; fits one B200 (40 GB)
    "cfg2": dict(popsize=100_000, dim=10_000),      # BASELINE configs[1]
    "cfg5": dict(popsize=1_000_000, dim=100_000),   # BASELINE configs[4]: 400 GB of samples, sharded over 2 / 4 / 8 GPUs
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="metric", choices=sorted(CONFIGS), help="workload: metric = PGPE 1M x 10k (default); cfg2 = 100k x 10k; "
                    "cfg5 = 1M x 100k row-sharded over the GPUs (materialised shards while they fit in HBM, else the lazy population)")
    ap.add_argument("--popsize", type=int, default=None)
    ap.add_argument("--dim", type=int, default=None)
    ap.add_argument("--lazy", type=int, default=-1, help="1/0: never materialise the population (Philox regeneration). Default: only when the shard does not fit")
    ap.add_argument("--cpu-sizes", default=None, help="comma-separated population sizes of the CPU-baseline samples (default: 2k,4k,8k rows x 10k "
                    "columns in our arm's bounded leg; 10k,30k,100k in the reference arm -- SURVEY 8(d))")
    ap.add_argument("--cpu-budget-s", type=float, default=None, help="wall-clock budget of the CPU leg (default 25 s in our arm, 200 s in the reference arm)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the short cfg2 / cfg3 / cfg4 legs of the default N = 1 line")
    ap.add_argument("--no-sharded-parity", action="store_true", help="skip the sharded-vs-unsharded parity leg at N > 1")
    ap.add_argument("--cuda-graph", type=int, default=-1, help="1/0: replay each generation from a CUDA graph. Default: 0 at N = 1 (kernels are timed live inside the timed region), 1 at N > 1 (the fused kernel is then timed stand-alone right after the timed region)")
    ap.add_argument("--peer", type=int, default=-1, help="1/0: at N > 1 move fitnesses and gradients between the GPUs from inside the producing kernels (NVLink peer memory, evotorch_b200/peer.py) instead of NCCL all_gather/all_reduce. Default: 1 at N > 1")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="after the timed steps, write what the last timed generation "
                    "computed as DIR/<name>.npy: center, stdev, mean_eval, the fitnesses and a fixed, seeded sample of population rows "
                    "(at most 64 MB in all); inputs are seeded, so two builds can be compared output for output")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs dumps the GPU path (--impl ours)")
    cfg = CONFIGS[a.config]
    a.popsize = cfg["popsize"] if a.popsize is None else a.popsize
    a.dim = cfg["dim"] if a.dim is None else a.dim
    return a


def metric_name(args) -> str:
    cfg = CONFIGS[args.config]
    if (args.popsize, args.dim) == (cfg["popsize"], cfg["dim"]):
        return METRIC_BY_CONFIG.get(args.config, METRIC)
    return f"PGPE generations/sec at popsize={args.popsize}xdim={args.dim} (Rastrigin, fp32)"


def workload_config(args, n_gpus, collectives="nccl"):
    how = {"nccl": "NCCL all_gather(fitness) + all_reduce(grad)",
           "peer": "fitness gather + gradient reduction fused into the producing kernels over NVLink peer memory (no NCCL in the loop)"}[collectives]
    return {
        "workload": f"PGPE(symmetric, ClipUp, centered ranking, stdev_max_change=0.2) on Rastrigin, popsize={args.popsize}, dim={args.dim}, fp32",
        "popsize": args.popsize,
        "dim": args.dim,
        "center_learning_rate": LR_MU,
        "stdev_learning_rate": LR_SIGMA,
        "stdev_init": STDEV_INIT,
        "parallelism": f"population row-sharded over {n_gpus} GPU(s); {how}" if n_gpus > 1 else "single GPU",
        "l2": "inputs larger than L2 (population %.1f GB >> 126 MB): no flush needed" % (4.0 * args.popsize * args.dim / 1e9 / n_gpus),
    }


# ----------------------------------------------------------------------------------------------------- CPU baseline
def cpu_reference_run(args, *, sizes, budget_s: float, max_steps: int, with_gpu_eager: bool) -> dict:
    """SURVEY 8(d) protocol for the reference's CPU path: time the reference's torch-CPU op sequence (oracle/ref_cpu_path.py,
    bit-identical to the live reference) with all host threads at several population sizes (full dimension), check that the
    time per generation is linear in the population size, and extrapolate to the workload's population from the least-squares
    line t(N) = a + b N (every op on the path is linear in N apart from the O(N log N) argsort of N floats, < 1 % of a
    generation).  `budget_s` bounds the leg: the number of timed generations per size is chosen from the first measurement."""
    import torch

    from oracle.ref_cpu_path import PGPEReferencePath

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sizes = sorted({min(int(n) - int(n) % 2, args.popsize) for n in sizes})
    t_leg = time.perf_counter()
    per_size, per_row_guess = [], None
    share = budget_s / sum(sizes)  # seconds of budget per sampled row, all sizes together
    for n in sizes:
        path = PGPEReferencePath(args.dim, n, center_learning_rate=LR_MU, stdev_learning_rate=LR_SIGMA, stdev_init=STDEV_INIT, seed=SEED)
        path.step()  # generation 0 only samples and evaluates: allocation + first touch of the population, not timed
        t0 = time.perf_counter()
        path.step()  # first full generation (also the warm-up of the update ops)
        first = time.perf_counter() - t0
        per_row_guess = first / n
        k = int(max(1, min(max_steps, (share * n - first) / max(first, 1e-9))))
        times = []
        for _ in range(k):
            t0 = time.perf_counter()
            path.step()
            times.append(time.perf_counter() - t0)
        times.sort()
        per_size.append({"popsize": n, "timed_steps": k, "median_s": times[len(times) // 2], "min_s": times[0], "first_step_s": first})
        del path
    xs = [float(r["popsize"]) for r in per_size]
    ys = [r["median_s"] for r in per_size]
    if len(xs) >= 2:
        mx, my = sum(xs) / len(xs), sum(ys) / len(ys)
        b = sum((x - mx) * (y - my) for x, y in zip(xs, ys)) / sum((x - mx) ** 2 for x in xs)
        a = my - b * mx
    else:
        a, b = 0.0, ys[0] / xs[0]
    fit_kind = "t(N) = a + b*N seconds per generation, least squares over the medians"
    if a < 0.0 or b <= 0.0:  # noisy tiny samples: a negative fixed cost is unphysical -> line through the origin
        a, b = 0.0, sum(x * y for x, y in zip(xs, ys)) / sum(x * x for x in xs)
        fit_kind = "t(N) = b*N (least squares through the origin: the unconstrained fit had a negative intercept or slope)"
    resid = max(abs((a + b * x) - y) / y for x, y in zip(xs, ys))
    t_full = a + b * args.popsize
    prop = ys[-1] * args.popsize / xs[-1]  # plain proportional scaling of the largest sample, for comparison
    linearity = {"fit": fit_kind, "a_s": a, "b_s_per_row": b,
                 "max_rel_residual": resid, "extrapolated_s_per_generation": t_full, "proportional_from_largest_s": prop,
                 "per_row_us": [1e6 * y / x for x, y in zip(xs, ys)]}
    torch_eager_gpu = None
    if with_gpu_eager and torch.cuda.is_available():
        # the same torch op sequence, eager, on this GPU ("PyTorch path" comparator, SURVEY 8(d)); bounded sample, scaled linearly
        try:
            n_gpu = min(100_000, args.popsize, int(1e9 // args.dim))
            n_gpu -= n_gpu % 2
            gpath = PGPEReferencePath(args.dim, n_gpu, center_learning_rate=LR_MU, stdev_learning_rate=LR_SIGMA, stdev_init=STDEV_INIT, seed=SEED,
                                      device="cuda")
            for _ in range(3):
                gpath.step()
            torch.cuda.synchronize()
            g0 = time.perf_counter()
            for _ in range(10):
                gpath.step()
            torch.cuda.synchronize()
            gdt = (time.perf_counter() - g0) / 10
            torch_eager_gpu = {"value": (1.0 / gdt) * (n_gpu / args.popsize), "unit": UNIT,
                               "sample": f"10 generations at popsize={n_gpu} x dim={args.dim} ({1e3 * gdt:.2f} ms each), scaled linearly in popsize "
                                         f"to {args.popsize}; the reference's torch op sequence, eager, on cuda:0"}
            del gpath
            torch.cuda.empty_cache()
        except Exception as exc:  # e.g. out of memory for the temporaries: report, do not fail the bench
            torch_eager_gpu = {"unavailable": repr(exc)[:200]}
    direct = next((r for r in per_size if r["popsize"] == 100_000 and args.dim == 10_000), None)
    return {
        "value": 1.0 / t_full,
        "unit": UNIT,
        "cores": cores,
        "kind": "port",
        "extrapolated": True,
        # BASELINE config 2 (PGPE 100 k x 10 k) is one of the sampled sizes: measured directly, nothing extrapolated
        "cfg2_direct": None if direct is None else {"generations_per_s": 1.0 / direct["median_s"], "median_s": direct["median_s"], "min_s": direct["min_s"]},
        "linearity": linearity,
        "samples": per_size,
        "torch_eager_gpu": torch_eager_gpu,
        "sample": ("generations of the reference's torch-CPU op sequence at popsize " + ", ".join(str(r["popsize"]) for r in per_size)
                   + f" x dim={args.dim} (medians {', '.join('%.3f s' % r['median_s'] for r in per_size)}); least-squares line in popsize, "
                   f"max residual {100 * resid:.1f} %, EXTRAPOLATED to popsize={args.popsize}; torch {torch.__version__} CPU, "
                   f"{torch.get_num_threads()} threads; leg took {time.perf_counter() - t_leg:.0f} s"),
        "sample_ms_per_step": 1e3 * ys[-1],
    }


def cpu_sizes(args, default_elems) -> list:
    if args.cpu_sizes:
        return [int(x) for x in args.cpu_sizes.split(",") if x]
    return [max(2, int(e // args.dim)) for e in default_elems]  # same element counts for any dimension


# ----------------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.lines, self.proc, self.thread = [], None, None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
            # nvidia-smi takes a moment to start (NVML initialisation over all GPUs of the box, during which driver calls of this process
            # can stall): wait for its first sample so that none of that falls into the timed region
            deadline = time.perf_counter() + 5.0
            while not self.lines and time.perf_counter() < deadline and self.proc.poll() is None:
                time.sleep(0.01)
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self, t_begin: float, t_end: float) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        for t, line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            inside = t_begin <= t <= t_end + 0.1
            try:
                if inside:
                    sm.append(float(parts[1]))
                smax = float(parts[2])
            except ValueError:
                continue
            if inside:
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------- our arm
def measured_peak_gbs() -> tuple:
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def run_ours(args):
    import torch
    import torch.distributed as dist

    from evotorch_b200 import Problem, ops
    from evotorch_b200.algorithms import PGPE
    from evotorch_b200.distributions import SymmetricSeparableGaussian
    from evotorch_b200.objectives import rastrigin
    from evotorch_b200.optimizers import ClipUp
    from evotorch_b200.tools import modify_tensor

    # NCCL prints its version banner to STDOUT at NCCL_DEBUG=VERSION (set in some images): keep stdout = the one JSON line
    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
        os.environ["NCCL_DEBUG"] = "WARN"
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    N, D, K, W = args.popsize, args.dim, args.steps, max(args.warmup, 3)

    def barrier_sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- does the shard fit?  materialised population = 4 N D / world bytes; else the lazy (Philox-regenerating) population
    free_b, total_b = torch.cuda.mem_get_info()
    shard_bytes = 4.0 * (N // world) * D
    lazy = (shard_bytes > 0.85 * total_b) if args.lazy < 0 else bool(args.lazy)
    if world > 1:  # every rank must take the same decision
        t = torch.tensor([int(lazy)], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        lazy = bool(t.item())
    problem = Problem("min", rastrigin, initial_bounds=(-5.12, 5.12), solution_length=D, device=dev, seed=SEED, lazy_population=lazy)
    collectives, px = "nccl", None
    if world > 1 and (args.peer == 1 or args.peer < 0):
        try:
            from evotorch_b200.peer import enable_peer_exchange

            px = enable_peer_exchange(problem, N)
            collectives = "peer"
        except Exception as exc:  # e.g. CUDA IPC not permitted in this container: keep the NCCL collectives (still the GPU path)
            print(f"[bench] peer exchange unavailable ({exc!r}); using NCCL collectives", file=sys.stderr)
    searcher = PGPE(problem, popsize=N, center_learning_rate=LR_MU, stdev_learning_rate=LR_SIGMA, stdev_init=STDEV_INIT,
                    distributed=(world > 1))
    use_graph = (world > 1) if args.cuda_graph < 0 else args.cuda_graph == 1
    if use_graph:
        searcher.enable_cuda_graph()
    for _ in range(W):
        searcher.step()

    # ---- device-resident timing (value) + live per-kernel timing (roofline)
    clocks = ClockSampler(local_rank) if rank == 0 else None  # started (and warmed up) BEFORE the barrier: rank 0 must not enter late
    barrier_sync()
    launches0 = ops.launch_count()
    ops.enable_timers()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_begin = time.perf_counter()
    ev0.record()
    for _ in range(K):
        searcher.step()
    ev1.record()
    barrier_sync()
    t_end = time.perf_counter()
    elapsed_ms = max_over_ranks(ev0.elapsed_time(ev1))
    timers = ops.timer_results()
    ops.disable_timers()
    launches = ops.launch_count() - launches0
    clock_info = clocks.stop(t_begin, t_end) if clocks is not None else None
    mean_eval = float(searcher.status["mean_eval"])
    value = K / (elapsed_ms / 1e3)
    if args.dump_outputs and rank == 0:  # before anything below launches into the population's buffers
        dump_outputs(searcher, args.dump_outputs)

    # ---- roofline of the dominant kernel (fused sample + evaluate): algorithmic bytes = the population written once
    n_local = N // world
    peak, peak_src = measured_peak_gbs()
    kern = {}
    for name, (cnt, ms) in timers.items():
        kern[name] = {"launches_timed": cnt, "ms": ms}
    if "sample_eval" not in timers:  # CUDA-graph mode: kernels are not individually timed; time the fused kernel on its own
        pop = searcher._population if searcher._population is not None else next(iter(problem._grad_batches.values()))
        d0 = searcher._distribution
        ops.enable_timers()
        for _ in range(5):
            ops.sample_eval(problem.evok_objective_id, None if lazy else pop._data, d0.mu, d0.sigma, n_rows=len(pop), symmetric=True, seed=1,
                            stream_id=12345, f=pop._evdata.view(-1))
        torch.cuda.synchronize()
        timers = dict(timers, **ops.timer_results())
        ops.disable_timers()
        kern = {name: {"launches_timed": cnt, "ms": ms, "note": "timed stand-alone after the run (CUDA-graph mode)"} for name, (cnt, ms) in timers.items()}
    fused_ms = timers["sample_eval"][1]
    fused_bytes = 4.0 * n_local * D + 4.0 * n_local
    achieved = fused_bytes / (fused_ms * 1e-3) / 1e9
    # DRAM traffic of the kernel from the committed ncu --set full capture (profiles/traffic.json), scaled by rows x columns
    traffic, traffic_note = None, "no capture"
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
            cap = json.load(fh)["sample_eval"]
        if lazy:
            traffic_note = "lazy population: the kernel stores nothing (fitnesses only); the figure is MODEL bandwidth (bytes a materialising kernel would write)"
        else:
            traffic = cap["ratio"] * fused_bytes
            traffic_note = (f"dram__bytes_read+write = {cap['ratio']:.4f} x algorithmic bytes in {cap['source']} "
                            f"(captured at popsize {cap['capture']['popsize']}, scaled linearly to this launch)")
    except Exception:
        pass
    roofline = {"kernel": "evok::sample_eval_kernel<RASTRIGIN, symmetric, %s, vec4>" % ("no store (lazy)" if lazy else "store"), "bound": "hbm",
                "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_note": traffic_note, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": fused_bytes, "ms_per_launch": fused_ms,
                "timing": ("CUDA events around every launch inside the timed region" if not use_graph else
                           "generations replayed from a CUDA graph: the kernel was timed stand-alone (5 launches, CUDA events) right after the timed region"),
                "share_of_step": fused_ms / (elapsed_ms / K)}
    for gname in ("grad", "grad_regen"):
        if gname in timers:
            g_ms = timers[gname][1]
            g_bytes = 4.0 * (n_local // 2) * D
            kern[gname].update({"algorithmic_bytes": g_bytes, "achieved_gbs": g_bytes / (g_ms * 1e-3) / 1e9,
                                "frac": g_bytes / (g_ms * 1e-3) / 1e9 / peak})
    model_bytes = 10.0 * n_local * D  # SURVEY.md 8(d): write X + read X (evaluate) + read the + rows (gradient)
    traffic_bytes = 0.0 if lazy else 6.0 * n_local * D  # what this engine actually moves: evaluation is fused into the write

    # ---- end to end: host-resident distribution -> device generation -> gradients back to the host, every step
    e2e = None
    if not args.no_e2e:
        del searcher
        torch.cuda.empty_cache()
        mu_host = torch.empty(D, dtype=torch.float32).pin_memory()
        sigma_host = torch.empty(D, dtype=torch.float32).pin_memory()
        mu_host.copy_(torch.empty(D).uniform_(-5.12, 5.12, generator=torch.Generator().manual_seed(SEED)))
        sigma_host.fill_(STDEV_INIT)
        hdist = SymmetricSeparableGaussian({"mu": mu_host, "sigma": sigma_host, "divide_mu_grad_by": "num_directions",
                                            "divide_sigma_grad_by": "num_directions"})
        assert hdist.mu.data_ptr() == mu_host.data_ptr() and hdist.mu.is_pinned()  # the distribution lives in the pinned buffers
        hopt = ClipUp(solution_length=D, dtype=torch.float32, stepsize=LR_MU, device="cpu")

        def e2e_step():
            # H2D: mu, sigma (pinned) -> device inside sample_and_compute_gradients; D2H: gradients + mean fitness
            res = problem.sample_and_compute_gradients(hdist, N, ranking_method="centered")[0]
            _ = float(res["mean_eval"])
            upd = hdist.update_parameters(res["gradients"], learning_rates={"sigma": LR_SIGMA}, optimizers={"mu": hopt})
            new_sigma = modify_tensor(sigma_host, upd.sigma, max_change=0.2)
            mu_host.copy_(upd.mu)
            sigma_host.copy_(new_sigma)

        for _ in range(W):
            e2e_step()
        barrier_sync()
        t0 = time.perf_counter()
        for _ in range(K):
            e2e_step()
        barrier_sync()
        e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
        h2d = 2 * D * 4
        d2h = 2 * D * 4 + 4
        e2e = {"value": K / (e2e_ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "ms_per_step": e2e_ms / K,
               "api": "Problem.sample_and_compute_gradients(host-resident SymmetricSeparableGaussian) + update_parameters/modify_tensor on the host"}
    else:
        del searcher
        torch.cuda.empty_cache()

    # ---- N > 1: parity of the sharded generation with the unsharded one (same seed), measured in this very run
    sharded_parity = None
    if world > 1 and not args.no_sharded_parity:
        try:
            sharded_parity = sharded_parity_leg(dev, use_peer=(px is not None))
        except Exception as exc:
            sharded_parity = {"error": repr(exc)[:300]}

    def finish():
        # leave without tearing the NCCL communicators down (teardown after graph-captured collectives can hang); every rank
        # has passed the final barrier and rank 0 has flushed its JSON line
        sys.stdout.flush()
        sys.stderr.flush()
        if world > 1:
            os._exit(0)

    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    if rank != 0:
        finish()
        return

    line = {
        "metric": metric_name(args),
        "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": elapsed_ms / K,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dict(workload_config(args, world, collectives), cuda_graph=bool(use_graph), lazy_population=bool(lazy), name=args.config),
        "impl": "ours",
        "gpu_launches": int(launches), "clocks": clock_info, "e2e": e2e, "roofline": roofline, "kernels": kern,
        "whole_generation": {"model_bytes_per_gen_per_gpu": model_bytes, "model_gbs": model_bytes * value / 1e9,
                             "model_frac_of_peak": model_bytes * value / 1e9 / peak,
                             "moved_bytes_per_gen_per_gpu": traffic_bytes, "moved_gbs": traffic_bytes * value / 1e9,
                             "note": "model = SURVEY 8(d) 10*N*D bytes (unfused write+read+half read); moved = 6*N*D (evaluation fused into the sampling write; 0 with the lazy population)"},
        "mean_eval_after": mean_eval,
    }
    if sharded_parity is not None:
        line["sharded_parity"] = sharded_parity
    if px is not None:
        if px.timed_out():
            raise RuntimeError("a peer-exchange wait timed out during the run: the numbers above are invalid")
        line["peer_exchange"] = {"wait_timeouts": 0, "buffer_bytes": px.nbytes}
    if world == 1 and not args.no_other_configs and args.config == "metric":
        line["other_configs"] = other_config_legs(dev, peak)
    if not args.no_cpu_baseline and world == 1:
        line["cpu_baseline"] = cpu_reference_run(args, sizes=cpu_sizes(args, (2e7, 4e7, 8e7)), budget_s=args.cpu_budget_s or 25.0, max_steps=3,
                                                 with_gpu_eager=True)
    emit(line)
    finish()


DUMP_BYTES = 64 << 20


def dump_outputs(searcher, directory: str) -> None:
    """What a caller of `searcher.step()` receives after the last step, as float32 / float64 .npy files: the distribution's
    center and stdev, mean_eval, and, where this process holds the population, its fitnesses and a sample of its rows.
    Samples are drawn with a fixed seed so that they name the same rows in every run; together they stay within DUMP_BYTES."""
    import numpy as np
    import torch

    os.makedirs(directory, exist_ok=True)
    status = searcher.status
    out = {"center": status["center"], "stdev": status["stdev"], "mean_eval": np.float64(status["mean_eval"])}
    pop = searcher.population  # None when the population is row-sharded over ranks
    if pop is not None:
        n, d = len(pop), pop.solution_length
        budget = (DUMP_BYTES - 8 * d - 64) // 4  # float32 elements left after center, stdev and mean_eval
        gen = torch.Generator().manual_seed(SEED)
        fitness = pop.evals[:, searcher.obj_index]
        n_fit = min(n, budget // 2)
        if n_fit < n:
            fitness = fitness[torch.randperm(n, generator=gen)[:n_fit].sort().values.to(fitness.device)]
        out["fitness"] = fitness
        n_rows = min(n, 512, max(1, (budget - n_fit) // d))
        rows = torch.randperm(n, generator=gen)[:n_rows].sort().values.tolist()
        out["population_rows"] = torch.stack([pop[i].values for i in rows])  # row by row: a lazy population regenerates them
    for name, value in out.items():
        arr = value.detach().float().cpu().numpy() if isinstance(value, torch.Tensor) else np.asarray(value)
        np.save(os.path.join(directory, f"{name}.npy"), arr)


def sharded_parity_leg(dev, use_peer: bool) -> dict:
    """Three distribution updates of PGPE at 100k x 1k, once row-sharded over the ranks (the collectives of the timed run) and once
    unsharded on every rank, same seed: the first population's ranking must be IDENTICAL (same Philox counters, global
    ranking) and mu / sigma must agree to fp32 summation order."""
    import torch
    import torch.distributed as dist

    from evotorch_b200 import Problem, ops
    from evotorch_b200.algorithms import PGPE
    from evotorch_b200.objectives import rastrigin

    n, d, gens, seed = 100_000, 1_000, 3, 17
    world, rank = dist.get_world_size(), dist.get_rank()

    def make(distributed):
        prob = Problem("min", rastrigin, initial_bounds=(-5.12, 5.12), solution_length=d, device=dev, seed=seed)
        if distributed and use_peer:
            from evotorch_b200.peer import enable_peer_exchange

            enable_peer_exchange(prob, n)
        return prob, PGPE(prob, popsize=n, center_learning_rate=LR_MU, stdev_learning_rate=LR_SIGMA, stdev_init=STDEV_INIT, distributed=distributed)

    prob_s, sh = make(True)
    prob_u, un = make(False)
    sh.step()
    un.step()
    # generation 0: the fitness vector of the sharded run (gathered here from the shards, whichever way the run exchanged them)
    # vs the unsharded population's
    shard = next(iter(prob_s._grad_batches.values()))
    local = shard.evals[:, 0].contiguous().clone()
    parts = [torch.empty_like(local) for _ in range(world)]
    dist.all_gather(parts, local)
    f_sharded = torch.cat(parts)
    f_un = un.population.evals[:, 0].contiguous()
    p1 = torch.empty(n, dtype=torch.int64, device=dev)
    p2 = torch.empty(n, dtype=torch.int64, device=dev)
    ops.rank(f_sharded.contiguous(), "centered", False, perm=p1)
    ops.rank(f_un, "centered", False, perm=p2)
    fitness_equal = bool(torch.equal(f_sharded, f_un))
    perm_equal = bool(torch.equal(p1, p2))
    for _ in range(gens - 1):
        sh.step()
        un.step()
    un.step()  # the single-process searcher only samples on its first step (gaussian.py:351-355); the sharded protocol updates on every step

    def rel(a, b):  # max-norm relative difference (element-wise ratios explode on the centre's near-zero components)
        return float((a - b).abs().max() / b.abs().max())

    out = torch.tensor([rel(sh.status["center"], un.status["center"]), rel(sh.status["stdev"], un.status["stdev"]),
                        0.0 if (fitness_equal and perm_equal) else 1.0], device=dev, dtype=torch.float64)
    dist.all_reduce(out, op=dist.ReduceOp.MAX)
    # every rank must also hold the SAME replicated distribution
    c = sh.status["center"].clone()
    c0 = c.clone()
    dist.broadcast(c0, src=0)
    same = torch.tensor([float(torch.equal(c, c0))], device=dev)
    dist.all_reduce(same, op=dist.ReduceOp.MIN)
    return {"workload": f"PGPE {n} x {d}, {gens} generations, seed {seed}: sharded over {world} ranks ({'peer exchange' if use_peer else 'NCCL'}) vs unsharded",
            "max_rel_diff_mu": float(out[0]), "max_rel_diff_sigma": float(out[1]), "first_generation_fitness_and_permutation_identical": bool(out[2] == 0.0),
            "replicated_state_identical_on_all_ranks": bool(same.item() == 1.0), "tolerance": 1e-5,
            "metric": "max |a - b| / max |b| over the vector",
            "ok": bool(out[0] < 1e-5 and out[1] < 1e-5 and out[2] == 0.0 and same.item() == 1.0)}


def other_config_legs(dev, peak_gbs: float) -> dict:
    """Short device-timed legs of the other single-GPU BASELINE configs (driver-timed with the headline line): cfg2 PGPE
    100k x 10k, cfg3 CMA-ES D = 1024 popsize 4096 (sphere), cfg4 batched MLP(376-256-17) forward over 65 536 policies."""
    import torch

    from evotorch_b200 import Problem, ops
    from evotorch_b200.algorithms import CMAES, PGPE
    from evotorch_b200.objectives import rastrigin, sphere

    out = {}

    def timed(fn, reps):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    try:  # ---- cfg2
        n, d = 100_000, 10_000
        s = PGPE(Problem("min", rastrigin, initial_bounds=(-5.12, 5.12), solution_length=d, device=dev, seed=SEED), popsize=n,
                 center_learning_rate=LR_MU, stdev_learning_rate=LR_SIGMA, stdev_init=STDEV_INIT)
        for _ in range(3):
            s.step()
        ops.enable_timers()
        ms = timed(s.step, 20)
        tm = ops.timer_results()
        ops.disable_timers()
        se_ms = tm["sample_eval"][1]
        out["cfg2_pgpe_100k_x_10k"] = {"generations_per_s": 1e3 / ms, "ms_per_step": ms, "steps": 20, "fused_kernel_ms": se_ms,
                                       "fused_kernel_gbs": 4.0 * n * d / se_ms / 1e6, "fused_kernel_frac_of_hbm_peak": 4.0 * n * d / se_ms / 1e6 / peak_gbs,
                                       "model_10ND_gbs": 10.0 * n * d / ms / 1e6}
        s.enable_cuda_graph()
        for _ in range(3):
            s.step()
        out["cfg2_pgpe_100k_x_10k"]["cuda_graph_generations_per_s"] = 1e3 / timed(s.step, 20)
        del s
        torch.cuda.empty_cache()
    except Exception as exc:
        out["cfg2_pgpe_100k_x_10k"] = {"error": repr(exc)[:300]}
    try:  # ---- cfg3
        d, n = 1024, 4096
        c = CMAES(Problem("min", sphere, initial_bounds=(-3, 3), solution_length=d, device=dev, seed=SEED), stdev_init=1.0, popsize=n)
        for _ in range(5):
            c.step()
        ms = timed(c.step, 20)
        flops = 2.0 * n * d * d * 2 + d**3 / 3.0
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
                tf32_peak = float(json.load(fh)["bf16_tflops"]) / 2.0
        except Exception:
            tf32_peak = 1100.0
        out["cfg3_cmaes_1024_x_4096"] = {"generations_per_s": 1e3 / ms, "ms_per_step": ms, "steps": 20, "useful_flop_per_generation": flops,
                                         "useful_tflops": flops / ms / 1e9, "tensor_flop_per_generation_3xtf32": 3 * 2.0 * n * d * d * 2,
                                         "frac_of_tf32_peak_3x": 3 * 2.0 * n * d * d * 2 / ms / 1e9 / tf32_peak, "tf32_peak_tflops": tf32_peak,
                                         "mean_eval": float(c.status["mean_eval"])}
        c.enable_cuda_graph()  # the same generation replayed from one CUDA graph (cuSOLVER Cholesky included)
        for _ in range(3):
            c.step()
        if c._graph is not None:
            ms_g = timed(c.step, 20)
            out["cfg3_cmaes_1024_x_4096"].update({"cuda_graph_generations_per_s": 1e3 / ms_g, "cuda_graph_ms_per_step": ms_g,
                                                  "cuda_graph_frac_of_tf32_peak_3x": 3 * 2.0 * n * d * d * 2 / ms_g / 1e9 / tf32_peak})
        del c
        torch.cuda.empty_cache()
    except Exception as exc:
        out["cfg3_cmaes_1024_x_4096"] = {"error": repr(exc)[:300]}
    try:  # ---- cfg4
        from evotorch_b200.neuroevolution import Policy

        net = torch.nn.Sequential(torch.nn.Linear(376, 256), torch.nn.Tanh(), torch.nn.Linear(256, 17))
        pol = Policy(net)
        NP = 65536
        P = torch.empty(NP, pol.parameter_length, device=dev).normal_(0, 0.1)
        obs = torch.randn(NP, 376, device=dev)
        pol.set_parameters(P)
        for _ in range(3):
            pol(obs)
        ms = timed(lambda: pol(obs), 10)
        gb = 4.0 * NP * pol.parameter_length / 1e9
        out["cfg4_mlp_376_256_17_x_65536"] = {"ms_per_forward": ms, "gbs": gb / ms * 1e3, "frac_of_hbm_peak": gb / ms * 1e3 / peak_gbs,
                                              "observations_per_policy": 1, "activation": "tanh", "params_per_policy": pol.parameter_length}
        # the same population on ONE shared minibatch of 256 observations (SupervisedNE, common_minibatch): the first layer of all
        # 65 536 networks is a single (16.8 M x 376) x (376 x 256) product on the tcgen05 GEMM (3xTF32, weights read once)
        try:
            Bm = 256
            xb = torch.randn(Bm, 376, device=dev)
            for _ in range(2):
                y = pol.forward_shared(P, xb)
            ms_b = timed(lambda: pol.forward_shared(P, xb), 5)
            useful = 2.0 * NP * Bm * (376 * 256 + 256 * 17)
            tensor = 3 * 2.0 * NP * Bm * 376 * 256
            try:
                with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
                    tf32_peak = float(json.load(fh)["bf16_tflops"]) / 2.0
            except Exception:
                tf32_peak = 1100.0
            out["cfg4_mlp_376_256_17_x_65536"]["shared_minibatch_B256"] = {
                "ms_per_forward": ms_b, "useful_tflops_fp32_equivalent": useful / ms_b / 1e9, "tensor_tflops_3xtf32": tensor / ms_b / 1e9,
                "frac_of_tf32_peak": tensor / ms_b / 1e9 / tf32_peak, "tf32_peak_tflops": tf32_peak, "parameter_gbs": gb / ms_b * 1e3,
                "observations_per_policy": Bm}
            del y, xb
        except Exception as exc:
            out["cfg4_mlp_376_256_17_x_65536"]["shared_minibatch_B256"] = {"error": repr(exc)[:300]}
        del P, obs, pol
        torch.cuda.empty_cache()
    except Exception as exc:
        out["cfg4_mlp_376_256_17_x_65536"] = {"error": repr(exc)[:300]}
    return out


def run_reference(args):
    """The reference arm: the reference's own CPU implementation of the path (its torch-CPU op sequence, restated in
    oracle/ref_cpu_path.py and checked bit-identical against the real reference in the build container), all host threads,
    same metric / config, SURVEY 8(d) protocol: populations of 10k / 30k / 100k rows at the full dimension, linearity check,
    extrapolation to the workload's population from the fitted line.  Rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    n_gpus = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    base = cpu_reference_run(args, sizes=cpu_sizes(args, (1e8, 3e8, 1e9)), budget_s=args.cpu_budget_s or 200.0, max_steps=max(1, min(args.steps, 5)),
                             with_gpu_eager=False)
    line = {
        "metric": metric_name(args), "value": base["value"], "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": 1e3 / base["value"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": dict(workload_config(args, n_gpus), name=args.config), "impl": "reference",
        "cpu_baseline": base,
        "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


_RESULT_FD = None


def claim_stdout():
    """stdout must carry exactly ONE JSON line, but libraries write there too (NCCL prints its version banner to stdout when
    the image sets NCCL_DEBUG): keep a private duplicate of the real stdout for the result and point fd 1 at stderr."""
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_RESULT_FD, data)


if __name__ == "__main__":
    a = parse_args()
    claim_stdout()
    try:
        if a.impl == "reference":
            run_reference(a)
        else:
            run_ours(a)
    except BaseException:
        import traceback

        traceback.print_exc()
        sys.stderr.flush()
        raise
