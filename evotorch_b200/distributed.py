"""Population sharding over the GPUs of one box with torch.distributed (NCCL over NVLink; gloo in the CPU tests).

This replaces the reference's Ray-actor path (`Problem.sample_and_compute_gradients`, core.py:2762-3073 and
`GaussianSearchAlgorithm._step_distributed`, algorithms/distributed/gaussian.py:199-272).  One process per GPU
(launched with torchrun).  Per generation each rank

  1. samples and evaluates its own contiguous row shard (K1+K2).  The Philox counter of a draw is a function of the
     GLOBAL row index, so the population is identical for every world size;
  2. all-gathers the local fitness slice -> the full fitness vector (N floats: 4 MB at N = 1 M);
  3. ranks the full vector (K3, replicated) and keeps its slice of the utilities;
  4. reduces its partial gradients over its rows (K4) and all-reduces the stacked (mu, sigma) partials (2*D floats);
  5. applies the (replicated) update (K5).

Unlike the reference (which ranks *locally* per actor and averages the per-actor gradients), ranking is global, so an
R-GPU run reproduces the single-GPU run at the same population size up to fp32 summation order.
"""

from __future__ import annotations

import os
from typing import Optional

import torch
import torch.distributed as dist

from .tools.misc import split_workload
from .tools.ranking import rank


def world() -> tuple:
    """(rank, world_size) of the default process group; (0, 1) when torch.distributed is not initialised."""
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def shard_rows(popsize: int, world_size: int, rank_: int, symmetric: bool) -> tuple:
    """Contiguous row range [row0, row0 + n) of this rank; antithetic pairs are never split."""
    unit = 2 if symmetric else 1
    if popsize % unit != 0:
        raise ValueError(f"popsize ({popsize}) must be even for a symmetric distribution")
    shares = split_workload(popsize // unit, world_size)
    row0 = unit * sum(shares[:rank_])
    return row0, unit * shares[rank_], [unit * s for s in shares]


def all_gather_rows(local: torch.Tensor, counts: list) -> torch.Tensor:
    """Concatenate the 1-D `local` tensors of all ranks (possibly of different lengths `counts`) in rank order."""
    rank_, ws = world()
    if ws == 1:
        return local
    if len(set(counts)) == 1:
        out = torch.empty(sum(counts), dtype=local.dtype, device=local.device)
        dist.all_gather_into_tensor(out, local.contiguous())
        return out
    width = max(counts)
    padded = torch.zeros(width, dtype=local.dtype, device=local.device)
    padded[: local.numel()] = local
    gathered = torch.empty(ws * width, dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(gathered, padded)
    return torch.cat([gathered[r * width: r * width + counts[r]] for r in range(ws)])


def broadcast_seed(problem) -> None:
    """Make every rank draw from the same Philox key (rank 0's) -- required for the population to be rank-count invariant.
    With `rng="torch"` (CPU problems, non-fp32 dtypes) the noise comes from each rank's own torch generator, whose stream
    cannot be indexed by global row: the generators are then re-seeded with a per-rank offset of rank 0's seed, so that the
    shards hold DIFFERENT samples (the same seed on every rank would make the global population `world_size` duplicated
    blocks); the trajectory is then reproducible for a given world size, not across world sizes."""
    rank_, ws = world()
    if ws == 1 or getattr(problem, "_seed_synced", False):
        return
    t = torch.tensor([problem._philox_seed & 0x7FFFFFFFFFFFFFFF, problem._philox_stream], dtype=torch.int64, device=problem.device)
    dist.broadcast(t, src=0)
    problem._philox_seed, problem._philox_stream = int(t[0].item()), int(t[1].item())
    if problem.rng == "torch":
        problem.generator.manual_seed((problem._philox_seed + 0x9E3779B97F4A7C15 * (rank_ + 1)) & 0x7FFFFFFFFFFFFFFF)
    problem._seed_synced = True


def broadcast_search_state(tensors: list) -> None:
    """Replicated-update invariant: every rank must start from rank 0's distribution and optimizer state.  With
    `center_init=None` each rank draws its own centre (and with `seed=None` its own seed), so the searchers call this once
    before their first sharded generation (in place, src = rank 0)."""
    rank_, ws = world()
    if ws == 1:
        return
    for t in tensors:
        if isinstance(t, torch.Tensor) and t.numel() > 0:
            if t.is_contiguous():
                dist.broadcast(t, src=0)
            else:
                c = t.contiguous()
                dist.broadcast(c, src=0)
                t.copy_(c)


def _results_to_home(problem, grads: dict, mean_eval: torch.Tensor, home_device: torch.device) -> tuple:
    """Gradients and mean fitness on the distribution's device.  Device -> host goes through ONE packed copy into a pinned
    staging buffer and one stream synchronisation (instead of a blocking copy per tensor)."""
    if home_device == problem.device:
        return grads, mean_eval
    if home_device.type != "cpu" or problem.device.type != "cuda":
        return {k: v.to(home_device) for k, v in grads.items()}, mean_eval.to(home_device)
    keys = sorted(grads)
    sizes = [grads[k].numel() for k in keys]
    total = sum(sizes) + 1
    stage = problem.__dict__.get("_d2h_stage")
    if stage is None or stage[0].numel() != total:
        stage = problem.__dict__["_d2h_stage"] = (torch.empty(total, dtype=torch.float32).pin_memory(),
                                                  torch.empty(total, dtype=torch.float32, device=problem.device))
    host, dev = stage
    off = 0
    for k, n in zip(keys, sizes):
        dev[off:off + n].copy_(grads[k].reshape(-1))
        off += n
    dev[off:off + 1].copy_(mean_eval.reshape(1))
    host.copy_(dev, non_blocking=True)
    torch.cuda.current_stream(problem.device).synchronize()
    out, off = {}, 0
    for k, n in zip(keys, sizes):
        out[k] = host[off:off + n].clone().reshape(grads[k].shape)
        off += n
    return out, host[off].clone()


def _usable_peer_exchange(problem, dev_dist, popsize: int, ws: int):
    """The PeerExchange attached to `problem` (peer.enable_peer_exchange) if this generation can run on it."""
    peer = getattr(problem, "_peer_exchange", None)
    if peer is None or ws == 1:
        return None
    from . import ops

    ok = (peer.popsize == popsize and peer.world == ws and problem.evok_objective_id is not None and problem.rng == "philox"
          and len(problem.senses) == 1 and problem.eval_data_length == 0 and hasattr(dev_dist, "partial_gradients")
          and hasattr(dev_dist, "SYMMETRIC") and ops.uses_kernels(dev_dist.mu) and len(problem.before_eval_hook) == 0)
    if not ok:
        raise ValueError("the attached PeerExchange does not fit this generation (needs: same popsize and world size, a built-in "
                         "objective, rng='philox', one objective, a separable Gaussian on CUDA float32, no before_eval_hook)")
    return peer


def sharded_sample_and_gradients(problem, distribution, popsize: int, *, obj_index: int, ranking_method: Optional[str]) -> dict:
    """One sample -> evaluate -> (global) rank -> gradient pass over this rank's row shard; see the module docstring.
    Returns {"gradients", "num_solutions", "mean_eval"} like the reference's `_sample_and_compute_gradients`
    (core.py:3156-3301), with gradients on `distribution.device`."""
    from .core import LazySolutionBatch, SolutionBatch

    rank_, ws = world()
    home_device = distribution.device
    dev_dist = distribution.to(problem.device)
    symmetric = bool(getattr(dev_dist, "SYMMETRIC", False))
    if ws > 1 and not hasattr(dev_dist, "partial_gradients"):
        raise NotImplementedError(f"{type(dev_dist).__name__} cannot be sharded over ranks (full-covariance search is a small-D method)")
    row0, n_local, counts = shard_rows(popsize, ws, rank_, symmetric)
    broadcast_seed(problem)

    peer = _usable_peer_exchange(problem, dev_dist, popsize, ws)
    cache = problem.__dict__.setdefault("_grad_batches", {})
    batch = cache.get(n_local)
    if batch is None:
        if problem.lazy_population:
            batch = cache[n_local] = LazySolutionBatch(problem, n_local, device=problem.device)
        else:
            batch = cache[n_local] = SolutionBatch(problem, n_local, device=problem.device, empty=True)
        if peer is not None:  # the shard's fitness column IS its slice of the exchange buffer
            batch._evdata = peer.f_all[row0:row0 + n_local].view(n_local, 1)
    sense = problem.senses[obj_index]
    method = "raw" if ranking_method is None else ranking_method
    # sharded ranking: sort locally, exchange sorted keys, rank the local rows against the world (no GPU holds all fitnesses)
    sharded_rank = (peer is not None and method in ("centered", "linear", "nes") and dev_dist.accepts_local_weights(method)
                    and os.environ.get("EVOTORCH_B200_SHARDED_RANK", "0") == "1")  # opt-in: measured equal to the replicated sort at 8 GPUs
    problem.philox_row0 = row0
    try:
        problem.sample_and_evaluate(dev_dist, batch)
    finally:
        problem.philox_row0 = 0

    samples = batch.recipe if isinstance(batch, LazySolutionBatch) else batch.access_values(keep_evals=True)
    if sharded_rank:
        offsets = [0]
        for c in counts:
            offsets.append(offsets[-1] + c)
        scratch = problem.__dict__.setdefault("_grad_scratch", {})
        w_local = scratch.get(n_local)
        if w_local is None:
            w_local = scratch[n_local] = torch.empty(n_local, dtype=torch.float32, device=problem.device)
        w_local, mean_buf = peer.rank_sharded(batch._evdata.view(-1), method, sense == "max", offsets, w_local)
        dev_dist._peer = peer
        try:
            summed = dev_dist.partial_gradients(samples, w_local, row0, method, local_weights_of=popsize)  # already summed over the ranks
        finally:
            dev_dist._peer = None
        grads = dev_dist.finalize_gradients(summed, popsize)
        mean_eval = mean_buf.reshape(())  # live 1-element buffer: holds the latest generation's global mean fitness
        grads, mean_eval = _results_to_home(problem, grads, mean_eval, home_device)
        return {"gradients": grads, "num_solutions": popsize, "mean_eval": mean_eval}
    if peer is not None:
        # the fitness all-gather: the sampler wrote this rank's slice of f_all locally; one push kernel copies it to every peer
        # (coalesced 16-byte stores, one system fence per peer)
        peer.push_fitness(row0, n_local)
        f_all = peer.wait_fitness()
    else:
        f_local = batch.access_evals(obj_index)
        f_all = all_gather_rows(f_local.to(dev_dist.dtype), counts)
    weights_all = rank(f_all, method, higher_is_better=(sense == "max"))

    if peer is not None:
        dev_dist._peer = peer
        try:
            summed = dev_dist.partial_gradients(samples, weights_all, row0, method)  # already summed over the ranks
        finally:
            dev_dist._peer = None
        grads = dev_dist.finalize_gradients(summed, popsize)
    elif hasattr(dev_dist, "partial_gradients"):
        partial = dev_dist.partial_gradients(samples, weights_all, row0, method)
        if ws > 1:
            keys = sorted(partial)
            stacked = torch.stack([partial[k] for k in keys])
            dist.all_reduce(stacked, op=dist.ReduceOp.SUM)
            partial = {k: stacked[i] for i, k in enumerate(keys)}
        grads = dev_dist.finalize_gradients(partial, popsize)
    else:
        grads = dev_dist._compute_gradients(samples, weights_all, method)

    mean_eval = torch.mean(f_all)  # 0-dim tensor: converting it to float is the caller's (lazy) choice, no forced sync here
    grads, mean_eval = _results_to_home(problem, grads, mean_eval, home_device)
    return {"gradients": grads, "num_solutions": popsize, "mean_eval": mean_eval}


def adaptive_sample_and_gradients(problem, distribution, popsize: int, *, num_interactions: int, popsize_max: Optional[int], obj_index: int,
                                  ranking_method: Optional[str]) -> dict:
    """`_sample_and_compute_gradients` with an interaction-count threshold (core.py:3239-3282): batches of `popsize`
    solutions are sampled and evaluated until this process has made more than `num_interactions` simulator interactions (or
    holds `popsize_max` solutions); the gradients are computed over their concatenation (same kernels, K3 + K4, as the
    fixed-size path).  The number of solutions then differs from rank to rank and from generation to generation, which the
    global-ranking protocol of `sharded_sample_and_gradients` cannot shard: single-process only."""
    from .core import SolutionBatch

    if world()[1] > 1:
        raise NotImplementedError("adaptive population size (num_interactions) is not available with a population sharded over ranks: "
                                  "the global ranking needs a fixed, common population size")
    home_device = distribution.device
    dev_dist = distribution.to(problem.device)
    first = problem._get_local_interaction_count()
    batches, total = [], 0
    while True:
        batch = SolutionBatch(problem, popsize, device=problem.device, empty=True)
        problem.sample_and_evaluate(dev_dist, batch)
        batches.append(batch)
        total += popsize
        if problem._get_local_interaction_count() - first > num_interactions:
            break
        if popsize_max is not None and total >= popsize_max:
            break
    merged = batches[0] if len(batches) == 1 else SolutionBatch.cat(batches)
    grads = dev_dist.compute_gradients(merged.access_values(keep_evals=True), merged.access_evals(obj_index),
                                       objective_sense=problem.senses[obj_index], ranking_method=ranking_method)
    mean_eval = torch.mean(merged.access_evals(obj_index))
    if home_device != problem.device:
        grads = {k: v.to(home_device) for k, v in grads.items()}
        mean_eval = mean_eval.to(home_device)
    return {"gradients": grads, "num_solutions": len(merged), "mean_eval": mean_eval}
