"""Problem / SolutionBatch / Solution: the data model at the boundary of the hot path.

Mirrors the part of evotorch.core the distribution-based searchers touch (core.py:365-3411 `Problem`,
:3590-4601 `SolutionBatch`, :4742-5107 `Solution`).  A SolutionBatch is two ordinary torch tensors -- decision
values (N x D, row-major, `problem.dtype`) and evaluations (N x (objectives + eval_data_length), NaN = not
evaluated) -- which the kernels read and write in place.

Not carried over (out of scope, SURVEY.md section 8): Ray actors (`num_actors`), object-dtype problems,
multi-objective pareto utilities.  Population sharding across GPUs is done with torch.distributed instead of Ray
(see evotorch_b200/distributed.py).
"""

from __future__ import annotations

import math
from typing import Any, Callable, Iterable, Optional, Union

import torch

from . import ops
from .tools.cloning import Clonable
from .tools.hook import Hook
from .tools.readonlytensor import as_read_only_tensor
from .tools.misc import ensure_tensor_length_and_dtype, extract_generator, make_gaussian, make_uniform, to_torch_dtype

ObjectiveSense = Union[str, Iterable[str]]


class Problem(Clonable):
    """Definition of an optimisation problem (core.py:365).  `objective_func` receives either one solution (1-D tensor)
    or, with `vectorized=True` / an `@vectorized`-marked function, the whole N x D population.  Built-in objectives from
    `evotorch_b200.objectives` additionally carry an `evok_objective_id`, which lets the searchers fuse evaluation into the
    sampling kernel."""

    def __init__(self, objective_sense: ObjectiveSense, objective_func: Optional[Callable] = None, *, initial_bounds=None, bounds=None,
                 solution_length: Optional[int] = None, dtype=None, eval_dtype=None, device=None, eval_data_length: Optional[int] = None,
                 seed: Optional[int] = None, num_actors=None, actor_config=None, num_gpus_per_actor=None, num_subbatches=None,
                 subbatch_size=None, store_solution_stats: Optional[bool] = None, vectorized: Optional[bool] = None,
                 rng: Optional[str] = None, lazy_population: bool = False):
        if num_actors not in (None, 0, 1):
            # Drop-in behaviour for scripts written against the reference (e.g. its quick-start, tests/test_examples.py:29-78):
            # the request is accepted and mapped onto what replaces Ray here -- the ranks of torch.distributed when the script was
            # launched with torchrun (searchers built with distributed=True then shard the population over them), else this one
            # process, which evaluates the whole population with the vectorised / fused kernels.
            import warnings

            warnings.warn(
                f"num_actors={num_actors!r}: evotorch_b200 has no Ray actors. The population is evaluated by this process"
                " (or sharded over the torch.distributed ranks when launched with torchrun and distributed=True is given to the"
                " searcher; see evotorch_b200.distributed).", stacklevel=2)
        self._requested_num_actors = num_actors
        self._dtype = torch.float32 if dtype is None else to_torch_dtype(dtype)
        if eval_dtype is None:
            self._eval_dtype = self._dtype if self._dtype.is_floating_point else torch.float32
        else:
            self._eval_dtype = to_torch_dtype(eval_dtype)
        self._device = torch.device("cpu") if device is None else torch.device(device)
        if solution_length is None:
            raise ValueError(f"Together with a numeric dtype ({self._dtype!r}), expected to receive `solution_length` as an integer."
                             " However, `solution_length` is None.")
        self._solution_length = int(solution_length)

        if isinstance(objective_sense, str):
            senses = [objective_sense]
        else:
            senses = list(objective_sense)
            if len(senses) == 0:
                raise ValueError("Encountered an empty sequence via `objective_sense`.")
        for s in senses:
            if s not in ("min", "max"):
                raise ValueError(f"Invalid objective sense: {s!r}. Instead, please provide the objective sense as 'min' or 'max'.")
        self._senses = senses
        self._objective_sense = objective_sense

        self._initial_lower_bounds = self._initial_upper_bounds = None
        self._lower_bounds = self._upper_bounds = None
        if bounds is not None and initial_bounds is None:
            initial_bounds = bounds
        if initial_bounds is not None:
            self._initial_lower_bounds, self._initial_upper_bounds = self._process_bounds(initial_bounds)
        if bounds is not None:
            self._lower_bounds, self._upper_bounds = self._process_bounds(bounds)

        self._objective_func = objective_func
        if objective_func is None:
            if vectorized is not None:
                raise ValueError("This problem object received no external fitness function; `vectorized` must be left as None.")
            self._vectorized = None
        elif getattr(objective_func, "__evotorch_vectorized__", False):
            if vectorized is not None:
                raise ValueError("Received a fitness function that was decorated via @vectorized; `vectorized` must be left as None.")
            self._vectorized = True
        else:
            self._vectorized = bool(vectorized)

        self._eval_data_length = 0 if eval_data_length is None else int(eval_data_length)
        self._store_solution_stats = None if store_solution_stats is None else bool(store_solution_stats)
        self._best = self._worst = None
        self._best_evals = self._worst_evals = None
        self._after_eval_status: dict = {}
        self._before_eval_hook, self._after_eval_hook = Hook(), Hook()

        # RNG: a torch.Generator (used by generate_values and by the rng="torch" sampler) plus a Philox key for the kernels
        self._generator = torch.Generator(device=self._device)
        self._seed = None
        self.manual_seed(seed)
        if rng is None:
            rng = "philox" if self._device.type == "cuda" and self._dtype == torch.float32 else "torch"
        if rng not in ("philox", "torch"):
            raise ValueError(f"rng must be 'philox' or 'torch', got {rng!r}")
        self.rng = rng
        # "lazy population": never materialise the N x D matrix.  The fused kernel evaluates the samples straight from the
        # Philox counters and the gradient kernel regenerates them, so a generation needs O(N + D) memory (BASELINE config 5,
        # 1 M x 100 k = 400 GB of samples, then runs on a single GPU).  Only for built-in objectives + the Philox sampler.
        self.lazy_population = bool(lazy_population)

    # ------------------------------------------------------------------ construction helpers
    def _process_bounds(self, pair) -> tuple:
        lb, ub = pair
        out = []
        for b in (lb, ub):
            t = torch.as_tensor(b, dtype=self._dtype, device=self._device)
            if t.ndim not in (0, 1):
                raise ValueError(f"Lower and upper bounds are expected as scalars or as 1-dimensional vectors, got shape {tuple(t.shape)}.")
            if t.ndim == 1 and len(t) != self._solution_length:
                raise ValueError(f"Boundary vectors must have length {self._solution_length}, got {len(t)}.")
            out.append(t)
        return tuple(out)

    def manual_seed(self, seed: Optional[int] = None):
        """Seed the torch generator and the Philox key (core.py:1616)."""
        if seed is None:
            seed = int(torch.randint(0, 2**62, (1,)).item())
            self._seed = None
        else:
            self._seed = int(seed)
        self._generator.manual_seed(int(seed))
        self._philox_seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        self._philox_stream = 0
        self.philox_row0 = 0  # global index of the first local row when the population is sharded over ranks
        self.philox_stream_offset = None  # optional device-side generation counter (set while a CUDA graph is captured / replayed)

    def next_philox_stream(self) -> tuple:
        """(seed, stream_id) for the next kernel-sampled population; every call uses a fresh Philox stream."""
        sid = self._philox_stream
        self._philox_stream += 1
        return self._philox_seed, sid

    # ------------------------------------------------------------------ properties
    @property
    def dtype(self) -> torch.dtype:
        return self._dtype

    @property
    def eval_dtype(self) -> torch.dtype:
        return self._eval_dtype

    @property
    def device(self) -> torch.device:
        return self._device

    @property
    def generator(self) -> torch.Generator:
        return self._generator

    @property
    def has_own_generator(self) -> bool:
        return True

    @property
    def objective_sense(self) -> ObjectiveSense:
        return self._senses[0] if len(self._senses) == 1 else self._senses

    @property
    def senses(self) -> list:
        return self._senses

    @property
    def is_single_objective(self) -> bool:
        return len(self._senses) == 1

    @property
    def is_multi_objective(self) -> bool:
        return len(self._senses) > 1

    @property
    def solution_length(self) -> int:
        return self._solution_length

    @property
    def eval_data_length(self) -> int:
        return self._eval_data_length

    @property
    def initial_lower_bounds(self):
        return self._initial_lower_bounds

    @property
    def initial_upper_bounds(self):
        return self._initial_upper_bounds

    @property
    def lower_bounds(self):
        return self._lower_bounds

    @property
    def upper_bounds(self):
        return self._upper_bounds

    @property
    def num_actors(self) -> int:
        return 0

    @property
    def actors(self):
        return None

    @property
    def is_main(self) -> bool:
        return True

    @property
    def is_remote(self) -> bool:
        return False

    @property
    def before_eval_hook(self) -> Hook:
        return self._before_eval_hook

    @property
    def after_eval_hook(self) -> Hook:
        return self._after_eval_hook

    @property
    def before_grad_hook(self) -> Hook:
        """Called (no arguments) at the start of `sample_and_compute_gradients` (core.py:2204, :2889)."""
        return self.__dict__.setdefault("_before_grad_hook", Hook())

    @property
    def after_grad_hook(self) -> Hook:
        """Called with the list of result dictionaries of `sample_and_compute_gradients`; dictionaries it returns are
        merged into the problem's status (core.py:2212, :3070)."""
        return self.__dict__.setdefault("_after_grad_hook", Hook())

    def is_on_cpu(self) -> bool:
        return str(self._device) == "cpu"

    def kill_actors(self):
        """No-op: there are no Ray actors here (one process per GPU replaces them, distributed.py)."""

    @property
    def all_remote_problems(self):
        raise NotImplementedError("Ray actors are out of scope: shard the population over GPUs with torchrun (evotorch_b200/distributed.py)")

    @property
    def status(self) -> dict:
        return self._after_eval_status

    @property
    def stores_solution_stats(self) -> Optional[bool]:
        return self._store_solution_stats

    @property
    def evok_objective_id(self) -> Optional[int]:
        """Id of the fused evaluation kernel if the objective is one of evotorch_b200.objectives, else None."""
        return getattr(self._objective_func, "evok_objective_id", None)

    # ------------------------------------------------------------------ tensor makers (TensorMakerMixin subset)
    def _tm(self, dtype, device, use_eval_dtype=False):
        if dtype is None:
            dtype = self._eval_dtype if use_eval_dtype else self._dtype
        return to_torch_dtype(dtype), (self._device if device is None else torch.device(device))

    def _size(self, size, num_solutions):
        if num_solutions is not None:
            if len(size) > 0:
                raise ValueError("Provide either a size or `num_solutions`, not both.")
            return (int(num_solutions), self._solution_length)
        if len(size) == 1 and isinstance(size[0], (tuple, list, torch.Size)):
            return tuple(size[0])
        return tuple(int(s) for s in size)

    def make_tensor(self, data, *, dtype=None, device=None, use_eval_dtype: bool = False) -> torch.Tensor:
        dt, dev = self._tm(dtype, device, use_eval_dtype)
        return torch.as_tensor(data, dtype=dt, device=dev) if isinstance(data, torch.Tensor) else torch.tensor(data, dtype=dt, device=dev)

    def _target(self, size, num_solutions, out, dtype, device, use_eval_dtype) -> torch.Tensor:
        """The tensor a maker fills: `out` if given (then no size / dtype / device may be given), else a new one
        (tools/tensormaker.py:60-140)."""
        if out is not None:
            if len(size) > 0 or num_solutions is not None or dtype is not None or device is not None or use_eval_dtype:
                raise ValueError("When `out` is given, the arguments `size`, `num_solutions`, `dtype`, `device`, `use_eval_dtype` are not expected")
            return out
        dt, dev = self._tm(dtype, device, use_eval_dtype)
        return torch.empty(self._size(size, num_solutions), dtype=dt, device=dev)

    def make_empty(self, *size, num_solutions=None, out=None, dtype=None, device=None, use_eval_dtype: bool = False) -> torch.Tensor:
        return self._target(size, num_solutions, out, dtype, device, use_eval_dtype)

    def make_zeros(self, *size, num_solutions=None, out=None, dtype=None, device=None, use_eval_dtype: bool = False) -> torch.Tensor:
        return self._target(size, num_solutions, out, dtype, device, use_eval_dtype).zero_()

    def make_ones(self, *size, num_solutions=None, out=None, dtype=None, device=None, use_eval_dtype: bool = False) -> torch.Tensor:
        return self._target(size, num_solutions, out, dtype, device, use_eval_dtype).fill_(1)

    def make_nan(self, *size, num_solutions=None, out=None, dtype=None, device=None, use_eval_dtype: bool = False) -> torch.Tensor:
        return self._target(size, num_solutions, out, dtype, device, use_eval_dtype).fill_(float("nan"))

    def make_I(self, size=None, *, out=None, dtype=None, device=None, use_eval_dtype: bool = False) -> torch.Tensor:
        """Identity matrix: n x n with n = `size` (an int or a 1-tuple), the solution length by default, or filled into `out`
        (tools/tensormaker.py:427-508)."""
        if isinstance(size, tuple):
            if len(size) != 1:
                raise ValueError(f"When the size argument is given as a tuple, the method `make_I(...)` expects the tuple to have only one"
                                 f" element. The given tuple is {size}.")
            size = size[0]
        if out is not None:
            if size is not None or dtype is not None or device is not None or use_eval_dtype:
                raise ValueError("When `out` is given, the arguments `size`, `dtype`, `device`, `use_eval_dtype` are not expected")
            if out.ndim != 2 or out.shape[0] != out.shape[1]:
                raise ValueError(f"`out` was expected as a square matrix, but its shape is {tuple(out.shape)}")
            out.zero_()
            out.fill_diagonal_(1)
            return out
        dt, dev = self._tm(dtype, device, use_eval_dtype)
        return torch.eye(self._solution_length if size is None else int(size), dtype=dt, device=dev)

    def make_gaussian(self, *size, num_solutions=None, center=None, stdev=None, symmetric: bool = False, out=None, dtype=None,
                      device=None, use_eval_dtype: bool = False, generator=None) -> torch.Tensor:
        out = self._target(size, num_solutions, out, dtype, device, use_eval_dtype)
        return make_gaussian(out=out, center=center, stdev=stdev, symmetric=symmetric,
                             generator=self._generator if generator is None else generator)

    def make_uniform(self, *size, num_solutions=None, lb=None, ub=None, out=None, dtype=None, device=None, use_eval_dtype: bool = False,
                     generator=None) -> torch.Tensor:
        out = self._target(size, num_solutions, out, dtype, device, use_eval_dtype)
        return make_uniform(out=out, lb=lb, ub=ub, generator=self._generator if generator is None else generator)

    def make_randint(self, *size, n, num_solutions=None, out=None, dtype=None, device=None, use_eval_dtype: bool = False,
                     generator=None) -> torch.Tensor:
        """Uniform random integers in [0, n-1], as integers or as floats (tools/tensormaker.py:681-749)."""
        out = self._target(size, num_solutions, out, dtype, device, use_eval_dtype)
        gen = extract_generator(self._generator if generator is None else generator)
        n = int(n)
        if out.dtype.is_floating_point:
            out.copy_(torch.randint(0, n, out.shape, generator=gen, device=out.device, dtype=torch.int64))
        else:
            out.random_(0, n, generator=gen)
        return out

    def make_uniform_shaped_like(self, t: torch.Tensor, *, lb=None, ub=None) -> torch.Tensor:
        return self.make_uniform(out=torch.empty_like(t), lb=lb, ub=ub)

    def make_gaussian_shaped_like(self, t: torch.Tensor, *, center=None, stdev=None) -> torch.Tensor:
        return self.make_gaussian(out=torch.empty_like(t), center=center, stdev=stdev)

    def ensure_tensor_length_and_dtype(self, t: Any, *, allow_scalar: bool = False, about: Optional[str] = None) -> torch.Tensor:
        return ensure_tensor_length_and_dtype(t, self._solution_length, self._dtype, about=about, allow_scalar=allow_scalar,
                                              device=self._device)

    # ------------------------------------------------------------------ generation
    def generate_values(self, num_solutions: int) -> torch.Tensor:
        """Uniform samples within the initial bounds (core.py:1840-1909)."""
        result = torch.empty(int(num_solutions), self._solution_length, dtype=self._dtype, device=self._device)
        self._fill(result)
        return result

    def _fill(self, values: torch.Tensor):
        if self._initial_lower_bounds is None or self._initial_upper_bounds is None:
            raise RuntimeError(
                "The default implementation of the method `_fill(...)` does not know how to initialize solutions because it appears"
                " that this Problem object was not given neither `initial_bounds` nor `bounds` during the moment of initialization."
            )
        return self.make_uniform(out=values, lb=self._initial_lower_bounds, ub=self._initial_upper_bounds)

    def generate_batch(self, popsize: Optional[int] = None, *, empty: bool = False, center=None, stdev=None,
                       symmetric: bool = False) -> "SolutionBatch":
        if (center is None) != (stdev is None):
            raise ValueError("The arguments `center` and `stdev` were expected to be None or non-None at the same time.")
        if center is None:
            if symmetric:
                raise ValueError("The argument `symmetric` can be set as True only when `center` and `stdev` are provided.")
            return SolutionBatch(self, popsize, empty=empty, device=self._device)
        if empty:
            raise ValueError("When `center` and `stdev` are provided, the argument `empty` must be False.")
        result = SolutionBatch(self, popsize, device=self._device, empty=True)
        self.make_gaussian(out=result.access_values(), center=center, stdev=stdev, symmetric=symmetric)
        return result

    # ------------------------------------------------------------------ checks
    def ensure_numeric(self):
        if not (self._dtype.is_floating_point or self._dtype in (torch.int32, torch.int64, torch.int16, torch.int8)):
            raise ValueError("Expected a problem with numeric dtype.")

    def ensure_unbounded(self):
        if self._lower_bounds is not None or self._upper_bounds is not None:
            raise ValueError("Expected an unbounded problem. However, this problem object has its `lower_bounds` and/or `upper_bounds` set.")

    def ensure_single_objective(self):
        if len(self._senses) != 1:
            raise ValueError(f"Expected a single-objective problem, but this problem has {len(self._senses)} objectives.")

    def normalize_obj_index(self, obj_index: Optional[int] = None) -> int:
        """None -> 0 for single-objective problems; negative indices wrap (core.py:2672)."""
        n = len(self._senses)
        if obj_index is None:
            if n == 1:
                return 0
            raise ValueError("This problem has multiple objectives: `obj_index` must be given.")
        obj_index = int(obj_index)
        if not (-n <= obj_index < n):
            raise IndexError(f"Objective index out of range: {obj_index}")
        return obj_index % n

    # ------------------------------------------------------------------ evaluation
    @torch.no_grad()
    def evaluate(self, x: Union["SolutionBatch", "Solution"]):
        """Evaluate a batch in place (core.py:2532-2571): hooks, `_evaluate_batch`, best/worst bookkeeping."""
        if isinstance(x, Solution):
            batch = x.to_batch()
        elif isinstance(x, SolutionBatch):
            batch = x
        else:
            raise TypeError(f"The method `evaluate(...)` expected a Solution or a SolutionBatch as its argument, got {type(x)!r}.")
        self._before_eval_hook(batch)
        self._evaluate_all(batch)
        self._finish_evaluation(batch)

    @property
    def aux_device(self) -> torch.device:
        """Where `@on_aux_device` fitness functions run: the first visible GPU for a host-resident problem (if there is a GPU),
        else the problem's own device (core.py:1657-1692)."""
        if self._device.type == "cpu":
            return torch.device("cuda") if torch.cuda.is_available() else self._device
        return self._device

    def _device_of_fitness_function(self) -> Optional[torch.device]:
        """The device requested by `@on_device` / `@on_cuda` / `@on_aux_device` (or a plain `.device` attribute) on the objective
        function or on an overridden `_evaluate_batch` / `_evaluate`; None if there is no such request (core.py:2502-2530)."""
        for fn in (self._objective_func, self._evaluate_batch, self._evaluate):
            if fn is None:
                continue
            if getattr(fn, "__evotorch_on_aux_device__", False):
                return self.aux_device
            if hasattr(fn, "device"):
                return torch.device(fn.device)
        return None

    def _evaluate_all(self, batch: "SolutionBatch"):
        """Evaluate on the device the fitness function asks for: the batch is moved there, evaluated, and the results are
        copied back (core.py:2573-2585)."""
        wanted = self._device_of_fitness_function()
        if wanted is None or torch.device(wanted) == batch.device:
            self._evaluate_batch(batch)
            return
        moved = batch.to(wanted)
        self._evaluate_batch(moved)
        batch._evdata[:] = moved._evdata.to(batch.device)

    def _finish_evaluation(self, batch: "SolutionBatch"):
        self._after_eval_status = {}
        self._after_eval_status.update(self._get_best_and_worst(batch))
        self._after_eval_status.update(self._extra_status(batch))
        self._after_eval_status.update(self._after_eval_hook.accumulate_dict(batch))

    def _extra_status(self, batch: "SolutionBatch") -> dict:
        """Override point: problem-specific status items (core.py `_extra_status`)."""
        return {}

    def _evaluate_batch(self, batch: "SolutionBatch"):
        """Override point (core.py:2602-2611).  Built-in objectives run the K2 row-reduction kernel."""
        if self._vectorized and self._objective_func is not None:
            result = self._objective_func(batch.values)
            if isinstance(result, tuple):
                batch.set_evals(*result)
            else:
                batch.set_evals(result)
        else:
            for sln in batch:
                self._evaluate(sln)

    def _evaluate(self, solution: "Solution"):
        if self._objective_func is None:
            raise NotImplementedError
        result = self._objective_func(solution.values)
        if isinstance(result, tuple):
            solution.set_evals(*result)
        else:
            solution.set_evals(result)

    def _get_best_and_worst(self, batch: "SolutionBatch") -> dict:
        """Track best/worst solutions; on by default only for CPU batches, like the reference (core.py:2335-2400)."""
        if self._store_solution_stats is None:
            self._store_solution_stats = str(batch.device) == "cpu"
        if not self._store_solution_stats:
            return {}
        nobjs = len(self._senses)
        if self._best is None:
            self._best, self._worst = [None] * nobjs, [None] * nobjs
            self._best_evals = [math.inf if s == "min" else -math.inf for s in self._senses]
            self._worst_evals = [-math.inf if s == "min" else math.inf for s in self._senses]
        for i, sense in enumerate(self._senses):
            scores = batch.access_evals(i)
            ibest, iworst = batch.argbest(i), batch.argworst(i)
            best_score, worst_score = float(scores[ibest]), float(scores[iworst])
            better = best_score < self._best_evals[i] if sense == "min" else best_score > self._best_evals[i]
            worse = worst_score > self._worst_evals[i] if sense == "min" else worst_score < self._worst_evals[i]
            if better:
                self._best_evals[i], self._best[i] = best_score, batch[int(ibest)].clone()
            if worse:
                self._worst_evals[i], self._worst[i] = worst_score, batch[int(iworst)].clone()
        if nobjs == 1:
            return dict(best=self._best[0], worst=self._worst[0], best_eval=float(self._best[0].evals[0]),
                        worst_eval=float(self._worst[0].evals[0]))
        return {"best": self._best, "worst": self._worst}

    # ------------------------------------------------------------------ pickling (core.py:2711-2734)
    _TRANSIENT = ("_peer_exchange", "_grad_batches", "_grad_scratch", "_d2h_stage")

    def __getstate__(self) -> dict:
        """Device-mapped and cached objects (peer-exchange buffers, gradient batches, the CUDA-graph generation counter) are
        not part of a pickled problem; the Philox key and the host-side generation counter are, so an unpickled problem
        continues the same random stream."""
        state = {k: v for k, v in self.__dict__.items() if k not in self._TRANSIENT}
        state["philox_stream_offset"] = None
        return state

    # ------------------------------------------------------------------ fused sample + evaluate, gradient service
    def sample_and_evaluate(self, distribution, batch: "SolutionBatch"):
        """Fill `batch` with samples of `distribution` and evaluate it.  With a built-in objective, the Philox sampler and
        a separable Gaussian this is ONE kernel (K1+K2 fused: the population is written once and evaluated from registers);
        otherwise `distribution.sample(out=...)` followed by `evaluate` (gaussian.py:292-295 of the reference)."""
        obj = self.evok_objective_id
        if isinstance(batch, LazySolutionBatch):
            if not (obj is not None and self.rng == "philox" and len(self._senses) == 1 and hasattr(distribution, "SYMMETRIC")
                    and ops.uses_kernels(distribution.mu)):
                raise ValueError("a lazy population needs a built-in objective, rng='philox', a separable Gaussian and CUDA float32")
            n = len(batch)
            if distribution.SYMMETRIC and n % 2 != 0:
                raise ValueError(f"Symmetric sampling cannot be done if the number of solutions is odd: {n}")
            seed, stream_id = self.next_philox_stream()
            mu, sigma = distribution.mu.contiguous(), distribution.sigma.contiguous()
            batch.recipe = PhiloxRecipe(seed=seed, stream_id=stream_id, row0=self.philox_row0, n_rows=n, solution_length=self._solution_length,
                                        symmetric=distribution.SYMMETRIC, stream_offset=self.philox_stream_offset, mu=mu, sigma=sigma)
            # the hook runs AFTER the new population is defined (core.py:2559 of the reference calls it inside evaluate(), after
            # distribution.sample): `batch.values` regenerates the new samples from the recipe.  A lazy batch is read-only.
            self._before_eval_hook(batch)
            ops.sample_eval(obj, None, mu, sigma, n_rows=n, symmetric=distribution.SYMMETRIC, seed=seed, stream_id=stream_id,
                            row0=self.philox_row0, f=batch._evdata.view(-1), stream_offset=self.philox_stream_offset)
            self._finish_evaluation(batch)
            return
        values = batch.access_values()
        # before-eval hooks must see (and may edit) the freshly sampled values before they are evaluated (core.py:2559 of the
        # reference: the hook is called inside evaluate(), after distribution.sample): with hooks registered the sampling and the
        # evaluation stay two kernels with the hook in between
        fused = (obj is not None and self.rng == "philox" and ops.uses_kernels(values) and len(self._senses) == 1
                 and hasattr(distribution, "SYMMETRIC") and ops.uses_kernels(distribution.mu) and len(self._before_eval_hook) == 0)
        if not fused:
            distribution.sample(out=values, generator=self)
            self.evaluate(batch)
            return
        n = values.shape[0]
        if distribution.SYMMETRIC and n % 2 != 0:
            raise ValueError(f"Symmetric sampling cannot be done if the leftmost dimension of the target tensor is odd: {tuple(values.shape)}")
        seed, stream_id = self.next_philox_stream()
        evdata = batch._evdata
        direct = evdata.shape[1] == 1 and evdata.dtype == torch.float32 and evdata.is_contiguous()
        f = evdata.view(-1) if direct else torch.empty(n, dtype=torch.float32, device=values.device)
        ops.sample_eval(obj, values, distribution.mu.contiguous(), distribution.sigma.contiguous(), n_rows=n,
                        symmetric=distribution.SYMMETRIC, seed=seed, stream_id=stream_id, row0=self.philox_row0, f=f,
                        stream_offset=self.philox_stream_offset)
        if not direct:
            batch.set_evals(f)
        self._finish_evaluation(batch)

    def sample_and_compute_gradients(self, distribution, popsize: int, *, num_interactions: Optional[int] = None,
                                     popsize_max: Optional[int] = None, obj_index: Optional[int] = None,
                                     ranking_method: Optional[str] = None, with_stats: bool = True,
                                     ensure_even_popsize: bool = False):
        """Sample `popsize` solutions from `distribution`, evaluate them, and return the gradients of the distribution
        parameters (core.py:2762-3073).  The distribution may live on another device than the problem (e.g. a host-resident
        distribution driving a CUDA problem, like the reference's `dist_on_cpu` protocol at core.py:2958): its parameters are
        copied to the problem device, the gradients are returned on the distribution's device.
        When torch.distributed is initialised with more than one rank, every rank samples and evaluates its own row shard,
        fitnesses are all-gathered for a GLOBAL ranking and the partial gradients are all-reduced (see distributed.py); this
        replaces the reference's Ray actors, which rank locally per actor."""
        from .distributed import adaptive_sample_and_gradients, sharded_sample_and_gradients

        popsize = int(popsize)
        if ensure_even_popsize and popsize % 2 != 0:
            popsize += 1
        obj_index = self.normalize_obj_index(obj_index)
        hooks = self.__dict__
        if len(hooks.get("_before_grad_hook", ())) >= 1:
            hooks["_before_grad_hook"]()
        if num_interactions is not None:  # adaptive population size (core.py:3239-3282)
            result = adaptive_sample_and_gradients(self, distribution, popsize, num_interactions=int(num_interactions),
                                                   popsize_max=None if popsize_max is None else int(popsize_max), obj_index=obj_index,
                                                   ranking_method=ranking_method)
        else:
            result = sharded_sample_and_gradients(self, distribution, popsize, obj_index=obj_index, ranking_method=ranking_method)
        if len(hooks.get("_after_grad_hook", ())) >= 1:
            self._after_eval_status = hooks["_after_grad_hook"].accumulate_dict([result])
        return [result] if with_stats else result["gradients"]

    def _get_local_interaction_count(self) -> int:
        """Simulator interactions made so far by this process (core.py:2736-2747; RL problems override it).  The default reads
        the `total_interaction_count` status item."""
        if "total_interaction_count" in self._after_eval_status:
            return int(self._after_eval_status["total_interaction_count"])
        raise NotImplementedError

    def compare_solutions(self, a: "Solution", b: "Solution", obj_index: Optional[int] = None) -> float:
        i = self.normalize_obj_index(obj_index)
        sign = 1.0 if self._senses[i] == "max" else -1.0
        return sign * float(a.evals[i] - b.evals[i])

    def is_better(self, a, b, obj_index=None) -> bool:
        return self.compare_solutions(a, b, obj_index) > 0

    def is_worse(self, a, b, obj_index=None) -> bool:
        return self.compare_solutions(a, b, obj_index) < 0


class SolutionBatch:
    """A population: decision values + evaluation results as two torch tensors (core.py:3590-4601)."""

    def __init__(self, problem: Optional[Problem] = None, popsize: Optional[int] = None, *, device=None, slice_of=None,
                 like: Optional["SolutionBatch"] = None, merging_of: Iterable = None, empty: Optional[bool] = None):
        if slice_of is not None:
            source, sl = slice_of
            self._data = source._data[sl]
            self._evdata = source._evdata[sl]
            self._senses = source._senses
            self._num_objs = source._num_objs
            return
        if merging_of is not None:
            batches = list(merging_of)
            self._data = torch.cat([b._data for b in batches], dim=0)
            self._evdata = torch.cat([b._evdata for b in batches], dim=0)
            self._senses = batches[0]._senses
            self._num_objs = batches[0]._num_objs
            return
        if like is not None and problem is None:
            popsize = len(like) if popsize is None else int(popsize)
            device = like.device if device is None else device
            self._data = torch.empty(popsize, like._data.shape[1], dtype=like._data.dtype, device=device)
            self._evdata = torch.full((popsize, like._evdata.shape[1]), float("nan"), dtype=like._evdata.dtype, device=device)
            self._senses, self._num_objs = like._senses, like._num_objs
            return
        if problem is None or popsize is None:
            if like is not None and problem is not None and popsize is None:
                popsize = len(like)
            else:
                raise ValueError("SolutionBatch needs `problem` and `popsize` (or `like`, `slice_of`, `merging_of`).")
        device = problem.device if device is None else torch.device(device)
        popsize = int(popsize)
        self._senses = problem.senses
        self._num_objs = len(problem.senses)
        self._data = torch.empty(popsize, problem.solution_length, dtype=problem.dtype, device=device)
        self._evdata = torch.full((popsize, self._num_objs + problem.eval_data_length), float("nan"), dtype=problem.eval_dtype,
                                  device=device)
        if not empty:
            problem._fill(self._data)

    # ------------------------------------------------------------------ access
    def __len__(self) -> int:
        return self._data.shape[0]

    def __iter__(self):
        for i in range(len(self)):
            yield self[i]

    def __getitem__(self, i):
        if isinstance(i, slice):
            return SolutionBatch(slice_of=(self, i))
        if isinstance(i, (list, torch.Tensor)):
            return self.take(i)
        i = int(i)
        n = len(self)
        if not (-n <= i < n):
            raise IndexError(f"Solution index out of range: {i}")
        return Solution(self, i % n)

    @property
    def device(self) -> torch.device:
        return self._data.device

    @property
    def dtype(self) -> torch.dtype:
        return self._data.dtype

    values_dtype = dtype

    @property
    def eval_dtype(self) -> torch.dtype:
        return self._evdata.dtype

    @property
    def values_shape(self) -> torch.Size:
        return self._data.shape

    @property
    def eval_shape(self) -> torch.Size:
        return self._evdata.shape

    @property
    def solution_length(self) -> int:
        return self._data.shape[1]

    @property
    def senses(self) -> list:
        return self._senses

    @property
    def objective_sense(self):
        return self._senses[0] if len(self._senses) == 1 else self._senses

    @property
    def values(self) -> torch.Tensor:
        """The N x D decision values as a ReadOnlyTensor sharing storage with what the kernels wrote (core.py:4135-4164);
        `access_values()` gives the mutable tensor."""
        return as_read_only_tensor(self._data)

    @property
    def evals(self) -> torch.Tensor:
        """The N x (objectives + eval data) evaluation results as a ReadOnlyTensor (core.py:4101-4125)."""
        return as_read_only_tensor(self._evdata)

    def access_values(self, *, keep_evals: bool = False) -> torch.Tensor:
        """Mutable view of the decision values; evaluations are forgotten (NaN) unless `keep_evals` (core.py:4166-4195)."""
        if not keep_evals:
            self.forget_evals()
        return self._data

    def access_evals(self, obj_index: Optional[int] = None) -> torch.Tensor:
        """Mutable view of the evaluations, optionally of one objective column (core.py:4127-4164)."""
        return self._evdata if obj_index is None else self._evdata[:, self._normalize_obj_index(obj_index)]

    def forget_evals(self, *, solutions=None):
        if solutions is None:
            self._evdata.fill_(float("nan"))
        else:
            self._evdata[solutions] = float("nan")

    def _normalize_obj_index(self, i) -> int:
        if i is None:
            if self._num_objs != 1:
                raise ValueError("The objective index was expected as an integer (multi-objective batch).")
            return 0
        i = int(i)
        if not (-self._num_objs <= i < self._num_objs):
            raise IndexError(f"Objective index out of range: {i}")
        return i % self._num_objs

    def set_values(self, values: Any, *, solutions=None):
        """Overwrite decision values (and forget the affected evaluations) (core.py:3950-3964)."""
        if solutions is None:
            solutions = slice(None, None, None)
        self._data[solutions] = torch.as_tensor(values, dtype=self._data.dtype, device=self._data.device)
        self._evdata[solutions] = float("nan")

    def set_evals(self, evals: torch.Tensor, eval_data: Optional[torch.Tensor] = None, *, solutions=None):
        """Store evaluation results: `evals` is N (single objective) or N x objectives; `eval_data` fills the extra columns
        (core.py:3966-4087)."""
        if solutions is None:
            solutions = slice(None, None, None)
        num_solutions = self._evdata[solutions].shape[0]
        evals = torch.as_tensor(evals, dtype=self._evdata.dtype, device=self._evdata.device)
        if evals.ndim == 1:
            if self._num_objs != 1 and eval_data is None and evals.shape[0] == num_solutions:
                raise ValueError("A 1-dimensional `evals` tensor can only be used with single-objective problems.")
            evals = evals.reshape(-1, 1)
        elif evals.ndim != 2:
            raise ValueError(f"`evals` was expected with 1 or 2 dimensions, got shape {tuple(evals.shape)}")
        if evals.shape[0] != num_solutions:
            raise ValueError(f"Number of evaluation results ({evals.shape[0]}) does not match the number of solutions ({num_solutions}).")
        total_cols = self._evdata.shape[1]
        if eval_data is not None:
            eval_data = torch.as_tensor(eval_data, dtype=self._evdata.dtype, device=self._evdata.device).reshape(num_solutions, -1)
            if evals.shape[1] != self._num_objs or eval_data.shape[1] != total_cols - self._num_objs:
                raise ValueError("Shapes of `evals` / `eval_data` do not match the problem's objectives / eval_data_length.")
            self._evdata[solutions, : self._num_objs] = evals
            self._evdata[solutions, self._num_objs:] = eval_data
        elif evals.shape[1] == total_cols:
            self._evdata[solutions] = evals
        elif evals.shape[1] == self._num_objs:
            self._evdata[solutions, : self._num_objs] = evals
            self._evdata[solutions, self._num_objs:] = float("nan")
        else:
            raise ValueError(f"`evals` has {evals.shape[1]} columns; expected {self._num_objs} or {total_cols}.")

    # ------------------------------------------------------------------ ordering
    def _sort_keys(self, obj_index) -> tuple:
        i = self._normalize_obj_index(obj_index)
        return self._evdata[:, i], self._senses[i] == "max"

    def argsort(self, obj_index: Optional[int] = None) -> torch.Tensor:
        """Indices from best to worst (core.py:3827-3844); stable tie-break (ascending index)."""
        keys, descending = self._sort_keys(obj_index)
        if ops.uses_kernels(keys):
            return ops.argsort(keys.contiguous(), descending)
        return torch.argsort(keys, descending=descending, stable=True)

    def argbest(self, obj_index: Optional[int] = None) -> torch.Tensor:
        keys, is_max = self._sort_keys(obj_index)
        return torch.argmax(keys) if is_max else torch.argmin(keys)

    def argworst(self, obj_index: Optional[int] = None) -> torch.Tensor:
        keys, is_max = self._sort_keys(obj_index)
        return torch.argmin(keys) if is_max else torch.argmax(keys)

    def utility(self, obj_index: Optional[int] = None, *, ranking_method: Optional[str] = None) -> torch.Tensor:
        """Utilities of the solutions (higher = better) (core.py:4208-4302)."""
        from .tools.ranking import rank

        keys, is_max = self._sort_keys(obj_index)
        return rank(keys, "raw" if ranking_method is None else ranking_method, higher_is_better=is_max)

    def utils(self, *, ranking_method: Optional[str] = None) -> torch.Tensor:
        """Utilities for every objective, shape (N, number of objectives) (core.py:4304-4346)."""
        return torch.stack([self.utility(i, ranking_method=ranking_method) for i in range(self._num_objs)], dim=1)

    # ------------------------------------------------------------------ restructuring
    def take(self, indices: Iterable) -> "SolutionBatch":
        idx = torch.as_tensor(indices, device=self._data.device)
        out = SolutionBatch(like=self, popsize=len(idx))
        out._data[:] = self._data[idx]
        out._evdata[:] = self._evdata[idx]
        return out

    def take_best(self, n: int, *, obj_index: Optional[int] = None) -> "SolutionBatch":
        return self.take(self.argsort(obj_index)[: int(n)])

    def split(self, num_pieces: Optional[int] = None, *, max_size: Optional[int] = None) -> list:
        """Contiguous row slices sharing storage with this batch (core.py:4348, SolutionBatchPieces :4603)."""
        n = len(self)
        if (num_pieces is None) == (max_size is None):
            raise ValueError("Provide exactly one of `num_pieces` and `max_size`.")
        if num_pieces is None:
            num_pieces = math.ceil(n / int(max_size))
        from .tools.misc import split_workload

        pieces, start = [], 0
        for share in split_workload(n, int(num_pieces)):
            pieces.append(SolutionBatch(slice_of=(self, slice(start, start + share))))
            start += share
        return pieces

    def concat(self, other: Union["SolutionBatch", Iterable]) -> "SolutionBatch":
        others = [other] if isinstance(other, SolutionBatch) else list(other)
        return SolutionBatch(merging_of=[self, *others])

    @staticmethod
    def cat(solution_batches: Iterable) -> "SolutionBatch":
        return SolutionBatch(merging_of=list(solution_batches))

    def to(self, device) -> "SolutionBatch":
        if torch.device(device) == self.device:
            return self
        out = SolutionBatch(like=self, device=device)
        out._data[:] = self._data.to(device)
        out._evdata[:] = self._evdata.to(device)
        return out

    def clone(self) -> "SolutionBatch":
        out = SolutionBatch(like=self)
        out._data[:] = self._data
        out._evdata[:] = self._evdata
        return out

    def __copy__(self) -> "SolutionBatch":  # copy.copy / copy.deepcopy give independent storage, like the reference (core.py:4391-4399)
        return self.clone()

    def __deepcopy__(self, memo) -> "SolutionBatch":
        return self.clone()

    def __repr__(self) -> str:
        return f"<SolutionBatch: {len(self)} x {self.solution_length}, {self.dtype}, {self.device}>"


class PhiloxRecipe:
    """How a population was (and can again be) generated: stands in for the N x D sample matrix in the gradient calls."""

    def __init__(self, *, seed: int, stream_id: int, row0: int, n_rows: int, solution_length: int, symmetric: bool,
                 stream_offset: Optional[torch.Tensor], mu: torch.Tensor, sigma: torch.Tensor):
        self.seed, self.stream_id, self.row0, self.n_rows = seed, stream_id, row0, n_rows
        self.solution_length, self.symmetric, self.stream_offset = solution_length, symmetric, stream_offset
        self.mu, self.sigma = mu, sigma

    @property
    def shape(self) -> tuple:
        return (self.n_rows, self.solution_length)

    def materialize(self) -> torch.Tensor:
        """Regenerate the decision values (allocates n_rows x solution_length floats)."""
        out = torch.empty(self.n_rows, self.solution_length, dtype=torch.float32, device=self.mu.device)
        ops.sample_eval(ops.OBJ_NONE, out, self.mu, self.sigma, n_rows=self.n_rows, symmetric=self.symmetric, seed=self.seed,
                        stream_id=self.stream_id, row0=self.row0, stream_offset=self.stream_offset)
        return out


class LazySolutionBatch(SolutionBatch):
    """A population that exists only as fitnesses + a PhiloxRecipe.  `values` / `access_values()` regenerate the decision
    values on demand (every call allocates); everything evaluation-related behaves like a SolutionBatch."""

    def __init__(self, problem: "Problem", popsize: int, *, device=None):
        device = problem.device if device is None else torch.device(device)
        self._senses = problem.senses
        self._num_objs = len(problem.senses)
        self._popsize, self._solution_length = int(popsize), problem.solution_length
        self._values_dtype = problem.dtype
        self._evdata = torch.full((int(popsize), self._num_objs + problem.eval_data_length), float("nan"), dtype=problem.eval_dtype,
                                  device=device)
        self.recipe: Optional[PhiloxRecipe] = None

    @property
    def _data(self) -> torch.Tensor:
        if self.recipe is None:
            raise ValueError("This lazy population has not been sampled yet.")
        return self.recipe.materialize()

    def __len__(self) -> int:
        return self._popsize

    @property
    def device(self) -> torch.device:
        return self._evdata.device

    @property
    def dtype(self) -> torch.dtype:
        return self._values_dtype

    values_dtype = dtype

    @property
    def solution_length(self) -> int:
        return self._solution_length

    @property
    def values_shape(self) -> torch.Size:
        return torch.Size((self._popsize, self._solution_length))

    def access_values(self, *, keep_evals: bool = False) -> torch.Tensor:
        if not keep_evals:
            raise ValueError("The decision values of a lazy population are read-only (they are a function of the Philox counters).")
        return self._data

    def set_values(self, values: Any, *, solutions=None):
        raise ValueError("The decision values of a lazy population are read-only (they are a function of the Philox counters).")

    def __getitem__(self, i):
        if isinstance(i, (slice, list, torch.Tensor)):
            raise NotImplementedError("slicing a lazy population is not supported; use `.values` to materialise it")
        i = int(i) % self._popsize
        out = SolutionBatch(like=None, problem=None, popsize=None, slice_of=(_Materialized(self, i), slice(0, 1)))
        return Solution(out, 0)

    def __repr__(self) -> str:
        return f"<LazySolutionBatch: {self._popsize} x {self._solution_length}, {self.device}>"


class _Materialized:
    """One regenerated row of a lazy population, shaped like a SolutionBatch source for `slice_of`."""

    def __init__(self, lazy: LazySolutionBatch, i: int):
        r = lazy.recipe
        first = (i // 2) * 2 if r.symmetric else i
        rows = 2 if r.symmetric else 1
        block = torch.empty(rows, r.solution_length, dtype=torch.float32, device=r.mu.device)
        ops.sample_eval(ops.OBJ_NONE, block, r.mu, r.sigma, n_rows=rows, symmetric=r.symmetric, seed=r.seed, stream_id=r.stream_id,
                        row0=r.row0 + first, stream_offset=r.stream_offset)
        self._data = block[i - first: i - first + 1]
        self._evdata = lazy._evdata[i: i + 1]
        self._senses, self._num_objs = lazy._senses, lazy._num_objs


class Solution:
    """One row of a SolutionBatch, sharing its storage (core.py:4742-5107)."""

    def __init__(self, parent: SolutionBatch, index: int):
        self._batch = parent[int(index): int(index) + 1]

    @property
    def values(self) -> torch.Tensor:
        return as_read_only_tensor(self._batch._data[0])

    @property
    def evals(self) -> torch.Tensor:
        return as_read_only_tensor(self._batch._evdata[0])

    @property
    def evaluation(self) -> torch.Tensor:
        return as_read_only_tensor(self._batch._evdata[0])

    def access_values(self, *, keep_evals: bool = False) -> torch.Tensor:
        return self._batch.access_values(keep_evals=keep_evals)[0]

    def access_evals(self) -> torch.Tensor:
        return self._batch.access_evals()[0]

    def set_values(self, values: Any):
        self._batch.set_values(torch.as_tensor(values, dtype=self._batch.dtype, device=self._batch.device).reshape(1, -1))

    def set_evals(self, evals, eval_data=None):
        evals = torch.as_tensor(evals, dtype=self._batch.eval_dtype, device=self._batch.device).reshape(1, -1)
        if eval_data is not None:
            eval_data = torch.as_tensor(eval_data, dtype=self._batch.eval_dtype, device=self._batch.device).reshape(1, -1)
        self._batch.set_evals(evals, eval_data)

    set_evaluation = set_evals

    @property
    def is_evaluated(self) -> bool:
        n = self._batch._num_objs
        return not bool(torch.any(torch.isnan(self._batch._evdata[0, :n])))

    @property
    def senses(self) -> list:
        return self._batch.senses

    @property
    def objective_sense(self):
        return self._batch.objective_sense

    @property
    def dtype(self) -> torch.dtype:
        return self._batch.dtype

    @property
    def eval_dtype(self) -> torch.dtype:
        return self._batch.eval_dtype

    @property
    def device(self) -> torch.device:
        return self._batch.device

    @property
    def shape(self) -> torch.Size:
        return self.values.shape

    def __len__(self) -> int:
        return self._batch.solution_length

    def __iter__(self):
        return iter(self.values)

    def __getitem__(self, i):
        return self.values[i]

    def clone(self) -> "Solution":
        return Solution(self._batch.clone(), 0)

    def __copy__(self) -> "Solution":
        return self.clone()

    def __deepcopy__(self, memo) -> "Solution":
        return self.clone()

    def to(self, device) -> "Solution":
        return Solution(self._batch.to(device), 0)

    def to_batch(self) -> SolutionBatch:
        return self._batch

    def __repr__(self) -> str:
        return f"<Solution values={self.values}, evals={self.evals}>"
