"""Exercises the public helpers that the reference's own unit tests cover (hooks, ranking, the optimizer classes, read-only
tensors, the decorators, `expects_ndim` / `rowwise` and the functional optimizers) with fixed, seeded inputs, and returns
everything observable as numpy arrays.

The same code runs against the reference (`probe("evotorch")`, in tests/golden/gen_reference_api_golden.py, which stores
the result as reference_api_golden.npz) and against this package (`probe("evotorch_b200")`, in
tests/test_reference_unit_tests.py), so the test compares this package with the reference output for output.
"""

import importlib

import numpy as np
import torch

GROUPS = ("hook_ranking_optimizers_read_only", "decorators_expects_ndim_functional")


def _np(x):
    if isinstance(x, torch.Tensor):
        return x.detach().cpu().numpy().copy()
    return np.asarray(x)


def _raises(fn) -> bool:
    try:
        fn()
    except Exception:
        return True
    return False


def _hook_ranking_optimizers_read_only(pkg: str) -> dict:
    Hook = importlib.import_module(pkg + ".tools.hook").Hook
    rank = importlib.import_module(pkg + ".tools.ranking").rank
    opt = importlib.import_module(pkg + ".optimizers")
    ro = importlib.import_module(pkg + ".tools.readonlytensor")
    out = {}

    # Hook: positional / keyword arguments stored in the hook come first, dict and list results accumulate
    h = Hook([lambda a, b, c=0: {"sum": a + b + c}, lambda a, b, c=0: {"prod": a * b * c}], args=[2], kwargs={"c": 5})
    res = h(3)
    out["hook/dict_keys"] = np.array(sorted(res))
    out["hook/dict_values"] = np.array([res[k] for k in sorted(res)], dtype=np.float64)
    hl = Hook([lambda x: [x, x + 1], lambda x: [10 * x]])
    out["hook/list"] = np.array(hl(4), dtype=np.float64)
    out["hook/none_result"] = np.array(Hook([lambda: None])() is None)
    h2 = Hook()
    h2.append(lambda x: {"y": 2 * x})
    out["hook/len_after_append"] = np.array(len(h2))
    out["hook/appended"] = np.array(h2(7)["y"], dtype=np.float64)

    # ranking: every method, both senses, on a seeded vector with ties
    g = torch.Generator().manual_seed(3)
    x = torch.randn(11, generator=g)
    x[7] = x[2]
    for method in ("centered", "linear", "nes", "normalized", "raw"):
        for hib in (True, False):
            out[f"rank/{method}/{hib}"] = _np(rank(x, method, higher_is_better=hib))

    # the optimizer classes: ascent steps on seeded gradients
    D = 6
    grads = torch.randn(6, D, generator=g)
    cases = {
        "clipup": lambda: opt.ClipUp(solution_length=D, dtype=torch.float32, stepsize=0.3, momentum=0.8, max_speed=0.5),
        "clipup_default_speed": lambda: opt.ClipUp(solution_length=D, dtype=torch.float32, stepsize=0.1),
        "adam": lambda: opt.Adam(solution_length=D, dtype=torch.float32, stepsize=0.05),
        "adam_betas": lambda: opt.Adam(solution_length=D, dtype=torch.float32, stepsize=0.02, beta1=0.8, beta2=0.99, epsilon=1e-6),
        "sgd": lambda: opt.SGD(solution_length=D, dtype=torch.float32, stepsize=0.1),
        "sgd_momentum": lambda: opt.SGD(solution_length=D, dtype=torch.float32, stepsize=0.1, momentum=0.9),
    }
    for name, make in cases.items():
        o = make()
        out[f"optimizer/{name}"] = np.stack([_np(o.ascent(gr)) for gr in grads])
    for s in ("clipup", "clipsgd", "clipsga", "adam", "sgd", "sga"):
        out[f"optimizer_class/{s}"] = np.array(opt.get_optimizer_class(s).__name__)
    out["optimizer_class/unknown_raises"] = np.array(_raises(lambda: opt.get_optimizer_class("no_such_optimizer")))

    # read-only tensors: reads and out-of-place arithmetic work, writes raise
    t = ro.as_read_only_tensor(torch.arange(6.0))
    writes = {
        "add_": lambda: t.add_(1.0),
        "mul_": lambda: t.mul_(2.0),
        "zero_": lambda: t.zero_(),
        "copy_": lambda: t.copy_(torch.ones(6)),
        "setitem": lambda: t.__setitem__(0, 5.0),
    }
    for name, fn in writes.items():
        out[f"read_only/{name}_raises"] = np.array(_raises(fn))
    out["read_only/values_after_writes"] = _np(torch.as_tensor(t.clone()))
    out["read_only/plus_one"] = _np(torch.as_tensor(t + 1))
    out["read_only/sum"] = _np(torch.as_tensor(t.sum()))
    out["read_only/clone_is_writable"] = np.array(not _raises(lambda: torch.as_tensor(t.clone()).add_(1.0)))
    return out


def _decorators_expects_ndim_functional(pkg: str) -> dict:
    dec = importlib.import_module(pkg + ".decorators")
    fn = importlib.import_module(pkg + ".algorithms.functional")
    out = {}

    # decorators: the attribute each one sets, and that the function itself is returned unchanged
    def base(x):
        """doc"""
        return x

    for name in ("pass_info", "on_aux_device", "on_cuda", "vectorized"):
        f = getattr(dec, name)(base)
        attr = f"__evotorch_{name}__"
        out[f"decorator/{name}/attribute"] = np.array(bool(getattr(f, attr, False)))
        out[f"decorator/{name}/same_name_and_doc"] = np.array((f.__name__, f.__doc__) == ("base", "doc"))
        out[f"decorator/{name}/returns_input"] = np.array(f(3) == 3)
        out[f"decorator/{name}/too_many_args_raises"] = np.array(_raises(lambda: getattr(dec, name)(base, base)))

        def base(x):  # noqa: F811  (a fresh function for the next decorator)
            """doc"""
            return x

    for device in ("cpu", "cuda", "cuda:0", "cuda:1"):
        f = dec.on_device(device)(lambda x: x)
        out[f"decorator/on_device/{device}"] = np.array([str(f.device), bool(getattr(f, "__evotorch_on_device__", False))])
    for spec in (1, "0"):
        f = dec.on_cuda(spec)(lambda x: x)
        out[f"decorator/on_cuda/{spec}"] = np.array([str(f.device), bool(getattr(f, "__evotorch_on_device__", False))])

    # expects_ndim: core dimensions per argument, extra leading dimensions are batch dimensions (broadcast between arguments)
    g = torch.Generator().manual_seed(5)

    @dec.expects_ndim(1, 0)
    def scaled_norm(v, s):
        return torch.linalg.norm(v) * s

    v = torch.randn(4, generator=g)
    vb = torch.randn(3, 4, generator=g)
    vbb = torch.randn(2, 3, 4, generator=g)
    s = torch.randn(3, generator=g)
    out["expects_ndim/plain"] = _np(scaled_norm(v, torch.tensor(2.0)))
    out["expects_ndim/batched_vector"] = _np(scaled_norm(vb, torch.tensor(2.0)))
    out["expects_ndim/batched_scale"] = _np(scaled_norm(v, s))
    out["expects_ndim/matching_batches"] = _np(scaled_norm(vb, s))
    out["expects_ndim/multibatch"] = _np(scaled_norm(vbb, s))
    out["expects_ndim/python_scalar"] = _np(scaled_norm(vb, 3.0))

    @dec.expects_ndim(2, 1)
    def matvec(m, x):
        return m @ x

    m = torch.randn(2, 3, 4, generator=g)
    xs = torch.randn(4, generator=g)
    out["expects_ndim/matvec"] = _np(matvec(m, xs))

    @dec.rowwise
    def centred(x):
        return x - x.mean()

    out["rowwise/vector"] = _np(centred(v))
    out["rowwise/matrix"] = _np(centred(vb))
    out["rowwise/3d"] = _np(centred(vbb))
    out["rowwise/vectorized_flag"] = np.array(bool(getattr(centred, "__evotorch_vectorized__", False)))

    # functional optimizers: ask / tell on seeded gradients, single and batched centres
    grads = torch.randn(5, 3, 4, generator=g)
    c0 = torch.randn(3, 4, generator=g)
    for name, kw in (("adam", dict(center_learning_rate=0.1)), ("clipup", dict(center_learning_rate=0.2, max_speed=0.3)),
                     ("sgd", dict(center_learning_rate=0.1, momentum=0.5))):
        ask, tell = getattr(fn, name + "_ask"), getattr(fn, name + "_tell")
        for tag, center, gs in (("single", c0[0], grads[:, 0]), ("batched", c0, grads)):
            state = getattr(fn, name)(center_init=center, **kw)
            trail = []
            for gr in gs:
                state = tell(state, follow_grad=gr)
                trail.append(_np(ask(state)))
            out[f"functional/{name}/{tag}"] = np.stack(trail)
    return out


def probe(pkg: str, group: str) -> dict:
    """All observations of one group, computed with the package `pkg` (``"evotorch"`` or ``"evotorch_b200"``)."""
    return {"hook_ranking_optimizers_read_only": _hook_ranking_optimizers_read_only,
            "decorators_expects_ndim_functional": _decorators_expects_ndim_functional}[group](pkg)
