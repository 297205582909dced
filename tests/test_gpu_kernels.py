"""Parity of the sm_100a kernels (called through the C ABI of libevok.so via evotorch_b200.ops) against the numpy oracle
and the golden vectors produced by the real reference.  Needs a CUDA device: run with `-m gpu` on the B200 box."""

import os
import math

import numpy as np
import pytest
import torch

from oracle import es_oracle as O

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from evotorch_b200 import Problem, SolutionBatch, ops
    from evotorch_b200 import _native as nat
    from evotorch_b200.algorithms import CEM, PGPE, SNES
    from evotorch_b200.distributions import ExpSeparableGaussian, SeparableGaussian, SymmetricSeparableGaussian
    from evotorch_b200.objectives import ackley, rastrigin, sphere
    from evotorch_b200.optimizers import SGD, Adam, ClipUp
    from evotorch_b200.tools import modify_tensor, rank

DEV = "cuda"
METHODS = ("centered", "linear", "nes", "normalized", "raw")


def C(x, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(x), dtype=dtype).to(DEV)


def N(t):
    return t.detach().cpu().numpy()


def close(a, b, rtol=1e-5, atol=1e-6):
    np.testing.assert_allclose(np.asarray(a, np.float64), np.asarray(b, np.float64), rtol=rtol, atol=atol)


def test_library_is_loaded_and_is_the_in_tree_one():
    lib = nat.lib()
    assert lib.evok_abi_version() == 1
    assert nat.LIB_PATH.endswith("evotorch_b200/lib/libevok.so")


# ---------------------------------------------------------------------------------------------- K1 sampling
@pytest.mark.parametrize("symmetric", [True, False])
@pytest.mark.parametrize("n,D", [(64, 16), (10, 7), (6, 1), (48, 130), (2, 1000)])
def test_sampler_matches_philox_restatement(symmetric, n, D):
    rng = np.random.default_rng(D)
    mu = rng.standard_normal(D).astype(np.float32)
    sg = (np.abs(rng.standard_normal(D)) + 0.1).astype(np.float32)
    X = torch.empty(n, D, device=DEV)
    seed, sid = 0x1234_5678_9ABC_DEF0, 7
    ops.sample_eval(ops.OBJ_NONE, X, C(mu), C(sg), n_rows=n, symmetric=symmetric, seed=seed, stream_id=sid)
    ref = O.philox_population(mu, sg, n, symmetric, seed, sid)
    close(N(X), ref, rtol=0, atol=3e-5 * float(sg.max()) + 1e-6)
    if symmetric:
        close(N(X[0::2] + X[1::2]), np.broadcast_to(2 * mu, (n // 2, D)), rtol=0, atol=1e-5)
    # deterministic, and a different stream id gives a different population
    X2 = torch.empty_like(X)
    ops.sample_eval(ops.OBJ_NONE, X2, C(mu), C(sg), n_rows=n, symmetric=symmetric, seed=seed, stream_id=sid)
    assert torch.equal(X, X2)
    ops.sample_eval(ops.OBJ_NONE, X2, C(mu), C(sg), n_rows=n, symmetric=symmetric, seed=seed, stream_id=sid + 1)
    assert not torch.equal(X, X2)


@pytest.mark.parametrize("symmetric", [True, False])
def test_sampler_is_shard_and_geometry_independent(symmetric):
    n, D = 4096, 256
    mu = torch.linspace(-1, 1, D, device=DEV)
    sg = torch.full((D,), 0.5, device=DEV)
    whole = torch.empty(n, D, device=DEV)
    ops.sample_eval(ops.OBJ_NONE, whole, mu, sg, n_rows=n, symmetric=symmetric, seed=42, stream_id=3)
    for parts in ([1000, 3096], [512] * 8, [2, 4094]):
        row0, pieces = 0, []
        for m in parts:
            x = torch.empty(m, D, device=DEV)
            ops.sample_eval(ops.OBJ_NONE, x, mu, sg, n_rows=m, symmetric=symmetric, seed=42, stream_id=3, row0=row0)
            pieces.append(x)
            row0 += m
        assert torch.equal(torch.cat(pieces), whole)
    # a padded leading dimension (ldx > D) writes the same values
    wide = torch.zeros(n, D + 4, device=DEV)
    view = wide[:, :D]
    ops.sample_eval(ops.OBJ_NONE, view, mu, sg, n_rows=n, symmetric=symmetric, seed=42, stream_id=3)
    assert torch.equal(view, whole) and float(wide[:, D:].abs().max()) == 0.0


def test_sampler_statistics_and_argument_errors():
    n, D = 20000, 512
    mu = torch.zeros(D, device=DEV)
    sg = torch.ones(D, device=DEV)
    X = torch.empty(n, D, device=DEV)
    ops.sample_eval(ops.OBJ_NONE, X, mu, sg, n_rows=n, symmetric=False, seed=9, stream_id=0)
    z = X.double()
    assert abs(float(z.mean())) < 2e-3 and abs(float(z.std()) - 1) < 2e-3
    assert abs(float((z**3).mean())) < 1e-2 and abs(float((z**4).mean()) - 3) < 3e-2
    assert float(z.abs().max()) > 4.5  # tails are populated
    # column and row correlations vanish
    assert abs(float((z[:, 0] * z[:, 1]).mean())) < 0.03 and abs(float((z[0] * z[1]).mean())) < 0.2
    # Kolmogorov-Smirnov distance of a 1e6-sample against the normal CDF
    s = torch.sort(z.reshape(-1)[:1_000_000]).values
    cdf = 0.5 * (1 + torch.erf(s / math.sqrt(2)))
    ks = float((cdf - torch.arange(1, len(s) + 1, device=DEV, dtype=torch.float64) / len(s)).abs().max())
    assert ks < 2.5e-3
    with pytest.raises(ValueError):
        ops.sample_eval(ops.OBJ_NONE, torch.empty(5, D, device=DEV), mu, sg, n_rows=5, symmetric=True, seed=0, stream_id=0)
    with pytest.raises(ValueError):
        ops.sample_eval(ops.OBJ_NONE, torch.empty(4, D, device=DEV), mu, sg, n_rows=4, symmetric=True, seed=0, stream_id=0, row0=1)
    with pytest.raises(ValueError):
        ops.sample_eval(ops.OBJ_RASTRIGIN, None, mu, sg, n_rows=4, symmetric=True, seed=0, stream_id=0)  # f missing
    ops.sample_eval(ops.OBJ_NONE, torch.empty(0, D, device=DEV), mu, sg, n_rows=0, symmetric=True, seed=0, stream_id=0)  # empty is fine


# ---------------------------------------------------------------------------------------------- K2 evaluation
@pytest.mark.parametrize("objective", ["sphere", "rastrigin", "ackley"])
@pytest.mark.parametrize("n,D", [(64, 16), (33, 7), (5, 1), (17, 1003), (8, 10000)])
def test_eval_kernel_matches_oracle(objective, n, D):
    rng = np.random.default_rng(n * D)
    X = (rng.standard_normal((n, D)) * 2.5).astype(np.float32)
    X64 = X.astype(np.float64)
    if objective == "sphere":
        ref = (X64**2).sum(1)
    elif objective == "rastrigin":
        ref = O.rastrigin(X).astype(np.float64)
    else:
        ref = -20 * np.exp(-0.2 * np.sqrt((X64**2).mean(1))) - np.exp(np.cos(2 * np.pi * X64).mean(1)) + 20 + np.e
    got = N(ops.evaluate(ops.OBJECTIVE_IDS[objective], C(X)))
    # fp32 accumulation of D terms + fast cos: relative 1e-6 * sqrt(D) of the value scale (SURVEY.md section 7.3)
    close(got, ref, rtol=2e-6 * math.sqrt(D) + 2e-6, atol=2e-5)


@pytest.mark.parametrize("symmetric", [True, False])
@pytest.mark.parametrize("objective", ["sphere", "rastrigin", "ackley"])
def test_fused_sample_eval_is_consistent(symmetric, objective):
    n, D = 512, 1000
    oid = ops.OBJECTIVE_IDS[objective]
    rng = np.random.default_rng(5)
    mu = C(rng.uniform(-5.12, 5.12, D))
    sg = C(np.full(D, 1.0))
    X = torch.empty(n, D, device=DEV)
    f = torch.empty(n, device=DEV)
    ops.sample_eval(oid, X, mu, sg, n_rows=n, symmetric=symmetric, seed=77, stream_id=1, f=f)
    Xs = torch.empty_like(X)
    ops.sample_eval(ops.OBJ_NONE, Xs, mu, sg, n_rows=n, symmetric=symmetric, seed=77, stream_id=1)
    assert torch.equal(X, Xs)  # fusing the evaluation does not change the population
    f_lazy = torch.empty(n, device=DEV)
    ops.sample_eval(oid, None, mu, sg, n_rows=n, symmetric=symmetric, seed=77, stream_id=1, f=f_lazy)
    assert torch.equal(f, f_lazy)  # "lazy population": same fitness bits without materialising X
    X64 = N(X).astype(np.float64)
    if objective == "sphere":
        ref = (X64**2).sum(1)
    elif objective == "rastrigin":
        ref = 10.0 * D + (X64**2 - 10 * np.cos(2 * np.pi * X64)).sum(1)
    else:
        ref = -20 * np.exp(-0.2 * np.sqrt((X64**2).mean(1))) - np.exp(np.cos(2 * np.pi * X64).mean(1)) + 20 + np.e
    close(N(f), ref, rtol=1e-4, atol=1e-4)
    close(N(ops.evaluate(oid, X)), ref, rtol=1e-4, atol=1e-4)


# ---------------------------------------------------------------------------------------------- K3 ranking
@pytest.mark.parametrize("name", ["appxB", "reftest0", "reftest1", "rand257", "rand1000", "n2", "tied600"])
@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("hib", [True, False])
def test_rank_matches_reference_golden(golden, name, method, hib):
    f = golden[f"rank/{name}/f"]
    ref = golden[f"rank/{name}/{method}/{int(hib)}"]
    perm = torch.empty(len(f), dtype=torch.int64, device=DEV)
    got = N(ops.rank(C(f), method, hib, perm=perm))
    if method in ("centered", "linear", "raw"):
        np.testing.assert_array_equal(got, ref)  # bit exact against the reference's own output
    else:
        close(got, ref, rtol=3e-6, atol=3e-7)
    np.testing.assert_array_equal(N(perm), O.argsort_for_ranking(f, hib))  # bit-exact ranking indices


@pytest.mark.parametrize("n", [1, 2, 31, 1024, 1025, 2049, 4096, 4097, 8192, 8193, 100_003, 1_000_000])  # <= 8192: the single-launch counting rank; above: radix
@pytest.mark.parametrize("hib", [True, False])
def test_rank_large_with_ties_nan_and_signed_zero(n, hib):
    rng = np.random.default_rng(n)
    f = (rng.standard_normal(n) * 717 + 1.1e5).astype(np.float32)  # fp32 Rastrigin-like: massive collisions at large n
    if n > 100:
        f[::97] = 0.0
        f[1::97] = -0.0
        f[5::1013] = np.nan
        f[7::5003] = np.inf
        f[11::5003] = -np.inf
    perm = torch.empty(n, dtype=torch.int64, device=DEV)
    w = N(ops.rank(C(f), "centered", hib, perm=perm))
    order = O.argsort_for_ranking(f, hib)
    np.testing.assert_array_equal(N(perm), order)
    if n > 1:
        np.testing.assert_array_equal(w, O.rank_centered(f, hib))
    np.testing.assert_array_equal(N(ops.argsort(C(f), descending=not hib)), order)
    if n >= 31:
        close(N(ops.rank(C(f[np.isfinite(f)]), "nes", hib)), O.rank_nes(f[np.isfinite(f)], hib), rtol=2e-5, atol=2e-9)


def test_rank_properties_and_helpers():
    n = 300_000
    f = torch.randn(n, device=DEV) * 3
    w = ops.rank(f, "centered", False)
    # utilities are a permutation of the table, and monotone in fitness (lower f -> higher utility for "min")
    sw = torch.sort(w).values
    # IEEE division like torch-CPU / numpy (torch-CUDA multiplies by the reciprocal and can differ by 1 ulp, SURVEY appendix D)
    table = np.arange(n, dtype=np.float32) / np.float32(n - 1) - np.float32(0.5)
    np.testing.assert_array_equal(N(sw), table)
    order = torch.argsort(f, stable=True)
    fs, ws_ = f[order], w[order]
    strictly = fs[:-1] < fs[1:]  # among equal fitnesses the stable tie-break (ascending index) decides, checked elsewhere
    assert bool((ws_[:-1] > ws_[1:])[strictly].all())
    # weight adjustments
    w2 = ops.weights_adjust_(ops.rank(f, "nes", False).clone(), 1)
    assert abs(float(w2.double().sum())) < 1e-4
    w3 = ops.weights_adjust_(ops.rank(f, "linear", False).clone(), 2)
    assert abs(float(w3.abs().double().sum()) - 1) < 1e-5
    # elite mask = the k largest weights, ties by ascending index
    wt = torch.tensor([1.0, 5.0, 5.0, 2.0, 5.0, 0.0], device=DEV)
    assert ops.elite_mask(wt, 2).tolist() == [0, 1, 1, 0, 0, 0]
    assert ops.elite_mask(wt, 4).tolist() == [0, 1, 1, 1, 1, 0]
    # the counting path (n <= 8192) and the radix path (n > 8192) agree with torch on both sides of the switch
    for m in (5000, 8192, 8193, 20000):
        wm = torch.randn(m, device=DEV).round(decimals=1)  # plenty of ties
        ref = torch.zeros(m, device=DEV)
        ref[torch.argsort(wm, descending=True, stable=True)[: m // 3]] = 1
        assert torch.equal(ops.elite_mask(wm, m // 3), ref), m
        assert torch.equal(ops.argsort(wm, descending=False), torch.argsort(wm, stable=True)), m
    with pytest.raises(KeyError):
        ops.rank(f, "nope", True)


# ---------------------------------------------------------------------------------------------- K4 gradients
@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("sense", ["min", "max"])
def test_gradients_match_reference_golden(golden, method, sense):
    mu, sg = C(golden["grad/mu"]), C(golden["grad/sigma"])
    for div in ("num_directions", "num_solutions", "total_weight", "weight_stdev", None):
        extra = {} if div is None else {"divide_mu_grad_by": div, "divide_sigma_grad_by": div}
        d = SymmetricSeparableGaussian({"mu": mu, "sigma": sg, **extra})
        g = d.compute_gradients(C(golden["grad/Xsym"]), C(golden["grad/fsym"]), objective_sense=sense, ranking_method=method)
        scale = max(1.0, float(np.abs(golden[f"grad/sym/{method}/{sense}/{div}/sigma"]).max()))
        close(N(g["mu"]), golden[f"grad/sym/{method}/{sense}/{div}/mu"], rtol=2e-4, atol=2e-5 * scale)
        close(N(g["sigma"]), golden[f"grad/sym/{method}/{sense}/{div}/sigma"], rtol=2e-4, atol=2e-5 * scale)
        d = SeparableGaussian({"mu": mu, "sigma": sg, **extra})
        g = d.compute_gradients(C(golden["grad/Xns"]), C(golden["grad/fns"]), objective_sense=sense, ranking_method=method)
        scale = max(1.0, float(np.abs(golden[f"grad/sep/{method}/{sense}/{div}/sigma"]).max()))
        close(N(g["mu"]), golden[f"grad/sep/{method}/{sense}/{div}/mu"], rtol=2e-4, atol=2e-5 * scale)
        close(N(g["sigma"]), golden[f"grad/sep/{method}/{sense}/{div}/sigma"], rtol=2e-4, atol=2e-5 * scale)
    d = ExpSeparableGaussian({"mu": mu, "sigma": sg})
    g = d.compute_gradients(C(golden["grad/Xns"]), C(golden["grad/fns"]), objective_sense=sense, ranking_method=method)
    close(N(g["mu"]), golden[f"grad/exp/{method}/{sense}/mu"], rtol=2e-4, atol=2e-5)
    close(N(g["sigma"]), golden[f"grad/exp/{method}/{sense}/sigma"], rtol=2e-4, atol=5e-5)


@pytest.mark.parametrize("ratio", [0.5, 0.25, 0.1])
@pytest.mark.parametrize("sense", ["min", "max"])
def test_cem_gradients_match_reference_golden(golden, ratio, sense):
    d = SeparableGaussian({"mu": C(golden["grad/mu"]), "sigma": C(golden["grad/sigma"]), "parenthood_ratio": ratio})
    g = d.compute_gradients(C(golden["grad/Xns"]), C(golden["grad/fns"]), objective_sense=sense, ranking_method=None)
    close(N(g["mu"]), golden[f"grad/cem/{ratio}/{sense}/mu"], rtol=2e-5, atol=3e-6)
    close(N(g["sigma"]), golden[f"grad/cem/{ratio}/{sense}/sigma"], rtol=2e-5, atol=3e-6)


@pytest.mark.parametrize("form", ["separable", "symmetric", "exp", "moments"])
@pytest.mark.parametrize("n,D", [(2, 1), (6, 3), (64, 16), (130, 7), (1000, 130), (514, 1000), (4096, 1030), (256, 10000), (20000, 64)])
def test_grad_kernel_matches_oracle_ragged_shapes(form, n, D):
    rng = np.random.default_rng(n + D)
    mu = rng.standard_normal(D).astype(np.float32)
    sg = (np.abs(rng.standard_normal(D)) * 0.5 + 0.2).astype(np.float32)
    X = (mu + sg * rng.standard_normal((n, D))).astype(np.float32)
    w = (rng.standard_normal(n) / n).astype(np.float32)
    if form == "moments":
        w = (rng.random(n) < 0.3).astype(np.float32)
    fid = {"separable": ops.GRAD_SEPARABLE, "symmetric": ops.GRAD_SYMMETRIC, "exp": ops.GRAD_EXP, "moments": ops.GRAD_MOMENTS}[form]
    gm, gs = ops.grad(fid, C(X), C(w), C(mu), C(sg), 0.5, 2.0)
    w64, X64, mu64, sg64 = w.astype(np.float64), X.astype(np.float64), mu.astype(np.float64), sg.astype(np.float64)
    if form == "symmetric":
        eps = X64[0::2] - mu64
        a, b = (w64[0::2] - w64[1::2]) / 2, (w64[0::2] + w64[1::2]) / 2
        g = (eps**2 - sg64**2) / sg64
    else:
        eps = X64 - mu64
        a = b = w64
        g = {"separable": (eps**2 - sg64**2) / sg64, "exp": (eps / sg64) ** 2 - 1, "moments": eps**2}[form]
    ref_m = 0.5 * (a[:, None] * eps).sum(0)
    ref_s = 2.0 * (b[:, None] * g).sum(0)
    tol_m = 3e-6 * 0.5 * (np.abs(a)[:, None] * np.abs(eps)).sum(0).max() + 1e-9
    tol_s = 3e-6 * 2.0 * (np.abs(b)[:, None] * (np.abs(g) + 1)).sum(0).max() + 1e-9
    close(N(gm), ref_m, rtol=1e-4, atol=tol_m)
    close(N(gs), ref_s, rtol=1e-4, atol=tol_s)
    # a strided (padded) population gives identical bits
    wide = torch.zeros(n, D + 3, device=DEV)
    wide[:, :D] = C(X)
    gm2, gs2 = ops.grad(fid, wide[:, :D], C(w), C(mu), C(sg), 0.5, 2.0)
    close(N(gm2), N(gm), rtol=1e-5, atol=tol_m)
    close(N(gs2), N(gs), rtol=1e-5, atol=tol_s)


def test_grad_is_deterministic_linear_and_shard_additive():
    n, D = 8192, 2000
    g = torch.Generator(device=DEV).manual_seed(1)
    mu = torch.randn(D, device=DEV, generator=g)
    sg = torch.rand(D, device=DEV, generator=g) + 0.5
    X = mu + sg * torch.randn(n, D, device=DEV, generator=g)
    w1 = torch.randn(n, device=DEV, generator=g) / n
    w2 = torch.randn(n, device=DEV, generator=g) / n
    a1 = ops.grad(ops.GRAD_SYMMETRIC, X, w1, mu, sg, 1.0, 1.0)
    a1b = ops.grad(ops.GRAD_SYMMETRIC, X, w1, mu, sg, 1.0, 1.0)
    assert torch.equal(a1[0], a1b[0]) and torch.equal(a1[1], a1b[1])  # no atomics: bit-reproducible
    a2 = ops.grad(ops.GRAD_SYMMETRIC, X, w2, mu, sg, 1.0, 1.0)
    a12 = ops.grad(ops.GRAD_SYMMETRIC, X, w1 + w2, mu, sg, 1.0, 1.0)
    for k in range(2):
        close(N(a12[k]), N(a1[k] + a2[k]), rtol=1e-4, atol=2e-6)
    parts = [(0, 1000), (1000, 5000), (5000, 8192)]
    acc = [torch.zeros(D, device=DEV), torch.zeros(D, device=DEV)]
    for lo, hi in parts:
        p = ops.grad(ops.GRAD_SYMMETRIC, X[lo:hi], w1[lo:hi], mu, sg, 1.0, 1.0)
        acc[0] += p[0]
        acc[1] += p[1]
    for k in range(2):
        close(N(acc[k]), N(a1[k]), rtol=1e-4, atol=2e-6)
    # rows whose weights are zero are skipped without changing the result
    wz = w1.clone()
    wz[2000:6000] = 0
    z = ops.grad(ops.GRAD_SEPARABLE, X, wz, mu, sg, 1.0, 1.0)
    zz = ops.grad(ops.GRAD_SEPARABLE, torch.cat([X[:2000], X[6000:]]), torch.cat([wz[:2000], wz[6000:]]), mu, sg, 1.0, 1.0)
    for k in range(2):
        close(N(z[k]), N(zz[k]), rtol=1e-4, atol=2e-6)


@pytest.mark.parametrize("symmetric", [True, False])
def test_grad_regen_equals_materialised_path(symmetric):
    n, D = 2048, 1000
    mu = torch.linspace(-2, 2, D, device=DEV)
    sg = torch.rand(D, device=DEV) + 0.3
    X = torch.empty(n, D, device=DEV)
    row0 = 512
    ops.sample_eval(ops.OBJ_NONE, X, mu, sg, n_rows=n, symmetric=symmetric, seed=5, stream_id=9, row0=row0)
    w = torch.randn(n, device=DEV) / n
    form = ops.GRAD_SYMMETRIC if symmetric else ops.GRAD_SEPARABLE
    a = ops.grad(form, X, w, mu, sg, 1.0, 1.0)
    b = ops.grad_regen(form, w, mu, sg, seed=5, stream_id=9, row0=row0, scale_mu=1.0, scale_sigma=1.0)
    for k in range(2):
        close(N(b[k]), N(a[k]), rtol=2e-4, atol=3e-6)


# ---------------------------------------------------------------------------------------------- K5 updates
def test_optimizer_kernels_match_reference_golden(golden):
    grads = golden["opt/grads"]
    for i in range(4):
        ss, mom, ms = golden[f"opt/clipup/{i}/cfg"]
        opt = ClipUp(solution_length=12, dtype="float32", stepsize=ss, momentum=mom, max_speed=None if ms < 0 else ms, device=DEV)
        got = np.stack([N(opt.ascent(C(g))) for g in grads])
        close(got, golden[f"opt/clipup/{i}/steps"], rtol=3e-6, atol=3e-7)
        # fused mu += step gives the same trajectory
        opt2 = ClipUp(solution_length=12, dtype="float32", stepsize=ss, momentum=mom, max_speed=None if ms < 0 else ms, device=DEV)
        m = torch.zeros(12, device=DEV)
        for g in grads:
            opt2.ascent_into_(C(g), m)
        close(N(m), golden[f"opt/clipup/{i}/steps"].sum(0), rtol=1e-5, atol=1e-6)
    for tag, kw in (("adam/0", dict(stepsize=0.05)), ("adam/1", dict(stepsize=0.01, beta1=0.8, beta2=0.95, epsilon=1e-6))):
        opt = Adam(solution_length=12, dtype="float32", device=DEV, **kw)
        close(np.stack([N(opt.ascent(C(g))) for g in grads]), golden[f"opt/{tag}/steps"], rtol=1e-5, atol=1e-7)
    for tag, kw in (("sgd/0", dict(stepsize=0.1)), ("sgd/1", dict(stepsize=0.1, momentum=0.8))):
        opt = SGD(solution_length=12, dtype="float32", device=DEV, **kw)
        close(np.stack([N(opt.ascent(C(g))) for g in grads]), golden[f"opt/{tag}/steps"], rtol=3e-6, atol=1e-7)
    # a large vector exercises the multi-iteration single-CTA reductions
    D = 100_003
    g = torch.randn(D, device=DEV)
    opt = ClipUp(solution_length=D, dtype="float32", stepsize=0.5, device=DEV)
    ref = O.ClipUp(D, 0.5)
    for _ in range(4):
        close(N(opt.ascent(g)), ref.ascent(N(g)), rtol=1e-5, atol=1e-8)


def test_sigma_update_kernel_matches_modify_tensor(golden):
    xo, xt = golden["modify/r/orig"], golden["modify/r/target"]
    s = C(np.abs(xo) + 0.1)
    g = C(xt)
    for exp_form in (False, True):
        for kw in ({}, {"max_change": 0.2}, {"lb": 0.05, "ub": 1.0, "max_change": 0.5}, {"lb": C(np.full(16, 0.3))},
                   {"ub": C(np.linspace(0.2, 2.0, 16))}, {"max_change": C(np.linspace(0.01, 0.9, 16))}):
            cur = s.clone()
            ops.sigma_update_(cur, g, 0.3, exp_form, **kw)
            target = s * torch.exp(0.5 * 0.3 * g) if exp_form else s + 0.3 * g
            ref = modify_tensor(s, target, **kw)
            close(N(cur), N(ref), rtol=2e-6, atol=1e-7)
    # the reference's own known answers
    x = C([10, 11, 12])
    for kw, ans in (({"lb": 5}, [5, 21, 22]), ({"lb": 5, "ub": 20}, [5, 20, 20]), ({"max_change": 0.5}, [5, 16.5, 18]),
                    ({"lb": 7, "ub": 17, "max_change": 0.5}, [7, 16.5, 17])):
        cur = x.clone()
        ops.sigma_update_(cur, C([-10, 10, 10]), 1.0, False, **kw)
        assert cur.tolist() == ans


# ---------------------------------------------------------------------------------------------- whole generations
TRAJ = {
    "pgpe": lambda p, mu, sg: PGPE(p, popsize=32, center_learning_rate=0.5, stdev_learning_rate=0.1, center_init=mu, stdev_init=sg),
    "pgpe_max": lambda p, mu, sg: PGPE(p, popsize=32, center_learning_rate=0.5, stdev_learning_rate=0.1, center_init=mu, stdev_init=sg),
    "pgpe_nonsym_adam": lambda p, mu, sg: PGPE(p, popsize=30, center_learning_rate=0.05, stdev_learning_rate=0.1, center_init=mu,
                                                stdev_init=sg, symmetric=False, optimizer="adam"),
    "pgpe_nes_rank": lambda p, mu, sg: PGPE(p, popsize=32, center_learning_rate=0.3, stdev_learning_rate=0.1, center_init=mu,
                                             stdev_init=sg, ranking_method="nes", optimizer=None, stdev_min=0.01, stdev_max=2.0),
    "snes": lambda p, mu, sg: SNES(p, popsize=24, center_init=mu, stdev_init=sg),
    "snes_clipup": lambda p, mu, sg: SNES(p, popsize=24, center_init=mu, stdev_init=sg, optimizer="clipup", center_learning_rate=0.2,
                                           stdev_max_change=0.3),
    "cem": lambda p, mu, sg: CEM(p, popsize=40, parenthood_ratio=0.25, center_init=mu, stdev_init=sg, stdev_max_change=0.5),
}


@pytest.mark.parametrize("tag", sorted(TRAJ))
def test_seeded_reference_trajectory_through_the_cuda_searcher(golden, tag):
    """Feed the reference's recorded populations (X_t, f_t) to the CUDA searcher generation by generation: its
    rank -> gradient -> update kernels must reproduce the reference's (mu_{t+1}, sigma_{t+1}) within 1e-5 relative."""
    mu, sg, X, f = (golden[f"traj/{tag}/{k}"] for k in ("mu", "sigma", "X", "f"))
    T, n, D = X.shape
    sense = "max" if tag == "pgpe_max" else "min"
    prob = Problem(sense, rastrigin, initial_bounds=(-5.12, 5.12), solution_length=D, device=DEV, seed=11)
    s = TRAJ[tag](prob, C(mu[0]), C(sg[0]))
    s.step()  # generation 1: sample + evaluate only (with our own Philox population, replaced below)
    for t in range(T - 1):
        s._population.set_values(C(X[t]))
        s._population.set_evals(C(f[t]))
        s.step()
        close(N(s.status["center"]), mu[t + 1], rtol=1e-5, atol=2e-6)
        close(N(s.status["stdev"]), sg[t + 1], rtol=1e-5, atol=2e-6)


@pytest.mark.parametrize("algo", ["pgpe", "pgpe_nonsym", "snes", "cem"])
def test_cuda_searchers_optimise_and_are_seed_deterministic(algo):
    def make(seed):
        prob = Problem("min", rastrigin, initial_bounds=(-5.12, 5.12), solution_length=200, device=DEV, seed=seed)
        if algo == "pgpe":
            return PGPE(prob, popsize=2000, center_learning_rate=0.5, stdev_learning_rate=0.1, stdev_init=1.0)
        if algo == "pgpe_nonsym":
            return PGPE(prob, popsize=2000, center_learning_rate=0.5, stdev_learning_rate=0.1, stdev_init=1.0, symmetric=False)
        if algo == "snes":
            return SNES(prob, popsize=2000, stdev_init=3.0)
        return CEM(prob, popsize=2000, parenthood_ratio=0.2, stdev_init=3.0)

    a, b, c = make(4), make(4), make(5)
    a.step()
    first = a.status["mean_eval"]
    a.run(60)
    b.run(61)
    c.run(61)
    assert a.status["mean_eval"] < 0.7 * first
    assert torch.equal(a.status["center"], b.status["center"]) and torch.equal(a.status["stdev"], b.status["stdev"])
    assert not torch.equal(a.status["center"], c.status["center"])
    assert a.population.values.is_cuda and a.population.evals.shape == (2000, 1)
    assert math.isfinite(a.status["pop_best_eval"]) and a.status["pop_best"].values.shape == (200,)


@pytest.mark.parametrize("algo", ["pgpe", "pgpe_plain_nonsym", "snes", "cem"])
def test_cuda_graph_replay_is_bit_identical_to_eager(algo):
    def make():
        prob = Problem("min", rastrigin, initial_bounds=(-5.12, 5.12), solution_length=300, device=DEV, seed=21)
        if algo == "pgpe":
            return PGPE(prob, popsize=1000, center_learning_rate=0.5, stdev_learning_rate=0.1, stdev_init=1.0)
        if algo == "pgpe_plain_nonsym":
            return PGPE(prob, popsize=1000, center_learning_rate=0.1, stdev_learning_rate=0.1, stdev_init=1.0, symmetric=False, optimizer=None,
                        ranking_method="nes", stdev_min=0.01, stdev_max=3.0)
        if algo == "snes":
            return SNES(prob, popsize=1000, stdev_init=2.0)
        return CEM(prob, popsize=1000, parenthood_ratio=0.25, stdev_init=2.0, stdev_max_change=0.5)

    eager, graph = make(), make().enable_cuda_graph()
    seen = []
    graph.after_step_hook.append(lambda: seen.append(1) or {})
    for gen in range(12):
        eager.step()
        graph.step()
        assert torch.equal(eager.status["center"], graph.status["center"]), gen
        assert torch.equal(eager.status["stdev"], graph.status["stdev"]), gen
        assert torch.equal(eager.population.values, graph.population.values), gen
        assert torch.equal(eager.population.evals, graph.population.evals), gen
    assert graph._graph is not None and len(seen) == 12
    assert graph.status["mean_eval"] == eager.status["mean_eval"]
    # status tensors read in graph mode are snapshots, not views of the live buffers
    c = graph.status["center"]
    graph.step()
    assert not torch.equal(c, graph.status["center"])
    # an Adam-driven searcher is not capturable (host-side bias correction) and silently keeps stepping eagerly
    prob = Problem("min", rastrigin, initial_bounds=(-5.12, 5.12), solution_length=64, device=DEV, seed=3)
    adam = PGPE(prob, popsize=200, center_learning_rate=0.05, stdev_learning_rate=0.1, stdev_init=1.0, optimizer="adam").enable_cuda_graph()
    adam.run(4)
    assert adam._graph is None and adam.step_count == 4


def test_user_objective_and_torch_rng_paths_on_cuda():
    def my_sphere(x):
        return torch.sum(x * x, dim=-1)

    prob = Problem("min", my_sphere, initial_bounds=(-3, 3), solution_length=64, device=DEV, seed=1, vectorized=True)
    s = PGPE(prob, popsize=500, center_learning_rate=0.3, stdev_learning_rate=0.1, stdev_init=1.0)
    s.step()
    m0 = s.status["mean_eval"]
    s.run(40)
    assert s.status["mean_eval"] < 0.5 * m0
    prob_t = Problem("min", sphere, initial_bounds=(-3, 3), solution_length=64, device=DEV, seed=1, rng="torch")
    st = PGPE(prob_t, popsize=500, center_learning_rate=0.3, stdev_learning_rate=0.1, stdev_init=1.0)
    st.run(3)
    X = st.population.values
    close(N(X[0::2] + X[1::2]), np.broadcast_to(2 * N(st.status["center"]), (250, 64)), rtol=0, atol=1e-5)


@pytest.mark.parametrize("M,N,K", [(128, 256, 32), (4096, 1024, 1024), (1024, 1024, 4096), (100, 70, 36), (129, 257, 40), (12, 6, 6), (300, 513, 1000)])
def test_tcgen05_gemm_matches_float64(M, N, K):
    g = torch.Generator(device=DEV).manual_seed(M + N + K)
    A = torch.randn(M, K, device=DEV, generator=g)
    B = torch.randn(N, K, device=DEV, generator=g)
    ref = A.double() @ B.double().T
    C = ops.gemm_nt(A, B)
    scale = float(ref.abs().max())
    assert float((C.double() - ref).abs().max()) / scale < 3e-6  # fp32-SGEMM-class accuracy out of TF32 tensor cores (3xTF32)
    # exactly representable data must come out exact: proves the TMA / swizzle / descriptor data path
    Ai = torch.randint(-8, 9, (M, K), device=DEV, generator=g).float()
    Bi = torch.randint(-8, 9, (N, K), device=DEV, generator=g).float()
    assert torch.equal(ops.gemm_nt(Ai, Bi).double(), Ai.double() @ Bi.double().T)
    # fused affine epilogue and strided operands
    alpha = torch.tensor([0.37], device=DEV)
    bias = torch.randn(N, device=DEV, generator=g)
    C2 = torch.empty(M, N, device=DEV)
    wide = torch.zeros(M, K + 4, device=DEV)
    wide[:, :K] = A
    C1 = ops.gemm_nt(wide[:, :K], B, out2=C2, alpha=alpha, bias=bias)
    assert float((C1.double() - ref).abs().max()) / scale < 3e-6
    assert float((C2.double() - (0.37 * ref + bias.double())).abs().max()) / scale < 3e-6
    w = torch.randn(M, device=DEV, generator=g)
    assert torch.equal(ops.transpose_scale(A, w), (A * w[:, None]).T.contiguous())


def test_cmaes_on_cuda_reproduces_reference_trajectory(golden):
    """The reference's CMA-ES run (its z draws recorded) through the CUDA searcher: GEMM sampling, K2 evaluation, K3 ranking,
    K4 weighted recombination, rank-mu SYRK and Cholesky must reproduce (m, sigma, C, A, paths)."""
    from evotorch_b200.algorithms import CMAES

    Z = golden["cmaes/Z"]
    T, n, D = Z.shape
    prob = Problem("min", sphere, initial_bounds=(-3, 3), solution_length=D, device=DEV, seed=3)
    c = CMAES(prob, stdev_init=1.0, popsize=n, center_init=C(golden["cmaes/m0"]))
    close(N(c.weights), golden["cmaes/weights"], rtol=2e-6, atol=1e-8)
    for t in range(T):
        zt = C(Z[t])

        def recorded_sample(num_samples=None, zt=zt):
            ys = zt @ c.A.T
            return zt, ys, c.m.unsqueeze(0) + c.sigma * ys

        c.sample_distribution = recorded_sample
        c.step()
        close(N(c.population.evals[:, 0]), golden["cmaes/f"][t], rtol=2e-5, atol=1e-5)
        close(N(c.m), golden["cmaes/m"][t], rtol=2e-5, atol=3e-6)
        close(float(c.sigma), golden["cmaes/sigma"][t][0], rtol=2e-5)
        close(N(c.C), golden["cmaes/C"][t], rtol=2e-5, atol=3e-6)
        close(N(c.A), golden["cmaes/A"][t], rtol=2e-5, atol=3e-6)
        close(N(c.p_sigma), golden["cmaes/p_sigma"][t], rtol=2e-5, atol=3e-6)
        close(N(c.p_c), golden["cmaes/p_c"][t], rtol=2e-5, atol=3e-6)
    # with its own Philox draws it optimises
    prob2 = Problem("min", sphere, initial_bounds=(-3, 3), solution_length=64, device=DEV, seed=1)
    c2 = CMAES(prob2, stdev_init=1.0, popsize=256)
    c2.step()
    m0 = c2.status["mean_eval"]
    c2.run(60)
    assert c2.status["mean_eval"] < 0.2 * m0


def test_xnes_on_cuda_matches_reference_golden(golden):
    from evotorch_b200.algorithms import XNES
    from evotorch_b200.distributions import ExpGaussian

    dist = ExpGaussian({"mu": C(golden["xnes/mu"]), "sigma": C(golden["xnes/A"]), "sigma_inv": C(golden["xnes/A_inv"])})
    for method in ("nes", "centered"):
        g = dist.compute_gradients(C(golden["xnes/X"]), C(golden["xnes/f"]), objective_sense="min", ranking_method=method)
        close(N(g["d"]), golden[f"xnes/{method}/d"], rtol=1e-4, atol=3e-6)
        close(N(g["M"]), golden[f"xnes/{method}/M"], rtol=1e-4, atol=6e-6)
        upd = dist.update_parameters(g, learning_rates={"mu": 1.0, "sigma": 0.3})
        close(N(upd.mu), golden[f"xnes/{method}/new_mu"], rtol=2e-5, atol=3e-6)
        close(N(upd.A), golden[f"xnes/{method}/new_A"], rtol=2e-5, atol=3e-6)
        close(N(upd.A_inv), golden[f"xnes/{method}/new_A_inv"], rtol=2e-5, atol=6e-6)
    x = dist.sample(64, generator=torch.Generator(device=DEV).manual_seed(0))
    close(N(dist.to_global_coordinates(dist.to_local_coordinates(x))), N(x), rtol=1e-4, atol=1e-4)
    prob = Problem("min", sphere, initial_bounds=(-3, 3), solution_length=12, device=DEV, seed=2)
    s = XNES(prob, popsize=64, stdev_init=1.0)
    s.step()
    m0 = s.status["mean_eval"]
    s.run(80)
    assert s.status["mean_eval"] < 0.2 * m0


# ---------------------------------------------------------------------------------------------- K8 batched policy forward
def test_policy_kernel_matches_reference_golden_and_oracle(golden):
    from evotorch_b200.neuroevolution import Policy

    net = torch.nn.Sequential(torch.nn.Linear(11, 8), torch.nn.Tanh(), torch.nn.Linear(8, 3))
    pol = Policy(net)
    pol.set_parameters(C(golden["policy/params"]))
    close(N(pol(C(golden["policy/obs"]))), golden["policy/act"], rtol=1e-5, atol=2e-6)  # the reference's vmap(functional_call)
    rng = np.random.default_rng(0)
    for dims, acts, n in (([376, 256, 17], ["tanh", "none"], 67), ([5, 1], ["none"], 9), ([33, 70, 9, 4], ["relu", "sigmoid", "tanh"], 40),
                          ([2048, 3, 2048], ["tanh", "none"], 3)):
        L = sum(dims[i] * dims[i + 1] + dims[i + 1] for i in range(len(acts)))
        P = (rng.standard_normal((n, L)) * 0.1).astype(np.float32)
        X = rng.standard_normal((n, dims[0])).astype(np.float32)
        got = N(ops.mlp_forward(C(P), C(X), dims, acts))
        h = X.astype(np.float64)
        off = 0
        for l, act in enumerate(acts):
            W = P[:, off:off + dims[l] * dims[l + 1]].reshape(n, dims[l + 1], dims[l]).astype(np.float64)
            off += dims[l] * dims[l + 1]
            b = P[:, off:off + dims[l + 1]].astype(np.float64)
            off += dims[l + 1]
            h = np.einsum("noi,ni->no", W, h) + b
            h = {"tanh": np.tanh, "relu": lambda v: np.maximum(v, 0), "sigmoid": lambda v: 1 / (1 + np.exp(-v)), "none": lambda v: v}[act](h)
        close(got, h, rtol=2e-5, atol=2e-5)
        if dims == [376, 256, 17]:
            assert L == 100881  # cfg4: rows are only 4-byte aligned (L is odd)
            close(got, O.mlp_policy_forward(P, X, 376, 256, 17, "tanh"), rtol=2e-5, atol=2e-5)
            net4 = torch.nn.Sequential(torch.nn.Linear(376, 256), torch.nn.Tanh(), torch.nn.Linear(256, 17))
            p4 = Policy(net4)
            p4.set_parameters(C(P))
            close(N(p4(C(X))), got, rtol=0, atol=0)
    with pytest.raises(ValueError):
        ops.mlp_forward(C(np.zeros((3, 10))), C(np.zeros((3, 5))), [5, 1], ["none"])


# ---------------------------------------------------------------------------------------------- full-size properties
def test_config2_size_properties():
    """BASELINE configs[1]: PGPE, Rastrigin, N = 100 000, D = 10 000 (4 GB population) -- size-independent properties."""
    n, D = 100_000, 10_000
    prob = Problem("min", rastrigin, initial_bounds=(-5.12, 5.12), solution_length=D, device=DEV, seed=0)
    s = PGPE(prob, popsize=n, center_learning_rate=0.5, stdev_learning_rate=0.1, stdev_init=1.0)
    s.step()
    X, f = s.population.values, s.population.evals[:, 0]
    mu, sg = s.status["center"], s.status["stdev"]
    # antithetic pairs mirror around mu (1 ulp of |x|)
    rows = torch.randint(0, n // 2, (64,), device=DEV)
    assert float((X[2 * rows] + X[2 * rows + 1] - 2 * mu).abs().max()) < 4e-6
    # fused fitness == stand-alone evaluation of the stored population
    f2 = ops.evaluate(ops.OBJ_RASTRIGIN, X)
    assert float(((f - f2).abs() / f2).max()) < 2e-6
    sub = torch.randint(0, n, (16,), device=DEV)
    close(N(f[sub]), O.rastrigin(N(X[sub])), rtol=3e-6)
    # sample moments of the perturbations
    z = ((X[0::2][:2000] - mu) / sg).double()
    assert abs(float(z.mean())) < 1e-3 and abs(float(z.std()) - 1) < 1e-3
    # ranks are a permutation of the utility table and sorted consistently with the fitnesses
    w = rank(f, "centered", higher_is_better=False)
    np.testing.assert_array_equal(N(torch.sort(w).values), np.arange(n, dtype=np.float32) / np.float32(n - 1) - np.float32(0.5))
    order = ops.argsort(f, descending=True)
    assert bool((f[order][:-1] >= f[order][1:]).all()) and bool((w[order][:-1] <= w[order][1:]).all())
    # gradient of the whole population == sum over 3 uneven shards; regenerated-from-Philox gradient agrees
    d = s._distribution
    whole = d._compute_gradients(X, w, "centered")
    acc = {k: torch.zeros(D, device=DEV) for k in ("mu", "sigma")}
    for lo, hi in ((0, 30_000), (30_000, 30_002), (30_002, n)):
        p = d.partial_gradients(X[lo:hi], w, lo, "centered")
        for k in acc:
            acc[k] += p[k]
    for k in acc:
        close(N(acc[k]), N(whole[k]), rtol=1e-3, atol=2e-7)
    regen = ops.grad_regen(ops.GRAD_SYMMETRIC, w, mu, sg, seed=prob._philox_seed, stream_id=prob._philox_stream - 1, row0=0,
                           scale_mu=1.0 / (n // 2), scale_sigma=1.0 / (n // 2))
    close(N(regen[0]), N(whole["mu"]), rtol=1e-3, atol=3e-7)
    close(N(regen[1]), N(whole["sigma"]), rtol=1e-3, atol=3e-7)
    # and a few generations make progress
    m0 = s.status["mean_eval"]
    s.run(5)
    assert s.status["mean_eval"] < m0


def test_metric_size_properties():
    """BASELINE metric size: PGPE, popsize 1 000 000 x dim 10 000 (40 GB population on one B200) -- size-independent properties."""
    free, _total = torch.cuda.mem_get_info()
    if free < 60e9:
        pytest.skip("needs 60 GB of free device memory")
    n, D = 1_000_000, 10_000
    prob = Problem("min", rastrigin, initial_bounds=(-5.12, 5.12), solution_length=D, device=DEV, seed=7)
    s = PGPE(prob, popsize=n, center_learning_rate=0.5, stdev_learning_rate=0.1, stdev_init=1.0)
    s.step()
    X, f = s.population.values, s.population.evals[:, 0]
    mu, sg = s.status["center"], s.status["stdev"]
    assert X.shape == (n, D) and bool(torch.isfinite(f).all())
    rows = torch.randint(0, n // 2, (256,), device=DEV)
    assert float((X[2 * rows] + X[2 * rows + 1] - 2 * mu).abs().max()) < 4e-6  # antithetic pairs
    sub = torch.randint(0, n, (64,), device=DEV)
    close(N(f[sub]), O.rastrigin(N(X[sub])), rtol=3e-6)  # fused fitness vs the float64 oracle on stored rows
    # the last rows / columns were written (no tail bug at the full size) and follow the Philox restatement
    tail = O.philox_population(N(mu), N(sg), 4, True, prob._philox_seed, 0, row0=n - 4)
    close(N(X[n - 4:]), tail, rtol=0, atol=5e-5)
    # ranking at N = 1 M with massive fp32 ties: bit-exact permutation of the utility table, stable order
    perm = torch.empty(n, dtype=torch.int64, device=DEV)
    w = ops.rank(f, "centered", False, perm=perm)
    np.testing.assert_array_equal(N(torch.sort(w).values), np.arange(n, dtype=np.float32) / np.float32(n - 1) - np.float32(0.5))
    np.testing.assert_array_equal(N(perm), O.argsort_for_ranking(N(f), False))
    assert len(torch.unique(f)) < n  # there ARE ties at this size (SURVEY section 7.2)
    # gradients: whole population == sum of 8 GPU-like shards; a full generation then moves the distribution
    d = s._distribution
    whole = d._compute_gradients(X, w, "centered")
    acc = {k: torch.zeros(D, device=DEV) for k in ("mu", "sigma")}
    for r in range(8):
        lo, hi = r * n // 8, (r + 1) * n // 8
        p = d.partial_gradients(X[lo:hi], w, lo, "centered")
        for k in acc:
            acc[k] += p[k]
    for k in acc:
        close(N(acc[k]), N(whole[k]), rtol=1e-3, atol=1e-7)
    s.step()
    assert not torch.equal(s.status["center"], mu) and bool(torch.isfinite(s.status["stdev"]).all())


# ------------------------------------------------------------------------------------------------ lazy (never materialised) population
@pytest.mark.parametrize("algo", ["pgpe", "pgpe_plain_nonsym", "snes", "cem"])
@pytest.mark.parametrize("graph", [False, True])
def test_lazy_population_matches_materialised(algo, graph):
    """`Problem(lazy_population=True)`: fitnesses come straight from the Philox counters (X = NULL) and the gradient kernel
    regenerates the samples.  The trajectory must agree with the materialised population to fp32 reduction-order noise."""
    from evotorch_b200.core import LazySolutionBatch

    def make(lazy):
        prob = Problem("min", rastrigin, initial_bounds=(-5.12, 5.12), solution_length=515, device=DEV, seed=33, lazy_population=lazy)
        if algo == "pgpe":
            s = PGPE(prob, popsize=2000, center_learning_rate=0.5, stdev_learning_rate=0.1, stdev_init=1.0)
        elif algo == "pgpe_plain_nonsym":
            s = PGPE(prob, popsize=2000, center_learning_rate=0.1, stdev_learning_rate=0.1, stdev_init=1.0, symmetric=False, optimizer=None,
                     ranking_method="nes", stdev_min=0.01, stdev_max=3.0)
        elif algo == "snes":
            s = SNES(prob, popsize=2000, stdev_init=2.0)
        else:
            s = CEM(prob, popsize=2000, parenthood_ratio=0.25, stdev_init=2.0, stdev_max_change=0.5)
        return s.enable_cuda_graph() if (graph and lazy) else s

    full, lazy = make(False), make(True)
    for gen in range(6):
        full.step()
        lazy.step()
        assert isinstance(lazy.population, LazySolutionBatch)
        # same population, bit for bit (both are pure functions of (seed, generation, row, column, mu, sigma)) while mu/sigma agree
        if gen == 0:
            assert torch.equal(full.population.values, lazy.population.values)
            assert torch.equal(full.population.evals, lazy.population.evals)
        # (a different summation order inside the gradient kernel; a flipped near-tie in the ranking amplifies it a little per generation)
        torch.testing.assert_close(lazy.status["center"], full.status["center"], rtol=0, atol=2e-4)
        torch.testing.assert_close(lazy.status["stdev"], full.status["stdev"], rtol=0, atol=2e-4)
    if graph:
        assert lazy._graph is not None
    # the regenerated values are consistent with the fitnesses the fused kernel produced
    vals = lazy.population.values
    torch.testing.assert_close(ops.evaluate(ops.OBJ_RASTRIGIN, vals), lazy.population.evals.view(-1), rtol=2e-6, atol=1e-3)
    sol = lazy.population[7]
    assert torch.equal(sol.values, vals[7]) and torch.equal(sol.evals, lazy.population.evals[7])
    with pytest.raises(ValueError):
        lazy.population.access_values()


def test_lazy_population_needs_builtin_objective():
    prob = Problem("min", lambda x: x.sum(-1), initial_bounds=(-1, 1), solution_length=16, device=DEV, vectorized=True, lazy_population=True)
    with pytest.raises(ValueError, match="lazy population"):
        SNES(prob, popsize=64, stdev_init=1.0).step()


def test_lazy_population_runs_where_the_matrix_cannot_exist():
    """popsize 8192 x dim 1M = 33 GB of samples per generation, never written.  Checks the footprint stays O(N + D) and the
    search makes progress."""
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    prob = Problem("min", sphere, initial_bounds=(-1.0, 1.0), solution_length=1_000_000, device=DEV, seed=5, lazy_population=True)
    s = PGPE(prob, popsize=8192, center_learning_rate=0.2, stdev_learning_rate=0.1, stdev_init=0.1)
    s.step()
    first = s.status["mean_eval"]
    for _ in range(3):
        s.step()
    assert s.status["mean_eval"] < first
    assert torch.cuda.max_memory_allocated() < 2 * 1024 ** 3


# ------------------------------------------------------------------------------------------------ peer exchange (single-rank exercise of the kernels)
@pytest.fixture
def single_rank_group(tmp_path):
    import torch.distributed as dist

    if dist.is_initialized():
        pytest.skip("a process group already exists")
    dist.init_process_group("gloo", init_method=f"file://{tmp_path}/pg", rank=0, world_size=1)
    yield
    dist.destroy_process_group()


def test_peer_exchange_push_kernel_single_rank(single_rank_group):
    """World size 1 runs the very same kernels as the multi-GPU exchange (fitness push + flag raise, flag wait, gradient push,
    slot reduction); the results must equal the plain kernels bit for bit, generation after generation, also from a CUDA graph.
    (2- and 8-GPU parity: scripts/check_peer_exchange.py, profiles/r01_peer_exchange_*.txt.)"""
    from evotorch_b200.peer import PeerExchange

    n, d = 4096, 515
    px = PeerExchange(n, d, torch.device(DEV), timeout_ns=2_000_000_000)
    g = torch.Generator(device="cpu").manual_seed(3)
    mu = (torch.rand(d, generator=g) * 4 - 2).to(DEV)
    sigma = (torch.rand(d, generator=g) + 0.5).to(DEV)
    X, Xp = torch.empty(n, d, device=DEV), torch.empty(n, d, device=DEV)
    f = torch.empty(n, device=DEV)

    def generation(gen):
        ops.sample_eval(ops.OBJ_RASTRIGIN, Xp, mu, sigma, n_rows=n, symmetric=True, seed=9, stream_id=gen, f=px.f_all[0:n])
        px.push_fitness(0, n)
        f_all = px.wait_fitness()
        w = ops.rank(f_all, "centered", False)
        ops.grad_push(ops.GRAD_SYMMETRIC, Xp, w, mu, sigma, scale_mu=2.0 / n, scale_sigma=2.0 / n, peer=px)
        return f_all, w, px.reduce_gradients()

    for gen in range(3):
        f_all, w, (gmu, gsig) = generation(gen)
        ops.sample_eval(ops.OBJ_RASTRIGIN, X, mu, sigma, n_rows=n, symmetric=True, seed=9, stream_id=gen, f=f)
        rmu, rsig = ops.grad(ops.GRAD_SYMMETRIC, X, w, mu, sigma, 2.0 / n, 2.0 / n)
        assert torch.equal(X, Xp) and torch.equal(f, f_all), gen
        assert torch.equal(gmu, rmu) and torch.equal(gsig, rsig), gen
    assert px._epochs.tolist() == [3, 3] and not px.timed_out()
    # the regenerating (lazy) producer and CUDA-graph replay
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        w = ops.rank(px.f_all, "centered", False)
        ops.grad_push(ops.GRAD_SYMMETRIC, None, w, mu, sigma, scale_mu=2.0 / n, scale_sigma=2.0 / n, peer=px, seed=9, stream_id=2, row0=0)
        px.reduce_gradients()
        side.synchronize()
        with torch.cuda.graph(graph, stream=side):
            ops.grad_push(ops.GRAD_SYMMETRIC, None, w, mu, sigma, scale_mu=2.0 / n, scale_sigma=2.0 / n, peer=px, seed=9, stream_id=2, row0=0)
            out = px.reduce_gradients()
    for _ in range(3):
        graph.replay()
    torch.cuda.synchronize()
    torch.testing.assert_close(out[0], rmu, rtol=0, atol=2e-6)
    torch.testing.assert_close(out[1], rsig, rtol=0, atol=2e-6)
    assert px._epochs.tolist() == [3, 7] and not px.timed_out()
    px.close()


def test_peer_wait_times_out_instead_of_hanging(single_rank_group):
    from evotorch_b200.peer import PeerExchange

    px = PeerExchange(64, 8, torch.device(DEV), timeout_ns=20_000_000)  # 20 ms
    px.wait_fitness()  # nobody raised the flag
    assert px.timed_out()
    px.close()


@pytest.mark.parametrize("mode", ["eager", "graph", "lazy_graph"])
def test_checkpoint_resume_is_bit_identical_on_gpu(tmp_path, mode):
    """A searcher pickled mid-run (PicklingLogger(checkpoint=True)) continues exactly like the uninterrupted one: the
    sampler is counter based, the captured CUDA graph is dropped from the pickle and re-captured after loading."""
    from evotorch_b200.logging import PicklingLogger

    def make():
        prob = Problem("min", rastrigin, initial_bounds=(-5.12, 5.12), solution_length=200, device=DEV, seed=4, lazy_population=mode.startswith("lazy"))
        s = PGPE(prob, popsize=500, center_learning_rate=0.4, stdev_learning_rate=0.1, stdev_init=1.0)
        return s.enable_cuda_graph() if mode.endswith("graph") else s

    straight = make()
    straight.run(11)
    s = make()
    logger = PicklingLogger(s, interval=5, directory=str(tmp_path), prefix="gpu", verbose=False, checkpoint=True)
    s.run(5)
    data = logger.unpickle_last_file()
    assert data["center"].device.type == "cpu" and torch.equal(data["center"], s.status["center"].cpu())
    resumed = PicklingLogger.resume(logger.last_file_name)
    assert resumed._graph is None and resumed.step_count == 5
    resumed.run(6)
    assert (resumed._graph is not None) == mode.endswith("graph")
    assert torch.equal(resumed.status["center"], straight.status["center"])
    assert torch.equal(resumed.status["stdev"], straight.status["stdev"])
    assert resumed.status["mean_eval"] == straight.status["mean_eval"]


def _searcher_variants():
    import importlib.util

    spec = importlib.util.spec_from_file_location("searcher_variants", os.path.join(os.path.dirname(__file__), "golden", "searcher_variants.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.mark.parametrize("tag", sorted(t for t in _searcher_variants().VARIANTS if not t.startswith("xnes")))
def test_searcher_option_variants_through_the_cuda_kernels(tag):
    """The option variants of `tests/golden/searcher_variants.py` (SGD with momentum, stdev bounds, no max-change, ClipUp config,
    normalized / linear / raw ranking, SNES without learning-rate scaling, Adam on SNES, CEM bounds / maximisation): the
    reference's recorded populations go through the CUDA rank -> gradient -> update kernels generation by generation."""
    mod = _searcher_variants()
    algo, d, sense, fn, kw, gens = mod.VARIANTS[tag]
    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "searcher_variants_golden.npz"))
    mu, sg, X, f = (gold[f"{tag}/{k}"] for k in ("mu", "sigma", "X", "f"))
    kw = {k: v for k, v in kw.items() if k not in ("stdev_init", "radius_init")}
    prob = Problem(sense, mod.objective(fn), initial_bounds=(-5.12, 5.12), solution_length=d, device=DEV, seed=11, vectorized=True)
    s = {"PGPE": PGPE, "SNES": SNES, "CEM": CEM}[algo](prob, center_init=C(mu[0]), stdev_init=C(sg[0]), **kw)
    s.step()
    assert len(s.population) == X.shape[1]
    for t in range(gens - 1):
        s._population.set_values(C(X[t]))
        s._population.set_evals(C(f[t]))
        s.step()
        close(N(s.status["center"]), mu[t + 1], rtol=2e-5, atol=3e-6)
        close(N(s.status["stdev"]), sg[t + 1], rtol=2e-5, atol=3e-6)
