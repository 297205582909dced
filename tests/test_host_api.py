"""The host-side mirror of the reference API on CPU tensors (BASELINE config 1 path): seeded trajectories of the package
must reproduce the REAL reference's trajectories recorded in tests/golden (same torch RNG stream => same populations)."""

import os
import math

import numpy as np
import pytest
import torch

from evotorch_b200 import Problem, SolutionBatch
from evotorch_b200.algorithms import CEM, PGPE, SNES, XNES
from evotorch_b200.distributions import ExpSeparableGaussian, SeparableGaussian, SymmetricSeparableGaussian
from evotorch_b200.logging import PandasLogger, StdOutLogger
from evotorch_b200.optimizers import SGD, Adam, ClipUp, get_optimizer_class
from evotorch_b200.tools import modify_tensor, rank


def rastrigin(x: torch.Tensor) -> torch.Tensor:
    n = x.shape[1]
    return 10 * n + torch.sum((x**2) - 10 * torch.cos(2 * np.pi * x), 1)


def sphere(x: torch.Tensor) -> torch.Tensor:
    return torch.sum(x**2, dim=-1)


def T(x):
    return torch.as_tensor(np.asarray(x), dtype=torch.float32)


MAKERS = {
    "pgpe": (lambda p: PGPE(p, popsize=32, center_learning_rate=0.5, stdev_learning_rate=0.1, stdev_init=1.0), 8, "min", rastrigin),
    "pgpe_max": (lambda p: PGPE(p, popsize=32, center_learning_rate=0.5, stdev_learning_rate=0.1, stdev_init=1.0), 8, "max", rastrigin),
    "pgpe_nonsym_adam": (lambda p: PGPE(p, popsize=30, center_learning_rate=0.05, stdev_learning_rate=0.1, stdev_init=1.0,
                                         symmetric=False, optimizer="adam"), 8, "min", rastrigin),
    "pgpe_nes_rank": (lambda p: PGPE(p, popsize=32, center_learning_rate=0.3, stdev_learning_rate=0.1, radius_init=4.0,
                                      ranking_method="nes", optimizer=None, stdev_min=0.01, stdev_max=2.0), 8, "min", rastrigin),
    "snes": (lambda p: SNES(p, popsize=24, stdev_init=2.0), 8, "min", rastrigin),
    "snes_clipup": (lambda p: SNES(p, popsize=24, stdev_init=2.0, optimizer="clipup", center_learning_rate=0.2,
                                    stdev_max_change=0.3), 8, "min", rastrigin),
    "cem": (lambda p: CEM(p, popsize=40, parenthood_ratio=0.25, stdev_init=2.0, stdev_max_change=0.5), 8, "min", rastrigin),
}


@pytest.mark.parametrize("tag", sorted(MAKERS))
def test_cpu_trajectory_matches_reference(golden, tag):
    make, D, sense, fn = MAKERS[tag]
    prob = Problem(sense, fn, initial_bounds=(-5.12, 5.12), solution_length=D, vectorized=True, seed=11, dtype=torch.float32)
    s = make(prob)
    mus, sigs = golden[f"traj/{tag}/mu"], golden[f"traj/{tag}/sigma"]
    for t in range(len(mus)):
        s.step()
        np.testing.assert_allclose(s.status["center"].numpy(), mus[t], rtol=1e-5, atol=2e-6)
        np.testing.assert_allclose(s.status["stdev"].numpy(), sigs[t], rtol=1e-5, atol=2e-6)
        np.testing.assert_allclose(s.population.values.numpy(), golden[f"traj/{tag}/X"][t], rtol=1e-5, atol=5e-6)
        np.testing.assert_allclose(s.population.evals[:, 0].numpy(), golden[f"traj/{tag}/f"][t], rtol=1e-5, atol=1e-4)
    assert s.step_count == len(mus) and s.status["iter"] == len(mus)
    for key in ("best", "worst", "best_eval", "worst_eval", "center", "stdev", "mean_eval", "pop_best", "pop_best_eval", "median_eval"):
        assert key in s.status
    assert math.isfinite(s.status["mean_eval"]) and math.isfinite(s.status["pop_best_eval"])


def test_xnes_cpu_trajectory(golden):
    prob = Problem("min", sphere, initial_bounds=(-5.12, 5.12), solution_length=5, vectorized=True, seed=11, dtype=torch.float32)
    s = XNES(prob, popsize=16, stdev_init=1.5)
    for t in range(5):
        s.step()
        np.testing.assert_allclose(s.status["center"].numpy(), golden["traj/xnes/mu"][t], rtol=2e-4, atol=2e-5)
        np.testing.assert_allclose(s.status["stdev"].numpy(), golden["traj/xnes/sigma"][t], rtol=2e-4, atol=2e-5)


def test_readme_snes_config1_runs_on_cpu():
    # BASELINE.json configs[0]: SNES, Rastrigin, dim=100, popsize=1000, CPU (reference README.md:76-116)
    prob = Problem("min", rastrigin, initial_bounds=(-5.12, 5.12), solution_length=100, vectorized=True, seed=1)
    s = SNES(prob, popsize=1000, stdev_init=10.0)
    log = PandasLogger(s)
    s.run(30)
    df = log.to_dataframe()
    assert len(df) == 30 and df["mean_eval"].iloc[-1] < df["mean_eval"].iloc[0]


@pytest.mark.parametrize("method", ["centered", "linear", "nes", "normalized", "raw"])
@pytest.mark.parametrize("name", ["appxB", "rand257", "rand1000", "tied600"])
def test_rank_cpu_matches_reference(golden, method, name):
    f = T(golden[f"rank/{name}/f"])
    for hib in (True, False):
        got = rank(f, method, higher_is_better=hib).numpy()
        np.testing.assert_allclose(got, golden[f"rank/{name}/{method}/{int(hib)}"], rtol=3e-6, atol=3e-7)
    with pytest.raises(KeyError):
        rank(f, "nope", higher_is_better=True)


def test_distribution_api_and_errors(golden):
    mu, sg = T(golden["grad/mu"]), T(golden["grad/sigma"])
    d = SymmetricSeparableGaussian({"mu": mu, "sigma": sg, "divide_mu_grad_by": "num_directions", "divide_sigma_grad_by": "num_directions"})
    g = d.compute_gradients(T(golden["grad/Xsym"]), T(golden["grad/fsym"]), objective_sense="min", ranking_method="centered")
    np.testing.assert_allclose(g["mu"].numpy(), golden["grad/sym/centered/min/num_directions/mu"], rtol=2e-4, atol=2e-6)
    np.testing.assert_allclose(g["sigma"].numpy(), golden["grad/sym/centered/min/num_directions/sigma"], rtol=2e-4, atol=2e-6)
    with pytest.raises(ValueError):
        d.compute_gradients(T(golden["grad/Xsym"]), T(golden["grad/fsym"]), objective_sense="up")
    with pytest.raises(ValueError):
        d.compute_gradients(T(golden["grad/Xsym"]), T(golden["grad/fsym"][:-1]), objective_sense="min")
    with pytest.raises(ValueError):
        d.sample(out=torch.empty(4, 3))
    with pytest.raises(ValueError):
        d.sample(out=torch.empty(5, 16))  # odd number of rows for a symmetric distribution
    with pytest.raises(ValueError):
        d.sample(4, out=torch.empty(4, 16))
    with pytest.raises(ValueError):
        SeparableGaussian({"mu": mu, "sigma": sg, "bogus": 1})
    x = d.sample(6, generator=torch.Generator().manual_seed(0))
    np.testing.assert_allclose((x[0::2] + x[1::2]).numpy(), np.broadcast_to(2 * mu.numpy(), (3, 16)), atol=1e-5)
    upd = d.update_parameters(g, learning_rates={"mu": 0.1, "sigma": 0.2})
    assert upd is not d and torch.equal(d.mu, mu)
    np.testing.assert_allclose(upd.mu.numpy(), (mu + 0.1 * g["mu"]).numpy(), rtol=1e-6)
    e = ExpSeparableGaussian({"mu": mu, "sigma": sg})
    ge = e.compute_gradients(T(golden["grad/Xns"]), T(golden["grad/fns"]), objective_sense="max", ranking_method="centered")
    np.testing.assert_allclose(ge["sigma"].numpy(), golden["grad/exp/centered/max/sigma"], rtol=2e-4, atol=5e-5)
    for ratio in (0.5, 0.25, 0.1):
        c = SeparableGaussian({"mu": mu, "sigma": sg, "parenthood_ratio": ratio})
        gc = c.compute_gradients(T(golden["grad/Xns"]), T(golden["grad/fns"]), objective_sense="min", ranking_method=None)
        np.testing.assert_allclose(gc["mu"].numpy(), golden[f"grad/cem/{ratio}/min/mu"], rtol=1e-4, atol=2e-6)
        np.testing.assert_allclose(gc["sigma"].numpy(), golden[f"grad/cem/{ratio}/min/sigma"], rtol=1e-4, atol=5e-6)


def test_partial_gradients_add_up(golden):
    mu, sg = T(golden["grad/mu"]), T(golden["grad/sigma"])
    X, f = T(golden["grad/Xsym"]), T(golden["grad/fsym"])
    for cls, extra, method in ((SymmetricSeparableGaussian, {"divide_mu_grad_by": "num_directions", "divide_sigma_grad_by": "num_directions"}, "nes"),
                               (SeparableGaussian, {"parenthood_ratio": 0.25}, "raw"), (ExpSeparableGaussian, {}, "centered")):
        d = cls({"mu": mu, "sigma": sg, **extra})
        w = rank(f, method, higher_is_better=False)
        whole = d._compute_gradients(X, w, method)
        parts = [d.partial_gradients(X[a:b], w, a, method) for a, b in ((0, 20), (20, 44), (44, 64))]
        summed = {k: sum(p[k] for p in parts) for k in parts[0]}
        fin = d.finalize_gradients(summed, 64)
        for k in whole:
            np.testing.assert_allclose(fin[k].numpy(), whole[k].numpy(), rtol=2e-5, atol=2e-6)


def test_optimizers_cpu(golden):
    grads = golden["opt/grads"]
    for i in range(4):
        ss, mom, ms = golden[f"opt/clipup/{i}/cfg"]
        opt = ClipUp(solution_length=12, dtype="float32", stepsize=ss, momentum=mom, max_speed=None if ms < 0 else ms)
        got = np.stack([opt.ascent(T(g)).numpy() for g in grads])
        np.testing.assert_allclose(got, golden[f"opt/clipup/{i}/steps"], rtol=2e-6, atol=2e-7)
    opt = Adam(solution_length=12, dtype="float32", stepsize=0.05)
    np.testing.assert_allclose(np.stack([opt.ascent(T(g)).numpy() for g in grads]), golden["opt/adam/0/steps"], rtol=5e-6, atol=1e-7)
    opt = SGD(solution_length=12, dtype="float32", stepsize=0.1, momentum=0.8)
    np.testing.assert_allclose(np.stack([opt.ascent(T(g)).numpy() for g in grads]), golden["opt/sgd/1/steps"], rtol=2e-6, atol=1e-7)
    # API validation mirrored from the reference's tests/test_optimizers.py:25-43, :115-138
    with pytest.raises(ValueError):
        ClipUp(solution_length=3, dtype="float32", stepsize=-1.0)
    with pytest.raises(ValueError):
        ClipUp(solution_length=3, dtype="float32", stepsize=0.1, momentum=1.5)
    with pytest.raises(ValueError):
        Adam(solution_length=3, dtype="float32", beta1=0.9)
    c = ClipUp(solution_length=3, dtype="float32", stepsize=0.1)
    assert c.param_groups[0]["max_speed"] == pytest.approx(0.2)
    c.param_groups[0]["lr"] = 0.3
    assert c.param_groups[0]["lr"] == 0.3
    with pytest.raises(ValueError):
        c.param_groups[0]["momentum"] = 2.0
    assert get_optimizer_class("clipup") is ClipUp and get_optimizer_class("adam") is Adam and get_optimizer_class("sga") is SGD
    assert get_optimizer_class("clipup", {"max_speed": 0.7})(solution_length=2, dtype="float32", stepsize=0.1).param_groups[0]["max_speed"] == 0.7
    with pytest.raises(ValueError):
        get_optimizer_class("nope")


def test_modify_tensor_known_answers():
    x, t = T([10, 11, 12]), T([0, 21, 22])
    assert modify_tensor(x, t, lb=5).tolist() == [5, 21, 22]
    assert modify_tensor(x, t, lb=5, ub=20).tolist() == [5, 20, 20]
    assert modify_tensor(x, t, max_change=0.5).tolist() == [5, 16.5, 18]
    assert modify_tensor(x, t, lb=7, ub=17, max_change=0.5).tolist() == [7, 16.5, 17]
    with pytest.raises(IndexError):
        modify_tensor(x, t, lb=T([1, 2]))


def test_solution_batch_semantics():
    prob = Problem("max", sphere, initial_bounds=(-1, 1), solution_length=4, vectorized=True, seed=3, eval_data_length=2)
    b = SolutionBatch(prob, 6)
    assert b.values.shape == (6, 4) and b.evals.shape == (6, 3) and torch.isnan(b.evals).all()
    assert float(b.values.min()) >= -1 and float(b.values.max()) <= 1
    prob.evaluate(b)
    assert not torch.isnan(b.evals[:, 0]).any() and torch.isnan(b.evals[:, 1:]).all()
    assert int(b.argbest()) == int(torch.argmax(b.evals[:, 0])) and int(b.argworst()) == int(torch.argmin(b.evals[:, 0]))
    assert b.argsort().tolist() == torch.argsort(b.evals[:, 0], descending=True, stable=True).tolist()
    v = b.access_values(keep_evals=True)
    assert not torch.isnan(b.evals[:, 0]).any()
    v = b.access_values()
    assert torch.isnan(b.evals).all() and v.data_ptr() == b.values.data_ptr()
    b.set_evals(torch.arange(6.0), torch.ones(6, 2))
    assert b.evals[:, 0].tolist() == [0, 1, 2, 3, 4, 5] and b[2].evals.tolist() == [2, 1, 1]
    s = b[5].clone()
    b.set_values(torch.zeros(6, 4))
    assert torch.isnan(b.evals).all() and s.evals[0] == 5 and s.is_evaluated and not b[0].is_evaluated
    pieces = b.split(4)
    assert [len(p) for p in pieces] == [2, 2, 1, 1] and pieces[0].values.data_ptr() == b.values.data_ptr()
    assert len(SolutionBatch.cat(pieces)) == 6
    with pytest.raises(ValueError):
        b.set_evals(torch.zeros(5))
    with pytest.warns(UserWarning, match="no Ray actors"):  # accepted and mapped to this process / the torch.distributed ranks
        assert Problem("min", sphere, solution_length=3, num_actors=4).num_actors == 0
    with pytest.raises(ValueError):
        Problem("sideways", sphere, solution_length=3)
    bounded = Problem("min", sphere, bounds=(-1, 1), solution_length=3, vectorized=True)
    with pytest.raises(ValueError):
        SNES(bounded, stdev_init=1.0)
    with pytest.raises(ValueError):
        PGPE(prob, popsize=7, center_learning_rate=0.1, stdev_learning_rate=0.1, stdev_init=1.0)
    with pytest.raises(ValueError):
        PGPE(prob, popsize=8, center_learning_rate=0.1, stdev_learning_rate=0.1)


def test_builtin_objectives_on_cpu(golden):
    from evotorch_b200.objectives import ackley, rastrigin as rb, sphere as sb

    X = T(golden["grad/Xsym"])
    np.testing.assert_allclose(rb(X).numpy(), golden["grad/fsym"], rtol=1e-6)
    np.testing.assert_allclose(sb(X).numpy(), (X**2).sum(1).numpy(), rtol=1e-6)
    assert ackley(torch.zeros(2, 5)).abs().max() < 1e-5
    assert rb.evok_objective_id == 2 and rb.__evotorch_vectorized__
    prob = Problem("min", rb, initial_bounds=(-5.12, 5.12), solution_length=8, seed=11)
    s = PGPE(prob, popsize=32, center_learning_rate=0.5, stdev_learning_rate=0.1, stdev_init=1.0)
    s.run(3)
    np.testing.assert_allclose(s.status["center"].numpy(), golden["traj/pgpe/mu"][2], rtol=1e-5, atol=2e-6)


def test_stdout_logger(capsys):
    prob = Problem("min", sphere, initial_bounds=(-1, 1), solution_length=4, vectorized=True, seed=3)
    s = SNES(prob, stdev_init=1.0)
    StdOutLogger(s, interval=2)
    s.run(4)
    out = capsys.readouterr().out
    assert out.count("iter") == 2 and "mean_eval" in out


def test_cmaes_cpu_trajectory_matches_reference(golden):
    from evotorch_b200.algorithms import CMAES

    prob = Problem("min", sphere, initial_bounds=(-3, 3), solution_length=6, vectorized=True, seed=3, dtype=torch.float32)
    c = CMAES(prob, stdev_init=1.0, popsize=12)
    np.testing.assert_allclose(c.weights.numpy(), golden["cmaes/weights"], rtol=2e-6, atol=1e-8)
    consts = golden["cmaes/consts"]
    np.testing.assert_allclose([c.mu_eff, c.c_sigma, c.damp_sigma, c.c_c, c.c_1, c.c_mu, c.decompose_C_freq], consts, rtol=2e-6)
    for t in range(6):
        c.step()
        np.testing.assert_allclose(c.m.numpy(), golden["cmaes/m"][t], rtol=1e-5, atol=2e-6)
        np.testing.assert_allclose(float(c.sigma), golden["cmaes/sigma"][t][0], rtol=1e-5)
        np.testing.assert_allclose(c.C.numpy(), golden["cmaes/C"][t], rtol=1e-5, atol=2e-6)
        np.testing.assert_allclose(c.A.numpy(), golden["cmaes/A"][t], rtol=1e-5, atol=2e-6)
        np.testing.assert_allclose(c.p_sigma.numpy(), golden["cmaes/p_sigma"][t], rtol=1e-5, atol=2e-6)
        np.testing.assert_allclose(c.p_c.numpy(), golden["cmaes/p_c"][t], rtol=1e-5, atol=2e-6)
    assert "stepsize" in c.status and "center" in c.status and c.status["iter"] == 6
    big = CMAES(Problem("min", sphere, initial_bounds=(-3, 3), solution_length=1024, vectorized=True, seed=3), stdev_init=1.0, popsize=4096)
    ref = golden["cmaes/cfg3_consts"]
    np.testing.assert_allclose([big.mu_eff, big.c_sigma, big.damp_sigma, big.c_c, big.c_1, big.c_mu, big.decompose_C_freq,
                                float(torch.sum(big.weights))], ref, rtol=5e-6)
    sep = CMAES(Problem("min", sphere, initial_bounds=(-3, 3), solution_length=20, vectorized=True, seed=3), stdev_init=1.0, separable=True)
    sep.step()
    m0 = sep.status["mean_eval"]
    sep.run(40)
    assert sep.status["mean_eval"] < m0 and sep.C.ndim == 1


def test_policy_cpu_matches_reference(golden):
    from evotorch_b200.neuroevolution import Policy, count_parameters, fill_parameters, parameter_vector

    net = torch.nn.Sequential(torch.nn.Linear(11, 8), torch.nn.Tanh(), torch.nn.Linear(8, 3))
    pol = Policy(net)
    assert pol.parameter_length == int(golden["policy/dims"][3]) == count_parameters(net)
    pol.set_parameters(T(golden["policy/params"]))
    np.testing.assert_allclose(pol(T(golden["policy/obs"])).numpy(), golden["policy/act"], rtol=1e-5, atol=2e-6)
    # one shared flat vector == filling the module (the reference's tests/test_net.py idea)
    flat = T(golden["policy/params"][0])
    pol.set_parameters(flat)
    fill_parameters(net, flat)
    np.testing.assert_allclose(pol(T(golden["policy/obs"])).numpy(), net(T(golden["policy/obs"])).detach().numpy(), rtol=1e-6, atol=1e-6)
    assert torch.equal(parameter_vector(net), flat)
    with pytest.raises(ValueError):
        pol.set_parameters(torch.zeros(5))
    with pytest.raises(ValueError):
        Policy(net)(torch.zeros(2, 11))


def test_searcher_pickles_and_resumes_identically():
    import pickle

    prob = Problem("min", sphere, initial_bounds=(-1, 1), solution_length=5, seed=3, vectorized=True)
    s = PGPE(prob, popsize=10, center_learning_rate=0.1, stdev_learning_rate=0.1, stdev_init=1.0)
    s.run(3)
    clone = pickle.loads(pickle.dumps(s))  # the reference checkpoints by pickling (logging.py:369-376, tools/cloning.py:258)
    s.run(2)
    clone.run(2)
    assert torch.equal(s.status["center"], clone.status["center"]) and torch.equal(s.status["stdev"], clone.status["stdev"])


def test_bench_reference_arm_prints_one_json_line():
    import json
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--cpu-sizes", "64,128,256", "--cpu-budget-s", "2", "--dim", "200", "--popsize", "1000"], capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "dtype", "data",
                "config", "impl", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["value"] > 0
    lin = d["cpu_baseline"]["linearity"]  # SURVEY 8(d): several population sizes, a fitted line, its residual, an extrapolated value
    assert [r["popsize"] for r in d["cpu_baseline"]["samples"]] == [64, 128, 256] and lin["max_rel_residual"] >= 0
    assert abs(1.0 / lin["extrapolated_s_per_generation"] - d["value"]) < 1e-9 * d["value"] and d["cpu_baseline"]["extrapolated"] is True


def _load_dir(path):
    return {f[:-4]: np.load(os.path.join(path, f)) for f in sorted(os.listdir(path))}


def test_bench_dump_outputs_are_float_bounded_and_seeded(tmp_path, monkeypatch):
    import bench
    from evotorch_b200 import objectives

    def run():
        s = PGPE(Problem("min", objectives.rastrigin, initial_bounds=(-5.12, 5.12), solution_length=40, device="cpu", seed=0), popsize=600,
                 center_learning_rate=0.5, stdev_learning_rate=0.1, stdev_init=1.0)
        s.run(3)
        return s

    s = run()
    bench.dump_outputs(s, str(tmp_path / "a"))
    bench.dump_outputs(run(), str(tmp_path / "b"))
    a, b = _load_dir(tmp_path / "a"), _load_dir(tmp_path / "b")
    assert sorted(a) == ["center", "fitness", "mean_eval", "population_rows", "stdev"]
    for name in a:
        assert a[name].dtype in (np.float32, np.float64), name
        np.testing.assert_array_equal(a[name], b[name], err_msg=name)
    np.testing.assert_array_equal(a["center"], s.status["center"].numpy())
    np.testing.assert_array_equal(a["fitness"], s.population.evals[:, 0].numpy())
    X = s.population.values.numpy()
    assert a["population_rows"].shape == (512, 40) and all((X == r).all(1).any() for r in a["population_rows"])
    # a smaller budget samples the fitnesses and rows instead of exceeding it
    monkeypatch.setattr(bench, "DUMP_BYTES", 4000)
    bench.dump_outputs(s, str(tmp_path / "c"))
    c = _load_dir(tmp_path / "c")
    assert sum(v.nbytes for v in c.values()) <= 4000 and 0 < len(c["fitness"]) < 600 and len(c["population_rows"]) >= 1
    assert np.isin(c["fitness"], a["fitness"]).all()


@pytest.mark.gpu
def test_bench_dump_outputs_of_the_timed_path(tmp_path):
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    dumps = []
    for tag in ("a", "b"):
        r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "2", "--warmup", "1", "--popsize", "20000", "--dim",
                            "1000", "--no-cpu-baseline", "--no-e2e", "--no-other-configs", "--dump-outputs", str(tmp_path / tag)],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        dumps.append(_load_dir(tmp_path / tag))
    a, b = dumps
    assert sorted(a) == ["center", "fitness", "mean_eval", "population_rows", "stdev"]
    assert a["fitness"].shape == (20000,) and a["population_rows"].shape == (512, 1000) and a["center"].shape == (1000,)
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    for name in a:
        assert a[name].dtype in (np.float32, np.float64) and np.isfinite(a[name]).all(), name
        np.testing.assert_allclose(a[name], b[name], rtol=1e-6, atol=1e-6, err_msg=name)


# ------------------------------------------------------------------------------------------------ pickling / checkpoints (SURVEY 8 f4)
def test_pickling_logger_files_items_and_resume(tmp_path, capsys):
    import pickle

    from evotorch_b200.logging import PicklingLogger

    def make():
        prob = Problem("min", rastrigin, initial_bounds=(-5.12, 5.12), solution_length=12, vectorized=True, seed=11)
        return PGPE(prob, popsize=40, center_learning_rate=0.3, stdev_learning_rate=0.1, stdev_init=1.0)

    straight = make()
    straight.run(9)

    s = make()
    logger = PicklingLogger(s, interval=3, directory=str(tmp_path / "ckpt"), prefix="run", items_to_save=("center", "stdev", "best", "nope"),
                            checkpoint=True)
    s.run(4)
    files = sorted(os.listdir(tmp_path / "ckpt"))
    assert files == ["run_generation000003.pickle", "run_generation000004.pickle"]  # every 3rd generation + the end of the run
    assert logger.last_generation == 4 and logger.last_file_name.endswith("run_generation000004.pickle")
    assert "Saved to" in capsys.readouterr().out
    data = logger.unpickle_last_file()
    assert set(data) >= {"center", "stdev", "best", "beginning_time", "now", "elapsed", "searcher"} and "nope" not in data
    assert torch.equal(data["center"], s.status["center"]) and data["center"].device.type == "cpu"
    assert data["best"].shape == (12,)  # a Solution is stored as its decision values
    # resume from the generation-3 file: the continued run must be the uninterrupted run, bit for bit
    resumed = PicklingLogger.resume(str(tmp_path / "ckpt" / "run_generation000003.pickle"))
    assert resumed.step_count == 3
    resumed.run(6)
    assert torch.equal(resumed.status["center"], straight.status["center"])
    assert torch.equal(resumed.status["stdev"], straight.status["stdev"])
    # the resumed searcher keeps checkpointing through its (re-bound) logger
    assert "run_generation000009.pickle" in os.listdir(tmp_path / "ckpt")
    # plain pickles of problem and searcher round-trip too
    clone = pickle.loads(pickle.dumps(s))
    clone.step(); s.step()
    assert torch.equal(clone.status["center"], s.status["center"])
    with pytest.raises(KeyError):
        lg = PicklingLogger(s, interval=1, directory=str(tmp_path / "plain"), prefix="p", verbose=False)
        PicklingLogger.resume(lg.save())


def test_lazy_population_and_peer_exchange_fail_loudly_without_their_prerequisites():
    """Neither feature has a CPU stand-in: a lazy population needs the fused Philox sampler (CUDA float32 + built-in objective),
    a peer exchange needs an initialised process group."""
    from evotorch_b200.core import LazySolutionBatch
    from evotorch_b200.objectives import rastrigin as builtin_rastrigin
    from evotorch_b200.peer import PeerExchange

    prob = Problem("min", builtin_rastrigin, initial_bounds=(-1, 1), solution_length=8, lazy_population=True, seed=1)
    searcher = SNES(prob, popsize=10, stdev_init=1.0)
    with pytest.raises(ValueError, match="lazy population"):
        searcher.step()
    batch = LazySolutionBatch(prob, 10)
    assert len(batch) == 10 and batch.values_shape == (10, 8) and "LazySolutionBatch" in repr(batch)
    with pytest.raises(ValueError):
        batch.values  # not sampled yet
    with pytest.raises(ValueError):
        batch.set_values(torch.zeros(10, 8))
    with pytest.raises(RuntimeError, match="process group"):
        PeerExchange(10, 8, torch.device("cpu"))


def test_gradient_hooks_randint_and_misc_problem_api():
    """core.py:2204-2226 (before / after grad hooks around sample_and_compute_gradients), tensormaker.py:681 (make_randint),
    core.py:3303 (is_on_cpu), core.py:4304 (SolutionBatch.utils)."""
    prob = Problem("min", rastrigin, initial_bounds=(-5.12, 5.12), solution_length=6, vectorized=True, seed=2)
    calls = []
    prob.before_grad_hook.append(lambda: calls.append("before"))
    prob.after_grad_hook.append(lambda results: {"grad_calls": len(calls), "n": results[0]["num_solutions"]})
    dist = SymmetricSeparableGaussian({"mu": torch.zeros(6), "sigma": torch.ones(6), "divide_mu_grad_by": "num_directions",
                                       "divide_sigma_grad_by": "num_directions"})
    out = prob.sample_and_compute_gradients(dist, 20, ranking_method="centered")
    assert calls == ["before"] and prob.status == {"grad_calls": 1, "n": 20} and set(out[0]["gradients"]) == {"mu", "sigma"}
    assert prob.is_on_cpu() and prob.kill_actors() is None
    with pytest.raises(NotImplementedError):
        prob.all_remote_problems
    r = prob.make_randint(1000, n=7)
    assert r.dtype == prob.dtype and r.min() >= 0 and r.max() <= 6 and set(r.tolist()) == set(range(7))
    ri = prob.make_randint(5, 3, n=4, dtype=torch.int64)
    assert ri.shape == (5, 3) and ri.dtype == torch.int64 and int(ri.max()) < 4
    batch = SolutionBatch(prob, popsize=9)
    prob.evaluate(batch)
    u = batch.utils(ranking_method="centered")
    assert u.shape == (9, 1) and torch.equal(u[:, 0], batch.utility(0, ranking_method="centered"))


def _shifted_to_maximise(x):
    return -torch.sum((x - 1.5) ** 2 * torch.arange(1, x.shape[-1] + 1, dtype=x.dtype), dim=-1)


@pytest.mark.parametrize("tag", ["separable", "no_active", "csa_squared_bounds", "maximise_default_popsize", "ratios_no_limit"])
def test_cmaes_option_variants_match_reference(tag):
    """Every CMA-ES option of the reference (cmaes.py:90-606): separable covariance, no active weights, squared CSA with
    step-size bounds, maximisation with the default population size, hyper-parameter ratios without the decomposition limit.
    Same seed -> same torch-generator stream on CPU, so the trajectories are compared step by step."""
    import os

    from evotorch_b200.algorithms import CMAES

    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "cmaes_variants_golden.npz"))
    cfg = {
        "separable": ("min", sphere, 8, dict(stdev_init=1.0, popsize=14, separable=True)),
        "no_active": ("min", sphere, 6, dict(stdev_init=0.7, popsize=10, active=False)),
        "csa_squared_bounds": ("min", sphere, 6, dict(stdev_init=1.0, popsize=12, csa_squared=True, stdev_min=0.6, stdev_max=1.1)),
        "maximise_default_popsize": ("max", _shifted_to_maximise, 7, dict(stdev_init=2.0)),
        "ratios_no_limit": ("min", sphere, 5, dict(stdev_init=1.0, popsize=16, c_1_ratio=0.5, c_mu_ratio=2.0, c_sigma_ratio=1.5, damp_sigma_ratio=0.8,
                                                   c_c_ratio=1.2, c_m=0.9, limit_C_decomposition=False)),
    }[tag]
    sense, fn, d, kw = cfg
    prob = Problem(sense, fn, initial_bounds=(-3, 3), solution_length=d, vectorized=True, seed=11, dtype=torch.float32)
    c = CMAES(prob, **kw)
    assert c.popsize == int(gold[f"{tag}/popsize"])
    for t in range(7):
        c.step()
        np.testing.assert_allclose(c.population.evals[:, 0].numpy(), gold[f"{tag}/f"][t], rtol=2e-5, atol=2e-5)
        np.testing.assert_allclose(c.m.numpy(), gold[f"{tag}/m"][t], rtol=2e-5, atol=5e-6)
        np.testing.assert_allclose(float(c.sigma), float(gold[f"{tag}/sigma"][t]), rtol=2e-5)
        np.testing.assert_allclose(c.C.numpy(), gold[f"{tag}/C"][t], rtol=5e-5, atol=5e-6)
        np.testing.assert_allclose(c.p_sigma.numpy(), gold[f"{tag}/p_sigma"][t], rtol=5e-5, atol=5e-6)
        np.testing.assert_allclose(c.p_c.numpy(), gold[f"{tag}/p_c"][t], rtol=5e-5, atol=5e-6)


def _variant_table():
    import importlib.util

    spec = importlib.util.spec_from_file_location("searcher_variants", os.path.join(os.path.dirname(__file__), "golden", "searcher_variants.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.mark.parametrize("tag", sorted(_variant_table().VARIANTS))
def test_searcher_option_variants_match_reference(tag):
    """One seeded reference trajectory per searcher option not covered by `reference_golden.npz`: SGD with momentum, radius_init,
    stdev bounds, no max-change, ClipUp configuration, normalized / linear / raw ranking, scale_learning_rate=False, default
    population sizes, Adam on SNES, CEM bounds and maximisation, XNES learning rates (gaussian.py:543-1405)."""
    mod = _variant_table()
    algo, d, sense, fn, kw, gens = mod.VARIANTS[tag]
    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "searcher_variants_golden.npz"))
    prob = Problem(sense, mod.objective(fn), initial_bounds=(-5.12, 5.12), solution_length=d, vectorized=True, seed=11, dtype=torch.float32)
    s = {"PGPE": PGPE, "SNES": SNES, "CEM": CEM, "XNES": XNES}[algo](prob, **kw)
    tol = dict(rtol=3e-4, atol=3e-5) if algo == "XNES" else dict(rtol=2e-5, atol=3e-6)
    for t in range(gens):
        s.step()
        assert len(s.population) == int(gold[f"{tag}/popsize"])
        np.testing.assert_allclose(s.population.evals[:, 0].numpy(), gold[f"{tag}/f"][t], rtol=2e-5, atol=2e-4)
        np.testing.assert_allclose(s.status["center"].numpy(), gold[f"{tag}/mu"][t], **tol)
        np.testing.assert_allclose(s.status["stdev"].numpy(), gold[f"{tag}/sigma"][t], **tol)


def test_decorators_and_device_aware_evaluation():
    """decorators.py:170-960: vectorized / rowwise / expects_ndim / on_device / on_cuda / on_aux_device markers and how `Problem`
    honours them (core.py:2502-2585).  (The reference's own tests/test_decorators.py, test_expects_ndim.py and test_func_alg.py pass
    against this package through scripts/run_reference_tests.py.)"""
    from evotorch_b200.decorators import expects_ndim, on_aux_device, on_cuda, on_device, pass_info, rowwise, vectorized

    @rowwise
    def norm2(x):
        return torch.sum(x**2)

    assert norm2(torch.ones(4)).shape == () and norm2(torch.ones(3, 4)).shape == (3,) and norm2(torch.ones(2, 3, 4)).shape == (2, 3)
    prob = Problem("min", norm2, initial_bounds=(-1, 1), solution_length=4, seed=1)  # marked vectorized by @rowwise
    batch = SolutionBatch(prob, popsize=6)
    prob.evaluate(batch)
    torch.testing.assert_close(batch.evals[:, 0], (batch.values**2).sum(-1))

    @expects_ndim(2, 1, None)
    def affine(a, b, tag):
        assert tag == "x" and a.ndim == 2 and b.ndim == 1
        return a @ b

    assert affine(torch.ones(4, 3), torch.ones(3), "x").shape == (4,)
    assert affine(torch.ones(5, 7, 4, 3), torch.ones(7, 3), "x").shape == (5, 7, 4)  # batch dims align on the right
    assert affine(np.ones((4, 3), dtype=np.float32), torch.ones(3), "x").shape == (4,)
    with pytest.raises(ValueError):
        affine(torch.ones(3), torch.ones(3), "x")
    assert expects_ndim(lambda v, s: v * s, (1, 0))(torch.ones(2, 3), 2.0).shape == (2, 3)  # scalars become tensors

    assert vectorized(lambda x: x).__evotorch_vectorized__ and vectorized()(lambda x: x).__evotorch_vectorized__
    assert pass_info(lambda **k: None).__evotorch_pass_info__ and on_aux_device(lambda x: x).__evotorch_on_aux_device__
    assert on_cuda(lambda x: x).device == torch.device("cuda") and on_cuda(1)(lambda x: x).device == torch.device("cuda:1")

    seen = []

    @on_device("cpu")
    @vectorized
    def f(x):
        seen.append(x.device)
        return x.sum(-1)

    p2 = Problem("min", f, initial_bounds=(-1, 1), solution_length=3, seed=1)
    assert p2._device_of_fitness_function() == torch.device("cpu") and p2.aux_device.type in ("cpu", "cuda")
    b2 = SolutionBatch(p2, popsize=4)
    p2.evaluate(b2)
    assert seen == [torch.device("cpu")] and not torch.isnan(b2.evals).any()


def test_values_and_evals_are_read_only_tensors():
    """core.py:4101-4164 + tools/readonlytensor.py: `.values` / `.evals` share storage with the population but refuse in-place
    modification; library functions fed with them still return ordinary tensors."""
    import copy

    from evotorch_b200.tools import ReadOnlyTensor, as_read_only_tensor, storage_ptr

    prob = Problem("min", sphere, initial_bounds=(-1, 1), solution_length=4, vectorized=True, seed=1)
    batch = SolutionBatch(prob, popsize=6)
    prob.evaluate(batch)
    v, e = batch.values, batch.evals
    assert isinstance(v, ReadOnlyTensor) and isinstance(e, ReadOnlyTensor) and isinstance(batch[0].values, ReadOnlyTensor)
    assert storage_ptr(v) == storage_ptr(batch.access_values(keep_evals=True))  # a view, not a copy
    with pytest.raises(TypeError):
        v[0] = 1.0
    with pytest.raises(TypeError):
        v += 1
    with pytest.raises(AttributeError):
        v.zero_()
    with pytest.raises(TypeError):
        torch.add(v, 1, out=v)
    with pytest.raises(ValueError):
        v.numpy()[0, 0] = 3.0  # the numpy view is read-only too
    assert type(v.clone()) is torch.Tensor and type(v[[0, 2]]) is torch.Tensor  # copies are ordinary tensors
    assert isinstance(v[1:3], ReadOnlyTensor) and isinstance(v.reshape(-1), ReadOnlyTensor)  # views stay read-only
    assert isinstance(copy.deepcopy(v), ReadOnlyTensor) and torch.equal(copy.deepcopy(v), v)
    # reading works everywhere, and results of the library's own functions are writable tensors
    w = rank(e[:, 0], "centered", higher_is_better=False)
    assert type(w) is torch.Tensor
    w += 1
    dist = SymmetricSeparableGaussian({"mu": torch.zeros(4), "sigma": torch.ones(4)})
    grads = dist.compute_gradients(v, e[:, 0], objective_sense="min", ranking_method="centered")
    assert all(type(g) is torch.Tensor for g in grads.values())
    batch.access_values()[:] = 0.5  # the sanctioned way to write
    assert float(batch.values[0, 0]) == 0.5 and torch.isnan(batch.evals).all()
    x = torch.arange(3.0)
    assert storage_ptr(as_read_only_tensor(x)) == storage_ptr(x)


# ---------------------------------------------------------------------------------------------- round 2: drop-in gaps
@pytest.mark.parametrize("algo", ["snes", "pgpe", "cem"])
def test_reference_quickstart_with_actors_and_distributed_runs_unchanged(algo):
    """The reference's own quick-start (tests/test_examples.py:29-78) passes `num_actors=2` and `distributed=True`; with one
    process that maps to the ordinary generation (a warning says so) and the status carries the same keys."""
    def sphere1(x):
        return torch.sum(x.pow(2.0))

    with pytest.warns(UserWarning, match="no Ray actors"):
        problem = Problem("min", sphere1, solution_length=10, initial_bounds=(-1, 1), num_actors=2)
    kw = {"snes": (SNES, {"stdev_init": 5, "distributed": True}),
          "pgpe": (PGPE, {"popsize": 10, "center_learning_rate": 0.01, "stdev_learning_rate": 0.1, "radius_init": 0.27, "distributed": True}),
          "cem": (CEM, {"popsize": 10, "parenthood_ratio": 0.1, "radius_init": 0.27, "distributed": True})}[algo]
    searcher = kw[0](problem, **kw[1])
    searcher.run(2)
    assert "center" in searcher.status and searcher.step_count == 2


class _CountingProblem(Problem):
    """A stand-in for an RL problem: every evaluated solution costs `cost` simulator interactions (vecgymne.py reports them
    as the `total_interaction_count` status item)."""

    def __init__(self, cost, **kw):
        super().__init__("min", lambda x: torch.sum(x * x, dim=-1), initial_bounds=(-1, 1), solution_length=5, vectorized=True, seed=1, **kw)
        self._cost, self._count = cost, 0

    def _evaluate_batch(self, batch):
        super()._evaluate_batch(batch)
        self._count += self._cost * len(batch)

    def _extra_status(self, batch):
        return {"total_interaction_count": self._count}


def test_adaptive_population_size_follows_the_reference_loop():
    """gaussian.py:299-349: populations of `popsize` are sampled until MORE than `num_interactions` interactions were made
    (or `popsize_max` solutions exist); the generation's population is their concatenation."""
    prob = _CountingProblem(cost=3)
    s = PGPE(prob, popsize=10, center_learning_rate=0.1, stdev_learning_rate=0.1, stdev_init=1.0, num_interactions=100)
    s.step()
    assert len(s.population) == 40  # 10 solutions = 30 interactions; 30, 60, 90 are not > 100, 120 is
    m0 = s.status["mean_eval"]
    s.run(15)
    assert len(s.population) == 40 and s.status["mean_eval"] < m0
    capped = PGPE(_CountingProblem(cost=3), popsize=10, center_learning_rate=0.1, stdev_learning_rate=0.1, stdev_init=1.0, num_interactions=100,
                  popsize_max=20)
    capped.run(2)
    assert len(capped.population) == 20
    with pytest.raises(ValueError):
        PGPE(prob, popsize=10, center_learning_rate=0.1, stdev_learning_rate=0.1, stdev_init=1.0, popsize_max=20)
    # the gradient service (core.py:3239-3282) with the same thresholds
    prob2 = _CountingProblem(cost=3)
    dist = SymmetricSeparableGaussian({"mu": torch.zeros(5), "sigma": torch.ones(5), "divide_mu_grad_by": "num_directions",
                                       "divide_sigma_grad_by": "num_directions"})
    prob2.evaluate(prob2.generate_batch(2))  # the status item exists from the first evaluation on
    out = prob2.sample_and_compute_gradients(dist, 10, num_interactions=100, ranking_method="centered")[0]
    assert out["num_solutions"] == 40 and set(out["gradients"]) == {"mu", "sigma"}
    out = prob2.sample_and_compute_gradients(dist, 10, num_interactions=100, popsize_max=30, ranking_method="centered")[0]
    assert out["num_solutions"] == 30


def test_local_weight_conditions_and_policy_guards():
    """Sharded ranking is only legal when a shard's gradient needs nothing but its own rows' utilities; Policy rejects stateful nets."""
    from evotorch_b200.distributions import ExpSeparableGaussian, SeparableGaussian
    from evotorch_b200.neuroevolution import Policy

    mu, sg = torch.zeros(4), torch.ones(4)
    sym = SymmetricSeparableGaussian({"mu": mu, "sigma": sg, "divide_mu_grad_by": "num_directions", "divide_sigma_grad_by": "num_directions"})
    assert sym.accepts_local_weights("centered") and not sym.accepts_local_weights("nes") and not sym.accepts_local_weights("raw")
    assert not SeparableGaussian({"mu": mu, "sigma": sg, "divide_mu_grad_by": "total_weight"}).accepts_local_weights("centered")
    assert not SeparableGaussian({"mu": mu, "sigma": sg, "parenthood_ratio": 0.5}).accepts_local_weights("centered")
    exp = ExpSeparableGaussian({"mu": mu, "sigma": sg})
    assert exp.accepts_local_weights("nes") and not exp.accepts_local_weights("centered")
    # gradients from a shard's own utilities == the slice-based partial gradients
    g = torch.Generator().manual_seed(0)
    X = torch.randn(12, 4, generator=g)
    w = torch.randn(12, generator=g)
    a = sym.partial_gradients(X[4:8], w, 4, "centered")
    b = sym.partial_gradients(X[4:8], w[4:8].clone(), 4, "centered", local_weights_of=12)
    assert torch.equal(a["mu"], b["mu"]) and torch.equal(a["sigma"], b["sigma"])
    with pytest.raises(ValueError):
        sym.partial_gradients(X[4:8], w[4:8].clone(), 4, "nes", local_weights_of=12)
    with pytest.raises(NotImplementedError):
        Policy(torch.nn.Sequential(torch.nn.LSTM(3, 4)))
