"""oracle/ref_cpu_path.py (the torch-CPU restatement timed as the CPU baseline) against the real reference: golden
trajectories, bit for bit."""

import hashlib
import os

import numpy as np
import pytest

from oracle.ref_cpu_path import PGPEReferencePath

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("tag,sense", [("pgpe", "min"), ("pgpe_max", "max")])
def test_port_reproduces_golden_trajectory(golden, tag, sense):
    p = PGPEReferencePath(8, 32, center_learning_rate=0.5, stdev_learning_rate=0.1, stdev_init=1.0, seed=11, sense=sense)
    for t in range(len(golden[f"traj/{tag}/mu"])):
        p.step()
        np.testing.assert_allclose(p.mu.numpy(), golden[f"traj/{tag}/mu"][t], rtol=1e-6, atol=1e-6)
        np.testing.assert_allclose(p.sigma.numpy(), golden[f"traj/{tag}/sigma"][t], rtol=1e-6, atol=1e-6)
        np.testing.assert_allclose(p.X.numpy(), golden[f"traj/{tag}/X"][t], rtol=1e-6, atol=2e-6)


def test_port_is_bit_identical_to_the_reference_trajectory():
    """Eight generations at 300 dims x popsize 200 against the reference's own run (tests/golden/gen_ref_cpu_port_golden.py):
    centre, stdev and every population must be identical bit for bit."""
    with np.load(os.path.join(ROOT, "tests", "golden", "ref_cpu_port_golden.npz")) as z:
        gold = {k: z[k] for k in z.files}
    p = PGPEReferencePath(300, 200, center_learning_rate=0.5, stdev_learning_rate=0.1, stdev_init=1.0, seed=5)
    for t in range(len(gold["center"])):
        p.step()
        np.testing.assert_array_equal(p.mu.numpy(), gold["center"][t], err_msg=f"generation {t}")
        np.testing.assert_array_equal(p.sigma.numpy(), gold["stdev"][t], err_msg=f"generation {t}")
        X = p.X.numpy()
        np.testing.assert_array_equal(X[:16], gold["population_rows"][t], err_msg=f"generation {t}")
        assert hashlib.sha256(np.ascontiguousarray(X, dtype=np.float32).tobytes()).hexdigest() == gold["population_sha256"][t], t
