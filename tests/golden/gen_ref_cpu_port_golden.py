"""Golden trajectory of the REAL reference's PGPE on Rastrigin (300 dims, popsize 200, seed 5, 8 generations, CPU fp32), which
oracle/ref_cpu_path.py must reproduce bit for bit:

    PYTHONPATH=tests/golden/_refstubs:<reference checkout>/src EVOTORCH_VERBOSE_LEVEL=0 python tests/golden/gen_ref_cpu_port_golden.py

Centre and stdev are stored whole.  The populations (1.9 MB in all) are stored as SHA-256 digests of their bytes, which keeps
the comparison exact, plus their first 16 rows, which show where a mismatch lies.
"""

import hashlib
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import evotorch  # noqa: E402  (the reference)
from evotorch import Problem  # noqa: E402
from evotorch.algorithms import PGPE  # noqa: E402

from oracle.ref_cpu_path import rastrigin  # noqa: E402

assert not os.path.abspath(evotorch.__file__).startswith(os.path.dirname(os.path.dirname(HERE))), evotorch.__file__  # the reference, not this package
prob = Problem("min", rastrigin, initial_bounds=(-5.12, 5.12), solution_length=300, vectorized=True, seed=5, dtype=torch.float32)
s = PGPE(prob, popsize=200, center_learning_rate=0.5, stdev_learning_rate=0.1, stdev_init=1.0)
center, stdev, digests, rows = [], [], [], []
for t in range(8):
    s.step()
    X = s.population.values.numpy()
    center.append(s.status["center"].numpy().copy())
    stdev.append(s.status["stdev"].numpy().copy())
    digests.append(hashlib.sha256(np.ascontiguousarray(X, dtype=np.float32).tobytes()).hexdigest())
    rows.append(X[:16].copy())
np.savez_compressed(os.path.join(HERE, "ref_cpu_port_golden.npz"), center=np.stack(center), stdev=np.stack(stdev),
                    population_sha256=np.array(digests), population_rows=np.stack(rows))
