"""Golden observations of the reference's public helpers (tests/golden/reference_api_probe.py run against the REAL reference):

    PYTHONPATH=tests/golden/_refstubs:<reference checkout>/src EVOTORCH_VERBOSE_LEVEL=0 python tests/golden/gen_reference_api_golden.py
"""

import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

import evotorch  # noqa: E402  (the reference)
from reference_api_probe import GROUPS, probe  # noqa: E402

assert not os.path.abspath(evotorch.__file__).startswith(os.path.dirname(os.path.dirname(HERE))), evotorch.__file__  # the reference, not this package
out = {f"{group}/{key}": value for group in GROUPS for key, value in probe("evotorch", group).items()}
np.savez_compressed(os.path.join(HERE, "reference_api_golden.npz"), **out)
print(len(out), "arrays")
