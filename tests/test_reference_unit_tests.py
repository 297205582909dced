"""The public helpers that the reference's own unit tests cover (hooks, ranking, the optimizer classes, read-only tensors,
the decorators, `expects_ndim` / `rowwise`, the functional optimizers) must behave as the reference does: every
observation of tests/golden/reference_api_probe.py on this package equals the reference's, stored in
tests/golden/reference_api_golden.npz by tests/golden/gen_reference_api_golden.py."""

import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))

from reference_api_probe import GROUPS, probe  # noqa: E402


@pytest.mark.parametrize("group", GROUPS)
def test_public_helpers_match_reference(group):
    with np.load(os.path.join(HERE, "golden", "reference_api_golden.npz")) as z:
        expected = {k[len(group) + 1:]: z[k] for k in z.files if k.startswith(group + "/")}
    got = probe("evotorch_b200", group)
    assert sorted(got) == sorted(expected)
    for key, want in expected.items():
        have = np.asarray(got[key])
        assert have.shape == want.shape, key
        if want.dtype.kind in "fc":
            np.testing.assert_allclose(have, want, rtol=1e-6, atol=1e-6, err_msg=key)
        else:
            np.testing.assert_array_equal(have, want, err_msg=key)
