import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")

MODEL_CASES = [
    "painn_aspirin_b4",
    "schnet_ethanol_b1",
    "schnet_qm9_b8",
    "schnet_qm9_b8_padded",
    "schnet_qm9_b8_forces",
    "painn_box_216",
    "painn_bessel_shared",
    "schnet_box_216",
    "painn_md_ethanol_trained",
]


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: test needs a CUDA device (run on the B200 box with -m gpu)")


def load_case(name):
    """Load a golden fixture -> (spec, params, inputs, ref32, ref64)."""
    from schnetpack_b200 import synthetic as S

    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    spec = json.loads(str(z["spec_json"]))
    inputs = {k[3:]: z[k] for k in z.files if k.startswith("in:")}
    ref32 = {k[6:]: z[k] for k in z.files if k.startswith("ref32:")}
    ref64 = {k[6:]: z[k] for k in z.files if k.startswith("ref64:")}
    params = {k[6:]: z[k] for k in z.files if k.startswith("param:")}
    if not params:
        params = S.init_params(spec, int(z["seed"]))
    return spec, params, inputs, ref32, ref64


def rel_err(a, b):
    """max-norm relative error  max|a-b| / max|b|  (the 1e-5 'relative fp32' criterion of BASELINE.json)."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-30))


def flat_sample(a, k=1024):
    """A fixed sample of at most ``k`` elements of ``a`` (flattened; every element when there are no more than ``k``).
    Recorded reference outputs too large to store whole are kept as this sample plus their max-norm, so that a test can
    still form the ``rel_err`` of the full array's scale.  ``RandomState`` keeps its stream fixed across numpy versions."""
    a = np.asarray(a).reshape(-1)
    if a.size <= k:
        return a
    return a[np.sort(np.random.RandomState(a.size).choice(a.size, k, replace=False))]


@pytest.fixture(scope="session")
def primitives():
    return np.load(os.path.join(GOLDEN, "primitives.npz"))
