import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def oracle():
    """The CPU oracle bindings (test infrastructure)."""
    from oracle import oracle as O
    O.build()
    return O


@pytest.fixture(scope="session")
def golden():
    with open(os.path.join(GOLDEN_DIR, "golden.json")) as f:
        return json.load(f)


@pytest.fixture(scope="session")
def golden_inputs(golden, oracle):
    """name -> uint8 array; committed fixtures plus regenerated synthetic frames."""
    z = np.load(os.path.join(GOLDEN_DIR, "fixtures.npz"))
    inputs = {k: z[k] for k in z.files}
    for k, c in golden["synth"].items():
        inputs[k] = oracle.synth_ecg(c["first"], c["n"], c["bps"], c["ch"], c["ns"]).reshape(-1)
    return inputs


def has_ref():
    return os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libref.so"))
