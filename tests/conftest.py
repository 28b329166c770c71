import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run on the GPU box with -m gpu)")


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN


@pytest.fixture(scope="session")
def golden(oracle):
    """load(name) -> tests/golden/<name>.npz as a dict, with the seeded inputs the fixture does not store regenerated
    (fdsr_oracle.golden_inputs) after checking each against the float64 sum stored as `<input>_sum`."""
    def load(name):
        with np.load(os.path.join(GOLDEN, name + ".npz")) as z:
            g = dict(z)
        for k, v in oracle.golden_inputs(name).items():
            assert abs(float(v.double().sum()) - float(g[k + "_sum"])) < 1e-6, f"{name}: {k} differs from the fixture's"
            g[k] = v.numpy()
        return g
    return load


@pytest.fixture(scope="session")
def oracle():
    import fdsr_oracle
    return fdsr_oracle


@pytest.fixture(scope="session")
def schedule(oracle):
    return oracle.schedule_tables(oracle.make_beta_schedule(**oracle.DEFAULT_SCHEDULE))
