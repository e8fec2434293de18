import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with -m gpu)")
    config.addinivalue_line("markers", "slow: full-size property tests")


@pytest.fixture(scope="session")
def oracle():
    import oracle_lib
    oracle_lib.build_oracle()
    return oracle_lib.Oracle()


@pytest.fixture(scope="session")
def lambda_reads():
    from raven_b200 import seqio
    return seqio.ReadSet.load(os.path.join(ROOT, "tests", "golden", "lambda_reads.npz"))


@pytest.fixture(scope="session")
def gpu_engine():
    from raven_b200 import engine
    return engine.Engine(device=0)
