import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def oracle():
    import oracle_lib
    oracle_lib.build(ref=True)
    return oracle_lib.Oracle()


@pytest.fixture(scope="session")
def reference(oracle):
    import oracle_lib
    if not oracle_lib.Reference.available():
        pytest.skip("oracle/_ref not built (reference sources absent)")
    return oracle_lib.Reference()
