import os
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def oracle_libs():
    """Build (if needed) and load the oracle: the compiled reference when present, and the C restatement."""
    import oracle
    if not oracle.available("port") or (oracle.reference_dir() and not oracle.available("ref")):
        oracle.build()
    libs = {"port": oracle.load("port")}
    if oracle.available("ref"):
        libs["ref"] = oracle.load("ref")
    return libs


@pytest.fixture(scope="session")
def orc(oracle_libs):
    """The checker: oracle/_ref (unmodified reference sources) when it exists, else the restatement."""
    return oracle_libs.get("ref", oracle_libs["port"])


@pytest.fixture(scope="session")
def cuda_lib():
    from shermbot_navigation_b200 import build, nuslam
    if build.stale():
        build.build()
    return nuslam
