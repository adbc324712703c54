import os
import sys

import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def port():
    from oracle_lib import Port
    return Port()


@pytest.fixture(scope="session")
def ref():
    from oracle_lib import Ref, have_ref
    if not have_ref():
        pytest.skip("oracle/_ref not built (it is compiled from the original project's sources, see oracle/Makefile)")
    return Ref()


@pytest.fixture(scope="session")
def tmpdir_session(tmp_path_factory):
    return str(tmp_path_factory.mktemp("synth"))
