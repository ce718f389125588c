import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def find_fixture(name):
    """Path of a GGUF test model: the synthetic stand-ins for tinyllamas-stories-15M of tests/synth_model.py."""
    from tests.synth_model import model_path
    return model_path(name)


@pytest.fixture
def fixture_path():
    return find_fixture
