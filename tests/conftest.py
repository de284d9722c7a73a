import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def port():
    from oracle import oracle_lib
    return oracle_lib.Port()


@pytest.fixture(scope="session")
def corpora():
    from tools import corpus
    cache = {}

    def get(kind, n, seed=None):
        key = (kind, n, seed)
        if key not in cache:
            cache[key] = corpus.make(kind, n, seed)
        return cache[key]
    return get
