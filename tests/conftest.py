import os
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with `-m gpu`)")


@pytest.fixture(scope="session")
def lib():
    """The product library. Built on demand; never replaced by anything else."""
    from ipt_b200 import build, capi

    build.build()
    return capi.load()


@pytest.fixture(scope="session")
def oracle():
    import oracle_lib

    return oracle_lib.load_oracle()


@pytest.fixture(scope="session")
def ref():
    """The compiled reference (oracle/_ref). Skips where neither the prebuilt .so nor the IPT_REFERENCE sources exist."""
    import oracle_lib

    r = oracle_lib.load_ref()
    if r is None:
        pytest.skip("oracle/_ref/libipt_ref.so not available (no IPT_REFERENCE sources to build it from)")
    return r


@pytest.fixture(scope="session")
def ref_or_none():
    """The compiled reference where it is built, else None (tests then compare with its stored outputs)."""
    import oracle_lib

    return oracle_lib.load_ref()


@pytest.fixture(scope="session")
def pins():
    """tests/golden/pin_live.npz: the reference's outputs the live pins compare with."""
    import numpy as np
    from helpers import PINS

    return np.load(PINS)


@pytest.fixture(scope="session")
def has_gpu(lib):
    return lib.ipt_device_count() > 0
