import os
import sys

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "avisynth-jincresize_b200"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def native_built():
    """Build the host-side artefacts once per session (the CUDA libraries are built by __graft_entry__.build())."""
    import subprocess

    subprocess.run(["make", "-s", "host"], cwd=REPO, check=True)
    return True


@pytest.fixture(scope="session")
def have_ref(native_built):
    from oracle import ref as oref

    return oref.available()
