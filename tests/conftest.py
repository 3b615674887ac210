import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


def _make(*targets):
    subprocess.run(["make", "-s", "-C", ROOT, *targets], check=True, stdout=subprocess.DEVNULL)


@pytest.fixture(scope="session", autouse=True)
def built():
    """CPU-side artefacts every test may need: the oracle restatements and the generator.
    The CUDA library itself is built by `make` / __graft_entry__.build(); the prebuilt .so travels to the GPU box."""
    _make("oracle", "tools")
    if not os.path.exists(os.path.join(ROOT, "stochasticsim_b200", "lib", "libssb200.so")):
        _make("all")
    return True


@pytest.fixture(scope="session")
def ref_dir():
    """oracle/_ref/: the UNMODIFIED reference, compiled from the upstream stochasticSim sources that STOCHASTICSIM_SRC points to
    (they are not part of this repository); None if absent."""
    d = os.path.join(ROOT, "oracle", "_ref")
    src = os.environ.get("STOCHASTICSIM_SRC", "")
    if src and os.path.exists(os.path.join(src, "tncCountsProfile.c")) and not os.path.exists(os.path.join(d, "stochasticSpike")):
        _make("ref", "REFERENCE=" + os.path.abspath(src))
    return d if os.path.exists(os.path.join(d, "tncCountsProfile")) else None
