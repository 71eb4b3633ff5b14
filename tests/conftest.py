import importlib.util
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on a B200 with `pytest -m gpu`)")
    config.addinivalue_line("markers", "multigpu: needs >= 2 CUDA devices")


GOLDEN = os.path.join(ROOT, "tests", "golden", "ref_golden.npz")


def golden_module(name):
    """tests/golden/<name>.py: the scripts that minted the golden files also define their seeded inputs."""
    spec = importlib.util.spec_from_file_location(name, os.path.join(ROOT, "tests", "golden", name + ".py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.fixture(scope="session")
def golden():
    """The reference's outputs (tests/golden/ref_golden.npz) together with the seeded inputs they came from."""
    g = dict(np.load(GOLDEN))
    g.update(golden_module("make_golden").inputs())
    return g


def rel_close(got, want, rtol=1e-4, atol_scale=1e-5, what=""):
    """The parity bar of BASELINE.json's north_star: 1e-4 relative fp32.  `atol_scale`
    * max|want| absorbs cancellation in sums (an fp32 sum of d terms is only good to
    ~d*eps*sum|x|, so elements that cancel to ~0 cannot meet a pure relative bound —
    the reference's own atomics-ordered sums do not either)."""
    got = np.asarray(got, dtype=np.float64)
    want = np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    scale = np.abs(want).max() if want.size else 0.0
    err = np.abs(got - want)
    bound = rtol * np.abs(want) + atol_scale * scale + 1e-30
    bad = err > bound
    assert not bad.any(), "%s: %d/%d elements off; worst err %.3e at %s (want %.6g got %.6g)" % (
        what, int(bad.sum()), bad.size, float(err.max()), np.unravel_index(err.argmax(), err.shape),
        float(want.flat[err.argmax()]), float(got.flat[err.argmax()]))
