import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests", "golden")):
    if p not in sys.path:
        sys.path.insert(0, p)

import cases  # noqa: E402  (tests/golden, on the path above)

RTOL, ATOL = 1e-4, 1e-5  # BASELINE.json north_star: fp32 parity bound for NMF outputs / input grads


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box via gpurun)")


def tol_ratio(got, ref, rtol=RTOL, atol=ATOL):
    """max |got-ref| / (atol + rtol*|ref|); parity holds when <= 1.  A sampled golden output (cases.Sample) is compared
    with ``got`` at its indices: ``got`` has the full shape (all of it must be finite), or is a Sample of the same
    indices."""
    if isinstance(ref, cases.Sample) and isinstance(got, cases.Sample):
        assert got.full_shape == ref.full_shape and np.array_equal(got.index, ref.index)
    elif isinstance(ref, cases.Sample):
        got = np.asarray(got, dtype=np.float64)
        assert got.shape == ref.full_shape, (got.shape, ref.full_shape)
        if not np.isfinite(got).all():
            return float("inf")
        got = got.reshape(-1)[ref.index]
    got = np.asarray(got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    assert got.shape == ref.shape, (got.shape, ref.shape)
    if not np.isfinite(got).all():
        return float("inf")
    return float(np.max(np.abs(got - ref) / (atol + rtol * np.abs(ref)))) if got.size else 0.0


def assert_close(got, ref, rtol=RTOL, atol=ATOL, what=""):
    r = tol_ratio(got, ref, rtol, atol)
    assert r <= 1.0, f"{what}: max err / tol = {r:.3g} (rtol={rtol}, atol={atol})"


@pytest.fixture(scope="session")
def golden():
    d = os.path.join(ROOT, "tests", "golden")
    return {k: cases.load_golden(d, k) for k in ("nmf", "sw", "fused", "block", "model")}
