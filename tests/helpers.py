"""Shared helpers for the parity tests."""
import pathlib

import numpy as np
import torch

GOLDEN = pathlib.Path(__file__).parent / "golden"

# North-star tolerance (BASELINE.json): "within 1e-4 relative fp32 for rendered RGB/depth, pointmaps and
# Gaussian gradients".  Relative to the tensor's scale (max |ref|), which is how a field of values that
# crosses zero has to be compared.
RTOL = 1e-4


def rel_err(a, b):
    a = np.asarray(a.detach().cpu() if isinstance(a, torch.Tensor) else a, dtype=np.float64)
    b = np.asarray(b.detach().cpu() if isinstance(b, torch.Tensor) else b, dtype=np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    if a.size == 0:
        return 0.0
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-20))


def assert_close(a, b, rtol=RTOL, what="", max_outlier_frac=0.0):
    """|a-b| <= rtol * max|b| element-wise; `max_outlier_frac` admits the rare elements where a discrete
    decision (alpha<1/255 skip, T<=1e-4 stop) flips between two fp32 evaluations of exp()."""
    a64 = np.asarray(a.detach().cpu() if isinstance(a, torch.Tensor) else a, dtype=np.float64)
    b64 = np.asarray(b.detach().cpu() if isinstance(b, torch.Tensor) else b, dtype=np.float64)
    assert a64.shape == b64.shape, (what, a64.shape, b64.shape)
    if a64.size == 0:
        return
    scale = max(np.abs(b64).max(), 1e-20)
    bad = np.abs(a64 - b64) > rtol * scale
    frac = bad.mean()
    assert frac <= max_outlier_frac, (f"{what}: {bad.sum()} of {bad.size} elements exceed rtol={rtol} "
                                      f"(max rel err {np.abs(a64 - b64).max() / scale:.3e})")


def golden_sample(n, k, seed=0):
    """Fixed sample of k flat indices out of n, shared by tests/golden/make_reference_builds_golden.py and the tests that
    read what it stored."""
    return np.random.default_rng(seed).choice(n, size=min(k, n), replace=False)


def reference_builds():
    """Seeded samples of what the reference's own CUDA extensions computed on the tests' inputs (written on a B200 by
    tests/golden/make_reference_builds_golden.py)."""
    return np.load(GOLDEN / "reference_builds.npz")
