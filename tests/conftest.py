"""pytest configuration: registers the `gpu` marker and shared helpers.

`-m "not gpu"` = oracle-vs-golden, host logic, C-ABI symbol checks (runs in the CPU build container).
`-m gpu`       = CUDA-vs-oracle / CUDA-vs-golden parity through the C-ABI (runs on a B200 box).
"""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu on the GPU box")


def golden(name):
    return dict(np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False))


def paper_weights_path():
    """A copy of the reference's weights/paper_weights.pth as .npz, if one is available (it is an input artefact,
    70 MB, git-ignored; see tests/golden/export_paper_weights.py)."""
    p = os.path.join(ROOT, "weights", "paper_weights.npz")
    return p if os.path.exists(p) else None


def assert_close(a, b, rtol, atol=0.0, name="", norm_rel=None):
    """|a-b| <= atol + rtol*|b| elementwise, or (norm_rel) max|a-b| <= norm_rel * max|b|."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, f"{name}: shape {a.shape} vs {b.shape}"
    assert np.all(np.isfinite(a)), f"{name}: non-finite values"
    err = np.abs(a - b)
    if norm_rel is not None:
        scale = max(np.abs(b).max(), 1e-30)
        assert err.max() <= norm_rel * scale + atol, (
            f"{name}: max|err| {err.max():.3e} > {norm_rel:g} * max|ref| {scale:.3e} (+{atol:g})")
        return
    bad = err > atol + rtol * np.abs(b)
    assert not bad.any(), (f"{name}: {bad.sum()} / {bad.size} elements out of tolerance; max err {err.max():.3e}, "
                           f"max ref {np.abs(b).max():.3e}")


def quat_align(qa, qb):
    """Flip qa's sign per quaternion to match qb (eigh sign ambiguity, SURVEY Appendix C.1)."""
    s = np.sign(np.sum(qa * qb, axis=-1, keepdims=True))
    s[s == 0] = 1
    return qa * s
