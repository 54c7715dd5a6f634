import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

GOLDEN = Path(__file__).resolve().parent / "golden"


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with `-m gpu`)")


def infonce_inputs(B: int, M: int, D: int, seed: int, unit: bool = True):
    """The seeded (buyer [B,D], pos [B,D], neg [B,M,D]) f32 inputs of the infonce_*.npz golden cases."""
    rng = np.random.default_rng(seed)
    b = rng.standard_normal((B, D)).astype(np.float32)
    p = rng.standard_normal((B, D)).astype(np.float32)
    n = rng.standard_normal((B, M, D)).astype(np.float32)
    if unit:                          # the towers L2-normalise their outputs (buyer_tower.py:66,99; item tower likewise)
        b /= np.linalg.norm(b, axis=1, keepdims=True)
        p /= np.linalg.norm(p, axis=1, keepdims=True)
        n /= np.maximum(np.linalg.norm(n, axis=2, keepdims=True), 1e-12)
    return b, p, n


def golden(name: str):
    g = dict(np.load(GOLDEN / name, allow_pickle=False))
    if "input_seed" in g:
        # buyer and pos are not stored (that keeps the file under 1 MB): they are regenerated from the seed, and
        # neg, drawn after them from the same generator and stored, checks that the regeneration is exact
        B, M, D = g["neg"].shape
        b, p, n = infonce_inputs(B, M, D, int(g["input_seed"]), bool(g["input_unit"]))
        assert np.array_equal(n, g["neg"]), f"{name}: the seeded generator no longer reproduces the stored inputs"
        g.update(buyer=b, pos=p)
    return g


@pytest.fixture(scope="session")
def native_lib():
    """The C-ABI library; builds it if this checkout has not been built yet."""
    from two_tower_model_v2_b200 import _native
    if not _native.LIB_PATH.exists():
        import __graft_entry__
        __graft_entry__.build()
    return _native.load()


def rel_err(a, b):
    """Norm-wise: max|a-b| / max|b| (the whole tensor's largest element is the scale)."""
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def elem_rel_err(a, b, floor_frac=1.0):
    """Element-wise: max over elements of |a-b| / max(|b|, floor), floor = floor_frac * rms of that ROW of b: every
    element is held to the relative tolerance, except that elements below the row's typical magnitude (rms; 0.051 for
    a unit vector in D = 384) are held to tolerance * rms absolute - the reference's own fp32-vs-fp64 noise (2e-7 of
    the largest element) is already 6e-6 relative on an element at 0.1 rms, so a smaller floor would test fp32 itself."""
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    rms = np.sqrt((b * b).mean(axis=-1, keepdims=True))
    floor = np.maximum(floor_frac * rms, 1e-30)
    return float((np.abs(a - b) / np.maximum(np.abs(b), floor)).max())
