import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run with -m gpu on the B200 box)")


def rel_l2(a, b):
    import numpy as np
    dt = np.complex128 if (np.iscomplexobj(a) or np.iscomplexobj(b)) else np.float64
    a = np.asarray(a, dtype=dt)
    b = np.asarray(b, dtype=dt)
    d = np.linalg.norm(b.ravel())
    return float(np.linalg.norm((a - b).ravel()) / (d if d > 0 else 1.0))


def _reduce(f, stride, nblk=16):
    import numpy as np
    n = f.shape[0]
    b = n // nblk
    f64 = f.astype(np.float64).reshape(nblk, b, nblk, b)
    return np.ascontiguousarray(f[::stride, ::stride]), np.stack([f64.sum(axis=(1, 3)), (f64 * f64).sum(axis=(1, 3))])


def check_golden(got, gold, name, stride, tol):
    """`got` against a field stored as <name>_sub / <name>_blk (tests/golden/make_golden_headline.py reduce_field)"""
    import numpy as np
    sub, blk = _reduce(got, stride)
    assert rel_l2(sub, gold[f"{name}_sub"]) < tol, (name, rel_l2(sub, gold[f"{name}_sub"]))
    # the full field enters through the block sums and sums of squares (16 x 16 blocks of (n / 16)^2 points)
    assert rel_l2(blk[1], gold[f"{name}_blk"][1]) < 2 * tol, (name, "block sums of squares")
    scale = np.sqrt(gold[f"{name}_blk"][1].sum() * got.size)          # |sum| <= sqrt(N * sum of squares)
    assert np.abs(blk[0] - gold[f"{name}_blk"][0]).max() < tol * scale, (name, "block sums")
