"""CPU tests (no GPU) of the kNN feature: the fp64 oracle against render()'s reference kNN helper, the K = int(n ** 0.5)
expression of post_process, and argument rejection of ogs_knn_segmented and knn_points without a device."""
import ctypes as C
import math
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import knn as oracle  # noqa: E402
from opengaussian_b200 import knn, renderer  # noqa: E402


@pytest.mark.parametrize("n", [1, 2, 10, 37, 500, 3000])
def test_oracle_matches_reference_knn(n):
    x = np.random.default_rng(n).standard_normal((n, 3)).astype(np.float32)
    K = oracle.sqrt_k(n)
    d, idx, _ = oracle.knn(x, x, K)
    ref = renderer._knn_mean_dists(torch.from_numpy(x).double(), K).numpy()
    np.testing.assert_allclose(d, ref, rtol=1e-12, atol=1e-12)
    assert (idx[:, 0] == np.arange(n)).all()                  # the self-match, at distance 0
    keep, per_point, thr = oracle.post_process_keep(x)
    t = torch.from_numpy(ref)
    assert np.isclose(thr, float(t.mean() + t.std()), rtol=1e-12, equal_nan=True)     # NaN for n = 1
    assert (keep == (per_point < thr)).all()


def test_oracle_kdtree_matches_brute_force():
    x = np.random.default_rng(1).standard_normal((oracle.BRUTE_MAX + 500, 3)).astype(np.float32)
    d, idx, tie = oracle.knn(x[:300], x, 40)                   # k-d tree
    small = x[: oracle.BRUTE_MAX]
    d2, idx2, _ = oracle.knn(x[:300], small, 40)               # brute force over a subset: distances can only grow
    assert (d <= d2 + 1e-15).all()
    full = ((x[:300, None, :].astype(np.float64) - x[None].astype(np.float64)) ** 2).sum(-1)
    np.testing.assert_allclose(d, np.sort(full, 1)[:, :40], rtol=1e-12, atol=0)
    assert (idx[~tie] == np.argsort(full, 1, kind="stable")[~tie, :40]).all()


def test_sqrt_k_matches_reference_expression():
    ks = np.arange(1, math.isqrt(200_000_000) + 1, dtype=np.int64)
    n = np.concatenate([ks * ks - 1, ks * ks, ks * ks + 1,
                        np.random.default_rng(0).integers(0, 200_000_001, 20000)])
    n = np.unique(n[n >= 0])
    got = knn.sqrt_k(torch.from_numpy(n)).numpy()
    want = np.array([int(torch.tensor(int(v)) ** 0.5) for v in n])
    assert (got == want).all(), n[got != want][:10]
    # where the float32 expression and the integer square root part: the reference's value is kept
    assert int(knn.sqrt_k(torch.tensor([4097 * 4097 - 1]))[0]) == 4097 != math.isqrt(4097 * 4097 - 1)


@pytest.fixture(scope="module")
def lib():
    from opengaussian_b200 import _lib, build
    build.build()
    return _lib.lib()


def test_knn_segmented_rejects_bad_arguments_without_device(lib):
    f = lib.ogs_knn_segmented
    buf = (C.c_float * 8)()
    p = C.cast(buf, C.c_void_p)
    assert f(-1, None, None, 0, None, None, None, 0, p, None, None, None, None, None) == -1
    assert b"bad sizes" in lib.ogs_last_error()
    assert f(4, None, None, 1, p, p, p, 0, p, None, None, None, None, None) == -1        # queries without q / q_seg
    assert f(4, p, p, -1, p, p, p, 0, p, None, None, None, None, None) == -1             # S < 0
    assert f(4, p, p, 1, p, None, p, 0, p, None, None, None, None, None) == -1           # no offsets
    assert f(4, p, p, 1, p, p, p, 0, None, None, None, p, None, None) == -1              # half a neighbour list
    assert f(4, p, p, 1, p, p, p, 0, None, None, None, p, p, None) == -1                 # list with k_max = 0
    assert b"k_max" in lib.ogs_last_error()
    assert f(4, p, p, 1, p, p, p, 4, None, None, None, None, None, None) == -1           # no output
    assert b"no output" in lib.ogs_last_error()
    assert f(0, None, None, 0, None, None, None, 0, p, None, None, None, None, None) == 0  # nothing to do


def test_knn_points_argument_errors():
    from opengaussian_b200._lib import OgsError
    with pytest.raises(ValueError, match="only D = 3"):
        knn.knn_points(torch.zeros(1, 4, 2), torch.zeros(1, 5, 2))
    with pytest.raises(ValueError):
        knn.knn_points(torch.zeros(1, 4, 3), torch.zeros(2, 5, 3))
    with pytest.raises(OgsError, match="no CPU path"):
        knn.knn_points(torch.zeros(1, 4, 3), torch.zeros(1, 5, 3), K=2)
    with pytest.raises(OgsError, match="no CPU path"):
        knn.slot_knn_sums(torch.zeros(4, 3), torch.zeros(4, dtype=torch.int32), 1)


def test_compat_package_exposes_knn_points():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, os.path.join(root, "compat", "knn"))
    try:
        from pytorch3d.ops import knn_points
    finally:
        sys.path.pop(0)
        for m in ("pytorch3d.ops", "pytorch3d"):
            sys.modules.pop(m, None)
    assert knn_points is knn.knn_points
