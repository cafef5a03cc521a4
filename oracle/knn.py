"""fp64 CPU oracle of exact k-nearest-neighbour search and of render()'s post_process outlier rule -- TEST
INFRASTRUCTURE ONLY (see oracle/__init__.py).

Squared distances are computed in float64 from the float32 coordinates (exact differences, no cancellation): numpy
brute force for small clouds, scipy.spatial.cKDTree for large ones.  The outlier rule restates the reference's
post_process (gaussian_renderer/__init__.py:315-322) as opengaussian_b200.renderer._post_process states it:
K = int(n ** 0.5) on a count tensor; mean and unbiased std over all n * K values of the [n, K] distance matrix; keep
the points whose mean over K is below mean + std.
"""
import numpy as np
import torch

BRUTE_MAX = 4096          # candidates up to which the oracle uses brute force


def knn(q, p, K):
    """q [Q,3], p [M,3] (array-likes) -> (dists [Q,k] float64 ascending, idx [Q,k] int64, tie [Q] bool), k = min(K, M).
    Ties in distance are ordered by index.  tie[i]: two of the k + 1 nearest distances of row i agree to a relative
    1e-6 (float32 resolution), so that a float32 computation may order or select them differently."""
    q = np.asarray(q, dtype=np.float32).astype(np.float64)
    p = np.asarray(p, dtype=np.float32).astype(np.float64)
    Q, M = q.shape[0], p.shape[0]
    k = min(K, M)
    k1 = min(k + 1, M)
    if M <= BRUTE_MAX:
        chunk = max(1, (1 << 22) // max(M, 1))
        dd, ii = np.zeros((0, k1)), np.zeros((0, k1), np.int64)
        for i0 in range(0, Q, chunk):
            di = ((q[i0:i0 + chunk, None, :] - p[None, :, :]) ** 2).sum(-1)
            order = np.lexsort((np.broadcast_to(np.arange(M), di.shape), di), axis=-1)[:, :k1]
            dd = np.concatenate((dd, np.take_along_axis(di, order, 1)))
            ii = np.concatenate((ii, order))
    else:
        from scipy.spatial import cKDTree
        dist, ii = cKDTree(p).query(q, k=k1, workers=-1)
        dist, ii = dist.reshape(Q, k1), ii.reshape(Q, k1)
        dd = ((q[:, None, :] - p[ii]) ** 2).sum(-1)            # exact squares from the coordinates
        order = np.lexsort((ii, dd), axis=-1)
        dd, ii = np.take_along_axis(dd, order, 1), np.take_along_axis(ii, order, 1)
    gaps = np.diff(dd, axis=1) <= 1e-6 * np.maximum(dd[:, 1:], 1e-30)
    tie = gaps.any(axis=1) if k1 > 1 else np.zeros(Q, bool)
    return dd[:, :k], ii[:, :k].astype(np.int64), tie


def sqrt_k(n):
    """The reference's K for a cloud of n points: int(n ** 0.5) with n a count tensor (float32 square root)."""
    return int(torch.tensor(n) ** 0.5)


def knn_sums(p):
    """Per point of the cloud p [n,3]: (sum, sum of squares) of its K = sqrt_k(n) smallest squared distances."""
    n = len(p)
    if n == 0:
        return np.zeros(0), np.zeros(0)
    d, _, _ = knn(p, p, sqrt_k(n))
    return d.sum(1), (d * d).sum(1)


def post_process_keep(p):
    """The reference's outlier rule on one cloud p [n,3] -> (keep [n] bool, per-point mean [n], threshold)."""
    n = len(p)
    d, _, _ = knn(p, p, sqrt_k(n))
    per_point = d.mean(1)
    thr = d.mean() + d.std(ddof=1)
    return per_point < thr, per_point, thr
