"""Exact k-nearest-neighbour search on the B200 (csrc/knn.cu, C ABI ogs_knn_segmented).

``knn_points`` is a drop-in for ``pytorch3d.ops.knn_points`` as pytorch3d documents it:

* ``p1 [N,P1,D]``, ``p2 [N,P2,D]``, optional ``lengths1 [N]`` / ``lengths2 [N]`` (int64; the rows of cloud n beyond
  them are padding).  D must be 3, the only dimension OpenGaussian uses; anything else is a ValueError.
* Returns ``KNN(dists [N,P1,K], idx [N,P1,K] int64, knn [N,P1,K,3] or None)``: squared distances of the K nearest
  points of ``p2[n, :lengths2[n]]`` to each ``p1[n, i]``, ascending; ties in distance go to the lower index.  A query
  that is also a candidate finds itself at distance 0.
* Padding: where ``lengths2[n] < K`` the entries from ``lengths2[n]`` on, and every entry of the rows
  ``i >= lengths1[n]``, hold 0 in ``dists``, ``idx`` and ``knn``.
* ``dists`` is differentiable in ``p1`` and ``p2`` (when grad is enabled and either requires it, it is recomputed from
  ``idx`` with torch ops, and autograd differentiates that); ``idx`` is not.  ``knn`` (``return_nn=True``) is the
  gathered ``p2`` rows, differentiable the same way.
* ``version`` selects among pytorch3d's kernels and is ignored here; ``return_sorted=False`` still returns sorted
  neighbours (an ordering pytorch3d's unsorted result may also have).
* CUDA tensors only.

``slot_knn_sums`` serves render()'s post_process for every leaf of a view in one launch.
"""
from collections import namedtuple

import torch

from . import _lib

KNN = namedtuple("KNN", ["dists", "idx", "knn"])


def _launch(q, q_seg, S, p, p_off, k_seg, k_max=0, sum_=None, sumsq=None, nn_dist=None, nn_idx=None):
    _lib.launch("ogs_knn_segmented", q.device, q.shape[0], _lib.ptr(q), _lib.ptr(q_seg), S, _lib.ptr(p), _lib.ptr(p_off),
                _lib.ptr(k_seg), k_max, None, _lib.ptr(sum_), _lib.ptr(sumsq), _lib.ptr(nn_dist), _lib.ptr(nn_idx))


def sqrt_k(n):
    """K = int(n ** 0.5) for an int64 tensor of counts, evaluated as the reference's post_process evaluates it on a
    count tensor: ``n ** 0.5`` is float32, then truncated.  From n = 4097**2 - 1 on this differs from an integer
    square root for some n just below a square; the reference's value is the one kept."""
    return (n.to(torch.int64) ** 0.5).to(torch.int32)


def knn_points(p1, p2, lengths1=None, lengths2=None, K=1, version=-1, return_nn=False, return_sorted=True):
    """pytorch3d.ops.knn_points for D = 3 (see the module docstring for the contract)."""
    if p1.dim() != 3 or p2.dim() != 3 or p1.shape[0] != p2.shape[0]:
        raise ValueError("knn_points: p1 and p2 must be [N, P, D] with the same N")
    if p1.shape[2] != p2.shape[2]:
        raise ValueError("knn_points: p1 and p2 must have the same point dimension")
    if p1.shape[2] != 3:
        raise ValueError(f"knn_points: only D = 3 is supported (got D = {p1.shape[2]})")
    if K < 1:
        raise ValueError("knn_points: K must be at least 1")
    if not (p1.is_cuda and p2.is_cuda):
        raise _lib.OgsError("knn_points needs CUDA tensors (no CPU path)")
    N, P1, P2, dev = p1.shape[0], p1.shape[1], p2.shape[1], p1.device
    len1 = torch.full((N,), P1, dtype=torch.int64, device=dev) if lengths1 is None else lengths1.to(dev, torch.int64)
    len2 = torch.full((N,), P2, dtype=torch.int64, device=dev) if lengths2 is None else lengths2.to(dev, torch.int64)
    len1, len2 = len1.clamp(0, P1), len2.clamp(0, P2)
    dists = torch.zeros(N, P1, K, dtype=torch.float32, device=dev)
    idx = torch.zeros(N, P1, K, dtype=torch.int64, device=dev)
    if N * P1 > 0 and P2 > 0:
        # segment 2n = p2[n, :len2[n]], segment 2n + 1 = the padding behind it: CSR offsets over the flat p2
        start = torch.arange(N, device=dev, dtype=torch.int64) * P2
        p_off = torch.stack((start, start + len2), 1).reshape(-1)
        p_off = torch.cat((p_off, p_off.new_full((1,), N * P2)))
        k_seg = torch.stack((len2.clamp(max=K), torch.zeros_like(len2)), 1).reshape(-1).to(torch.int32)
        rows = torch.arange(P1, device=dev)
        q_seg = torch.where(rows[None, :] < len1[:, None], 2 * torch.arange(N, device=dev)[:, None], -1)
        q = p1.detach().float().contiguous().view(-1, 3)
        p = p2.detach().float().contiguous().view(-1, 3)
        _launch(q, q_seg.to(torch.int32).view(-1), 2 * N, p, p_off, k_seg, K, nn_dist=dists, nn_idx=idx)
    need_grad = torch.is_grad_enabled() and (p1.requires_grad or p2.requires_grad)
    knn = None
    if return_nn or need_grad:
        valid = (torch.arange(K, device=dev)[None, None, :] < len2.clamp(max=K)[:, None, None]) & \
                (torch.arange(P1, device=dev)[None, :, None] < len1[:, None, None])
        knn = p2[torch.arange(N, device=dev)[:, None, None], idx] if P2 > 0 else p2.new_zeros(N, P1, K, 3)
        knn = knn * valid.unsqueeze(-1)
        if need_grad:
            dists = ((p1.unsqueeze(2) - knn) ** 2).sum(-1) * valid
    return KNN(dists.to(p1.dtype), idx, knn if return_nn else None)


def slot_knn_sums(points, subset, S):
    """For each point i with subset[i] = s in [0, S): the sum and the sum of squares (fp64) of the squared distances to
    its K_s nearest points of slot s (itself included), K_s = sqrt_k(n_s) with n_s the slot's size.  -> (sum [P],
    sumsq [P], n [S] int64, K [S] int32); points of no slot get 0.  One launch for all slots, no host read."""
    if not points.is_cuda:
        raise _lib.OgsError("slot_knn_sums needs CUDA tensors (no CPU path)")
    dev, P = points.device, points.shape[0]
    key = torch.where((subset >= 0) & (subset < S), subset, S).to(torch.int32)
    order = torch.sort(key, stable=True).indices
    seg = key[order].contiguous()
    n = torch.zeros(S + 1, dtype=torch.int64, device=dev).index_add_(0, key.long(), torch.ones_like(key, dtype=torch.int64))
    p_off = torch.cat((n.new_zeros(1), torch.cumsum(n, 0)))
    k = sqrt_k(n[:S])
    k_seg = torch.cat((k, k.new_zeros(1)))          # segment S: the points of no slot, as candidates of nobody
    pts = points.detach().float()[order].contiguous()
    s1 = torch.empty(P, dtype=torch.float64, device=dev)
    s2 = torch.empty(P, dtype=torch.float64, device=dev)
    if P > 0:
        _launch(pts, seg, S + 1, pts, p_off, k_seg, sum_=s1, sumsq=s2)
    sum_ = torch.empty_like(s1).index_copy_(0, order, s1)
    sumsq = torch.empty_like(s2).index_copy_(0, order, s2)
    return sum_, sumsq, n[:S], k
