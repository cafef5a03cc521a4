"""GPU tests of the segmented kNN kernel (csrc/knn.cu): knn_points against the fp64 oracle, the per-point sums of
render()'s post_process, and render()'s all-leaves plan against the per-leaf _post_process loop."""
import os
import sys
import types

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import knn as oracle  # noqa: E402
from opengaussian_b200 import knn, renderer, synth  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")


def _check_cloud(q, p, d, idx, K, what):
    """One cloud's rows against the oracle: distances to 1e-6 relative, indices equal outside oracle ties."""
    od, oi, tie = oracle.knn(q, p, K)
    k = od.shape[1]
    d, idx = d[:, :k].cpu().double().numpy(), idx[:, :k].cpu().numpy()
    np.testing.assert_allclose(d, od, rtol=1e-6, atol=1e-12, err_msg=what)
    bad = (idx != oi).any(1)
    assert not (bad & ~tie).any(), (what, np.nonzero(bad & ~tie)[0][:5])
    print(f"{what}: {int(tie.sum())} of {len(tie)} rows with ties, {int(bad.sum())} of them ordered differently")
    return k


@pytest.mark.parametrize("case", ["single", "k_above_p2", "duplicates", "k316"])
def test_knn_points_vs_oracle(case):
    g = torch.Generator().manual_seed(7)
    if case == "single":
        p1, p2, K = torch.randn(1, 1, 3, generator=g), torch.randn(1, 1, 3, generator=g), 1
    elif case == "k_above_p2":
        p1, p2, K = torch.randn(1, 50, 3, generator=g), torch.randn(1, 7, 3, generator=g), 12
    elif case == "duplicates":
        base = torch.randint(0, 6, (1, 3000, 3), generator=g).float() * 0.25      # many exact duplicates and ties
        p1, p2, K = base, base, 40
    else:
        p1 = torch.rand(1, 100_000, 3, generator=g) * 4 - 2
        p2, K = p1, 316
    r = knn.knn_points(p1.to(DEV), p2.to(DEV), K=K, return_nn=True)
    assert r.dists.shape == (1, p1.shape[1], K) and r.idx.dtype == torch.int64 and r.knn.shape == (1, p1.shape[1], K, 3)
    k = _check_cloud(p1[0].numpy(), p2[0].numpy(), r.dists[0], r.idx[0], K, case)
    assert (r.dists[0, :, k:] == 0).all() and (r.idx[0, :, k:] == 0).all() and (r.knn[0, :, k:] == 0).all()
    assert torch.equal(r.knn[0, :, :k], p2.to(DEV)[0][r.idx[0, :, :k]])
    if case == "k316":
        print(f"pairs {p1.shape[1] * p2.shape[1]:.3e}")


def test_knn_points_batched_lengths_and_grad():
    g = torch.Generator().manual_seed(3)
    N, P1, P2, K = 4, 300, 500, 17
    p1, p2 = torch.randn(N, P1, 3, generator=g), torch.randn(N, P2, 3, generator=g)
    len1, len2 = torch.tensor([300, 120, 0, 77]), torch.tensor([500, 9, 250, 1])
    a = p1.to(DEV).requires_grad_()
    b = p2.to(DEV).requires_grad_()
    r = knn.knn_points(a, b, lengths1=len1.to(DEV), lengths2=len2.to(DEV), K=K)
    assert r.knn is None
    for n in range(N):
        l1, l2 = int(len1[n]), int(len2[n])
        if l1:
            _check_cloud(p1[n, :l1].numpy(), p2[n, :l2].numpy(), r.dists[n, :l1].detach(), r.idx[n, :l1], K, f"cloud {n}")
        k = min(K, l2)
        assert (r.dists[n, l1:] == 0).all() and (r.idx[n, l1:] == 0).all()            # padded rows
        assert (r.dists[n, :, k:] == 0).all() and (r.idx[n, :, k:] == 0).all()        # fewer than K candidates
    # the gradient equals autograd through the gathered points
    w = torch.randn(N, P1, K, device=DEV)
    ga, gb = torch.autograd.grad((r.dists * w).sum(), (a, b))
    a2, b2 = p1.to(DEV).requires_grad_(), p2.to(DEV).requires_grad_()
    valid = (torch.arange(K, device=DEV)[None, None] < len2.to(DEV).clamp(max=K)[:, None, None]) & \
            (torch.arange(P1, device=DEV)[None, :, None] < len1.to(DEV)[:, None, None])
    nn = torch.stack([b2[n][r.idx[n]] for n in range(N)])
    ref = ((a2.unsqueeze(2) - nn) ** 2).sum(-1) * valid
    ra, rb = torch.autograd.grad((ref * w).sum(), (a2, b2))
    torch.testing.assert_close(ga, ra)
    torch.testing.assert_close(gb, rb)
    with torch.no_grad():
        r2 = knn.knn_points(a, b, lengths1=len1.to(DEV), lengths2=len2.to(DEV), K=K)
    torch.testing.assert_close(r2.dists, r.dists.detach(), rtol=1e-6, atol=1e-7)
    assert torch.equal(r2.idx, r.idx)


def _grid_leaves(n_leaves=300, seed=0):
    """Leaves of 10 to 20 000 points (log-uniform sizes) with coordinates on a 1/1024 grid in [-1, 1]: there
    cdist's matrix-product form and the direct form compute every squared distance exactly, so the plan comparison
    checks the selection and the statistics rather than cdist's cancellation error."""
    g = torch.Generator().manual_seed(seed)
    sizes = torch.exp(torch.rand(n_leaves, generator=g) * (np.log(20000) - np.log(10)) + np.log(10)).long()
    sizes[:3] = torch.tensor([10, 20000, 11])
    leaf = torch.repeat_interleave(torch.arange(n_leaves), sizes)
    centre = (torch.rand(n_leaves, 3, generator=g) * 1.2 - 0.6)[leaf]
    spread = (torch.rand(n_leaves, 1, generator=g) * 0.3 + 0.05)[leaf]
    xyz = (centre + torch.randn(leaf.shape[0], 3, generator=g) * spread).clamp(-1, 1)
    xyz = torch.round(xyz * 1024) / 1024
    perm = torch.randperm(leaf.shape[0], generator=g)
    return xyz[perm], leaf[perm]


def test_slot_sums_vs_oracle():
    xyz, leaf = _grid_leaves(40, seed=1)
    s1, s2, n, k = knn.slot_knn_sums(xyz.to(DEV), leaf.to(DEV).int(), 40)
    assert torch.equal(n.cpu(), torch.bincount(leaf, minlength=40))
    for s in range(40):
        rows = (leaf == s).nonzero()[:, 0]
        o1, o2 = oracle.knn_sums(xyz[rows].numpy())
        assert int(k[s]) == oracle.sqrt_k(len(rows))
        np.testing.assert_allclose(s1[rows.to(DEV)].cpu().numpy(), o1, rtol=1e-6)
        np.testing.assert_allclose(s2[rows.to(DEV)].cpu().numpy(), o2, rtol=1e-6)
    # a slot map with points of no slot: their sums are 0 and they are nobody's candidates
    sub = torch.where(leaf < 20, leaf, -1).int().to(DEV)
    t1, _, _, _ = knn.slot_knn_sums(xyz.to(DEV), sub, 20)
    assert torch.equal(t1[sub >= 0], s1[sub >= 0]) and (t1[sub < 0] == 0).all()


def _loop_slots(subset, S, means3D):
    """The per-leaf loop the segmented pass replaces: _post_process once per slot (same interface as
    renderer._post_process_slots)."""
    counts = []
    for k in range(S):
        filt = subset == k
        post = renderer._post_process(filt, means3D)
        subset = torch.where(filt & ~post, -1, subset).to(torch.int32)
        counts.append(int(post.sum()))
    return subset, counts


def test_plan_leaves_vs_per_leaf_loop(monkeypatch):
    xyz, leaf = _grid_leaves()
    P = xyz.shape[0]
    xyz, leaf = xyz.to(DEV), leaf.to(DEV)
    viewed = torch.ones(P, dtype=torch.bool, device=DEV)
    lerf = list(range(300))
    args = (leaf, lerf, None, None, viewed, viewed, False, True, xyz)
    ids, sub = renderer._plan_leaves(*args)
    with monkeypatch.context() as m:
        m.setattr(renderer, "_post_process_slots", _loop_slots)
        ids_ref, sub_ref = renderer._plan_leaves(*args)
    assert ids == ids_ref and len(ids) > 250
    # points whose mean over K lies within 1e-5 relative of their leaf's threshold may fall either way
    s1, s2, n, k = knn.slot_knn_sums(xyz, leaf.int(), 300)
    tot = torch.zeros(300, dtype=torch.float64, device=DEV).index_add_(0, leaf, s1)
    tot2 = torch.zeros_like(tot).index_add_(0, leaf, s2)
    cnt = (n * k).double()
    thr = (tot / cnt + ((tot2 - tot * tot / cnt) / (cnt - 1)).sqrt())[leaf]
    near = ((s1 / k[leaf] - thr).abs() <= 1e-5 * thr)
    diff = sub != sub_ref
    print(f"plan: {P} points, {len(ids)} leaves kept, {int(diff.sum())} points differ, {int(near.sum())} near threshold")
    assert not (diff & ~near).any()
    assert int(near.sum()) < 1e-4 * P
    # a leaf with no points: dropped here, where the per-leaf loop raises
    ids2, sub2 = renderer._plan_leaves(leaf, lerf + [999], None, None, viewed, viewed, False, True, xyz)
    assert ids2 == ids and torch.equal(sub2, sub)
    # one selected leaf: the same call with one slot
    sel = torch.tensor([1], device=DEV)
    one = renderer._plan_leaves(leaf, [1], sel, None, viewed, viewed, False, True, xyz)
    with monkeypatch.context() as m:
        m.setattr(renderer, "_post_process_slots", _loop_slots)
        one_ref = renderer._plan_leaves(leaf, [1], sel, None, viewed, viewed, False, True, xyz)
    assert one[0] == one_ref[0] == [1]
    assert not ((one[1] != one_ref[1]) & ~near).any()


KEYS = ["render", "alpha", "depth", "silhouette", "ins_feat", "cluster_imgs", "cluster_silhouettes", "leaf_clusters_imgs",
        "leaf_cluster_silhouettes", "occured_leaf_id", "cluster_occur", "viewspace_points", "visibility_filter", "radii"]
PIPE = types.SimpleNamespace(debug=False, compute_cov3D_python=False, convert_SHs_python=False)


def _equal(a, b, key):
    if isinstance(a, list):
        assert isinstance(b, list) and len(a) == len(b), key
        for x, y in zip(a, b):
            _equal(x, y, key)
    elif isinstance(a, torch.Tensor):
        assert torch.equal(a.detach(), b.detach()), key
    else:
        assert a == b, key


def test_render_post_process_all_leaves_vs_loop(monkeypatch):
    P = 200_000
    gs = synth.make_gaussians(P, "blender", 3, scale_mult=1.0)
    gs["means3D"] = torch.round(gs["means3D"] * 512) / 512      # exact distances in both forms (see _grid_leaves)
    cam = synth.orbit_cameras(3, 4.0, 200, 150, 0.69, 1.0)[0]
    model = synth.SynthModel(gs, DEV)
    leaf_idx = torch.randint(0, 640, (P,), generator=torch.Generator().manual_seed(0)).to(DEV)
    c = types.SimpleNamespace(FoVx=cam.FoVx, FoVy=cam.FoVy, image_height=cam.image_height, image_width=cam.image_width,
                              world_view_transform=cam.world_view_transform.to(DEV),
                              full_proj_transform=cam.full_proj_transform.to(DEV),
                              camera_center=cam.camera_center.to(DEV), bClusterOccur=None)
    bg = torch.tensor([0.1, 0.3, 0.2], device=DEV)
    kw = dict(leaf_cluster_idx=leaf_idx, post_process=True, better_vis=True, rescale=False, root_num=65, leaf_num=10)
    with torch.no_grad():
        torch.manual_seed(0)
        new = renderer.render(c, model, PIPE, bg, 1000, **kw)
        with monkeypatch.context() as m:
            m.setattr(renderer, "_post_process_slots", _loop_slots)
            torch.manual_seed(0)
            old = renderer.render(c, model, PIPE, bg, 1000, **kw)
    assert list(new.keys()) == KEYS
    assert len(new["occured_leaf_id"]) > 100
    for key in KEYS:
        _equal(new[key], old[key], key)
