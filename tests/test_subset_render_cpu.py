"""CPU tests (no GPU) of render()'s batched cluster / leaf passes: the planner reproduces the reference loop's choice of
subsets (gaussian_renderer/__init__.py:173-236,245-356) as one partition of the Gaussians, and the C entry point
ogs_raster_forward_subsets rejects bad arguments without touching a device."""
import ctypes as C

import pytest
import torch

from opengaussian_b200 import renderer


def _scene(P=3000, seed=0, n_clusters=12, leaf_num=4):
    g = torch.Generator().manual_seed(seed)
    cluster_idx = torch.randint(0, n_clusters, (P,), generator=g)
    # skewed cluster sizes: some clusters fall under the 100-point and 10-point thresholds
    small = torch.rand(P, generator=g) < 0.5
    cluster_idx = torch.where(small & (cluster_idx % 3 == 0), cluster_idx, cluster_idx - cluster_idx % 3)
    cluster_idx[cluster_idx == 3] = torch.where(torch.rand(int((cluster_idx == 3).sum()), generator=g) < 0.1, 3, 4)
    leaf_idx = cluster_idx * leaf_num + torch.randint(0, leaf_num, (P,), generator=g)
    viewed = torch.rand(P, generator=g) < 0.8
    scales = torch.rand(P, 3, generator=g) * 0.7
    xyz = torch.randn(P, 3, generator=g)
    return cluster_idx, leaf_idx, viewed, scales, xyz


def _check_partition(ids, subset, filters):
    assert subset.dtype == torch.int32
    assert len(ids) == len(filters)
    union = torch.zeros_like(subset, dtype=torch.bool)
    for k, f in enumerate(filters):
        assert torch.equal(subset == k, f), k
        union |= f
    assert torch.equal(subset >= 0, union)


def _loop_clusters(cluster_idx, viewed, scale_filter, better_vis, selected_root_id, occur):
    """The reference's coarse loop (:187-236) up to the rasterizer call."""
    ids, filters = [], []
    for idx in range(int(cluster_idx.max()) + 1):
        if not better_vis and idx != selected_root_id:
            continue
        if occur is not None and occur[idx] == False:  # noqa: E712
            continue
        f = (cluster_idx == idx) & viewed
        if better_vis:
            f = f & scale_filter
            if f.sum() < 100:
                continue
        ids.append(idx)
        filters.append(f)
    return ids, filters


@pytest.mark.parametrize("better_vis,selected_root_id,with_occur", [(True, None, False), (True, None, True),
                                                                   (False, 4, False), (False, 5, True)])
def test_cluster_plan_matches_loop(better_vis, selected_root_id, with_occur):
    cluster_idx, _, viewed, scales, _ = _scene()
    n = int(cluster_idx.max()) + 1
    occur = torch.tensor([i % 4 != 1 for i in range(n)]) if with_occur else None
    scale_filter = (scales < 0.5).all(dim=1)
    ids, subset = renderer._plan_clusters(cluster_idx, n, viewed, scale_filter, better_vis, selected_root_id, occur)
    want_ids, filters = _loop_clusters(cluster_idx, viewed, scale_filter, better_vis, selected_root_id, occur)
    assert ids == want_ids
    if better_vis:
        assert 0 < len(ids) < n          # the 100-point rule dropped some clusters
    _check_partition(ids, subset, filters)


def _loop_leaves(leaf_idx, lerf_range, selected_leaf_id, pre_mask, viewed, scale_filter, better_vis, post_process, xyz):
    """The reference's leaf loop (:300-345) up to the rasterizer call."""
    ids, filters = [], []
    for leaf in lerf_range:
        if selected_leaf_id is None:
            f = leaf_idx == leaf
        else:
            f = (leaf_idx.unsqueeze(1) == selected_leaf_id).any(dim=1)
        if pre_mask is not None:
            f = f & pre_mask
        f = f & viewed
        if better_vis:
            f = f & scale_filter
            if f.sum() < 100:
                continue
        if post_process:
            d = renderer._knn_mean_dists(xyz[f], int(f.sum() ** 0.5))
            mask = (d.mean(dim=-1) < d.mean() + d.std()).squeeze()
            f[f != 0] = mask
        if f.sum() < 10:
            continue
        ids.append(leaf)
        filters.append(f)
        if selected_leaf_id is not None:
            break
    return ids, filters


@pytest.mark.parametrize("case", ["all", "root", "better_vis", "pre_mask", "post_process", "selected", "selected_post",
                                  "selected_empty"])
def test_leaf_plan_matches_loop(case):
    cluster_idx, leaf_idx, viewed, scales, xyz = _scene(seed=1)
    leaf_num, root_num = 4, int(cluster_idx.max()) + 1
    scale_filter = (scales < 0.6).all(dim=1)
    better_vis = case == "better_vis"
    pre_mask = (xyz[:, 0] > -0.5) if case == "pre_mask" else None
    post_process = case in ("post_process", "selected_post")
    selected = None
    lerf_range = list(range(root_num * leaf_num)) if case != "root" else list(range(4 * leaf_num, 5 * leaf_num))
    if case == "post_process":          # the outlier removal needs a non-empty leaf (the reference's kNN fails on none)
        lerf_range = sorted(set(leaf_idx[viewed & scale_filter].tolist()))
    if case.startswith("selected"):
        selected = torch.tensor([13, 17] if case != "selected_empty" else [1000])
        lerf_range = selected.tolist()
    ids, subset = renderer._plan_leaves(leaf_idx, lerf_range, selected, pre_mask, viewed, scale_filter, better_vis,
                                        post_process, xyz)
    want_ids, filters = _loop_leaves(leaf_idx, lerf_range, selected, pre_mask, viewed, scale_filter, better_vis,
                                     post_process, xyz)
    assert ids == want_ids
    if case == "selected_empty":
        assert ids == []
    else:
        assert len(ids) > 0
    if case == "all":
        assert len(ids) < len(lerf_range)   # the 10-point rule dropped leaves
    _check_partition(ids, subset, filters)


@pytest.fixture(scope="module")
def lib():
    from opengaussian_b200 import build, _lib
    build.build()
    return _lib.lib()


def test_forward_subsets_argument_validation_without_device(lib):
    from opengaussian_b200 import _lib
    ri = _lib.RasterInputs()
    ri.P, ri.W, ri.H = 4, 16, 16
    fake = 256                                       # never dereferenced: every check runs before device work
    ri.bg = ri.viewmatrix = ri.projmatrix = ri.campos = fake
    ri.means3D = ri.opacities = ri.colors_precomp = ri.scales = ri.rotations = fake
    out = _lib.SubsetOutputs(fake, None, fake)
    cb = _lib.ALLOC_FN(lambda u, n, t: None)
    subset = C.c_void_p(fake)

    def call(sub, S, o=out):
        return lib.ogs_raster_forward_subsets(C.byref(ri), sub, S, C.byref(o), cb, None, None)

    assert call(None, 4) == -1 and b"subset is NULL" in lib.ogs_last_error()
    assert call(subset, 0) == -1 and b"out of range" in lib.ogs_last_error()
    assert call(subset, _lib.MAX_SUBSETS + 1) == -1 and b"out of range" in lib.ogs_last_error()
    ri.act_flags = _lib.ACT_OPACITY_SIGMOID
    assert call(subset, 4) == -1 and b"act_flags" in lib.ogs_last_error()
    ri.act_flags = 0
    assert call(subset, 4, _lib.SubsetOutputs(None, None, fake)) == -1 and b"outputs" in lib.ogs_last_error()
    ri.shs = fake                                    # the forward's own checks come first, with its message
    assert call(subset, 4) == -2 and b"excatly one of either SHs or precomputed colors" in lib.ogs_last_error()
