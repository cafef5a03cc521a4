"""All cluster / leaf subsets of a view in one rasterizer call (GaussianRasterizer.forward_subsets, C ABI
ogs_raster_forward_subsets) and render()'s batched no-grad passes built on it.  A subset's images must be BIT-identical
to a separate forward over that subset's rows, and render()'s dict must be identical, key for key, to the per-subset
loop (gaussian_renderer/__init__.py:173-236,245-356)."""
import math
import types

import pytest
import torch

from opengaussian_b200 import renderer, synth
from opengaussian_b200.rasterizer import GaussianRasterizationSettings, GaussianRasterizer

pytestmark = pytest.mark.gpu

KEYS = ["render", "alpha", "depth", "silhouette", "ins_feat", "cluster_imgs", "cluster_silhouettes",
        "leaf_clusters_imgs", "leaf_cluster_silhouettes", "occured_leaf_id", "cluster_occur", "viewspace_points",
        "visibility_filter", "radii"]
PIPE = types.SimpleNamespace(debug=False, compute_cov3D_python=False, convert_SHs_python=False)


def _rasterizer(cam, bg, dev, sh_degree=3):
    rs = GaussianRasterizationSettings(
        image_height=int(cam.image_height), image_width=int(cam.image_width), tanfovx=math.tan(cam.FoVx * 0.5),
        tanfovy=math.tan(cam.FoVy * 0.5), bg=bg, scale_modifier=1.0, viewmatrix=cam.world_view_transform.to(dev),
        projmatrix=cam.full_proj_transform.to(dev), sh_degree=sh_degree, campos=cam.camera_center.to(dev),
        prefiltered=False, debug=False)
    return GaussianRasterizer(rs)


def _voxel_ids(xyz, n):
    """Spatially coherent subsets: the cells of an n x n x n grid over the points' bounding box."""
    lo, hi = xyz.min(0).values, xyz.max(0).values
    c = ((xyz - lo) / (hi - lo) * n).long().clamp(0, n - 1)
    return (c[:, 0] * n + c[:, 1]) * n + c[:, 2]


def _gs(gs, dev):
    return {k: v.to(dev) if isinstance(v, torch.Tensor) else v for k, v in gs.items()}


def _check_against_separate_forwards(rast, g, subset, S, sh, bg, ebg=None):
    """forward_subsets vs GaussianRasterizer.forward on each slot's gathered rows: bit-identical."""
    kw = dict(shs=g["shs"]) if sh else dict(colors_precomp=g["ins_feat"][:, :3], extra_feats=g["ins_feat"][:, 3:6],
                                            extra_bg=ebg)
    with torch.no_grad():
        color, depth, alpha, extra = rast.forward_subsets(g["means3D"], g["opacities"], subset, S, scales=g["scales"],
                                                          rotations=g["rotations"], **kw)
    H, W = rast.raster_settings.image_height, rast.raster_settings.image_width
    assert color.shape == (S, 3, H, W) and depth.shape == (S, 1, H, W) and alpha.shape == (S, 1, H, W)
    assert (extra is None) == sh and (sh or extra.shape == (S, 3, H, W))
    for k in range(S):
        idx = subset == k
        args = dict(means3D=g["means3D"][idx], means2D=torch.zeros_like(g["means3D"][idx]),
                    opacities=g["opacities"][idx], scales=g["scales"][idx], rotations=g["rotations"][idx])
        if sh:
            want = rast(shs=g["shs"][idx], **args)
        else:
            want = rast(colors_precomp=g["ins_feat"][idx, :3], extra_feats=g["ins_feat"][idx, 3:6], extra_bg=ebg, **args)
        assert torch.equal(color[k], want[0]), k
        assert torch.equal(depth[k], want[2]), k
        assert torch.equal(alpha[k], want[3]), k
        if not sh:
            assert torch.equal(extra[k], want[4]), k
        if not bool(idx.any()):                                 # empty slot: the background, alpha 0
            assert torch.equal(color[k], bg[:, None, None].expand(3, H, W)) and float(alpha[k].abs().max()) == 0.0
    return color, alpha


@pytest.mark.parametrize("sh", [False, True])
def test_forward_subsets_equals_separate_forwards(sh):
    dev = torch.device("cuda")
    P = 6000
    g = _gs(synth.make_gaussians(P, "blender", 4, scale_mult=1.2), dev)
    cam = synth.orbit_cameras(3, 4.0, 150, 110, 0.69, 1.0)[1]             # 150 x 110: not a multiple of 16
    bg = torch.tensor([0.2, 0.5, 0.8], device=dev)
    ebg = torch.tensor([0.3, 0.1, 0.7], device=dev)
    rast = _rasterizer(cam, bg, dev)
    gen = torch.Generator(device=dev).manual_seed(1)

    # 9 slots: slot 5 empty, slot 8 holds exactly one Gaussian, ~10 % not rendered
    subset = torch.randint(0, 8, (P,), device=dev, generator=gen, dtype=torch.int32)
    subset[subset == 5] = 4
    subset[torch.rand(P, device=dev, generator=gen) < 0.1] = -1
    subset[1234] = 8
    _check_against_separate_forwards(rast, g, subset, 9, sh, bg, ebg)
    # coherent subsets
    _check_against_separate_forwards(rast, g, _voxel_ids(g["means3D"], 3).int(), 27, sh, bg, ebg)
    # S = 1, all Gaussians excluded, and an id outside [0, S) counts as excluded
    _check_against_separate_forwards(rast, g, torch.zeros(P, dtype=torch.int32, device=dev), 1, sh, bg, ebg)
    color, alpha = _check_against_separate_forwards(rast, g, torch.full((P,), -1, dtype=torch.int32, device=dev), 3,
                                                    sh, bg, ebg)
    assert float(alpha.abs().max()) == 0.0
    out_of_range = subset.clone()
    out_of_range[:100] = 9
    out_of_range[100:150] = -7
    _check_against_separate_forwards(rast, g, out_of_range, 9, sh, bg, ebg)
    # S = 640 with most slots empty (the reference's root_num x leaf_num)
    used = torch.randperm(640, generator=torch.Generator().manual_seed(2))[:20].to(dev).int()
    many = used[torch.randint(0, 20, (P,), device=dev, generator=gen)]
    _check_against_separate_forwards(rast, g, many, 640, sh, bg, ebg)


def test_forward_subsets_long_tile_lists():
    """300 k Gaussians at 800 x 800 in 64 spatial cells: tile lists run over many 256-entry blend rounds."""
    dev = torch.device("cuda")
    gs, cams = synth.make_scene("blender_300k_800", n_views=2)
    g = _gs(gs, dev)
    bg = torch.tensor([0.1, 0.3, 0.2], device=dev)
    rast = _rasterizer(cams[0], bg, dev)
    subset = _voxel_ids(g["means3D"], 4).int()
    subset[::97] = -1
    color, alpha = _check_against_separate_forwards(rast, g, subset, 64, False, bg, torch.tensor([0.5, 0.5, 0.5],
                                                                                                   device=dev))
    assert float(alpha.amax()) > 0.5


def test_forward_subsets_rejects_grad():
    dev = torch.device("cuda")
    g = _gs(synth.make_gaussians(100, "blender", 0), dev)
    rast = _rasterizer(synth.orbit_cameras(1, 4.0, 32, 32, 0.69)[0], torch.zeros(3, device=dev), dev)
    feat = g["ins_feat"][:, :3].clone().requires_grad_(True)
    subset = torch.zeros(100, dtype=torch.int32, device=dev)
    with pytest.raises(RuntimeError, match="no backward"):
        rast.forward_subsets(g["means3D"], g["opacities"], subset, 1, colors_precomp=feat, scales=g["scales"],
                             rotations=g["rotations"])
    with pytest.raises(Exception, match="excatly one of either SHs or precomputed colors"):
        rast.forward_subsets(g["means3D"], g["opacities"], subset, 1, scales=g["scales"], rotations=g["rotations"])


# ---------------------------------------------------------------------------------------------------------------------
# render(): batched (no grad) against the per-subset loop (grad enabled, _ins_feat requiring grad)

def _render_scene(dev, P=20000, seed=3):
    gs = synth.make_gaussians(P, "blender", seed, scale_mult=1.0)
    cam = synth.orbit_cameras(3, 4.0, 200, 150, 0.69, 1.0)[0]
    xyz = gs["means3D"]
    cluster_idx = _voxel_ids(xyz, 4)                            # 64 coherent coarse clusters
    big = int(torch.bincount(cluster_idx).argmax())
    small = torch.nonzero(cluster_idx == (big + 1) % 64)[:50, 0]
    cluster_idx[small] = 64                                     # a cluster under the 100-point rule
    logit = torch.logit(gs["opacities"].clamp(1e-4, 1 - 1e-4))
    logit[cluster_idx == big] = math.log(0.004 / 0.996)         # a cluster whose silhouette stays <= 0.8
    order = torch.argsort(xyz[:, 0], stable=True)
    rank = torch.empty_like(order)
    rank[order] = torch.arange(P)
    leaf_idx = cluster_idx * 10 + rank % 10
    model = synth.SynthModel(gs, dev)
    model._opacity = logit.to(dev)
    c = types.SimpleNamespace(FoVx=cam.FoVx, FoVy=cam.FoVy, image_height=cam.image_height, image_width=cam.image_width,
                              world_view_transform=cam.world_view_transform.to(dev),
                              full_proj_transform=cam.full_proj_transform.to(dev),
                              camera_center=cam.camera_center.to(dev), bClusterOccur=None)
    return model, c, cluster_idx.to(dev), leaf_idx.to(dev), big


def _equal(a, b, key):
    if isinstance(a, list):
        assert isinstance(b, list) and len(a) == len(b), key
        for x, y in zip(a, b):
            _equal(x, y, key)
    elif isinstance(a, torch.Tensor):
        assert isinstance(b, torch.Tensor) and a.shape == b.shape and a.dtype == b.dtype, key
        assert torch.equal(a.detach(), b.detach()), key
    else:
        assert a == b, key


def _both_paths(model, cam, bg, seed, **kw):
    torch.manual_seed(seed)
    with torch.no_grad():
        fast = renderer.render(cam, model, PIPE, bg, 1000, **kw)
    torch.manual_seed(seed)
    loop = renderer.render(cam, model, PIPE, bg, 1000, **kw)        # _ins_feat requires grad: the loop
    assert list(fast.keys()) == KEYS
    for k in KEYS:
        _equal(fast[k], loop[k], k)
    return fast, loop


def _rescale_seed():
    for s in range(100):
        torch.manual_seed(s)
        if torch.rand(1) > 0.5:
            return s
    raise AssertionError


def test_render_batched_equals_loop():
    dev = torch.device("cuda")
    model, cam, cluster_idx, leaf_idx, low = _render_scene(dev)
    assert model._ins_feat.requires_grad
    bg = torch.tensor([0.1, 0.3, 0.2], device=dev)
    common = dict(cluster_idx=cluster_idx, root_num=65, leaf_num=10, rescale=False)

    # the coarse sweep of construct_pseudo_ins_feat: many clusters, some under 100 points, one too faint
    fast, loop = _both_paths(model, cam, bg, 0, render_cluster=True, better_vis=True, **common)
    n_kept = len(fast["cluster_imgs"])
    assert n_kept > 10 and loop["cluster_imgs"][0].requires_grad and not fast["cluster_imgs"][0].requires_grad
    assert not bool(fast["cluster_occur"][low]) and not bool(fast["cluster_occur"][64])
    # the same with render()'s rescale draw (scales * factor)
    s = _rescale_seed()
    fast, _ = _both_paths(model, cam, bg, s, render_cluster=True, better_vis=True, **dict(common, rescale=True))
    assert fast["ins_feat"] is not None
    # better_vis=False with selected_root_id, and per-root leaves
    for r in (int(cluster_idx[0]), low):
        _both_paths(model, cam, bg, 0, render_cluster=True, better_vis=False, selected_root_id=r,
                    leaf_cluster_idx=leaf_idx, **common)
    # all leaves; pre_mask; post_process + better_vis; seg_rgb; selected_leaf_id
    fast, _ = _both_paths(model, cam, bg, 0, leaf_cluster_idx=leaf_idx, **common)
    assert len(fast["occured_leaf_id"]) > 100
    pre_mask = model._xyz[:, 2] > 0
    _both_paths(model, cam, bg, 0, leaf_cluster_idx=leaf_idx, pre_mask=pre_mask, selected_root_id=5, **common)
    fast, _ = _both_paths(model, cam, bg, 0, leaf_cluster_idx=leaf_idx, post_process=True,
                          selected_root_id=int(cluster_idx[7]), **common)
    assert len(fast["occured_leaf_id"]) > 0
    fast, _ = _both_paths(model, cam, bg, 0, leaf_cluster_idx=leaf_idx, seg_rgb=True, selected_root_id=9, **common)
    assert fast["leaf_clusters_imgs"][0].shape == (6, 150, 200)
    vis = torch.nonzero(fast["radii"] > 0)[:, 0]
    sel = torch.tensor([int(leaf_idx[vis[0]]), int(leaf_idx[vis[1]])], device=dev)
    fast, _ = _both_paths(model, cam, bg, 0, leaf_cluster_idx=leaf_idx, selected_leaf_id=sel, post_process=True,
                          **common)
    assert fast["occured_leaf_id"] == [sel[0].item()]
    # a camera on which some clusters do not occur
    cam.bClusterOccur = torch.tensor([i % 5 != 2 for i in range(65)])
    fast, _ = _both_paths(model, cam, bg, 0, render_cluster=True, better_vis=True, **common)
    assert len(fast["cluster_imgs"]) < n_kept
    for r in (2, 3):                                             # cluster 2 does not occur: no leaf passes at all
        fast, _ = _both_paths(model, cam, bg, 0, leaf_cluster_idx=leaf_idx, selected_root_id=r, **common)
        assert (fast["occured_leaf_id"] == []) == (r == 2)


def test_gradient_pass_takes_the_loop():
    dev = torch.device("cuda")
    model, cam, cluster_idx, leaf_idx, _ = _render_scene(dev, P=8000)
    bg = torch.zeros(3, device=dev)
    torch.manual_seed(0)
    out = renderer.render(cam, model, PIPE, bg, 1000, cluster_idx=cluster_idx, render_cluster=True, better_vis=True,
                          rescale=False, root_num=65)
    assert out["cluster_imgs"] and out["cluster_imgs"][0].requires_grad
    out["cluster_imgs"][0].sum().backward()
    assert model._ins_feat.grad is not None and float(model._ins_feat.grad.abs().max()) > 0


def test_budget_split(monkeypatch):
    dev = torch.device("cuda")
    model, cam, cluster_idx, leaf_idx, _ = _render_scene(dev)
    bg = torch.tensor([0.1, 0.3, 0.2], device=dev)
    kws = (dict(cluster_idx=cluster_idx, render_cluster=True, better_vis=True, rescale=False, root_num=65),
           dict(cluster_idx=cluster_idx, leaf_cluster_idx=leaf_idx, rescale=False, root_num=65, leaf_num=10))
    outs = []
    calls = []
    real = GaussianRasterizer.forward_subsets

    def counting(self, *a, **k):
        calls.append(a[3] if len(a) > 3 else k["num_subsets"])
        return real(self, *a, **k)

    monkeypatch.setattr(GaussianRasterizer, "forward_subsets", counting)
    for budget in (renderer.SUBSET_BATCH_BYTES, 7 * (6 + 2) * 150 * 200 * 4):     # default; 7 slots per launch
        monkeypatch.setattr(renderer, "SUBSET_BATCH_BYTES", budget)
        for kw in kws:
            calls.clear()
            torch.manual_seed(0)
            with torch.no_grad():
                outs.append((renderer.render(cam, model, PIPE, bg, 1000, **kw), list(calls)))
    for (a, ca), (b, cb) in zip(outs[:2], outs[2:]):
        assert len(ca) == 1 and len(cb) > 4 and max(cb) == 7 and sum(cb) == ca[0]
        for k in KEYS:
            _equal(a[k], b[k], k)
    assert len(outs[0][0]["cluster_imgs"]) > 7 and len(outs[1][0]["occured_leaf_id"]) > 100


def test_second_device():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    res = []
    for d in (0, 1):
        dev = torch.device("cuda", d)
        g = _gs(synth.make_gaussians(5000, "blender", 4, scale_mult=1.2), dev)
        rast = _rasterizer(synth.orbit_cameras(3, 4.0, 96, 80, 0.69, 1.0)[0], torch.tensor([0.2, 0.5, 0.8], device=dev),
                           dev)
        subset = _voxel_ids(g["means3D"], 2).int()
        with torch.cuda.device(0), torch.no_grad():
            color, depth, alpha, extra = rast.forward_subsets(
                g["means3D"], g["opacities"], subset, 8, colors_precomp=g["ins_feat"][:, :3],
                extra_feats=g["ins_feat"][:, 3:], scales=g["scales"], rotations=g["rotations"])
            assert torch.cuda.current_device() == 0
        res.append([t.cpu() for t in (color, depth, alpha, extra)])
    for a, b in zip(*res):
        assert torch.equal(a, b)


# ---------------------------------------------------------------------------------------------------------------------
# the reference's own render() (tests/golden/make_render_golden.py) for the cluster / leaf cases, on the batched path
def _golden_module():
    import importlib.util
    import os
    gdir = os.path.join(os.path.dirname(__file__), "golden")
    spec = importlib.util.spec_from_file_location("mrg_render", os.path.join(gdir, "make_render_golden.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m, os.path.join(gdir, "render_golden.npz")


@pytest.mark.parametrize("name", ["stage22_cluster", "stage3_all_leaves", "better_vis_seg_rgb"])
def test_batched_render_vs_reference_golden(name):
    import numpy as np
    m, path = _golden_module()
    gold = np.load(path)
    case = m.CASES[name]
    dev = torch.device("cuda")
    gs, cam, cluster_idx, leaf_idx = m.scene()
    pc = m.fill_model(types.SimpleNamespace(), gs, case.get("with_q", False))
    for k in ("_xyz", "_scaling", "_rotation", "_opacity", "_features_dc", "_features_rest", "_ins_feat", "_ins_feat_q"):
        setattr(pc, k, getattr(pc, k).detach().to(dev))
    model = synth.SynthModel.__new__(synth.SynthModel)
    model.__dict__.update(pc.__dict__)
    if model._ins_feat_q.numel() == 0:
        model._ins_feat_q = None
    kw = dict(case["kw"])
    if case.get("clusters"):
        kw["cluster_idx"] = cluster_idx.to(dev)
    if case.get("leaves"):
        kw["leaf_cluster_idx"] = leaf_idx.to(dev)
    if case.get("selected_leaf") is not None:
        kw["selected_leaf_id"] = torch.tensor(case["selected_leaf"], device=dev)
    kw.update(root_num=m.K1, leaf_num=m.K2)
    bg = torch.tensor([0.1, 0.3, 0.2], device=dev)
    c = types.SimpleNamespace(FoVx=cam.FoVx, FoVy=cam.FoVy, image_height=cam.image_height, image_width=cam.image_width,
                              world_view_transform=cam.world_view_transform.to(dev),
                              full_proj_transform=cam.full_proj_transform.to(dev),
                              camera_center=cam.camera_center.to(dev), bClusterOccur=None)
    torch.manual_seed(int(gold[f"{name}/seed"]))
    with torch.no_grad():
        out = renderer.render(c, model, PIPE, bg, 1000, **kw)
    assert list(out.keys()) == KEYS

    def img_close(got, want, what):                              # as test_render_gpu.test_render_vs_reference_golden
        want = torch.from_numpy(want).to(dev)
        assert got.shape == want.shape, (what, got.shape, want.shape)
        scale = max(1.0, float(want.abs().max()))
        diff = (got - want).abs().reshape(-1, want.shape[-2], want.shape[-1]).amax(0)
        bad = float((diff > 1e-5 * scale).float().mean())
        assert bad <= 0.03, (what, bad)
        assert float(diff.max()) < 0.05 * scale, (what, float(diff.max()))

    checked = 0
    for k in KEYS:
        if f"{name}/{k}/none" in gold:
            assert out[k] is None, k
            continue
        if f"{name}/{k}/len" in gold:
            n = int(gold[f"{name}/{k}/len"])
            assert isinstance(out[k], list) and len(out[k]) == n, (k, n)
            for i in range(n):
                want = gold[f"{name}/{k}/{i}"]
                if k == "occured_leaf_id":
                    assert int(out[k][i]) == int(want)
                else:
                    img_close(out[k][i], want, f"{k}[{i}]")
                checked += 1
            continue
        want = gold[f"{name}/{k}"]
        got = out[k]
        if k in ("radii", "visibility_filter", "cluster_occur"):
            assert np.array_equal(got.cpu().numpy(), want), k
        elif k == "viewspace_points":
            assert tuple(got.shape) == want.shape and float(got.abs().max()) == 0.0
        else:
            img_close(got, want, k)
        checked += 1
    assert checked >= 4
