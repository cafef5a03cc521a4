"""Differentiable subset rendering (GaussianRasterizer.forward_subsets_grad, C ABI ogs_raster_forward_subsets_state /
ogs_raster_backward_subsets) and render()'s gradient-carrying cluster / leaf passes built on it.  Images must be
BIT-identical to forward_subsets and to the per-subset loop; every gradient must equal the per-slot forward() +
backward() up to the order of the blend's atomic additions (helpers.grad_violations, no violation)."""
import math
import os
import sys
import types

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from helpers import grad_violations, to_oracle_cam  # noqa: E402
from opengaussian_b200 import _lib, renderer, synth  # noqa: E402
from opengaussian_b200.rasterizer import GaussianRasterizationSettings, GaussianRasterizer  # noqa: E402

pytestmark = pytest.mark.gpu

KEYS = ["render", "alpha", "depth", "silhouette", "ins_feat", "cluster_imgs", "cluster_silhouettes",
        "leaf_clusters_imgs", "leaf_cluster_silhouettes", "occured_leaf_id", "cluster_occur", "viewspace_points",
        "visibility_filter", "radii"]


def _pipe(batched=True):
    return types.SimpleNamespace(debug=False, compute_cov3D_python=False, convert_SHs_python=False,
                                 batched_subsets=batched)


def _rasterizer(cam, bg, dev, sh_degree=3):
    rs = GaussianRasterizationSettings(
        image_height=int(cam.image_height), image_width=int(cam.image_width), tanfovx=math.tan(cam.FoVx * 0.5),
        tanfovy=math.tan(cam.FoVy * 0.5), bg=bg, scale_modifier=1.0, viewmatrix=cam.world_view_transform.to(dev),
        projmatrix=cam.full_proj_transform.to(dev), sh_degree=sh_degree, campos=cam.camera_center.to(dev),
        prefiltered=False, debug=False)
    return GaussianRasterizer(rs)


def _voxel_ids(xyz, n):
    lo, hi = xyz.min(0).values, xyz.max(0).values
    c = ((xyz - lo) / (hi - lo) * n).long().clamp(0, n - 1)
    return (c[:, 0] * n + c[:, 1]) * n + c[:, 2]


def _gs(gs, dev):
    return {k: v.to(dev) if isinstance(v, torch.Tensor) else v for k, v in gs.items()}


def _cov3d(g):
    """[P,6] covariance from scales / rotations (xx, xy, xz, yy, yz, zz)."""
    q = torch.nn.functional.normalize(g["rotations"], dim=1)
    r, x, y, z = q.unbind(1)
    R = torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - r * z), 2 * (x * z + r * y),
                     2 * (x * y + r * z), 1 - 2 * (x * x + z * z), 2 * (y * z - r * x),
                     2 * (x * z - r * y), 2 * (y * z + r * x), 1 - 2 * (x * x + y * y)], 1).view(-1, 3, 3)
    M = R * g["scales"][:, None, :]
    S = M @ M.transpose(1, 2)
    return torch.stack([S[:, 0, 0], S[:, 0, 1], S[:, 0, 2], S[:, 1, 1], S[:, 1, 2], S[:, 2, 2]], 1).contiguous()


def _kw(g, sh, F, cov=False):
    kw = dict(opacities=g["opacities"])
    if cov:
        kw["cov3D_precomp"] = _cov3d(g)
    else:
        kw.update(scales=g["scales"], rotations=g["rotations"])
    if sh:
        kw["shs"] = g["shs"]
    else:
        kw["colors_precomp"] = g["ins_feat"][:, 3:6].contiguous()
    if F:
        kw["extra_feats"] = g["ins_feat"][:, :F].contiguous()
    return kw


def _subset_maps(P, dev, gen):
    """S -> slot map: -1 rows, empty slots, a one-Gaussian slot, and S = 640 with most slots empty."""
    maps = {}
    s7 = torch.randint(0, 6, (P,), device=dev, generator=gen, dtype=torch.int32)
    s7[s7 == 3] = 2                                           # slot 3 empty
    s7[torch.rand(P, device=dev, generator=gen) < 0.1] = -1
    s7[77] = 6                                                # slot 6 holds one Gaussian
    maps[7] = s7
    s1 = torch.zeros(P, dtype=torch.int32, device=dev)
    s1[::5] = -1
    maps[1] = s1
    maps[64] = torch.randint(-1, 64, (P,), device=dev, generator=gen, dtype=torch.int32)
    used = torch.randperm(640, generator=torch.Generator().manual_seed(2))[:20].to(dev).int()
    maps[640] = used[torch.randint(0, 20, (P,), device=dev, generator=gen)]
    return maps


# ---------------------------------------------------------------------------------------------------------------------
# 1. forward: bit-identical to forward_subsets

@pytest.mark.parametrize("sh", [False, True])
@pytest.mark.parametrize("F", [0, 2, 6])
def test_forward_equals_forward_subsets(sh, F):
    dev = torch.device("cuda")
    P = 6000
    g = _gs(synth.make_gaussians(P, "blender", 4, scale_mult=1.2), dev)
    cam = synth.orbit_cameras(3, 4.0, 150, 110, 0.69, 1.0)[1]             # 150 x 110: not a multiple of 16
    bg = torch.tensor([0.2, 0.5, 0.8], device=dev)
    ebg = torch.tensor([0.3, 0.1, 0.7, 0.4, 0.9, 0.6][:F], device=dev) if F else None
    rast = _rasterizer(cam, bg, dev)
    kw = _kw(g, sh, F)
    if F:
        kw["extra_bg"] = ebg
    leaves = {k: v.clone().requires_grad_(k != "extra_bg") for k, v in kw.items()}
    for S, subset in _subset_maps(P, dev, torch.Generator(device=dev).manual_seed(1)).items():
        with torch.no_grad():
            want = rast.forward_subsets(g["means3D"], subset=subset, num_subsets=S, **kw)
        got = rast.forward_subsets_grad(g["means3D"], subset=subset, num_subsets=S, **leaves)
        assert got[0].requires_grad and got[2].requires_grad
        for a, b in zip(got, want):
            assert (a is None) == (b is None) and (a is None or torch.equal(a.detach(), b)), S


def test_forward_long_tile_lists():
    """300 k Gaussians at 800 x 800 in 64 spatial cells: tile lists run over many 256-entry rounds, forward and back."""
    dev = torch.device("cuda")
    gs, cams = synth.make_scene("blender_300k_800", n_views=2)
    g = _gs(gs, dev)
    rast = _rasterizer(cams[0], torch.tensor([0.1, 0.3, 0.2], device=dev), dev)
    subset = _voxel_ids(g["means3D"], 4).int()
    subset[::97] = -1
    kw = _kw(g, False, 3)
    with torch.no_grad():
        want = rast.forward_subsets(g["means3D"], subset=subset, num_subsets=64, **kw)
    feat = kw["extra_feats"].clone().requires_grad_(True)
    got = rast.forward_subsets_grad(g["means3D"], subset=subset, num_subsets=64, **dict(kw, extra_feats=feat))
    for a, b in zip(got, want):
        assert torch.equal(a.detach(), b)
    assert float(want[2].amax()) > 0.5
    got[3].square().sum().backward()
    gf = feat.grad
    assert torch.isfinite(gf).all() and float(gf.abs().max()) > 0
    assert float(gf[subset < 0].abs().max()) == 0.0


# ---------------------------------------------------------------------------------------------------------------------
# 2. gradients against the per-slot forward() + backward()

def _per_slot_reference(rast, g, subset, S, kw, names, up):
    """Sum over slots of forward() + backward() on the rows of that slot, the gradients scattered back to [P, ...]."""
    P = g["means3D"].shape[0]
    want = {n: torch.zeros_like(kw[n] if n != "means3D" else g["means3D"]) for n in names}
    for k in range(S):
        idx = subset == k
        if not bool(idx.any()):
            continue
        args = {n: v[idx] for n, v in kw.items() if isinstance(v, torch.Tensor) and v.shape[0] == P}
        args["means3D"] = g["means3D"][idx]
        leaves = {n: args[n].clone().requires_grad_(True) for n in names}
        args.update(leaves)
        out = rast(means2D=torch.zeros_like(args["means3D"]), **args,
                   **({"extra_bg": kw["extra_bg"]} if "extra_bg" in kw else {}))
        loss = (out[0] * up["color"][k]).sum() + (out[2] * up["depth"][k]).sum() + (out[3] * up["alpha"][k]).sum()
        if len(out) > 4:
            loss = loss + (out[4] * up["feat"][k]).sum()
        loss.backward()
        for n in names:
            want[n][idx] = leaves[n].grad
    return want


@pytest.mark.parametrize("mode", ["features", "geometry_sh", "geometry_cov3D"])
def test_gradients_equal_per_slot_backward(mode):
    dev = torch.device("cuda")
    P = 6000
    g = _gs(synth.make_gaussians(P, "blender", 5, scale_mult=1.2), dev)
    cam = synth.orbit_cameras(3, 4.0, 150, 110, 0.69, 1.0)[0]
    rast = _rasterizer(cam, torch.tensor([0.2, 0.5, 0.8], device=dev), dev)
    H, W = 110, 150
    gen = torch.Generator(device=dev).manual_seed(7)
    if mode == "features":      # Stage 2.2: the geometry does not train, colour and feature channels do
        kw, names, F = _kw(g, False, 3), ["colors_precomp", "extra_feats"], 3
        kw["extra_bg"] = torch.tensor([0.3, 0.1, 0.7], device=dev)
    elif mode == "geometry_sh":
        kw, F = _kw(g, True, 6), 6
        names = ["means3D", "opacities", "scales", "rotations", "shs", "extra_feats"]
    else:
        kw, F = _kw(g, False, 2, cov=True), 2
        names = ["means3D", "opacities", "cov3D_precomp", "colors_precomp", "extra_feats"]
    for S, subset in ((7, _subset_maps(P, dev, gen)[7]), (27, _voxel_ids(g["means3D"], 3).int())):
        up = dict(color=torch.randn(S, 3, H, W, device=dev, generator=gen),
                  feat=torch.randn(S, F, H, W, device=dev, generator=gen),
                  depth=torch.randn(S, 1, H, W, device=dev, generator=gen),
                  alpha=torch.randn(S, 1, H, W, device=dev, generator=gen))
        leaves = {n: (kw[n] if n != "means3D" else g["means3D"]).clone().requires_grad_(True) for n in names}
        args = dict(kw, **leaves)
        means3D = args.pop("means3D", g["means3D"])
        color, depth, alpha, feat = rast.forward_subsets_grad(means3D, subset=subset, num_subsets=S, **args)
        ((color * up["color"]).sum() + (feat * up["feat"]).sum() + (depth * up["depth"]).sum() +
         (alpha * up["alpha"]).sum()).backward()
        want = _per_slot_reference(rast, g, subset, S, kw, names, up)
        outside = (subset < 0) | (subset >= S)
        for n in names:
            got = leaves[n].grad
            assert got is not None and torch.isfinite(got).all(), n
            frac, worst = grad_violations(got.cpu().numpy(), want[n].cpu().numpy())
            print(f"{mode} S={S} dL/d{n}: violating fraction {frac:.2e}, worst |diff|/tol {worst:.3f}")
            assert frac == 0.0, (n, frac, worst)
            if bool(outside.any()):
                assert float(got[outside].abs().max()) == 0.0, n


def test_double_backward_raises():
    dev = torch.device("cuda")
    g = _gs(synth.make_gaussians(500, "blender", 0), dev)
    rast = _rasterizer(synth.orbit_cameras(1, 4.0, 32, 32, 0.69)[0], torch.zeros(3, device=dev), dev)
    feat = g["ins_feat"][:, :3].clone().requires_grad_(True)
    color, _, _, _ = rast.forward_subsets_grad(g["means3D"], g["opacities"], torch.zeros(500, dtype=torch.int32,
                                                                                          device=dev), 1,
                                               colors_precomp=feat, scales=g["scales"], rotations=g["rotations"])
    (gf,) = torch.autograd.grad(color.square().sum(), feat, create_graph=True)
    with pytest.raises(RuntimeError):
        gf.sum().backward()


# ---------------------------------------------------------------------------------------------------------------------
# 3. independent pin: fp64 autograd of oracle/raster_torch.py per slot

def test_small_scene_vs_fp64_autograd():
    from opengaussian_b200 import debug
    from oracle import raster_torch
    dev = torch.device("cuda")
    P, W, H, S = 2000, 64, 48, 3
    gs = synth.make_gaussians(P, "blender", 0, scale_mult=2.5)
    cam = synth.orbit_cameras(4, 3.5, W, H, 0.9, 0.8)[0]
    bg = torch.tensor([0.2, 0.1, 0.3], device=dev)
    rs = GaussianRasterizationSettings(H, W, cam.tanfovx, cam.tanfovy, bg, 1.0, cam.world_view_transform.to(dev),
                                       cam.full_proj_transform.to(dev), 3, cam.camera_center.to(dev), False, False)
    rast = GaussianRasterizer(rs)
    g = _gs(gs, dev)
    subset = (torch.arange(P, device=dev) % 4).int() - 1         # slots 0..2 and -1
    names = ("means3D", "opacities", "scales", "rotations", "shs", "extra")
    leaves = {n: g["ins_feat" if n == "extra" else n].clone().requires_grad_(True) for n in names}
    args = {("extra_feats" if n == "extra" else n): v for n, v in leaves.items() if n != "means3D"}
    color, depth, alpha, feat = rast.forward_subsets_grad(leaves["means3D"], subset=subset, num_subsets=S, **args)
    gen = torch.Generator().manual_seed(9)
    want = {n: np.zeros(tuple(leaves[n].shape)) for n in names}
    loss = 0
    for k in range(S):
        idx = subset == k
        sub = {n: v[idx] for n, v in g.items() if isinstance(v, torch.Tensor) and v.shape[0] == P}
        out = debug.forward_with_state(rs, sub["means3D"], sub["opacities"], shs=sub["shs"], scales=sub["scales"],
                                       rotations=sub["rotations"], extra=sub["ins_feat"])
        idc = idx.cpu()
        d = lambda n: gs["ins_feat" if n == "extra" else n][idc].double().requires_grad_(True)  # noqa: E731
        lv = {n: d(n) for n in names}
        m2 = torch.zeros(int(idc.sum()), 3, dtype=torch.float64, requires_grad=True)
        col64, dep64, alp64 = raster_torch.render(
            to_oracle_cam(cam), out["radii"].cpu().numpy(), out["point_list"].cpu().numpy().view(np.uint32),
            out["ranges"].cpu().numpy().view(np.uint32).reshape(-1, 2), lv["means3D"], m2, lv["opacities"],
            scales=lv["scales"], rotations=lv["rotations"], shs=lv["shs"], extra=lv["extra"],
            bg=bg.cpu().numpy())
        got_img = torch.cat([color[k], feat[k]]).detach().double().cpu()
        clean = (got_img - col64.detach()).abs().amax(0) <= 2e-5     # pixels where no fp32 threshold decision flipped
        assert float((~clean).float().mean()) <= 0.03
        m = clean.double()
        gc = torch.randn(9, H, W, generator=gen, dtype=torch.float64) * m
        gd = torch.randn(H, W, generator=gen, dtype=torch.float64) * m
        ga = torch.randn(H, W, generator=gen, dtype=torch.float64) * m
        ((col64 * gc).sum() + (dep64 * gd).sum() + (alp64 * ga).sum()).backward()
        for n in names:
            want[n][idc.numpy()] = lv[n].grad.numpy()
        f = lambda a: a.float().to(dev)  # noqa: E731
        loss = loss + (color[k] * f(gc[:3])).sum() + (feat[k] * f(gc[3:])).sum() + (depth[k, 0] * f(gd)).sum() + \
            (alpha[k, 0] * f(ga)).sum()
    loss.backward()
    for n in names:
        got = leaves[n].grad.cpu().numpy()
        frac, worst = grad_violations(got, want[n])
        print(f"fp64 pin dL/d{n}: violating fraction {frac:.2e}, worst |diff|/tol {worst:.3f}")
        assert frac == 0.0, (n, frac, worst)
        assert np.abs(got[(subset < 0).cpu().numpy()]).max() == 0.0


# ---------------------------------------------------------------------------------------------------------------------
# 4. render() with grad (Stage 2.2): batched against the loop (pipe.batched_subsets = False)

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


def _roots(cluster_idx, big):
    """The two most populated coarse clusters other than the faint one and the under-100 one."""
    order = torch.bincount(cluster_idx).argsort(descending=True).tolist()
    return [r for r in order if r not in (big, 64)][:2]


def _forwards(calls):
    return calls.get("ogs_raster_forward", 0) + calls.get("ogs_raster_forward_cached", 0)


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


def _rescale_seed(drawn):
    for s in range(100):
        torch.manual_seed(s)
        if (torch.rand(1) > 0.5) == drawn:
            return s
    raise AssertionError


class _CountCalls:
    def __init__(self, monkeypatch):
        self.names = []
        real = _lib.launch

        def launch(name, device, *args):
            self.names.append(name)
            return real(name, device, *args)
        monkeypatch.setattr(_lib, "launch", launch)

    def take(self):
        n, self.names = self.names, []
        return {k: n.count(k) for k in set(n)}


def _grad_of(model, loss_fn, out):
    model._ins_feat.grad = None
    loss_fn(out).backward()
    g = model._ins_feat.grad.clone()
    model._ins_feat.grad = None
    return g


def _both(model, cam, bg, seed, counter, **kw):
    res = {}
    for batched in (False, True):
        torch.manual_seed(seed)
        counter.take()
        out = renderer.render(cam, model, _pipe(batched), bg, 1000, **kw)
        res[batched] = (out, counter.take())
    assert list(res[True][0].keys()) == KEYS
    for k in KEYS:
        _equal(res[True][0][k], res[False][0][k], k)
    return res


def _assert_grads_close(a, b, what):
    frac, worst = grad_violations(a.cpu().numpy(), b.cpu().numpy())
    print(f"{what}: violating fraction {frac:.2e}, worst |diff|/tol {worst:.3f}")
    assert frac == 0.0 and float(a.abs().max()) > 0, (what, frac, worst)


@pytest.mark.parametrize("rescale_drawn", [False, True])
def test_render_stage22_step_batched_equals_loop(monkeypatch, rescale_drawn):
    dev = torch.device("cuda")
    model, cam, cluster_idx, leaf_idx, big = _render_scene(dev)
    assert model._ins_feat.requires_grad and not model._xyz.requires_grad
    bg = torch.tensor([0.1, 0.3, 0.2], device=dev)
    counter = _CountCalls(monkeypatch)
    gen = torch.Generator(device=dev).manual_seed(5)
    mask = (torch.rand(150, 200, device=dev, generator=gen) > 0.3).float()
    target = torch.rand(6, 150, 200, device=dev, generator=gen)
    seed = _rescale_seed(rescale_drawn)
    for r in _roots(cluster_idx, big):
        res = _both(model, cam, bg, seed, counter, cluster_idx=cluster_idx, render_cluster=True, selected_root_id=r,
                    leaf_cluster_idx=leaf_idx, root_num=65, leaf_num=10, rescale=True)
        (fast, cf), (loop, cl) = res[True], res[False]
        n_leaves = len(fast["occured_leaf_id"])
        assert len(fast["cluster_imgs"]) == 1 and n_leaves >= 2
        assert fast["cluster_imgs"][0].requires_grad and fast["leaf_clusters_imgs"][0].requires_grad
        # one subset call per pass instead of one forward per subset
        assert cf.get("ogs_raster_forward_subsets_state") == 2 and "ogs_raster_forward_subsets" not in cf
        assert cl.get("ogs_raster_forward_subsets_state") is None
        assert _forwards(cl) == _forwards(cf) + 1 + n_leaves
        # the Stage 2.2 loss (a masked L2 on the root's feature image) and a loss over several leaf images
        l2 = lambda o: ((o["cluster_imgs"][0] - target) ** 2 * mask).mean()  # noqa: E731
        _assert_grads_close(_grad_of(model, l2, fast), _grad_of(model, l2, loop), f"root {r} masked L2")
        leaves = lambda o: sum(((img - target) ** 2).mean() * (i + 1)  # noqa: E731
                               for i, img in enumerate(o["leaf_clusters_imgs"][:4]))
        _assert_grads_close(_grad_of(model, leaves, fast), _grad_of(model, leaves, loop), f"root {r} leaves")


def test_render_coarse_sweep_with_grad(monkeypatch):
    dev = torch.device("cuda")
    model, cam, cluster_idx, _, low = _render_scene(dev)
    bg = torch.tensor([0.1, 0.3, 0.2], device=dev)
    counter = _CountCalls(monkeypatch)
    res = _both(model, cam, bg, 0, counter, cluster_idx=cluster_idx, render_cluster=True, better_vis=True,
                rescale=False, root_num=65)
    (fast, cf), (loop, cl) = res[True], res[False]
    n = len(fast["cluster_imgs"])
    assert n > 10 and fast["cluster_imgs"][0].requires_grad and not bool(fast["cluster_occur"][low])
    assert cf.get("ogs_raster_forward_subsets_state") == 1 and _forwards(cl) > _forwards(cf) + n
    loss = lambda o: sum(img.square().mean() for img in o["cluster_imgs"][::3])  # noqa: E731
    _assert_grads_close(_grad_of(model, loss, fast), _grad_of(model, loss, loop), "coarse sweep")


def test_trainable_geometry_keeps_the_loop(monkeypatch):
    dev = torch.device("cuda")
    model, cam, cluster_idx, leaf_idx, big = _render_scene(dev, P=8000)
    model._xyz.requires_grad_(True)
    counter = _CountCalls(monkeypatch)
    torch.manual_seed(0)
    out = renderer.render(cam, model, _pipe(), torch.zeros(3, device=dev), 1000, cluster_idx=cluster_idx,
                          render_cluster=True, selected_root_id=_roots(cluster_idx, big)[0], leaf_cluster_idx=leaf_idx,
                          rescale=False, root_num=65)
    assert "ogs_raster_forward_subsets_state" not in counter.take()
    out["cluster_imgs"][0].sum().backward()
    assert float(out["viewspace_points"].grad.abs().max()) > 0


# ---------------------------------------------------------------------------------------------------------------------
# 5. budget split under grad

def test_budget_split_with_grad(monkeypatch):
    dev = torch.device("cuda")
    model, cam, cluster_idx, leaf_idx, _ = _render_scene(dev)
    bg = torch.tensor([0.1, 0.3, 0.2], device=dev)
    calls = []
    real = GaussianRasterizer.forward_subsets_grad

    def counting(self, *a, **k):
        calls.append(a[3] if len(a) > 3 else k["num_subsets"])
        return real(self, *a, **k)

    monkeypatch.setattr(GaussianRasterizer, "forward_subsets_grad", counting)
    kw = dict(cluster_idx=cluster_idx, leaf_cluster_idx=leaf_idx, rescale=False, root_num=65, leaf_num=10)
    loss = lambda o: sum(img.square().mean() * (i % 5) for i, img in enumerate(o["leaf_clusters_imgs"]))  # noqa: E731
    outs = []
    for budget in (renderer.SUBSET_BATCH_BYTES, 7 * ((6 + 2) * 4 + 8) * 150 * 200):    # default; 7 slots per launch
        monkeypatch.setattr(renderer, "SUBSET_BATCH_BYTES", budget)
        calls.clear()
        torch.manual_seed(0)
        out = renderer.render(cam, model, _pipe(), bg, 1000, **kw)
        outs.append((out, list(calls), _grad_of(model, loss, out)))
    (a, ca, ga), (b, cb, gb) = outs
    assert len(a["occured_leaf_id"]) > 100
    assert len(ca) == 1 and len(cb) > 4 and max(cb) == 7 and sum(cb) == ca[0]
    for k in KEYS:
        _equal(a[k], b[k], k)
    _assert_grads_close(gb, ga, "split")


# ---------------------------------------------------------------------------------------------------------------------
# 6. a second device

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
        leaves = {k: g[k].clone().requires_grad_(True) for k in ("means3D", "opacities", "scales", "rotations")}
        feat = g["ins_feat"].clone().requires_grad_(True)
        with torch.cuda.device(0):
            color, depth, alpha, extra = rast.forward_subsets_grad(
                leaves["means3D"], leaves["opacities"], subset, 8, colors_precomp=feat[:, :3], extra_feats=feat[:, 3:],
                scales=leaves["scales"], rotations=leaves["rotations"])
            (color.square().sum() + extra.sum() + depth.sum() + alpha.sum()).backward()
            assert torch.cuda.current_device() == 0
        torch.cuda.synchronize(dev)
        res.append([t.detach().cpu() for t in (color, depth, alpha, extra, feat.grad)] +
                   [v.grad.cpu() for v in leaves.values()])
    for i, (a, b) in enumerate(zip(*res)):
        if i < 4:
            assert torch.equal(a, b)
        else:
            frac, worst = grad_violations(a.numpy(), b.numpy())
            assert frac == 0.0, (i, frac, worst)
