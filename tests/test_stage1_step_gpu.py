"""The Stage-1 training step as train.py drives it -- render() of a training camera, the SAM-mask statistics, cohesion
and separation losses, backward to `_ins_feat` (train.py:352-498) -- through the resident-view cache
(rasterizer.ViewCache) and the per-camera CUDA graph (graphs.GraphedViewStep), against a float64 restatement with no
CUDA arithmetic in it: oracle/raster_torch.render of the feature image and alpha on the CUDA path's own tile lists,
oracle/mask_stats for the per-mask means and the cohesion loss, helpers.separation_loss_fp64, autograd to `_ins_feat`.

Cameras are built the way scene/cameras.py:71-73 builds them (transposed, i.e. non-contiguous, view and projection
matrices), views are visited in several orders and accumulated, and losses are kept across later steps."""
import types

import numpy as np
import pytest
import torch

from helpers import grad_violations, min_rank_gap, separation_loss_fp64
from opengaussian_b200 import synth

pytestmark = pytest.mark.gpu

SCENE, N_VIEWS, MASKS = "plumbing_10k_256", 3, 12
PIPE = types.SimpleNamespace(debug=False, compute_cov3D_python=False, convert_SHs_python=False)
BORDER = 2e-5          # a pixel whose CUDA and float64 values differ by more: an fp32 skip / stop decision flipped
MAX_REMOVED = 0.03


def _reference_camera(c, dev):
    """scene/cameras.py:71-73: torch.tensor(getWorld2View2(R, T)).transpose(0, 1).cuda(), the projection matrix
    transposed the same way, their bmm, the centre from the inverse."""
    w2v = np.ascontiguousarray(c.world_view_transform.t().numpy())    # getWorld2View2's matrix (float32, C order)
    view = torch.tensor(w2v).transpose(0, 1).cuda(dev)
    proj = synth.projection_matrix(c.FoVx, c.FoVy).float().transpose(0, 1).cuda(dev)
    full = view.unsqueeze(0).bmm(proj.unsqueeze(0)).squeeze(0)
    centre = view.inverse()[3, :3]
    assert not view.is_contiguous() and not proj.is_contiguous()
    return types.SimpleNamespace(FoVx=c.FoVx, FoVy=c.FoVy, image_height=c.image_height, image_width=c.image_width,
                                 world_view_transform=view, projection_matrix=proj, full_proj_transform=full,
                                 camera_center=centre, bClusterOccur=None)


def _oracle_cam(cam, sh_degree):
    from oracle import raster as orc
    return orc.Camera(W=cam.image_width, H=cam.image_height, tanfovx=float(np.tan(cam.FoVx * 0.5)),
                      tanfovy=float(np.tan(cam.FoVy * 0.5)),
                      view=cam.world_view_transform.cpu().contiguous().numpy().reshape(-1).copy(),
                      proj=cam.full_proj_transform.cpu().contiguous().numpy().reshape(-1).copy(),
                      campos=cam.camera_center.cpu().contiguous().numpy().copy(), scale_modifier=1.0, sh_degree=sh_degree)


class _Scene:
    def __init__(self):
        from opengaussian_b200.rasterizer import GaussianRasterizationSettings
        self.dev = torch.device("cuda")
        gs, cams = synth.make_scene(SCENE, n_views=N_VIEWS)
        self.pc = synth.SynthModel(gs, self.dev, stage0=False)
        self.cams = [_reference_camera(c, self.dev) for c in cams]
        H, W = cams[0].image_height, cams[0].image_width
        self.sam = [synth.sam_like_id_map(MASKS, H, W, 4 + v).to(self.dev) for v in range(N_VIEWS)]
        self.bg = torch.zeros(3, device=self.dev)
        self.removed = []
        self._ref = {}
        self._raster64 = []
        # the CUDA step's images, the float64 raster of the same view, and the borderline pixels taken out of the masks
        pc = self.pc
        with torch.no_grad():
            geo = dict(means3D=pc._xyz, opacities=torch.sigmoid(pc._opacity), scales=torch.exp(pc._scaling),
                       rotations=torch.nn.functional.normalize(pc._rotation),
                       shs=torch.cat([pc._features_dc, pc._features_rest], 1))
        for i, cam in enumerate(self.cams):
            from opengaussian_b200 import debug
            from opengaussian_b200.renderer import render
            from oracle import raster_torch
            rs = GaussianRasterizationSettings(H, W, float(np.tan(cam.FoVx * 0.5)), float(np.tan(cam.FoVy * 0.5)),
                                               self.bg, 1.0, cam.world_view_transform, cam.full_proj_transform,
                                               pc.active_sh_degree, cam.camera_center, False, False)
            st = debug.forward_with_state(rs, geo["means3D"], geo["opacities"], shs=geo["shs"], scales=geo["scales"],
                                          rotations=geo["rotations"])
            with torch.no_grad():
                out = render(cam, pc, PIPE, self.bg, 1000, rescale=False)
            d = lambda t: t.detach().double().cpu()  # noqa: E731
            ins = d(pc._ins_feat).requires_grad_(True)
            extra = (torch.nn.functional.normalize(ins, dim=1) + 1) / 2      # renderer.py:214 / SynthModel.get_ins_feat
            P = ins.shape[0]
            img64, _, alpha64 = raster_torch.render(
                _oracle_cam(cam, pc.active_sh_degree), st["radii"].cpu().numpy(),
                st["point_list"].cpu().numpy().view(np.uint32), st["ranges"].cpu().numpy().view(np.uint32).reshape(-1, 2),
                d(geo["means3D"]), torch.zeros(P, 3, dtype=torch.float64), d(geo["opacities"]), scales=d(geo["scales"]),
                rotations=d(geo["rotations"]), colors_precomp=torch.zeros(P, 3, dtype=torch.float64), extra=extra,
                bg=np.zeros(3 + extra.shape[1]))
            feat64 = img64[3:]
            diff = torch.maximum((d(out["ins_feat"]) - feat64.detach()).abs().amax(0),
                                 (d(out["silhouette"])[0] - alpha64.detach()).abs())
            bad = diff > BORDER
            self.removed.append(float(bad.double().mean()))
            self.sam[i][0][bad.to(self.dev)] = -1            # level 0: in no mask, on both sides
            self._raster64.append((ins, feat64, alpha64))

    def view_loss(self, iteration):
        from opengaussian_b200.mask_stats import cohesion_loss, get_SAM_mask_and_feat, mask_feature_mean, separation_loss
        from opengaussian_b200.renderer import render

        def view_loss(i):                                # tests/test_graphs_gpu.py, the iteration a parameter
            out = render(self.cams[i], self.pc, PIPE, self.bg, iteration, rescale=False)
            _, m, _ = get_SAM_mask_and_feat(self.sam[i], level=0, num_mask=MASKS)
            mean = mask_feature_mean(out["ins_feat"], m, image_mask=out["silhouette"])
            return separation_loss(mean, iteration) + 0.1 * cohesion_loss(out["ins_feat"], m, mean)
        return view_loss

    def reference(self, i, iteration):
        """(loss, dL/d_ins_feat) of view i in float64, for the parameter values of the set-up."""
        key = (i, iteration)
        if key not in self._ref:
            from oracle import mask_stats as oms
            from opengaussian_b200.mask_stats import get_SAM_mask_and_feat
            ins, feat64, alpha64 = self._raster64[i]
            _, m, _ = get_SAM_mask_and_feat(self.sam[i], level=0, num_mask=MASKS)
            m = m.cpu()
            mean = oms.mask_feature_mean(feat64, m, image_mask=alpha64[None])
            gap = min_rank_gap(mean.detach())
            assert gap > 1e-5, f"view {i}: mask means too close to a rank flip ({gap:.2e})"
            loss = separation_loss_fp64(mean, iteration) + 0.1 * oms.cohesion_loss(feat64, m, mean)
            (grad,) = torch.autograd.grad(loss, ins, retain_graph=True)
            self._ref[key] = (float(loss), grad)
        return self._ref[key]


@pytest.fixture(scope="module")
def scene():
    s = _Scene()
    print(f"borderline pixels removed from the masks: {[f'{r:.2%}' for r in s.removed]}")
    assert max(s.removed) <= MAX_REMOVED
    yield s
    from opengaussian_b200 import rasterizer as rz
    rz.view_cache.clear()


@pytest.fixture
def fresh_cache():
    from opengaussian_b200 import rasterizer as rz
    rz.view_cache.clear()
    rz.view_cache.enabled = True
    yield rz.view_cache
    rz.view_cache.clear()


def _check(loss, grad, want_loss, want_grad, what):
    assert abs(float(loss) - want_loss) <= 1e-5 * abs(want_loss), (what, float(loss), want_loss)
    frac, worst = grad_violations(grad.detach().cpu().numpy(), want_grad.numpy(), 1e-3)
    assert frac == 0.0, (what, frac, worst)


def _step(scene, iteration):
    from opengaussian_b200.graphs import GraphedViewStep, geometry_guard
    return GraphedViewStep(scene.view_loss(iteration), [scene.pc._ins_feat], guard=geometry_guard(scene.pc))


@pytest.mark.parametrize("iteration", [1000, 40_000])
def test_reference_cameras_hit_the_cache_and_capture(scene, fresh_cache, iteration):
    vc = fresh_cache
    step = _step(scene, iteration)
    h0, m0 = vc.hits, vc.misses
    for epoch in range(4):                               # eager, capture + replay, replay, replay
        for i in range(N_VIEWS):
            loss = step(i)
            _check(loss, scene.pc._ins_feat.grad, *scene.reference(i, iteration), (epoch, i))
        assert len(vc) == N_VIEWS, (epoch, vc.stats())
    assert vc.misses - m0 == N_VIEWS and vc.hits - h0 >= N_VIEWS, vc.stats()
    assert step.stats() == dict(graphs=N_VIEWS, replays=3 * N_VIEWS, captures=N_VIEWS, eager=N_VIEWS)
    # a cached forward of a reference camera is bit-identical to an uncached one
    from opengaussian_b200.renderer import render
    for i in range(N_VIEWS):
        with torch.no_grad():
            hit = render(scene.cams[i], scene.pc, PIPE, scene.bg, iteration, rescale=False)
            cold = render(scene.cams[i], scene.pc, types.SimpleNamespace(view_cache=False, **vars(PIPE)), scene.bg,
                          iteration, rescale=False)
        for k in ("render", "ins_feat", "silhouette", "depth"):
            assert torch.equal(hit[k], cold[k]), (i, k)
    assert len(vc) == N_VIEWS


def _orders(kind, epochs, seed=7):
    fwd = list(range(N_VIEWS))
    if kind == "capture":
        return [fwd] * epochs
    if kind == "reverse":                                # captured in view order, replayed backwards
        return [fwd, fwd] + [fwd[::-1]] * (epochs - 2)
    g = torch.Generator().manual_seed(seed)
    return [torch.randperm(N_VIEWS, generator=g).tolist() for _ in range(epochs)]


@pytest.mark.parametrize("kind", ["capture", "reverse", "shuffle", "zero_grad"])
@pytest.mark.parametrize("iteration", [1000, 40_000])
def test_multi_view_accumulation_in_any_order(scene, fresh_cache, iteration, kind):
    step = _step(scene, iteration)
    refs = [scene.reference(i, iteration) for i in range(N_VIEWS)]
    want_loss = sum(r[0] for r in refs)
    want_grad = sum(r[1] for r in refs)
    p = scene.pc._ins_feat
    opt = torch.optim.SGD([p], lr=0.0)
    p.grad = None
    for epoch, order in enumerate(_orders(kind, 5)):
        if kind == "zero_grad":
            opt.zero_grad(set_to_none=False)
            losses = [step(i, accumulate=True) for i in order]
        else:
            losses = [step(order[0])] + [step(i, accumulate=True) for i in order[1:]]
        _check(sum(float(x) for x in losses), p.grad, want_loss, want_grad, (kind, epoch, order))
    assert step.stats()["graphs"] == N_VIEWS and step.stats()["replays"] == 4 * N_VIEWS
    p.grad = None


def test_kept_losses_survive_later_replays(scene, fresh_cache):
    step = _step(scene, 40_000)
    for _ in range(2):
        for i in range(N_VIEWS):
            step(i)
    kept = []
    for epoch, order in enumerate(_orders("shuffle", 3, seed=3)):
        for i in order:
            kept.append((i, step(i)))
    assert step.stats()["replays"] >= 3 * N_VIEWS
    for i, loss in kept:
        want = scene.reference(i, 40_000)[0]
        assert abs(float(loss) - want) <= 1e-5 * abs(want), (i, float(loss), want)


def test_in_place_camera_edit_misses_that_view_only(scene, fresh_cache):
    from opengaussian_b200.renderer import render
    vc = fresh_cache
    cam = scene.cams[1]
    saved = [t.clone() for t in (cam.world_view_transform, cam.full_proj_transform, cam.camera_center)]
    try:
        for _ in range(2):
            for i in range(N_VIEWS):
                with torch.no_grad():
                    render(scene.cams[i], scene.pc, PIPE, scene.bg, 1000, rescale=False)
        with torch.no_grad():
            before = render(cam, scene.pc, PIPE, scene.bg, 1000, rescale=False)["ins_feat"].clone()
        h0, m0 = vc.hits, vc.misses
        # move the camera 5 cm along its own x axis: view, full projection and centre, all in place
        shift = torch.eye(4, device=scene.dev)
        shift[3, 0] = 0.05
        with torch.no_grad():
            cam.world_view_transform.copy_(cam.world_view_transform @ shift)
            cam.full_proj_transform.copy_(cam.world_view_transform @ cam.projection_matrix)
            cam.camera_center.copy_(cam.world_view_transform.inverse()[3, :3])
        with torch.no_grad():
            moved = render(cam, scene.pc, PIPE, scene.bg, 1000, rescale=False)
            cold = render(cam, scene.pc, types.SimpleNamespace(view_cache=False, **vars(PIPE)), scene.bg, 1000,
                          rescale=False)
        # the entry under the old key can never match again and stays until the LRU budget evicts it
        assert vc.misses - m0 == 1 and len(vc) == N_VIEWS + 1
        assert torch.equal(moved["ins_feat"], cold["ins_feat"]) and torch.equal(moved["silhouette"], cold["silhouette"])
        assert not torch.equal(moved["ins_feat"], before)
        h1 = vc.hits
        for i in (0, 2, 1):
            with torch.no_grad():
                render(scene.cams[i], scene.pc, PIPE, scene.bg, 1000, rescale=False)
        assert vc.hits - h1 == 3 and vc.misses - m0 == 1, vc.stats()
    finally:
        with torch.no_grad():
            for t, s in zip((cam.world_view_transform, cam.full_proj_transform, cam.camera_center), saved):
                t.copy_(s)


def test_replay_follows_in_place_parameter_updates(scene, fresh_cache):
    """After optimizer-like in-place updates of `_ins_feat` the replays match the eager step on the new values (the
    eager step itself is pinned against float64 above)."""
    pc = scene.pc
    saved = pc._ins_feat.detach().clone()
    view_loss = scene.view_loss(40_000)
    step = _step(scene, 40_000)
    gen = torch.Generator(device=scene.dev).manual_seed(11)
    order_gen = torch.Generator().manual_seed(5)
    try:
        for _ in range(2):
            for i in range(N_VIEWS):
                step(i)
        for _ in range(3):
            with torch.no_grad():
                pc._ins_feat.add_(0.2 * torch.randn(pc._ins_feat.shape, device=scene.dev, generator=gen))
            want_loss, want_grad = 0.0, torch.zeros_like(pc._ins_feat)
            for i in range(N_VIEWS):
                pc._ins_feat.grad = None
                loss = view_loss(i)
                loss.backward()
                want_loss += float(loss)
                want_grad += pc._ins_feat.grad
            order = torch.randperm(N_VIEWS, generator=order_gen).tolist()
            losses = [step(order[0])] + [step(i, accumulate=True) for i in order[1:]]
            got = pc._ins_feat.grad
            assert abs(sum(float(x) for x in losses) - want_loss) <= 1e-5 * abs(want_loss)
            assert float((got - want_grad).abs().max()) <= 5e-5 * float(want_grad.abs().max())
        assert step.stats()["captures"] == N_VIEWS and step.stats()["replays"] >= 4 * N_VIEWS
    finally:
        with torch.no_grad():
            pc._ins_feat.copy_(saved)
        pc._ins_feat.grad = None
