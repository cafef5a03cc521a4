"""Several devices in one process: with cuda:0 current, every library call on cuda:1 tensors makes cuda:1 current for
the call (the library keys its per-device state on the current device, and CUDA refuses a launch into another
device's stream), gives the results the same call gives on cuda:0, and leaves cuda:0 current."""
import numpy as np
import pytest
import torch

from opengaussian_b200 import synth

pytestmark = pytest.mark.gpu

H, W = 96, 128


@pytest.fixture(autouse=True)
def two_devices():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    torch.cuda.set_device(0)
    yield
    torch.cuda.set_device(0)


def _on_both(fn):
    """fn(device) -> dict of tensors, run on cuda:0 and on cuda:1 with cuda:0 current; returns both on the host."""
    out = []
    for d in (0, 1):
        dev = torch.device("cuda", d)
        res = fn(dev)
        torch.cuda.synchronize(dev)
        assert torch.cuda.current_device() == 0
        for k, v in res.items():
            assert v.device == dev, k
        out.append({k: v.detach().cpu() for k, v in res.items()})
    return out


def _exact(a, b, keys):
    for k in keys:
        assert torch.equal(a[k], b[k]), k


def _close(a, b, keys):
    """The tolerance of test_two_threads_two_streams: atomically accumulated floats may differ in the last bits."""
    for k in keys:
        assert a[k].shape == b[k].shape, k
        assert float((a[k] - b[k]).abs().max()) <= 1e-5 * float(b[k].abs().max()), k


@pytest.mark.parametrize("M", [5, 40])       # below and above mask_stats.ID_MAP_MIN_MASKS: mask rows / id map
def test_mask_feature_mean_and_cohesion(M):
    from opengaussian_b200.mask_stats import ID_MAP_MIN_MASKS, cohesion_loss, mask_feature_mean
    assert (M < ID_MAP_MIN_MASKS) == (M == 5)
    g = torch.Generator().manual_seed(M)
    feat0 = torch.rand(6, H, W, generator=g)
    img0 = torch.rand(1, H, W, generator=g)
    mean0 = torch.rand(M, 6, generator=g)
    masks0 = synth.sam_like_masks(M, H, W, 1)

    def run(dev):
        masks = masks0.to(dev)
        feat = feat0.to(dev).requires_grad_(True)
        img = img0.to(dev).requires_grad_(True)
        mean = mask_feature_mean(feat, masks, image_mask=img)
        mean.pow(2).sum().backward()
        with torch.no_grad():
            _, var, cnt = mask_feature_mean(feat, masks, image_mask=img, return_var=True)
        feat_c = feat0.to(dev).requires_grad_(True)
        mean_c = mean0.to(dev).requires_grad_(True)
        lc = cohesion_loss(feat_c, masks, mean_c)
        lc.backward()
        return dict(mean=mean, dfeat=feat.grad, dimg=img.grad, var=var, cnt=cnt, cohesion=lc, dfeat_c=feat_c.grad,
                    dmean_c=mean_c.grad)

    a, b = _on_both(run)
    _exact(a, b, ["cnt"])
    _close(a, b, ["mean", "dfeat", "dimg", "var", "cohesion", "dfeat_c", "dmean_c"])


def test_separation_loss_and_calculate_iou():
    from opengaussian_b200.mask_stats import calculate_iou, separation_loss
    g = torch.Generator().manual_seed(2)
    mean0 = torch.rand(20, 6, generator=g)
    m1, m2 = synth.sam_like_masks(12, H, W, 3), synth.sam_like_masks(9, H, W, 4)

    def run(dev):
        mean = mean0.to(dev).requires_grad_(True)
        loss = separation_loss(mean, 100)
        loss.backward()
        return dict(loss=loss, dmean=mean.grad, iou=calculate_iou(m1.to(dev), m2.to(dev)))

    a, b = _on_both(run)
    _exact(a, b, ["iou"])
    _close(a, b, ["loss", "dmean"])


def test_batched_splat_ids():
    from opengaussian_b200.sam_footprints import batched_splat_ids
    gs = synth.make_gaussians(2000, "blender", 1, scale_mult=0.6)
    cam0 = synth.orbit_cameras(3, 4.0, W, H, 0.69, 1.0)[1]
    rs = np.random.RandomState(7)
    blocks = rs.permutation(((H + 12) // 13) * ((W + 16) // 17)).reshape((H + 12) // 13, (W + 16) // 17) % 37
    sam0 = torch.from_numpy(np.repeat(np.repeat(blocks, 13, axis=0), 17, axis=1)[:H, :W].astype(np.int64) - 1)

    def run(dev):
        return batched_splat_ids(cam0.to(dev), synth.SynthModel(gs, dev), torch.arange(5, 2000, 29), sam0.to(dev))

    a, b = _on_both(run)
    assert int(a["footprint_pixels"].gt(0).sum()) >= 10
    _exact(a, b, a.keys())


def test_rasterizer_forward_backward():
    from opengaussian_b200.rasterizer import GaussianRasterizationSettings, GaussianRasterizer
    gs = synth.make_gaussians(20_000, "blender", 5, scale_mult=1.0)
    cam0 = synth.orbit_cameras(2, 4.0, 256, 192, 0.69, 1.0)[0]
    keys = ("means3D", "opacities", "shs", "scales", "rotations")

    def run(dev):
        cam = cam0.to(dev)
        rs = GaussianRasterizationSettings(cam.image_height, cam.image_width, cam.tanfovx, cam.tanfovy,
                                           torch.zeros(3, device=dev), 1.0, cam.world_view_transform,
                                           cam.full_proj_transform, 3, cam.camera_center, False, False)
        leaves = {k: gs[k].to(dev).requires_grad_(True) for k in keys}
        color, radii, depth, alpha = GaussianRasterizer(rs)(means2D=torch.zeros_like(leaves["means3D"]), **leaves)
        (color.sum() + depth.sum()).backward()
        return dict(color=color, radii=radii, depth=depth, alpha=alpha, **{"d_" + k: leaves[k].grad for k in keys})

    a, b = _on_both(run)
    assert int(a["radii"].gt(0).sum()) > 1000
    _exact(a, b, ["color", "radii", "depth", "alpha"])
    _close(a, b, ["d_" + k for k in keys])


def test_kmeans_root_assign_and_fused_adam():
    from opengaussian_b200.kmeans_quantize import Quantize_kMeans
    from opengaussian_b200.optim import FusedAdam
    g = torch.Generator().manual_seed(5)
    feat0 = torch.rand(30_000, 6, generator=g)
    xyz0 = torch.rand(30_000, 3, generator=g) * 4 - 2
    grad0 = torch.randn(30_000, 6, generator=g)

    class _G:
        pass

    def run(dev):
        pc = _G()
        pc._ins_feat = feat0.to(dev).requires_grad_(True)
        pc._xyz = xyz0.to(dev)
        q = Quantize_kMeans(num_clusters=16, num_leaf_clusters=4, num_iters=5, dim=9)
        q.centers = torch.cat([feat0[:16], xyz0[:16] * 0.5], 1).to(dev)
        q.forward(pc, 0, assign=True, mode="root", pos_weight=0.5)
        p = torch.nn.Parameter(feat0.to(dev))
        opt = FusedAdam([p], lr=0.01, eps=1e-15)
        for _ in range(2):
            p.grad = grad0.to(dev)
            opt.step()
        return dict(ids=q.cls_ids, centers=q.centers, feat_q=pc._ins_feat_q, adam=p.data)

    a, b = _on_both(run)
    _exact(a, b, ["ids", "feat_q", "adam"])
    _close(a, b, ["centers"])
