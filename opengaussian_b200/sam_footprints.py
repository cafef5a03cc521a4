"""Single-splat footprints for the multi-view SAM-mask refiner (SURVEY.md section 8f rank 3).

``MultiViewSAMMaskRefiner`` (utils/sam_refinement_utils.py) asks, for every selected Gaussian and every camera
that sees it, "which SAM segment does this splat mostly cover?" -- ``get_splat_id_and_weights`` (:902-913): a
P = 1 rasterizer call with white view-independent SH (``render_single_gaussian`` :330-403), ``fix_image``
(:143-176), ``rgb_to_weight_map`` (:103-141) and a weighted ``torch.bincount`` over the whole image (:645-702),
in Python loops over Gaussians x cameras (:1177-1196, :1247-1275).

* ``render_single_gaussian`` / ``get_splat_id_and_weights``: the reference methods as functions, on the B200
  rasterizer (one splat per call; returns the full weight map that ``expand_masks`` needs).
* ``batched_splat_ids``: all selected Gaussians of ONE camera in one call (csrc/footprint.cu through
  ``ogs_splat_footprint_votes``): dominant id, "is the render visible", footprint size.  Same preprocess kernel
  and the same alpha arithmetic as the rasterizer, so the uint8 image the reference would quantise is reproduced
  pixel for pixel; votes are integer sums of the quantised weights (the reference sums float32 weights with
  atomics, which orders ids the same way up to float rounding).
"""
import ctypes as C
import math

import numpy as np
import torch

from . import _lib
from .rasterizer import GaussianRasterizationSettings, GaussianRasterizer

# colour of the white, view-independent SH the refiner renders with (features_dc = 1, features_rest = 0):
# max(SH_C0 * 1 + 0.5, 0) in float32, as the preprocess kernel evaluates it
WHITE_SH_COLOR = float(np.float32(0.28209479177387814) + np.float32(0.5))


def _settings(viewpoint_camera, sh_degree, scaling_modifier):
    return GaussianRasterizationSettings(
        image_height=int(viewpoint_camera.image_height), image_width=int(viewpoint_camera.image_width),
        tanfovx=math.tan(viewpoint_camera.FoVx * 0.5), tanfovy=math.tan(viewpoint_camera.FoVy * 0.5),
        bg=torch.zeros(3, dtype=torch.float32, device="cuda"), scale_modifier=scaling_modifier,
        viewmatrix=viewpoint_camera.world_view_transform, projmatrix=viewpoint_camera.full_proj_transform,
        sh_degree=sh_degree, campos=viewpoint_camera.camera_center, prefiltered=False, debug=False)


def render_single_gaussian(viewpoint_camera, pc, gaussian_idx, scaling_modifier=1.0, use_view_inv_white_shs=False,
                           override_color=None):
    """Reference :330-403: (rendered_image [3,H,W], radii [1], rendered_depth, rendered_alpha) of one Gaussian."""
    rasterizer = GaussianRasterizer(raster_settings=_settings(viewpoint_camera, pc.active_sh_degree, scaling_modifier))
    sl = slice(gaussian_idx, gaussian_idx + 1)
    means3D = pc.get_xyz[sl]
    means2D = torch.zeros_like(means3D, requires_grad=True)
    colors_precomp = None
    if override_color is not None:
        colors_precomp = override_color[sl] if override_color.ndim == 2 else override_color.unsqueeze(0)
    shs = pc.get_features[sl]
    if use_view_inv_white_shs:
        shs = torch.cat((torch.ones(1, 1, 3, device=shs.device), torch.zeros(1, shs.shape[1] - 1, 3, device=shs.device)), dim=1)
    return rasterizer(means3D=means3D, means2D=means2D, shs=shs if colors_precomp is None else None,
                      colors_precomp=colors_precomp, opacities=pc.get_opacity[sl], scales=pc.get_scaling[sl],
                      rotations=pc.get_rotation[sl], cov3D_precomp=None)


def fix_image(rendered_image):
    """Reference :143-176 for the [3,H,W] float case: [H,W,3] uint8."""
    if rendered_image.ndim == 3 and rendered_image.shape[0] == 3:
        rendered_image = rendered_image.permute(1, 2, 0)
    if rendered_image.dtype != torch.uint8:
        rendered_image = torch.clamp(rendered_image * 255, 0, 255).to(torch.uint8)
    return rendered_image.contiguous()


def rgb_to_weight_map(rendered_image):
    """Reference :103-141: [H,W,3] -> [H,W,1] weights, maximum exactly 1."""
    if rendered_image.dtype == torch.uint8:
        rendered_image = rendered_image.float() / 255.0
    elif rendered_image.max() > 1.0:
        rendered_image = rendered_image / 255.0
    weight_map = torch.mean(rendered_image, dim=2)
    max_val = weight_map.max()
    if max_val > 0:
        weight_map = weight_map / max_val
    return weight_map.unsqueeze(2)


def most_common_id_weighted(sam_mask, weight_matrix):
    """Reference :645-702 (get_most_common_id_in_mask_weighted)."""
    if weight_matrix.ndim == 3 and weight_matrix.shape[2] == 1:
        weight_matrix = weight_matrix.squeeze(2)
    ids, weights = sam_mask.flatten(), weight_matrix.flatten()
    min_id, max_id = int(ids.min()), int(ids.max())
    if min_id == max_id:
        return min_id
    offset = -min_id if min_id < 0 else 0
    counts = torch.bincount((ids + offset).long(), weights=weights, minlength=max_id + offset + 1)
    return int(torch.argmax(counts)) - offset


def get_splat_id_and_weights(camera, gaussians, gaussian_id, sam_mask):
    """Reference :902-913: (most dominant id, weight map [H,W,1], render visible?) of one splat in one camera."""
    rendered_image, _, _, _ = render_single_gaussian(camera, gaussians, gaussian_id, use_view_inv_white_shs=True)
    rendered_image = fix_image(rendered_image.detach())
    non_black_mask = torch.any(rendered_image != 0, dim=2)
    weights_mask = rgb_to_weight_map(rendered_image)
    return most_common_id_weighted(sam_mask, weights_mask), weights_mask, bool(non_black_mask.any())


def batched_splat_ids(camera, gaussians, gaussian_ids, sam_mask, scaling_modifier=1.0):
    """``get_splat_id_and_weights`` for ALL ``gaussian_ids`` (LongTensor [B]) of one camera in one call.

    Returns a dict of [B] tensors: ``dominant_id`` int64, ``visible`` bool (= ``non_black_mask.any()``),
    ``dominant_weight`` int32 (sum of the uint8 weights of that id), ``footprint_pixels`` int32, ``q_max`` int32
    (divide the integer weights by it to get ``rgb_to_weight_map``'s normalisation), ``radii`` int32.
    Splats whose footprint spans more than 128 distinct ids are redone with the one-splat path."""
    if not sam_mask.is_cuda:
        raise _lib.OgsError("batched_splat_ids needs CUDA tensors (no CPU path)")
    dev = sam_mask.device
    ids = torch.as_tensor(gaussian_ids, device=dev, dtype=torch.long).reshape(-1)
    B = int(ids.numel())
    H, W = int(camera.image_height), int(camera.image_width)
    assert tuple(sam_mask.shape) == (H, W), "sam_mask must be [H, W]"
    sam = sam_mask.detach().to(torch.int32).contiguous()
    f32 = lambda t: t.detach().float().contiguous()  # noqa: E731
    means = f32(gaussians.get_xyz[ids])
    opac = f32(gaussians.get_opacity[ids]).reshape(-1)
    scales = f32(gaussians.get_scaling[ids])
    rots = f32(gaussians.get_rotation[ids])
    view, proj = f32(camera.world_view_transform), f32(camera.full_proj_transform)
    lo, hi = int(sam.min()), int(sam.max())
    empty_id = lo if (lo < 0 or lo == hi) else 0          # argmax over all-zero counts (:686-695): index 0 of the shifted ids
    out = {k: torch.zeros(B, dtype=torch.int32, device=dev)
           for k in ("dominant_id", "dominant_weight", "footprint_pixels", "q_max", "radii")}
    if B > 0:
        inp = _lib.FootprintInputs(P=B, W=W, H=H, act_flags=0, means3D=means.data_ptr(), opacities=opac.data_ptr(),
                                   scales=scales.data_ptr(), rotations=rots.data_ptr(), scale_modifier=scaling_modifier,
                                   tanfovx=math.tan(camera.FoVx * 0.5), tanfovy=math.tan(camera.FoVy * 0.5),
                                   color=WHITE_SH_COLOR, viewmatrix=view.data_ptr(), projmatrix=proj.data_ptr(),
                                   sam_ids=sam.data_ptr(), empty_id=empty_id, reserved_=0)
        overflow = C.c_int32(0)
        _lib.launch("ogs_splat_footprint_votes", dev, C.byref(inp),
                    *(_lib.ptr(out[k]) for k in ("dominant_id", "dominant_weight", "footprint_pixels", "q_max", "radii")),
                    C.byref(overflow))
        if overflow.value:
            for j in torch.nonzero(out["dominant_weight"] < 0).flatten().tolist():
                did, wm, _ = get_splat_id_and_weights(camera, gaussians, int(ids[j]), sam_mask)
                out["dominant_id"][j] = did
                q = torch.round(wm.squeeze(2) * float(out["q_max"][j]))
                out["dominant_weight"][j] = int(q[sam_mask == did].sum())
    out["visible"] = out["footprint_pixels"] > 0
    out["dominant_id"] = out["dominant_id"].long()
    return out
