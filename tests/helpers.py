"""Shared helpers for the parity tests: small seeded scenes in oracle (numpy) form."""
import math

import numpy as np
import torch

from opengaussian_b200 import synth
from oracle import raster as orc


def small_scene(P=300, W=64, H=48, seed=0, kind="blender", fovx=0.9, radius=3.5, scale_mult=2.5, view=0,
                n_views=4, height=0.8):
    gs = synth.make_gaussians(P, kind, seed, scale_mult=scale_mult)
    cams = synth.orbit_cameras(n_views, radius, W, H, fovx, height)
    return gs, cams[view]


def to_oracle_cam(cam, sh_degree=3, scale_modifier=1.0):
    return orc.Camera(W=cam.image_width, H=cam.image_height, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy,
                      view=cam.world_view_transform.numpy().reshape(-1).copy(),
                      proj=cam.full_proj_transform.numpy().reshape(-1).copy(),
                      campos=cam.camera_center.numpy().copy(), scale_modifier=scale_modifier,
                      sh_degree=sh_degree)


def np_inputs(gs):
    return {k: (v.numpy() if isinstance(v, torch.Tensor) else v) for k, v in gs.items()}


def grad_violations(got, want, rtol=1e-3):
    """Per-element gradient check (BASELINE north_star: "gradients within 1e-3 relative"): an element passes when
    |got - want| <= rtol * |want| + rtol * rms(want).  Returns (violating fraction, worst |diff| / tolerance)."""
    got = np.asarray(got, np.float64).reshape(-1)
    want = np.asarray(want, np.float64).reshape(-1)
    if want.size == 0:
        return 0.0, 0.0
    rms = float(np.sqrt(np.mean(want * want)))
    tol = rtol * np.abs(want) + rtol * rms + 1e-30
    ratio = np.abs(got - want) / tol
    return float((ratio > 1.0).mean()), float(ratio.max())


def separation_loss_fp64(mean, iteration, rows=slice(None)):
    """train.py:123-155 (separation_loss) restated with the loss in float64, differentiable w.r.t. `mean` by autograd.
    The rank weights are computed as the reference computes them (`sorted_indices.float()`: float32), the ranks by a
    STABLE argsort, i.e. ties by column -- the CUDA kernel's rule; the reference's unstable argsort may order exact ties
    either way, which changes neither the value nor, for identical rows, the total gradient.  `rows` restricts the sum
    to those rows of the [N, N] matrix (each row's weights depend on that row only), so that a large N can be
    evaluated and differentiated a block of rows at a time; the slices' sums add up to the loss."""
    m = mean.double()
    N = m.shape[0]
    r = torch.arange(N)[rows]
    inv = 1.0 / ((m[r, None, :] - m[None, :, :]).pow(2).sum(2) + 1)
    inv = inv.masked_fill(r[:, None] == torch.arange(N)[None, :], 0)
    ranks = inv.detach().argsort(dim=1, stable=True).argsort(dim=1)
    w = (ranks.float() / (N - 1)) * (1.0 - 0.1) + 0.1
    if iteration is not None and iteration > 35000:
        w[w < 0.9] = 0.1
    return (inv * w.double()).sum() / (N * (N - 1))


def min_rank_gap(mean, rows=slice(None)):
    """Smallest relative gap between two DISTINCT inverse distances 1 / (|m_i - m_j|^2 + 1) within a row of `mean`
    (float64): above ~1e-6 no float32 rounding can reorder them, so the float32 kernel and a float64 reference rank
    every row the same way."""
    m = mean.double()
    N = m.shape[0]
    r = torch.arange(N)[rows]
    inv = 1.0 / ((m[r, None, :] - m[None, :, :]).pow(2).sum(2) + 1)
    inv = inv.masked_fill(r[:, None] == torch.arange(N)[None, :], 0)
    s = inv.sort(dim=1).values
    lo, hi = s[:, :-1], s[:, 1:]
    gap = (hi - lo) / hi.clamp(min=1e-300)
    gap = gap[hi != lo]
    return float(gap.min()) if gap.numel() else float("inf")
