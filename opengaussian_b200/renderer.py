"""``render()`` of OpenGaussian (reference gaussian_renderer/__init__.py:22-373) on the fused
B200 rasterizer: same signature, same 14-key return dict, same control flow for the coarse /
fine cluster passes -- but every group of reference passes that shares geometry is ONE launch of
the C-channel rasterizer:

  reference (Stage 1 / 2.1, :104-163)              here
  -------------------------------------------      -----------------------------------------
  pass 1  RGB (SH)                                 rescale_factor == 1 (always when
  pass 2  ins_feat[:, :3] as colours               rescale=False: Stage 1, render.py,
  pass 3  ins_feat[:, 3:6] as colours              pseudo-label construction):
  pass 4  SH again, only alpha kept (silhouette)       1 pass: RGB + 6 feature channels + depth + alpha
                                                   rescale_factor != 1 (Stage 2, p = 0.5):
                                                       RGB pass + 1 pass (6 feature channels + alpha)
  cluster / leaf passes: 2 x 3 channels (:203-225, :327-345)   1 pass with 6 channels

The feature channels get the same background as the reference gives them (bg_color applied to
each 3-channel group, because the reference reuses one rasterizer for all passes).  The CPU RNG
draws (`torch.rand(1)` at :121,124) are reproduced so that training stays in lock-step.
``fused=False`` falls back to the reference's literal pass structure (used by the parity test).
Cluster / leaf passes: all subsets of the call in ONE rasterizer call (_render_slots), with or without a gradient.
"""
import math

import torch

from . import knn
from .rasterizer import GaussianRasterizationSettings, GaussianRasterizer, pin_for_capture
from .rasterizer import view_cache as _view_cache


def _knn_mean_dists(x: torch.Tensor, K: int, chunk: int = 4096) -> torch.Tensor:
    """Squared distances to the K nearest neighbours (self included), like
    pytorch3d.ops.knn_points(x, x, K).dists[0] -- used only by post_process (:293-309)."""
    out = []
    for i in range(0, x.shape[0], chunk):
        d = torch.cdist(x[i:i + chunk], x) ** 2
        out.append(torch.topk(d, K, dim=1, largest=False).values)
    return torch.cat(out, 0)


_ZERO_SINKS = {}     # (P, device) -> (zeros [P,3], zeros [P,3]): the frozen-geometry stand-in for the screen-space gradient sink
_TILED_BG = {}       # device -> (signature of bg3, nb, tiled background, bg3)


def _zero_sink(xyz):
    """A zero `viewspace_points` tensor whose .grad is zeros, shared by every frozen-geometry render() of this model size
    (two 12 MB fills per call at 1 M Gaussians otherwise).  Nothing writes to it: the densification statistics that read
    it (train.py:598) only run while the positions train, and then render() builds a real gradient sink."""
    key = (xyz.shape[0], xyz.device, xyz.dtype)
    hit = _ZERO_SINKS.get(key)
    if hit is None:
        _ZERO_SINKS.clear()                      # one model size at a time
        hit = (torch.zeros_like(xyz), torch.zeros_like(xyz))
        hit[0].grad = hit[1]
        _ZERO_SINKS[key] = hit
    pin_for_capture(xyz.device, *hit)
    return hit[0]


def _tiled_bg(bg3, nb):
    """bg_color repeated over the feature channels (the reference reuses one rasterizer, hence one background, for all
    its 3-channel passes); cached per device and width on the background tensor's storage and version counter."""
    sig = (bg3.data_ptr(), bg3._version)
    hit = _TILED_BG.get((bg3.device, nb))
    if hit is None or hit[0] != sig:
        hit = (sig, torch.cat([bg3] * ((nb + 2) // 3))[:nb].contiguous(), bg3)     # keeps bg3 alive: the address stays its own
        _TILED_BG[(bg3.device, nb)] = hit
    pin_for_capture(bg3.device, hit[1])
    return hit[1]


def _feat_args(bg3, feat, shs):
    """The colour arguments of a feature pass: the SH colours (seg_rgb), `feat` as colours, or its first 3 channels as
    colours and the rest as extra channels."""
    if shs is not None:
        return dict(shs=shs)
    if feat.shape[-1] > 3:
        return dict(colors_precomp=feat[:, :3], extra_feats=feat[:, 3:], extra_bg=_tiled_bg(bg3, feat.shape[-1] - 3))
    return dict(colors_precomp=feat)


def _feat_image(color, extra, shs, dim):
    """The image of a feature pass from the rasterizer's colour and extra channels (channels at `dim`): with shs the RGB
    image duplicated, as the reference does."""
    if shs is not None:
        return torch.cat((color, color), dim=dim)
    if extra is not None:
        return torch.cat((color, extra), dim=dim)
    return color


def _feat_pass(rasterizer, bg3, means3D, means2D, opacity, scales, rotations, cov3D_precomp, feat, shs=None,
               fused=True):
    """One pass compositing all channels of `feat` ([n,3] or [n,6]) -> (image [F,H,W], alpha [1,H,W]).
    With shs given (seg_rgb) the RGB image is rendered and duplicated like the reference does.
    fused=False: the reference's literal two 3-channel passes."""
    if shs is None and not fused and feat.shape[-1] > 3:
        img, _, _, alpha = rasterizer(means3D=means3D, means2D=means2D, shs=None, colors_precomp=feat[:, :3],
                                      opacities=opacity, scales=scales, rotations=rotations,
                                      cov3D_precomp=cov3D_precomp)
        img2, _, _, alpha = rasterizer(means3D=means3D, means2D=means2D, shs=None, colors_precomp=feat[:, 3:],
                                       opacities=opacity, scales=scales, rotations=rotations,
                                       cov3D_precomp=cov3D_precomp)
        return torch.cat((img, img2), dim=0), alpha
    img, _, _, alpha, *extra = rasterizer(means3D=means3D, means2D=means2D, opacities=opacity, scales=scales,
                                          rotations=rotations, cov3D_precomp=cov3D_precomp,
                                          **_feat_args(bg3, feat, shs))
    return _feat_image(img, extra[0] if extra else None, shs, 0), alpha


# ---- the coarse-cluster and leaf passes of render(): a planning step and a render step ----
# The planners decide, in the reference's loop order, which clusters / leaves reach the rasterizer and with which rows;
# their filters are disjoint, so they are handed on as ONE int32 slot map `subset` ([P]: slot k or -1, the filter of
# slot k is subset == k).  The render step then runs either one rasterizer call for all slots
# (GaussianRasterizer.forward_subsets, or forward_subsets_grad when a gradient must reach the inputs) or the reference's
# one pass per slot (_subset_route says when).

# Output bytes of one subset call, S * ((C + 2) * 4 [+ 8 state bytes with grad]) * H * W; more slots are split.  This
# bounds what a call returns and keeps for its backward, not peak memory: the backward of a gradient-carrying call also
# receives upstream gradient images of the same size as the outputs the loss reads (plus zero planes for padding).
SUBSET_BATCH_BYTES = 4 << 30


def _slot_map(ids, base, slots):
    """int32 [P]: the position of ids[i] in `slots` where base[i] holds, else -1."""
    subset = torch.full(ids.shape, -1, dtype=torch.int32, device=ids.device)
    if slots:
        n = max(slots) + 1
        lut = torch.full((n,), -1, dtype=torch.int32, device=ids.device)
        lut[torch.tensor(slots, dtype=torch.long, device=ids.device)] = torch.arange(
            len(slots), dtype=torch.int32, device=ids.device)
        ok = base & (ids >= 0) & (ids < n)
        subset = torch.where(ok, lut[ids.clamp(0, n - 1).long()], subset)
    return subset


def _post_process(filter_idx, means3D):
    """The reference's per-leaf outlier removal (:315-322): keeps the points whose mean distance to their sqrt(n) nearest
    neighbours is below mean + std."""
    filter_idx = filter_idx.clone()
    nearest_k_distance = _knn_mean_dists(means3D[filter_idx].detach(), int(filter_idx.sum() ** 0.5))
    mean_d, std_d = nearest_k_distance.mean(), nearest_k_distance.std()
    mask = nearest_k_distance.mean(dim=-1) < mean_d + std_d
    mask = mask.squeeze()
    filter_idx[filter_idx != 0] = mask
    return filter_idx


def _post_process_slots(subset, S, means3D):
    """_post_process for every slot of the slot map `subset` at once (CUDA tensors) -> (subset with the removed points
    at -1, kept points per slot as a host list).  Per slot: K = int(n ** 0.5) as the reference computes it, mean and
    unbiased std over all n * K distances of the slot's kNN matrix (from fp64 per-point sums), keep a point when its
    mean over K is below mean + std.  One kNN launch for all slots and one host read.  An empty slot keeps 0 points
    (where _post_process raises, as the reference's kNN does on an empty cloud)."""
    if S == 0:
        return subset, []
    s1, s2, n, k = knn.slot_knn_sums(means3D.detach(), subset, S)
    inside = subset >= 0
    seg = subset.long().clamp_min(0)                  # the points of no slot have zero sums
    tot = torch.zeros(S, dtype=torch.float64, device=subset.device).index_add_(0, seg, s1)
    tot2 = torch.zeros_like(tot).index_add_(0, seg, s2)
    cnt = (n * k).double()
    mean = tot / cnt
    std = ((tot2 - tot * mean) / (cnt - 1)).clamp_min(0).sqrt()      # NaN for one value, as torch.std: nothing kept
    keep = inside & (s1 / k[seg] < (mean + std)[seg])
    kept = torch.zeros(S, dtype=torch.int64, device=subset.device).index_add_(0, seg, keep.long()).tolist()
    return torch.where(keep, subset, -1).to(torch.int32), kept


def _plan_clusters(cluster_idx, num_cluster, viewed_pts, scale_filter, better_vis, selected_root_id, cluster_occur_cam):
    """Coarse clusters of the loop :173-236 that reach the rasterizer, in loop order -> (cluster ids, slot map).  Filter of
    cluster idx: cluster_idx == idx, visible, and with better_vis all scales < 0.5 and at least 100 such points (the
    counts of all clusters come from one bincount).  The silhouette test (:222) is the render step's."""
    cand = []
    for idx in range(num_cluster):
        if not better_vis and idx != selected_root_id:
            continue
        if cluster_occur_cam is not None and cluster_occur_cam[idx] == False:  # noqa: E712
            continue
        cand.append(idx)
    base = viewed_pts & scale_filter if better_vis else viewed_pts
    if better_vis and cand:
        counts = torch.bincount(cluster_idx[base & (cluster_idx >= 0)], minlength=num_cluster).tolist()
        cand = [idx for idx in cand if counts[idx] >= 100]
    return cand, _slot_map(cluster_idx, base, cand)


def _plan_leaves(leaf_cluster_idx, lerf_range, selected_leaf_id, pre_mask, viewed_pts, scale_filter, better_vis,
                 post_process, means3D):
    """Leaves of the loop :245-356 that reach the rasterizer, in loop order -> (leaf ids = occured_leaf_id, slot map).
    Filter of leaf idx: leaf_cluster_idx == idx (with selected_leaf_id: any of those leaves), & pre_mask, visible; with
    better_vis all scales < 0.1 and at least 100 points; then post_process's outlier removal; then at least 10 points.
    With selected_leaf_id every iteration has the same filter and the loop stops after the first pass: at most one
    slot.  Without post_process the counts of all leaves come from one bincount.  On CUDA tensors post_process runs for
    all leaves at once (_post_process_slots); there a leaf with no points is dropped, where the per-leaf loop (CPU
    tensors) raises as the reference does."""
    base = viewed_pts if pre_mask is None else pre_mask & viewed_pts
    if better_vis:
        base = base & scale_filter
    if selected_leaf_id is not None:
        filt = (leaf_cluster_idx.unsqueeze(1) == selected_leaf_id).any(dim=1) & base
        if not lerf_range or (better_vis and filt.sum() < 100):
            return [], _slot_map(leaf_cluster_idx, filt, [])
        n_kept = None
        if post_process and filt.is_cuda:
            sub, (n_kept,) = _post_process_slots(torch.where(filt, 0, -1).to(torch.int32), 1, means3D)
            filt = sub == 0
        elif post_process:
            filt = _post_process(filt, means3D)
        if (filt.sum() if n_kept is None else n_kept) < 10:
            return [], _slot_map(leaf_cluster_idx, filt, [])
        return [lerf_range[0]], torch.where(filt, 0, -1).to(torch.int32)
    if not lerf_range:
        return [], _slot_map(leaf_cluster_idx, base, [])
    counts = torch.bincount(leaf_cluster_idx[base & (leaf_cluster_idx >= 0)], minlength=max(lerf_range) + 1).tolist()
    count = lambda idx: counts[idx] if 0 <= idx < len(counts) else 0          # noqa: E731
    cand = [idx for idx in lerf_range if not (better_vis and count(idx) < 100)]
    if not post_process:
        cand = [idx for idx in cand if count(idx) >= 10]
        return cand, _slot_map(leaf_cluster_idx, base, cand)
    subset = _slot_map(leaf_cluster_idx, base, cand)
    if subset.is_cuda:
        subset, counts = _post_process_slots(subset, len(cand), means3D)
        kept = [k for k, c in enumerate(counts) if c >= 10]
    else:
        kept = []
        for k, idx in enumerate(cand):
            filt = subset == k
            post = _post_process(filt, means3D)
            subset = torch.where(filt & ~post, -1, subset).to(torch.int32)
            if post.sum() >= 10:
                kept.append(k)
    lut = torch.full((len(cand) + 1,), -1, dtype=torch.int32, device=subset.device)     # renumber the kept slots
    lut[torch.tensor(kept, dtype=torch.long, device=subset.device)] = torch.arange(len(kept), dtype=torch.int32,
                                                                                  device=subset.device)
    subset = torch.where(subset >= 0, lut[subset.long()], subset)
    return [cand[k] for k in kept], subset


def _slot_route(fused, batched, means2D, *inputs):
    """_subset_route in the current grad mode: a gradient is needed when grad is enabled and one of `inputs` requires
    it."""
    needs_grad = torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in inputs)
    return _subset_route(fused, batched, needs_grad, means2D.requires_grad)


def _subset_route(fused, batched, needs_grad, means2D_grad):
    """How _render_slots renders its slots: "batched" (one forward_subsets call, no gradient), "batched_grad" (one
    forward_subsets_grad call) or "loop" (the reference's one rasterizer pass per slot).  The loop stays for fused=False
    (the reference's literal passes), for pipe.batched_subsets = False (batched=False), and when the screen-space points
    need a gradient (trainable geometry: the loop feeds viewspace_points.grad, a subset call has no means2D input).
    A single slot (the Stage 2.2 root pass) is batched too: the call preprocesses every Gaussian where the loop gathers
    the slot's rows, but the loop's filter, count read and gather cost more (2.83 -> 2.47 ms per step on a B200 at
    1 M Gaussians, DESIGN.md section 8 item 8)."""
    if not (fused and batched):
        return "loop"
    if not needs_grad:
        return "batched"
    return "loop" if means2D_grad else "batched_grad"


def _render_slots(rasterizer, bg3, ids, subset, means3D, means2D, opacity, scales, rotations, cov3D_precomp, feat, shs,
                  fused, keep_min_alpha=None, batched=True):
    """The images of the planned slots -> (images, silhouettes), lists in slot order, each entry as _feat_pass returns it.
    keep_min_alpha: keep only the slots whose silhouette exceeds it somewhere (the coarse loop's test, :222), and
    remove the others from `ids` in place.  batched=False: the loop (pipe.batched_subsets)."""
    imgs, sils = [], []
    route = _slot_route(fused, batched, means2D, means3D, opacity, scales, rotations, cov3D_precomp, feat, shs)
    if route != "loop":
        keep_ids = []
        for a, b, img, sil in _render_slots_batched(rasterizer, bg3, len(ids), subset, means3D, opacity, scales,
                                                    rotations, cov3D_precomp, feat, shs, route == "batched_grad"):
            if keep_min_alpha is not None:
                keep = (sil.amax(dim=(1, 2, 3)) > keep_min_alpha).tolist()       # one host read per launch
                sel = [k for k in range(b - a) if keep[k]]
                keep_ids += [ids[a + k] for k in sel]
                if len(sel) != b - a:
                    sel_t = torch.tensor(sel, dtype=torch.long, device=img.device)
                    img, sil = img.index_select(0, sel_t), sil.index_select(0, sel_t)
            imgs += list(img.unbind(0))
            sils += list(sil.unbind(0))
        if keep_min_alpha is not None:
            ids[:] = keep_ids
        return imgs, sils

    def filt(t, idx):
        return None if t is None else t[idx]

    keep_ids = []
    for k, idx in enumerate(ids):
        filter_idx = subset == k
        img, sil = _feat_pass(rasterizer, bg3, means3D[filter_idx], means2D[filter_idx], opacity[filter_idx],
                              scales[filter_idx], rotations[filter_idx], filt(cov3D_precomp, filter_idx),
                              feat[filter_idx], shs=filt(shs, filter_idx), fused=fused)
        if keep_min_alpha is not None and not sil.max() > keep_min_alpha:
            continue
        keep_ids.append(idx)
        imgs.append(img)
        sils.append(sil)
    ids[:] = keep_ids
    return imgs, sils


def _render_slots_batched(rasterizer, bg3, S, subset, means3D, opacity, scales, rotations, cov3D_precomp, feat, shs,
                          grad=False):
    """forward_subsets (grad: forward_subsets_grad) over slots [a, b) per launch, each launch's outputs and state within
    SUBSET_BATCH_BYTES: yields (a, b, images [b-a,F,H,W], silhouettes [b-a,1,H,W]) with the channel layout of
    _feat_pass."""
    rs = rasterizer.raster_settings
    H, W = int(rs.image_height), int(rs.image_width)
    kw = _feat_args(bg3, feat, shs)
    nb = kw["extra_feats"].shape[-1] if "extra_feats" in kw else 0
    per_launch = max(1, SUBSET_BATCH_BYTES // (((3 + nb + 2) * 4 + (8 if grad else 0)) * H * W))
    call = rasterizer.forward_subsets_grad if grad else rasterizer.forward_subsets
    for a in range(0, S, per_launch):
        b = min(S, a + per_launch)
        sub = subset if (a == 0 and b == S) else torch.where((subset >= a) & (subset < b), subset - a, -1)
        color, _, alpha, extra = call(means3D, opacity, sub, b - a, scales=scales, rotations=rotations,
                                      cov3D_precomp=cov3D_precomp, **kw)
        yield a, b, _feat_image(color, extra, shs, 1), alpha


def render(viewpoint_camera, pc, pipe, bg_color: torch.Tensor, iteration,
           scaling_modifier=1.0, override_color=None, visible_mask=None, mask_num=0,
           cluster_idx=None,       # per-point cluster id (coarse-level)
           leaf_cluster_idx=None,  # per-point cluster id (fine-level)
           rescale=True,           # re-scale (for enhance ins_feat)
           origin_feat=False,      # origin ins_feat (not quantized)
           render_feat_map=True,   # render image-level feat map
           render_color=True,      # render rgb image
           render_cluster=False,   # render cluster, stage 2.2
           better_vis=False,       # filter some points
           selected_root_id=None,  # coarse-level cluster id
           selected_leaf_id=None,  # fine-level cluster id (possibly more than one)
           pre_mask=None,
           seg_rgb=False,          # render cluster rgb, not feat
           post_process=False,     # post
           root_num=64, leaf_num=10,
           fused=True):
    """Render the scene.  Background tensor (bg_color) must be on GPU!
    ``pipe.view_cache = False`` keeps this call out of the frozen-geometry view cache (rasterizer.ViewCache).
    ``pipe.batched_subsets = False`` renders the cluster / leaf passes one rasterizer pass per subset, as the reference
    does, instead of one subset call per pass (same images; the gradients differ only in the order of float additions)."""
    if getattr(pipe, "view_cache", True) is False and _view_cache.enabled:
        with _view_cache.disabled():
            return render(viewpoint_camera, pc, pipe, bg_color, iteration, scaling_modifier, override_color, visible_mask,
                          mask_num, cluster_idx, leaf_cluster_idx, rescale, origin_feat, render_feat_map, render_color,
                          render_cluster, better_vis, selected_root_id, selected_leaf_id, pre_mask, seg_rgb, post_process,
                          root_num, leaf_num, fused)
    xyz = pc.get_xyz
    # Screen-space gradient sink (reference :45): its .grad feeds the densification statistics (train.py:598,
    # scene/gaussian_model.py:512-514), which only exist while the geometry trains.  From stage 1 on OpenGaussian
    # detaches the geometry (train.py:431-436); asking the rasterizer for dL/dmeans2D there forces the FULL geometry
    # backward (blend moments + preprocess chain, ~0.45 ms per step at 1 M Gaussians) for a tensor nobody reads.  So the
    # sink tracks gradients only when the positions do (or when pipe.viewspace_grad = True); otherwise it is a plain
    # zero tensor whose .grad is zeros, so that code reading viewspace_points.grad keeps working.
    track_vs = bool(xyz.requires_grad or getattr(pipe, "viewspace_grad", False))
    if track_vs:
        screenspace_points = torch.zeros_like(xyz, dtype=xyz.dtype, requires_grad=True, device=xyz.device) + 0
        try:
            screenspace_points.retain_grad()
        except Exception:
            pass
    else:
        screenspace_points = _zero_sink(xyz)

    tanfovx = math.tan(viewpoint_camera.FoVx * 0.5)
    tanfovy = math.tan(viewpoint_camera.FoVy * 0.5)
    raster_settings = GaussianRasterizationSettings(
        image_height=int(viewpoint_camera.image_height),
        image_width=int(viewpoint_camera.image_width),
        tanfovx=tanfovx, tanfovy=tanfovy, bg=bg_color, scale_modifier=scaling_modifier,
        viewmatrix=viewpoint_camera.world_view_transform, projmatrix=viewpoint_camera.full_proj_transform,
        sh_degree=pc.active_sh_degree, campos=viewpoint_camera.camera_center, prefiltered=False,
        debug=pipe.debug)
    rasterizer = GaussianRasterizer(raster_settings=raster_settings)

    means3D = xyz
    means2D = screenspace_points

    # probabilistically rescale (same RNG draws as the reference, :121-124)
    prob = torch.rand(1)
    rescale_factor = None         # 1.0: the reference builds a device scalar here every call (:122, a host->device copy)
    rescaled = False
    if prob > 0.5 and rescale:
        rescale_factor = torch.rand(1).to(xyz.device)
        rescaled = True
    one_pass = fused and render_color and render_feat_map and not rescaled

    # Raw-parameter path (SURVEY.md 8a9): when this call is exactly one fused pass over the whole model,
    # hand the PARAMETERS to the rasterizer and let preprocess apply the getters of
    # scene/gaussian_model.py:122-169 (exp / normalize / sigmoid, no get_features cat, no ins_feat
    # normalize) -- forward and backward -- instead of ~10 elementwise kernels and a 192 B/Gaussian copy.
    needs_activated = (render_cluster and cluster_idx is not None) or \
        (leaf_cluster_idx is not None and leaf_cluster_idx.numel() > 0)
    raw_names = ("_xyz", "_opacity", "_scaling", "_rotation", "_features_dc", "_features_rest", "_ins_feat")
    use_raw = (one_pass and not needs_activated and override_color is None and not pipe.compute_cov3D_python
               and not pipe.convert_SHs_python and all(hasattr(pc, n) for n in raw_names)
               and getattr(pipe, "raw_parameter_path", True))

    opacity = scales = rotations = cov3D_precomp = shs = colors_precomp = None
    if not use_raw:
        opacity = pc.get_opacity
        if pipe.compute_cov3D_python:
            cov3D_precomp = pc.get_covariance(scaling_modifier)
        else:
            scales = pc.get_scaling
            rotations = pc.get_rotation
        if override_color is None:
            if pipe.convert_SHs_python:
                from .sh import eval_sh
                shs_view = pc.get_features.transpose(1, 2).view(-1, 3, (pc.max_sh_degree + 1) ** 2)
                dir_pp = (pc.get_xyz - viewpoint_camera.camera_center.repeat(pc.get_features.shape[0], 1))
                dir_pp_normalized = dir_pp / dir_pp.norm(dim=1, keepdim=True)
                sh2rgb = eval_sh(pc.active_sh_degree, shs_view, dir_pp_normalized)
                colors_precomp = torch.clamp_min(sh2rgb + 0.5, 0.0)
            else:
                shs = pc.get_features
        else:
            colors_precomp = override_color

    def sc(s):
        return None if s is None else (s * rescale_factor if rescaled else s)

    rendered_image = radii = rendered_depth = rendered_alpha = None
    rendered_ins_feat = silhouette = None
    bg3 = bg_color.reshape(-1).float()
    batched = getattr(pipe, "batched_subsets", True)
    if use_raw:
        q = getattr(pc, "_ins_feat_q", None)
        raw_feat = pc._ins_feat if (origin_feat or q is None or len(q) == 0) else q
        nb = raw_feat.shape[-1]
        ebg = _tiled_bg(bg3, nb)
        rendered_image, radii, rendered_depth, rendered_alpha, rendered_ins_feat = rasterizer.forward_raw(
            means3D, means2D, pc._opacity, pc._features_dc, pc._features_rest, pc._scaling, pc._rotation,
            raw_ins_feat=raw_feat, extra_bg=ebg)
        silhouette = rendered_alpha
    elif one_pass:
        # ONE launch: RGB + feature channels + depth + alpha; silhouette == alpha (same geometry)
        ins_feat = (pc.get_ins_feat(origin=origin_feat) + 1) / 2
        nb = ins_feat.shape[-1]
        ebg = _tiled_bg(bg3, nb)
        rendered_image, radii, rendered_depth, rendered_alpha, rendered_ins_feat = rasterizer(
            means3D=means3D, means2D=means2D, shs=shs, colors_precomp=colors_precomp, opacities=opacity,
            scales=scales, rotations=rotations, cov3D_precomp=cov3D_precomp, extra_feats=ins_feat, extra_bg=ebg)
        silhouette = rendered_alpha
    else:
        if render_color:
            rendered_image, radii, rendered_depth, rendered_alpha = rasterizer(
                means3D=means3D, means2D=means2D, shs=shs, colors_precomp=colors_precomp, opacities=opacity,
                scales=scales, rotations=rotations, cov3D_precomp=cov3D_precomp)
        if render_feat_map:
            ins_feat = (pc.get_ins_feat(origin=origin_feat) + 1) / 2
            if fused:
                rendered_ins_feat, silhouette = _feat_pass(rasterizer, bg3, means3D, means2D, opacity, sc(scales),
                                                           rotations, cov3D_precomp, ins_feat)
            else:   # the reference's literal 3 passes (:129-163)
                rendered_ins_feat, _, _, _ = rasterizer(
                    means3D=means3D, means2D=means2D, shs=None, colors_precomp=ins_feat[:, :3], opacities=opacity,
                    scales=sc(scales), rotations=rotations, cov3D_precomp=cov3D_precomp)
                if ins_feat.shape[-1] > 3:
                    rendered_ins_feat2, _, _, _ = rasterizer(
                        means3D=means3D, means2D=means2D, shs=None, colors_precomp=ins_feat[:, 3:6],
                        opacities=opacity, scales=sc(scales), rotations=rotations, cov3D_precomp=cov3D_precomp)
                    rendered_ins_feat = torch.cat((rendered_ins_feat, rendered_ins_feat2), dim=0)
                _, _, _, silhouette = rasterizer(
                    means3D=means3D, means2D=means2D, shs=shs, colors_precomp=colors_precomp, opacities=opacity,
                    scales=sc(scales), rotations=rotations, cov3D_precomp=cov3D_precomp)

    # ---- [Stage 2.2] coarse cluster-level feature maps (:173-236) ----
    viewed_pts = radii > 0
    if cluster_idx is not None:
        num_cluster = cluster_idx.max() + 1
        cluster_occur = torch.zeros(num_cluster).to(torch.bool)
    else:
        cluster_occur = None
    if render_cluster and cluster_idx is not None and viewed_pts.sum() != 0:
        ins_feat = (pc.get_ins_feat(origin=origin_feat) + 1) / 2
        scale_filter = (scales < 0.5).all(dim=1)
        ids, subset = _plan_clusters(cluster_idx, int(num_cluster), viewed_pts, scale_filter, better_vis,
                                     selected_root_id, viewpoint_camera.bClusterOccur)
        rendered_clusters, rendered_cluster_silhouettes = _render_slots(
            rasterizer, bg3, ids, subset, means3D, means2D, opacity, sc(scales), rotations, cov3D_precomp, ins_feat,
            None, fused, keep_min_alpha=0.8, batched=batched)
        for idx in ids:
            cluster_occur[idx] = True
        if len(rendered_cluster_silhouettes) != 0:
            rendered_cluster_silhouettes = torch.vstack(rendered_cluster_silhouettes)
    else:
        rendered_clusters, rendered_cluster_silhouettes = None, None

    # ---- [Stage 2.2 & 3] fine cluster-level feature maps (:245-356) ----
    if leaf_cluster_idx is not None and leaf_cluster_idx.numel() > 0:
        ins_feat = (pc.get_ins_feat(origin=origin_feat) + 1) / 2
        scale_filter = (scales < 0.1).all(dim=1)
        if selected_leaf_id is None:
            if selected_root_id is not None:
                start_leaf = selected_root_id * leaf_num
                end_leaf = start_leaf + leaf_num
            else:
                start_leaf = 0
                end_leaf = root_num * leaf_num
            lerf_range = range(start_leaf, end_leaf)
        else:
            lerf_range = selected_leaf_id.tolist()
        skip_all = len(lerf_range) > 0 and viewpoint_camera.bClusterOccur is not None and \
            bool(viewpoint_camera.bClusterOccur[selected_root_id] == False)  # noqa: E712
        occured_leaf_id, subset = _plan_leaves(leaf_cluster_idx, [] if skip_all else list(lerf_range), selected_leaf_id,
                                               pre_mask, viewed_pts, scale_filter, better_vis, post_process, means3D)
        rendered_leaf_clusters, rendered_leaf_cluster_silhouettes = _render_slots(
            rasterizer, bg3, occured_leaf_id, subset, means3D, means2D, opacity, scales, rotations, cov3D_precomp,
            ins_feat, shs if seg_rgb else None, fused, batched=batched)
        if len(rendered_leaf_cluster_silhouettes) != 0:
            rendered_leaf_cluster_silhouettes = torch.vstack(rendered_leaf_cluster_silhouettes)
    else:
        rendered_leaf_clusters = None
        rendered_leaf_cluster_silhouettes = None
        occured_leaf_id = None

    return {"render": rendered_image,
            "alpha": rendered_alpha,
            "depth": rendered_depth,
            "silhouette": silhouette,
            "ins_feat": rendered_ins_feat,
            "cluster_imgs": rendered_clusters,
            "cluster_silhouettes": rendered_cluster_silhouettes,
            "leaf_clusters_imgs": rendered_leaf_clusters,
            "leaf_cluster_silhouettes": rendered_leaf_cluster_silhouettes,
            "occured_leaf_id": occured_leaf_id,
            "cluster_occur": cluster_occur,
            "viewspace_points": screenspace_points,
            "visibility_filter": viewed_pts,
            "radii": radii}
