"""Per-mask feature statistics and the Stage-1 losses (SURVEY.md section 8f rank 1) on the B200
streaming kernels of csrc/mask_stats.cu -- drop-ins for

* ``utils/opengs_utlis.py::mask_feature_mean`` (:240-283)  -- same signature and return values,
* ``train.py::cohesion_loss`` (:102-121) and ``train.py::separation_loss`` (:123-147),
* ``utils/opengs_utlis.py::pair_mask_feature_mean`` (:184-201),
* ``utils/opengs_utlis.py::calculate_iou`` (:90-123) and the small distance helpers
  ``calculate_pairwise_distances`` (:8-34) / ``calculate_distances`` (:36-58) used beside it by the
  Stage-3 association (train.py:870-882).

The reference expands ``feat_map [C,H,W]`` and ``gt_masks [M,H,W]`` to ``[M,C,H,W]`` float tensors
(processed in 5x5 Python chunks to dodge OOM); here every pass streams the M*H*W mask bytes once.
Both functions are differentiable (custom autograd, gradients to ``feat_map``, ``image_mask`` and the
mask means), because ``train.py:450-456`` back-propagates through them.
"""
import torch

from . import _lib


ID_MAP_MIN_MASKS = 16     # below this the M mask bytes per pixel are as cheap as building the id map


class _MaskSet:
    """Device-side forms of one ``gt_masks`` tensor: ``bytes`` [M,H*W] uint8 and, for M >= ID_MAP_MIN_MASKS, the id map
    ``ids`` [H*W] int16 with its device-side ``overlap`` flag (C ABI ogs_mask_id_map).  SAM masks are a partition of
    the image, so the four passes of a Stage-1 step read 2 B per pixel instead of M B; overlapping masks set the
    flag and the kernels walk the mask rows as before -- no host synchronisation either way."""
    __slots__ = ("bytes", "ids", "overlap")

    def __init__(self, gt_masks, ids=None):
        masks = gt_masks.detach()
        if masks.dtype != torch.bool:
            masks = masks != 0
        M = masks.shape[0]
        HW = masks.shape[1] * masks.shape[2]
        self.bytes = masks.contiguous().view(torch.uint8).view(M, HW)
        self.ids = self.overlap = None
        dev = masks.device
        if ids is not None and M <= 32767:
            self.ids = ids.detach().to(torch.int16).contiguous().view(HW)
            self.overlap = torch.zeros(1, dtype=torch.int32, device=dev)
        elif ID_MAP_MIN_MASKS <= M <= 32767 and HW > 0:
            self.ids = torch.empty(HW, dtype=torch.int16, device=dev)
            self.overlap = torch.empty(1, dtype=torch.int32, device=dev)
            _lib.launch("ogs_mask_id_map", dev, M, HW, _lib.ptr(self.bytes), _lib.ptr(self.ids), _lib.ptr(self.overlap))


# The mask set of the LAST gt_masks tensor seen: mask_feature_mean and cohesion_loss of one training step receive the
# same tensor (train.py:450-452).  The entry holds a strong reference to that tensor, so `is` cannot match a new
# tensor at a recycled address; an in-place edit bumps `_version` and misses.
_last = {"src": None, "version": -1, "set": None}


def register_mask_ids(gt_masks, ids):
    """Declare that ``gt_masks`` [M,H,W] is the one-hot expansion of ``ids`` [H,W] (-1 = no mask): the statistics
    passes on ``gt_masks`` then read the id map.  ``get_SAM_mask_and_feat`` below calls this."""
    if gt_masks.is_cuda:
        _last.update(src=gt_masks, version=gt_masks._version, set=_MaskSet(gt_masks, ids))


def _mask_set(gt_masks):
    if _last["src"] is gt_masks and _last["version"] == gt_masks._version:
        return _last["set"]
    ms = _MaskSet(gt_masks)
    _last.update(src=gt_masks, version=gt_masks._version, set=ms)
    return ms


def _prep(feat_map, gt_masks, image_mask=None):
    if not feat_map.is_cuda:
        raise _lib.OgsError("mask statistics need CUDA tensors (no CPU path)")
    Cn, H, W = feat_map.shape
    M = gt_masks.shape[0]
    assert tuple(gt_masks.shape[1:]) == (H, W), "gt_masks must be [num_mask, H, W]"
    feat = feat_map.detach().float().contiguous()
    ms = _mask_set(gt_masks)
    img = None
    if image_mask is not None:
        img = image_mask.detach().float().expand(1, H, W).contiguous().view(H * W)
    return feat, ms, img, M, Cn, H * W


def _mask_ptrs(ms):
    return _lib.ptr(ms.bytes), _lib.ptr(ms.ids), _lib.ptr(ms.overlap)


class _MaskMean(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feat_map, gt_masks, image_mask):
        feat, ms, img, M, Cn, HW = _prep(feat_map, gt_masks, image_mask)
        dev = feat.device
        sums = torch.empty(M, Cn, device=dev)
        counts = torch.empty(M, device=dev)
        _lib.launch("ogs_mask_mean_forward", dev, M, Cn, HW, _lib.ptr(feat), *_mask_ptrs(ms), _lib.ptr(img),
                    _lib.ptr(sums), _lib.ptr(counts))
        cnt = counts.clamp(min=1)
        mean = sums / cnt[:, None]
        ctx.save_for_backward(feat, img if img is not None else torch.empty(0, device=dev), counts, mean)
        ctx.ms = ms
        ctx.has_img = img is not None
        ctx.shape = feat_map.shape
        ctx.img_shape = None if image_mask is None else image_mask.shape
        ctx.mark_non_differentiable(counts)
        return mean, counts

    @staticmethod
    def backward(ctx, g_mean, _g_counts):
        feat, img, counts, mean = ctx.saved_tensors
        img = img if ctx.has_img else None
        M, Cn = mean.shape
        HW = feat.shape[1] * feat.shape[2]
        dev = feat.device
        G = (g_mean.float() / counts.clamp(min=1)[:, None]).contiguous()
        K = torch.where(counts > 1, (G * mean).sum(1), torch.zeros_like(counts)).contiguous()
        dfeat = torch.empty_like(feat)
        dimg = torch.empty(HW, device=dev) if img is not None else None
        _lib.launch("ogs_mask_mean_backward", dev, M, Cn, HW, _lib.ptr(feat), *_mask_ptrs(ctx.ms), _lib.ptr(img), _lib.ptr(G),
                    _lib.ptr(K), _lib.ptr(dfeat), _lib.ptr(dimg))
        g_img = None
        if dimg is not None and ctx.needs_input_grad[2]:
            g_img = dimg.view(1, feat.shape[1], feat.shape[2]).sum_to_size(ctx.img_shape)
        return dfeat.view(ctx.shape), None, g_img


def mask_feature_mean(feat_map, gt_masks, image_mask=None, return_var=False):
    """Average instance feature inside each mask: ``[num_mask, C]``; with ``return_var`` also the
    per-mask variance ``[num_mask]`` and pixel count ``[num_mask]`` (reference :240-283).  The mean is
    differentiable; the variance carries NO gradient (the reference's only ``return_var=True`` call site,
    train.py:689, runs inside the ``torch.no_grad()`` block of train.py:297)."""
    mean, counts = _MaskMean.apply(feat_map, gt_masks, image_mask)
    if not return_var:
        return mean
    feat, ms, img, M, Cn, HW = _prep(feat_map, gt_masks, image_mask)
    sq = torch.empty(M, Cn, device=feat.device)
    mean_d = mean.detach().contiguous()
    _lib.launch("ogs_mask_var_forward", feat.device, M, Cn, HW, _lib.ptr(feat), *_mask_ptrs(ms), _lib.ptr(img),
                _lib.ptr(mean_d), _lib.ptr(sq))
    cnt = counts.clamp(min=1)
    variance = (sq / cnt[:, None]).mean(dim=1)
    return mean, variance, cnt


class _Cohesion(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feat_map, gt_mask, feat_mean_stack):
        feat, ms, _, M, Cn, HW = _prep(feat_map, gt_mask)
        dev = feat.device
        mean = feat_mean_stack.detach().float().contiguous()
        dsum = torch.empty(M, device=dev)
        npix = torch.empty(M, device=dev)
        _lib.launch("ogs_cohesion_forward", dev, M, Cn, HW, _lib.ptr(feat), *_mask_ptrs(ms), _lib.ptr(mean), _lib.ptr(dsum),
                    _lib.ptr(npix))
        ctx.save_for_backward(feat, mean, npix)
        ctx.ms = ms
        ctx.shape = feat_map.shape
        return (dsum / npix.clamp(min=1)).mean() if M > 0 else feat.new_zeros(())

    @staticmethod
    def backward(ctx, g):
        feat, mean, npix = ctx.saved_tensors
        M, Cn = mean.shape
        HW = feat.shape[1] * feat.shape[2]
        dev = feat.device
        coef = (g.float() / (max(M, 1) * npix.clamp(min=1))).contiguous()
        dfeat = torch.empty_like(feat)
        dmean = torch.empty(M, Cn, device=dev)
        _lib.launch("ogs_cohesion_backward", dev, M, Cn, HW, _lib.ptr(feat), *_mask_ptrs(ctx.ms), _lib.ptr(mean),
                    _lib.ptr(coef), _lib.ptr(dfeat), _lib.ptr(dmean))
        return dfeat.view(ctx.shape), None, dmean


def cohesion_loss(feat_map, gt_mask, feat_mean_stack):
    """Intra-mask smoothing loss, Eq. (1) (reference train.py:102-121): mean over masks of the mean
    L2 distance of the mask's pixels to the mask's mean feature."""
    return _Cohesion.apply(feat_map, gt_mask, feat_mean_stack)


class _Separation(torch.autograd.Function):
    """separation_loss value + gradient in two kernel launches (C ABI ogs_separation_loss)."""

    @staticmethod
    def forward(ctx, mean, small_weights):
        m = mean.detach().float().contiguous()
        N, Cn = m.shape
        dev = m.device
        buf = torch.empty(N * N + N + 1 + N * Cn, dtype=torch.float32, device=dev)
        loss = buf[N * N + N:N * N + N + 1]
        dmean = buf[N * N + N + 1:].view(N, Cn)
        _lib.launch("ogs_separation_loss", dev, N, Cn, _lib.ptr(m), int(bool(small_weights)), _lib.ptr(buf), _lib.ptr(loss),
                    _lib.ptr(dmean))
        ctx.save_for_backward(dmean)
        return loss.reshape(())

    @staticmethod
    def backward(ctx, g):
        (dmean,) = ctx.saved_tensors
        return dmean * g, None


def separation_loss(feat_mean_stack, iteration=None):
    """Inter-mask contrastive loss, Eq. (2) (reference train.py:123-155).  On CUDA with 2 <= N: two kernel launches for
    value and gradient (csrc/separation.cu) instead of ~40 tiny torch kernels; otherwise the reference's expression."""
    N = feat_mean_stack.shape[0]
    if feat_mean_stack.is_cuda and N >= 2 and feat_mean_stack.shape[1] <= 16:
        return _Separation.apply(feat_mean_stack, iteration is not None and iteration > 35000)
    diff_squared = (feat_mean_stack.unsqueeze(1) - feat_mean_stack.unsqueeze(0)).pow(2).sum(2)
    inverse_distance = 1.0 / (diff_squared + 1)
    mask = torch.eye(N, device=feat_mean_stack.device).bool()
    inverse_distance = inverse_distance.masked_fill(mask, 0)
    sorted_indices = inverse_distance.argsort().argsort()
    loss_weight = (sorted_indices.float() / (N - 1)) * (1.0 - 0.1) + 0.1
    if iteration is not None and iteration > 35000:
        loss_weight[loss_weight < 0.9] = 0.1
    inverse_distance = inverse_distance * loss_weight
    return inverse_distance.sum() / (N * (N - 1))


def pair_mask_feature_mean(feat_map, masks):
    """Mean feature of N (map, mask) pairs: feat_map [N,C,H,W], masks [N,H,W] -> [N,C] (reference :184-201).
    One single-mask streaming pass per pair."""
    outs = []
    for i in range(feat_map.shape[0]):
        if not feat_map.is_cuda:
            raise _lib.OgsError("mask statistics need CUDA tensors (no CPU path)")
        feat = feat_map[i].detach().float().contiguous()
        Cn, HW = feat.shape[0], feat.shape[1] * feat.shape[2]
        mk = _MaskSet(masks[i:i + 1])              # one mask: no id map, and the step's cached mask set stays
        sums = torch.empty(1, Cn, device=feat.device)
        counts = torch.empty(1, device=feat.device)
        w = masks[i].detach().float().contiguous().view(HW)     # the reference multiplies by masks.float()
        _lib.launch("ogs_mask_mean_forward", feat.device, 1, Cn, HW, _lib.ptr(feat), *_mask_ptrs(mk), _lib.ptr(w),
                    _lib.ptr(sums), _lib.ptr(counts))
        outs.append(sums[0] / (counts[0] + 1e-6))
    return torch.stack(outs) if outs else feat_map.new_zeros(0, feat_map.shape[1])


def get_SAM_mask_and_feat(gt_sam_mask, level=3, filter_th=50, original_mask_feat=None, sample_mask=False, num_mask=None,
                          prev_max=None):
    """Per-view SAM masks from the 4-level id map ``gt_sam_mask`` [4,H,W] (reference utils/opengs_utlis.py:125-182):
    returns ``mask_id`` [H,W] (0 = invalid pixel, 1..num_mask), ``mask_bool`` [num_mask,H,W] (mask 0, the invalid pixels,
    excluded), optionally the masks' language features, and ``invalid_pix`` [H,W].  ``filter_th`` / ``sample_mask`` are
    unused, as in the reference.  Differences: ``mask_bool`` is a torch.bool tensor written by one kernel (C ABI
    ogs_sam_masks; the reference materialises an int64 one-hot, 8x the bytes, and re-derives mask_id with an argmax that
    returns it unchanged), and the id map is registered for the Stage-1 statistics passes (``register_mask_ids``).  ``num_mask`` (this level's mask
    count) and ``prev_max`` (the previous level's largest id) are properties of the view's SAM file: a trainer that
    stores them at load time passes them here and the call makes no device-to-host read (the reference does two per
    step, :138 and :146)."""
    if not gt_sam_mask.is_cuda:
        raise _lib.OgsError("get_SAM_mask_and_feat needs a CUDA id map (no CPU path)")
    dev = gt_sam_mask.device
    H, W = gt_sam_mask.shape[1:]
    HW = H * W
    level_ids = gt_sam_mask[level].to(torch.int32).contiguous()
    offset = 0
    if level > 0:
        offset = int(gt_sam_mask[level - 1].max().item() if prev_max is None else prev_max) + 1
    num = int((level_ids.max().item() - offset + 1) if num_mask is None else num_mask)
    num = max(num, 0)
    mask_id = torch.empty(H, W, dtype=torch.int64, device=dev)
    invalid_pix = torch.empty(H, W, dtype=torch.bool, device=dev)
    ids = torch.empty(HW, dtype=torch.int16, device=dev)
    mask_bool = torch.empty(num, H, W, dtype=torch.bool, device=dev)
    _lib.launch("ogs_sam_masks", dev, num, HW, _lib.ptr(level_ids), offset, _lib.ptr(mask_id), _lib.ptr(invalid_pix),
                _lib.ptr(ids), _lib.ptr(mask_bool))
    register_mask_ids(mask_bool, ids)
    if original_mask_feat is not None:
        max_ind = int(gt_sam_mask[level].max()) + 1
        min_ind = int(gt_sam_mask[level - 1].max()) + 1 if level > 0 else 0
        return mask_id, mask_bool, original_mask_feat.clone()[min_ind:max_ind, :], invalid_pix
    return mask_id, mask_bool, invalid_pix


def _as_mask_bytes(masks):
    if not masks.is_cuda:
        raise _lib.OgsError("calculate_iou needs CUDA tensors (no CPU path)")
    m = masks.detach()
    if m.dtype != torch.bool:
        m = m != 0
    return m.contiguous().view(torch.uint8)


def mask_pair_counts(masks1, masks2):
    """Integer statistics behind calculate_iou: (inter int32 [m,n], count1 int32 [n], count2 int32 [m])
    for masks1 [n,H,W] and masks2 [m,H,W]."""
    assert masks1.shape[1:] == masks2.shape[1:], "both mask sets must share H, W"
    a, b = _as_mask_bytes(masks1), _as_mask_bytes(masks2)
    n, m = a.shape[0], b.shape[0]
    HW = int(a.shape[1] * a.shape[2])
    dev = a.device
    inter = torch.empty(m, n, dtype=torch.int32, device=dev)
    counts = torch.empty(n + m, dtype=torch.int32, device=dev)
    if n + m > 0:
        nbytes = int(_lib.lib().ogs_mask_iou_scratch_bytes(n, m, HW))
        scratch = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=dev)
        _lib.launch("ogs_mask_pair_counts", dev, n, m, HW, _lib.ptr(a), _lib.ptr(b), _lib.ptr(scratch), _lib.ptr(inter),
                    _lib.ptr(counts))
    return inter, counts[:n], counts[n:]


def calculate_iou(masks1, masks2, base=None):
    """IoU matrix [m, n] between masks1 [n,H,W] and masks2 [m,H,W] (reference :90-123; ``base="former"`` divides
    by |masks1[i]|, ``"later"`` by |masks2[j]|, otherwise by the union).  Values equal the reference's float32
    sums exactly: all counts are integers below 2^24."""
    inter, c1, c2 = mask_pair_counts(masks1, masks2)
    intersection = inter.float()
    if base == "former":
        union = c1.float()[None, :] + 1e-6
    elif base == "later":
        union = c2.float()[:, None] + 1e-6
    else:
        union = (c1[None, :] + c2[:, None] - inter).float() + 1e-6
    return intersection / union


def calculate_pairwise_distances(tensor1, tensor2, metric=None):
    """L1 / L2 distances between every pair of rows of [m,D] and [n,D] (reference :8-34).  O(m n D): plain torch."""
    t1, t2 = tensor1.unsqueeze(1), tensor2.unsqueeze(0)
    if metric == "l1":
        return torch.abs(t1 - t2).sum(dim=2), None
    if metric == "l2":
        return None, torch.sqrt((t1 - t2).pow(2).sum(dim=2))
    return torch.abs(t1 - t2).sum(dim=2), torch.sqrt((t1 - t2).pow(2).sum(dim=2))


def calculate_distances(tensor1, tensor2, metric=None):
    """Row-wise L1 / L2 distances of two [N,D] tensors (reference :36-58)."""
    if metric == "l1":
        return torch.abs(tensor1 - tensor2).sum(dim=1)
    if metric == "l2":
        return torch.sqrt((tensor1 - tensor2).pow(2).sum(dim=1))
    return torch.abs(tensor1 - tensor2).sum(dim=1), torch.sqrt((tensor1 - tensor2).pow(2).sum(dim=1))
