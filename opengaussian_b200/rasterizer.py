"""Drop-in for the rasterizer package OpenGaussian imports as
``ashawkey_diff_gaussian_rasterization`` (gaussian_renderer/__init__.py:15,55-70,104-112;
utils/sam_refinement_utils.py:21,347-403): ``GaussianRasterizationSettings``,
``GaussianRasterizer`` and the autograd function behind them.

Same names, argument meaning, return tuple ``(color [3,H,W], radii [P] int32, depth [1,H,W],
alpha [1,H,W])`` and error messages as the upstream Python layer.  The compute is
libogs_b200.so (hand-written sm_100a CUDA behind the C ABI of include/ogs_b200.h); torch only
owns device memory and the stream.  Extension over upstream: ``extra_feats=[P,F]`` composites F
more per-Gaussian channels (OpenGaussian's ``ins_feat``) in the SAME pass and appends a fifth
return value ``feats [F,H,W]`` -- this is what lets ``render()`` replace its 4 passes by one.
"""
import collections
import ctypes as C
import itertools
import os
import threading
from typing import NamedTuple, Optional

import torch
import torch.nn as nn
from torch.autograd.function import once_differentiable

from . import _lib

_SUPPORTED_C = (3, 4, 6, 9, 12, 16)


class GaussianRasterizationSettings(NamedTuple):
    image_height: int
    image_width: int
    tanfovx: float
    tanfovy: float
    bg: torch.Tensor
    scale_modifier: float
    viewmatrix: torch.Tensor
    projmatrix: torch.Tensor
    sh_degree: int
    campos: torch.Tensor
    prefiltered: bool
    debug: bool


def _f32c(t: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    if t is None:
        return None
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def _none_if_empty(t):
    if t is None:
        return None
    if isinstance(t, torch.Tensor) and t.numel() == 0:
        return None
    return t


class _Alloc:
    """Allocation callback handed to the C ABI.  ONE process-wide ctypes thunk is created; the per-call
    state travels through the ABI's `alloc_user` pointer (a key into `_live`), so concurrent forwards from
    several Python threads / devices do not see each other.  Each forward owns a fresh dict that receives
    the torch buffers (kept alive by the autograd ctx).  No per-call ctypes objects and no reference cycles:
    buffers are released by refcount as soon as the graph dies (a cycle here would park ~100 MB per frame
    until the cyclic GC runs and force the caching allocator into cudaMalloc on every step)."""
    _live = {}
    _next = itertools.count(1)

    @staticmethod
    def _cb(user, nbytes, tag):
        bufs, device = _Alloc._live[user]
        t = torch.empty(max(int(nbytes), 1), dtype=torch.uint8, device=device)
        bufs[tag.decode()] = t
        return t.data_ptr()

    def __init__(self, device):
        self.bufs = {}
        self.key = next(_Alloc._next)
        _Alloc._live[self.key] = (self.bufs, device)
        self.fn = _ALLOC_THUNK
        self.user = C.c_void_p(self.key)

    def __del__(self):
        _Alloc._live.pop(self.key, None)


_ALLOC_THUNK = _lib.ALLOC_FN(_Alloc._cb)


def _sig(t):
    """Identity of a tensor's CONTENTS as far as torch can vouch for them: storage address, shape and the version
    counter that every in-place operation bumps (detach() / views share it with their base)."""
    return None if t is None else (t.data_ptr(), t._version, tuple(t.shape), tuple(t.stride()))


_CAM_COPIES = collections.OrderedDict()   # _sig(source) + dtype -> (contiguous fp32 copy, source), least recently used first
_CAM_COPIES_MAX = 4096                     # three matrices per camera at most; a copy costs one 512-byte block


def camera_inputs(viewmatrix, projmatrix, campos):
    """The camera part of a forward: ``(key, (viewmatrix, projmatrix, campos))`` -- the key taken from the CALLER's
    tensors (storage, version counter, shape, stride: the rule the geometry follows), the tensors as the C ABI needs them
    (contiguous float32).  The reference builds ``world_view_transform`` and the projection matrix transposed
    (scene/cameras.py:71-73), i.e. non-contiguous: their copies are made once per source tensor and reused while the
    source is unchanged, so the key, and the address a captured graph reads, repeat from one step to the next.  An
    in-place edit of the source (or of its base) bumps its version: new key, fresh copy."""
    key = (_sig(viewmatrix), _sig(projmatrix), _sig(campos))
    out = []
    for t, sig in zip((viewmatrix, projmatrix, campos), key):
        if t is None or (t.dtype == torch.float32 and t.is_contiguous()):
            out.append(t)
            continue
        sig = sig + (t.dtype,)
        hit = _CAM_COPIES.get(sig)
        if hit is not None:
            _CAM_COPIES.move_to_end(sig)
            out.append(hit[0])
            continue
        c = _f32c(t)
        if not (c.is_cuda and torch.cuda.is_current_stream_capturing()):   # a copy made inside a capture is the graph's
            _CAM_COPIES[sig] = (c, t)                                        # own memory: never handed out again
            while len(_CAM_COPIES) > _CAM_COPIES_MAX:
                _CAM_COPIES.popitem(last=False)
        out.append(c)
    return key, tuple(out)


def pin_for_capture(device, *tensors):
    """While graphs.GraphedViewStep captures on `device`, remembers `tensors` (library-internal cached buffers the
    captured kernels read) for as long as the graph lives; a no-op otherwise."""
    pins = _CAPTURE_PINS.get(device.index)
    if pins is not None:
        pins.append(tensors)


class _ViewEntry:
    __slots__ = ("geom_key", "state", "geom", "binning", "radii", "keep", "nbytes")


class ViewCache:
    """Per-camera reuse of everything the rasterizer derives from the GEOMETRY (SURVEY.md 8a4/a5: projected records,
    SH colours, radii, depth-sorted per-tile lists) while that geometry is frozen.

    From Stage 1 on OpenGaussian detaches xyz / scaling / rotation / opacity / SH and trains `_ins_feat` only
    (train.py:431-436), but the reference re-runs preprocess, duplication and the 64-bit sort on every render() of a
    training camera for 40 000 iterations.  Here a forward whose geometry parameters do not require grad leaves its
    geometry + binning buffers in this cache (exact-size copies: ~95 MB per view at 1 M Gaussians / 10 M duplicates;
    the default budget is 25 % of the device's memory, i.e. hundreds of views on a 180 GB B200, LRU beyond that), and
    the next forward of the same camera runs only the feature activation and the blend kernel
    (C ABI ogs_raster_forward_cached) -- bit-identical images, the usual backward.

    Admission: forwards on the model's own parameter tensors (raw-parameter mode, what render() uses for its fused pass)
    fill an entry at once; forwards on activated tensors only when the same tensors arrive twice in a row
    (`second_sighting`) -- the getters, the Stage-2 rescale draw and the cluster filters build new tensors per call.

    Validity is decided from what torch guarantees: an entry is keyed by the caller's camera tensors (camera_inputs;
    the reference's transposed matrices included) and matched against the geometry tensors' storage address, shape and
    VERSION COUNTER (bumped by every in-place op, shared by detach() and views -- so the per-iteration `.detach()` of
    train.py:431-436 still hits, an optimizer step or a densification misses).  The entry holds references to those tensors, so an address cannot be recycled while it is alive.
    NOT seen: writes through `tensor.data` or raw pointers -- call `view_cache.clear()` after such edits, or set
    `view_cache.enabled = False` (env OGS_VIEW_CACHE=0; per call: `pipe.view_cache = False` in render()).  The `radii`
    a cache hit returns alias the entry's copy: read-only, as every caller in the reference treats them."""

    def __init__(self):
        self.enabled = os.environ.get("OGS_VIEW_CACHE", "1") != "0"
        gb = os.environ.get("OGS_VIEW_CACHE_GB")
        self.max_bytes = None if gb is None else int(float(gb) * 2 ** 30)   # None: 25 % of the device, set on first use
        self._entries = collections.OrderedDict()      # camera key -> _ViewEntry, least recently used first
        self._sight = {}                               # device index -> (key, tensors) of the last unadmitted forward
        self._lock = threading.Lock()
        self.bytes = 0
        self.hits = self.misses = self.evictions = 0

    def clear(self):
        with self._lock:
            self._entries.clear()
            self._sight.clear()
            self.bytes = 0

    def second_sighting(self, device_index, key, keep) -> bool:
        """Admission rule for forwards that receive ACTIVATED tensors (the reference's own call convention): the getters
        of scene/gaussian_model.py:122-169 build new tensors on every call, so do the Stage-2 rescale draw and the
        cluster filters of render() -- geometry that will never be seen again must not cost an entry (two buffer copies,
        a host wait for the frame's duplicate count, the eviction of a useful view).  Such a forward is admitted only
        when the forward before it on this device had exactly the same key; the record holds that forward's tensors, so
        a recycled address cannot fake the match.  Raw-parameter forwards (the model's own parameter tensors) are
        admitted at once."""
        with self._lock:
            last = self._sight.get(device_index)
            if last is not None and last[0] == key:
                return True
            self._sight[device_index] = (key, keep)
            return False

    def disabled(self):
        """Context manager: forwards issued inside neither read nor fill the cache (render() uses it for
        ``pipe.view_cache = False``)."""
        return _CacheSwitch(self, False)

    def __len__(self):
        return len(self._entries)

    def stats(self):
        return dict(entries=len(self._entries), bytes=self.bytes, hits=self.hits, misses=self.misses,
                    evictions=self.evictions, max_bytes=self.max_bytes)

    @staticmethod
    def keys(rs, means3D, opacities, sh, sh_rest, colors_precomp, scales, rotations, cov3D, act_flags, n_feat_act,
             cam_key=None):
        """(camera key, geometry key) of a forward; ``cam_key`` is camera_inputs()'s key of the caller's camera tensors
        (default: taken from ``rs``)."""
        dev = means3D.device
        if cam_key is None:
            cam_key = (_sig(rs.viewmatrix), _sig(rs.projmatrix), _sig(rs.campos))
        cam = (dev.type, dev.index) + cam_key + (int(rs.image_height),
               int(rs.image_width), float(rs.tanfovx), float(rs.tanfovy), float(rs.scale_modifier),
               int(rs.sh_degree) if sh is not None else -1, bool(int(act_flags) & ~_lib.ACT_EXTRA_UNIT_HALF))
        geom = (_sig(means3D), _sig(opacities), _sig(sh), _sig(sh_rest), colors_precomp is not None, _sig(scales),
                _sig(rotations), _sig(cov3D), int(act_flags) & ~_lib.ACT_EXTRA_UNIT_HALF, bool(n_feat_act))
        return cam, geom

    def lookup(self, cam_key, geom_key):
        with self._lock:
            e = self._entries.get(cam_key)
            if e is not None and e.geom_key == geom_key:
                self._entries.move_to_end(cam_key)
                self.hits += 1
                return e
            self.misses += 1
            return None

    def insert(self, cam_key, entry: _ViewEntry, device=None):
        with self._lock:
            if self.max_bytes is None:
                total = torch.cuda.get_device_properties(device).total_memory if device is not None else 0
                self.max_bytes = int(0.25 * total)
            old = self._entries.pop(cam_key, None)          # same camera, other geometry: superseded
            if old is not None:
                self.bytes -= old.nbytes
            if entry.nbytes > self.max_bytes:
                return False
            while self._entries and self.bytes + entry.nbytes > self.max_bytes:
                _, ev = self._entries.popitem(last=False)
                self.bytes -= ev.nbytes
                self.evictions += 1
            self._entries[cam_key] = entry
            self.bytes += entry.nbytes
            return True


class _CacheSwitch:
    def __init__(self, cache, on):
        self.cache, self.on = cache, on

    def __enter__(self):
        self.prev, self.cache.enabled = self.cache.enabled, self.on
        return self.cache

    def __exit__(self, *exc):
        self.cache.enabled = self.prev
        return False


view_cache = ViewCache()
_BG_FULL = {}         # (device index, n_extra) -> (signature, [bg | extra_bg | 0] tensor, bg, extra_bg) of the last such forward
_CAPTURE_PINS = {}    # device index -> list that receives the cache buffers a CUDA-graph capture reads (graphs.GraphedViewStep)


def _fill_inputs(rs: GaussianRasterizationSettings, bg_full, means3D, opacities, shs, colors_precomp, scales,
                 rotations, cov3D_precomp, extra, n_extra, shs_rest=None, act_flags=0) -> _lib.RasterInputs:
    ri = _lib.RasterInputs()
    ri.P = means3D.shape[0]
    ri.sh_degree = int(rs.sh_degree)
    ri.M = 0 if shs is None else int(shs.shape[1]) + (0 if shs_rest is None else int(shs_rest.shape[1]))
    ri.act_flags = int(act_flags)
    ri.defer_capacity_check = int(_DEFER_CAPACITY)
    ri.shs_rest = _lib.ptr(shs_rest)
    ri.n_extra = n_extra
    ri.W = int(rs.image_width)
    ri.H = int(rs.image_height)
    ri.tanfovx = float(rs.tanfovx)
    ri.tanfovy = float(rs.tanfovy)
    ri.scale_modifier = float(rs.scale_modifier)
    ri.prefiltered = int(bool(rs.prefiltered))
    ri.debug = int(bool(rs.debug))
    ri.bg = _lib.ptr(bg_full)
    ri.viewmatrix = _lib.ptr(rs.viewmatrix)
    ri.projmatrix = _lib.ptr(rs.projmatrix)
    ri.campos = _lib.ptr(rs.campos)
    ri.means3D = _lib.ptr(means3D)
    ri.opacities = _lib.ptr(opacities)
    ri.shs = _lib.ptr(shs)
    ri.colors_precomp = _lib.ptr(colors_precomp)
    ri.scales = _lib.ptr(scales)
    ri.rotations = _lib.ptr(rotations)
    ri.cov3D_precomp = _lib.ptr(cov3D_precomp)
    ri.extra = _lib.ptr(extra)
    return ri


_FUSE_ACCUMULATE = False
_DEFER_CAPACITY = False
_GRAD_ARENA = {}      # device index -> flat fp32 tensor the backward carves its gradient buffer from (dist.GradArena)


def set_grad_arena(t: Optional[torch.Tensor]):
    """Registers (or, with None, removes) the flat float32 tensor from which the backward of this device carves the
    step's gradient buffer instead of allocating it -- opengaussian_b200.dist.GradArena passes its symmetric-memory
    buffer so that the gradient all-reduce can run through the NVSwitch multicast mapping.  The arena is reused by
    every step: gradients of the previous step that still alias it are overwritten by the next first backward."""
    if t is None:
        _GRAD_ARENA.clear()
    else:
        _GRAD_ARENA[t.device.index] = t


class deferred_capacity_check:
    """Context manager: forwards issued inside do NOT wait for their frame's (Gaussian, tile) duplicate count -- the one
    host<->device synchronisation of a frame (C ABI in->defer_capacity_check).  The caller must call
    ``capacity_overflowed(device)`` afterwards, from the same thread, and discard and redo everything computed from
    those frames when it returns True (the buffers were sized from a running estimate that proved too small; the
    estimate has been raised).  opengaussian_b200.dist.render_views_backward wraps a whole step this way."""

    def __init__(self, on: bool = True):
        self.on = on

    def __enter__(self):
        global _DEFER_CAPACITY
        self.prev = _DEFER_CAPACITY
        _DEFER_CAPACITY = self.on
        return self

    def __exit__(self, *exc):
        global _DEFER_CAPACITY
        _DEFER_CAPACITY = self.prev
        return False


def capacity_overflowed(device) -> bool:
    """Resolves every forward this thread issued on ``device`` under ``deferred_capacity_check``: True when at least
    one frame needed more (Gaussian, tile) entries than its buffers held -- its outputs are truncated."""
    with torch.cuda.device(device):
        rc = _lib.lib().ogs_raster_capacity_check()
    if rc < 0:
        _lib.check(rc, "ogs_raster_capacity_check")
    return rc == 1


def capacity_hint(device, new_hint: int = -1) -> int:
    """Reads (and with ``new_hint >= 0`` replaces; 0 = forget) this thread's running estimate of the number of
    (Gaussian, tile) entries per frame on ``device`` (C ABI ogs_raster_capacity_hint)."""
    with torch.cuda.device(device):
        return int(_lib.lib().ogs_raster_capacity_hint(int(new_hint)))


class fuse_grad_accumulation:
    """Context manager: while active, a backward whose differentiable inputs are ALL leaves that already
    hold a matching fp32 .grad adds its gradients straight into those tensors inside the preprocess-
    backward kernel and hands autograd `None` for them -- instead of writing fresh gradients that
    AccumulateGrad then adds in a separate read-read-write pass (0.08 ms per view at 1 M Gaussians).
    Used by opengaussian_b200.dist.render_views_backward for the 2nd..Vth view of a step.  Gradient hooks
    on those leaves do not see the fused contribution; anything that does not qualify falls back to the
    normal path."""

    def __init__(self, on: bool = True):
        self.on = on

    def __enter__(self):
        global _FUSE_ACCUMULATE
        self.prev = _FUSE_ACCUMULATE
        _FUSE_ACCUMULATE = self.on
        return self

    def __exit__(self, *exc):
        global _FUSE_ACCUMULATE
        _FUSE_ACCUMULATE = self.prev
        return False


def _fusable_grad(t, shape):
    g = t.grad
    return (t.is_leaf and g is not None and g.dtype == torch.float32 and g.is_contiguous() and g.device == t.device
            and tuple(g.shape) == tuple(shape))


def _check_inputs(means3D, shs, colors_precomp, scales, rotations, cov3D_precomp):
    """Upstream's argument rules (and messages) -> (shs, colors_precomp, scales, rotations, cov3D_precomp), an empty
    tensor standing for "not given" as upstream passes them."""
    if means3D.shape[0] > 0:
        shs, colors_precomp = _none_if_empty(shs), _none_if_empty(colors_precomp)
        scales, rotations, cov3D_precomp = _none_if_empty(scales), _none_if_empty(rotations), _none_if_empty(cov3D_precomp)
    if (shs is None and colors_precomp is None) or (shs is not None and colors_precomp is not None):
        raise Exception('Please provide excatly one of either SHs or precomputed colors!')
    if ((scales is None or rotations is None) and cov3D_precomp is None) or \
            ((scales is not None or rotations is not None) and cov3D_precomp is not None):
        raise Exception('Please provide exactly one of either scale/rotation pair or precomputed 3D covariance!')
    return shs, colors_precomp, scales, rotations, cov3D_precomp


def _pad_extra(extra, act_flags=0):
    """The extra channels padded with zero channels up to a compiled width (3 + F in _SUPPORTED_C) -> (extra, F padded).
    Raw channels (ACT_EXTRA_UNIT_HALF) are normalised as a whole, so they cannot be padded."""
    n = 0 if extra is None else int(extra.shape[1])
    if not n:
        return extra, 0
    c_tot = next((c for c in _SUPPORTED_C if c >= 3 + n), None)
    if c_tot is None:
        raise _lib.OgsError(f"extra_feats: at most {_SUPPORTED_C[-1] - 3} channels are supported")
    if c_tot == 3 + n:
        return extra, n
    if act_flags & _lib.ACT_EXTRA_UNIT_HALF:
        raise _lib.OgsError(f"raw extra_feats need 3 + F in {_SUPPORTED_C} (got F = {n})")
    return torch.cat([extra, extra.new_zeros(extra.shape[0], c_tot - 3 - n)], 1).contiguous(), c_tot - 3


def _bg_full(bg, extra_bg, n_extra):
    """The background of all 3 + n_extra channels, [bg | extra_bg | 0...] (extra_bg None: zeros); with extra channels
    cached per device and width, rebuilt only when bg or extra_bg changes (storage, version counter)."""
    bg = _f32c(bg).reshape(-1)
    if n_extra == 0:
        return bg
    dev = bg.device
    sig = (_sig(bg), _sig(extra_bg))
    hit = _BG_FULL.get((dev.index, n_extra))
    if hit is None or hit[0] != sig:
        if extra_bg is None:
            full = torch.cat([bg, bg.new_zeros(n_extra)])
        else:
            eb = _f32c(extra_bg).reshape(-1).to(dev)
            full = torch.cat([bg, eb, bg.new_zeros(n_extra - eb.numel())])
        hit = (sig, full, bg, extra_bg)            # the sources stay alive, so their addresses stay theirs
        _BG_FULL[(dev.index, n_extra)] = hit
    pin_for_capture(dev, hit[1])
    return hit[1]


def _prepare(rs, means3D, opacities, shs, colors_precomp, scales, rotations, cov3D_precomp, extra, extra_bg,
             sh_rest=None, act_flags=0):
    """The C-ABI arguments of a forward -> (inputs, F as given, F padded, background, camera key, camera, settings,
    inputs struct).  inputs: (means3D, opacities, shs, colors_precomp, scales, rotations, cov3D_precomp, extra,
    sh_rest) as contiguous float32, extra padded (_pad_extra); camera: camera_inputs(), which the settings now hold."""
    if means3D.device.type != "cuda":
        raise _lib.OgsError("GaussianRasterizer needs CUDA tensors (there is no CPU fallback)")
    means3D, opacities, shs, colors_precomp, scales, rotations, cov3D_precomp, extra, sh_rest = (
        _f32c(t) for t in (means3D, opacities, shs, colors_precomp, scales, rotations, cov3D_precomp, extra, sh_rest))
    if sh_rest is not None and shs is None:
        raise _lib.OgsError("shs_rest needs shs (= _features_dc)")
    n_extra_user = 0 if extra is None else int(extra.shape[1])
    extra, n_extra = _pad_extra(extra, act_flags)
    bg = _bg_full(rs.bg, extra_bg, n_extra)
    cam_key, cam = camera_inputs(rs.viewmatrix, rs.projmatrix, rs.campos)
    rs = rs._replace(viewmatrix=cam[0], projmatrix=cam[1], campos=cam[2])
    ri = _fill_inputs(rs, bg, means3D, opacities, shs, colors_precomp, scales, rotations, cov3D_precomp, extra, n_extra,
                      sh_rest, act_flags)
    inputs = (means3D, opacities, shs, colors_precomp, scales, rotations, cov3D_precomp, extra, sh_rest)
    return inputs, n_extra_user, n_extra, bg, cam_key, cam, rs, ri


def _grad_planes(grad_color, grad_feat, n_extra, shape, dev):
    """The image gradients of a backward for the C ABI -> (dL_dcolor, dL_dfeat), channels at dim -3 of images of
    `shape` without its channels ([H,W] or [S,H,W]).  With extra channels the feature gradient is always passed, with
    zero planes for the channels padded up to a compiled width or absent from the loss; with neither gradient, zero
    colour planes."""
    def planes(c):
        return (*shape[:-2], c, *shape[-2:])

    gc = _f32c(grad_color)
    gf = None
    if n_extra and grad_feat is not None and grad_feat.shape[-3] > 0:
        gf = _f32c(grad_feat)
        if gf.shape[-3] != n_extra:
            gf = torch.cat([gf, gf.new_zeros(planes(n_extra - gf.shape[-3]))], -3)
    if n_extra and gf is None:
        gf = torch.zeros(planes(n_extra), dtype=torch.float32, device=dev)
    if gc is None and gf is None:
        gc = torch.zeros(planes(3), dtype=torch.float32, device=dev)
    return gc, gf


class _RasterizeGaussians(torch.autograd.Function):
    @staticmethod
    def forward(ctx, means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp, extra,
                raster_settings, extra_bg=None, sh_rest=None, act_flags=0):
        L = _lib.lib()
        means2D_in = means2D
        act_flags = int(act_flags)
        (means3D, opacities, sh, colors_precomp, scales, rotations, cov3Ds_precomp, extra, sh_rest), n_extra_user, \
            n_extra, bg_full, cam_sig, cam, rs, ri = _prepare(
                raster_settings, means3D, opacities, sh, colors_precomp, scales, rotations, cov3Ds_precomp, extra,
                extra_bg, sh_rest, act_flags)
        cam_src = (raster_settings.viewmatrix, raster_settings.projmatrix, raster_settings.campos)
        dev = means3D.device
        P = means3D.shape[0]
        H, W = int(rs.image_height), int(rs.image_width)

        color_all = torch.empty(3 + n_extra, H, W, dtype=torch.float32, device=dev)
        depth = torch.empty(1, H, W, dtype=torch.float32, device=dev)
        alpha = torch.empty(1, H, W, dtype=torch.float32, device=dev)
        radii = torch.empty(P, dtype=torch.int32, device=dev)

        st = _lib.RasterState()
        alloc = _Alloc(dev)
        # Frozen geometry (OpenGaussian stages 1-3, train.py:431-436): reuse the camera's records and tile lists
        frozen = view_cache.enabled and P > 0 and not rs.debug and not any(
            t is not None and t.requires_grad for t in (means3D, sh, opacities, scales, rotations, cov3Ds_precomp, sh_rest))
        entry = cam_key = geom_key = None
        admit = False
        if frozen:
            n_feat_act = n_extra if (act_flags & _lib.ACT_EXTRA_UNIT_HALF) else 0
            cam_key, geom_key = ViewCache.keys(rs, means3D, opacities, sh, sh_rest, colors_precomp, scales, rotations,
                                               cov3Ds_precomp, act_flags, n_feat_act, cam_key=cam_sig)
            entry = view_cache.lookup(cam_key, geom_key)
            if entry is None:
                keep = cam_src + cam + (means3D, opacities, sh, sh_rest, scales, rotations, cov3Ds_precomp)
                admit = bool(act_flags & ~_lib.ACT_EXTRA_UNIT_HALF) or \
                    view_cache.second_sighting(dev.index, (cam_key, geom_key), keep)
        if entry is None and torch.cuda.is_current_stream_capturing():
            raise _lib.OgsError("GaussianRasterizer under CUDA-graph capture needs the view's geometry resident in "
                                "rasterizer.view_cache (frozen geometry, one eager visit first): a fresh forward reads "
                                "the frame's duplicate count back to the host")
        if entry is not None:
            pin_for_capture(dev, entry.geom, entry.binning, entry.radii, *cam)   # an evicted entry must not free what a graph reads
            radii = entry.radii.detach()     # a fresh tensor object over the first call's radii (this Function's own output)
            ro = _lib.RasterOutputs(_lib.ptr(color_all), _lib.ptr(depth), _lib.ptr(alpha), None)
            _lib.launch("ogs_raster_forward_cached", dev, C.byref(ri), C.byref(ro), alloc.fn, alloc.user,
                        C.byref(entry.state), C.byref(st))
            alloc.bufs["geom"], alloc.bufs["binning"] = entry.geom, entry.binning
        else:
            if admit:
                ri.defer_capacity_check = 0      # the entry needs this frame's duplicate count now
            ro = _lib.RasterOutputs(_lib.ptr(color_all), _lib.ptr(depth), _lib.ptr(alpha), _lib.ptr(radii))
            _lib.launch("ogs_raster_forward", dev, C.byref(ri), C.byref(ro), alloc.fn, alloc.user, C.byref(st))
            if admit and int(st.num_rendered) >= 0:
                gb, bb = C.c_int64(0), C.c_int64(0)
                _lib.check(L.ogs_raster_cached_bytes(C.byref(ri), st.num_rendered, C.byref(gb), C.byref(bb)),
                           "ogs_raster_cached_bytes")
                e = _ViewEntry()
                e.geom_key = geom_key
                e.geom = alloc.bufs["geom"][:gb.value].clone()          # exact-size copies: the forward's own buffers
                e.binning = alloc.bufs["binning"][:bb.value].clone()    # carry the capacity estimate's head room
                e.radii = radii.clone()      # the caller owns the tensor this call returns; later hits alias the entry's copy
                e.state = _lib.RasterState(e.geom.data_ptr(), e.binning.data_ptr(), None, st.num_rendered, gb.value,
                                           bb.value, 0, None)
                e.keep = keep
                e.nbytes = gb.value + bb.value + radii.numel() * 4
                view_cache.insert(cam_key, e, dev)

        # outputs a loss does not touch hand the backward None instead of a zero-filled image (Stage 1 has no colour
        # or depth loss: the kernel then runs its feature-channel-only form, C ABI dL_dcolor = NULL)
        ctx.set_materialize_grads(False)
        ctx.rs = rs
        ctx.bg_full = bg_full
        ctx.state = st
        ctx.bufs = alloc.bufs            # keeps geom/binning/image buffers alive
        ctx.n_extra = n_extra
        ctx.n_extra_user = n_extra_user
        ctx.num_rendered = int(st.num_rendered)
        ctx.act_flags = act_flags
        ctx.inputs_ref = (means3D, means2D_in)
        ctx.save_for_backward(means3D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp, extra, sh_rest)
        # colour and feature map are handed to autograd as TWO outputs (views of the one planar buffer the kernel
        # wrote): their gradients then arrive separately and go to the kernel as two pointers -- slicing one output
        # instead costs a zero-filled [C,H,W] gradient plus copies in the backward of every step
        color = color_all[:3]
        feat = color_all[3:3 + n_extra_user] if n_extra_user else color_all.new_empty(0, H, W)
        ctx.mark_non_differentiable(radii)
        return color, radii, depth, alpha, feat

    @staticmethod
    def backward(ctx, grad_color, _grad_radii, grad_depth, grad_alpha, grad_feat):
        L = _lib.lib()
        means3D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp, extra, sh_rest = ctx.saved_tensors
        rs = ctx.rs
        dev = means3D.device
        P = means3D.shape[0]
        n_extra = ctx.n_extra
        H, W = int(rs.image_height), int(rs.image_width)
        need = ctx.needs_input_grad   # means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3D, extra

        gc, gf = _grad_planes(grad_color, grad_feat, n_extra, (H, W), dev)
        gd, ga = _f32c(grad_depth), _f32c(grad_alpha)

        # All parameter gradients are carved out of ONE flat buffer (64-float aligned slices): autograd
        # adopts the views as .grad, and opengaussian_b200.dist.allreduce_gradients then reduces the whole
        # buffer with a single NCCL call instead of one per tensor.
        specs = []
        sources = []          # the input tensor each requested parameter gradient belongs to

        def want(flag, src, *shape):
            if not flag:
                return None
            n = 1
            for d in shape:
                n *= int(d)
            specs.append((len(specs), tuple(int(d) for d in shape), n))
            sources.append(src)
            return len(specs) - 1

        need_rest = sh_rest is not None and need[11]
        i_means3D = want(need[0], ctx.inputs_ref[0], P, 3)
        i_opac = want(need[4], opacities, *opacities.shape)
        i_sh = want((need[2] or need_rest) and sh is not None, sh, *(sh.shape if sh is not None else (0,)))
        i_sh_rest = want(need_rest, sh_rest, *(sh_rest.shape if sh_rest is not None else (0,)))
        i_colors = want(need[3] and colors_precomp is not None, colors_precomp, P, 3)
        i_scales = want(need[5] and scales is not None, scales, P, 3)
        i_rot = want(need[6] and rotations is not None, rotations, P, 4)
        i_cov = want(need[7] and cov3Ds_precomp is not None, cov3Ds_precomp, P, 6)
        i_extra = want(need[8] and extra is not None, extra, P, max(n_extra, 1))
        n_param = len(specs)
        i_means2D = want(need[1], None, P, 3)      # last: it is a per-view statistic, not all-reduced
        offs, total = [], 0
        for _, _, n in specs:
            offs.append(total)
            total += (n + 63) // 64 * 64
        # Gradient arena (dist.GradArena: symmetric memory for the in-switch all-reduce): the parameter gradients of
        # the FIRST backward of a step are carved from it -- only when every requested input is a leaf without a
        # .grad yet, so nothing that still aliases the arena can be overwritten; the per-view means2D gradient never
        # lives there.
        arena = _GRAD_ARENA.get(dev.index)
        param_total = offs[n_param] if i_means2D is not None else total
        use_arena = (arena is not None and 0 < param_total <= arena.numel() and n_param > 0 and
                     all(t is not None and t.is_leaf and t.grad is None for t in sources[:n_param]))
        if use_arena:
            flat = arena[:param_total]
            flat2 = torch.empty(P * 3, dtype=torch.float32, device=dev) if i_means2D is not None else None
        else:
            flat = torch.empty(max(total, 1), dtype=torch.float32, device=dev)
            flat2 = None

        def view(i):
            if i is None:
                return None
            _, shape, n = specs[i]
            if flat2 is not None and i == i_means2D:
                return flat2.view(shape)
            return flat[offs[i]:offs[i] + n].view(shape)

        g_means3D, g_opac, g_sh, g_sh_rest = view(i_means3D), view(i_opac), view(i_sh), view(i_sh_rest)
        g_colors, g_scales, g_rot, g_cov = view(i_colors), view(i_scales), view(i_rot), view(i_cov)
        g_extra, g_means2D = view(i_extra), view(i_means2D)
        # fused accumulation (see fuse_grad_accumulation): every requested gradient goes into the leaf's .grad
        accumulate = 0
        if _FUSE_ACCUMULATE and n_extra == ctx.n_extra_user:
            pairs = [(ctx.inputs_ref[0], g_means3D), (sh, g_sh), (colors_precomp, g_colors),
                     (opacities, g_opac), (scales, g_scales), (rotations, g_rot), (cov3Ds_precomp, g_cov),
                     (extra, g_extra), (sh_rest, g_sh_rest)]
            wanted = [(t, g) for t, g in pairs if g is not None]
            if wanted and all(_fusable_grad(t, g.shape) for t, g in wanted) and (need[2] or g_sh is None):
                accumulate = 1          # bit 0: the parameter gradients
                g_means3D = ctx.inputs_ref[0].grad if g_means3D is not None else None
                g_sh = sh.grad if g_sh is not None else None
                g_colors = colors_precomp.grad if g_colors is not None else None
                g_opac = opacities.grad if g_opac is not None else None
                g_scales = scales.grad if g_scales is not None else None
                g_rot = rotations.grad if g_rot is not None else None
                g_cov = cov3Ds_precomp.grad if g_cov is not None else None
                g_extra = extra.grad if g_extra is not None else None
                g_sh_rest = sh_rest.grad if g_sh_rest is not None else None
                # bit 1: means2D as well -- only when it is a shared leaf; render() feeds a fresh tensor per view,
                # whose gradient (a per-view densification statistic) is then returned to autograd as usual
                if g_means2D is not None and _fusable_grad(ctx.inputs_ref[1], g_means2D.shape):
                    accumulate |= 2
                    g_means2D = ctx.inputs_ref[1].grad
        scratch = torch.empty(L.ogs_raster_backward_scratch_floats(P, n_extra), dtype=torch.float32, device=dev)

        ri = _fill_inputs(rs, ctx.bg_full, means3D, opacities, sh, colors_precomp, scales, rotations,
                          cov3Ds_precomp, extra, n_extra, sh_rest, ctx.act_flags)
        gi = _lib.RasterGradsIn(_lib.ptr(gc), _lib.ptr(gd), _lib.ptr(ga), _lib.ptr(gf))
        go = _lib.RasterGradsOut(_lib.ptr(g_means3D), _lib.ptr(g_means2D), _lib.ptr(g_opac), _lib.ptr(g_sh),
                                 _lib.ptr(g_colors), _lib.ptr(g_scales), _lib.ptr(g_rot), _lib.ptr(g_cov),
                                 _lib.ptr(g_extra), _lib.ptr(g_sh_rest), _lib.ptr(scratch), accumulate, 0)
        _lib.launch("ogs_raster_backward", dev, C.byref(ri), C.byref(ctx.state), C.byref(gi), C.byref(go))
        if accumulate:       # already added into the leaves' .grad (means2D unless it was fused too)
            return (None, None if (accumulate & 2) else g_means2D) + (None,) * 11
        if g_extra is not None and n_extra != ctx.n_extra_user:
            g_extra = g_extra[:, :ctx.n_extra_user].contiguous()
        if not need[2]:
            g_sh = None
        return g_means3D, g_means2D, g_sh, g_colors, g_opac, g_scales, g_rot, g_cov, g_extra, None, None, g_sh_rest, None


def _forward_subsets(ctx, rs, subset, num_subsets, means3D, opacities, shs, colors_precomp, scales, rotations,
                     cov3D_precomp, extra, extra_bg):
    """One subset call -> (color [S,3,H,W], depth [S,1,H,W], alpha [S,1,H,W], feats [S,F,H,W]).  ctx None:
    ogs_raster_forward_subsets, forward only; else ogs_raster_forward_subsets_state, and ctx keeps what the backward
    needs."""
    inputs, n_extra_user, n_extra, bg, _, _, rs, ri = _prepare(
        rs, means3D, opacities, shs, colors_precomp, scales, rotations, cov3D_precomp, extra, extra_bg)
    means3D = inputs[0]
    dev = means3D.device
    P = means3D.shape[0]
    S = int(num_subsets)
    if tuple(subset.shape) != (P,):
        raise _lib.OgsError(f"subset must have shape [{P}], got {tuple(subset.shape)}")
    subset = subset.to(device=dev, dtype=torch.int32).contiguous()
    ri.defer_capacity_check = 0
    H, W = int(rs.image_height), int(rs.image_width)
    color_all = torch.empty(max(S, 0), 3 + n_extra, H, W, dtype=torch.float32, device=dev)
    depth = torch.empty(max(S, 0), 1, H, W, dtype=torch.float32, device=dev)
    alpha = torch.empty(max(S, 0), 1, H, W, dtype=torch.float32, device=dev)
    so = _lib.SubsetOutputs(_lib.ptr(color_all), _lib.ptr(depth), _lib.ptr(alpha))
    alloc = _Alloc(dev)
    args = (C.byref(ri), _lib.ptr(subset), S, C.byref(so), alloc.fn, alloc.user)
    if ctx is None:
        _lib.launch("ogs_raster_forward_subsets", dev, *args)
    else:
        st = _lib.RasterState()
        _lib.launch("ogs_raster_forward_subsets_state", dev, *args, C.byref(st))
        ctx.set_materialize_grads(False)
        ctx.rs, ctx.bg, ctx.state, ctx.bufs = rs, bg, st, alloc.bufs     # bufs: the state's geom/binning/image buffers
        ctx.S, ctx.n_extra, ctx.n_extra_user = S, n_extra, n_extra_user
        ctx.save_for_backward(*inputs[:8])
    feat = color_all[:, 3:3 + n_extra_user] if n_extra_user else color_all.new_empty(max(S, 0), 0, H, W)
    return color_all[:, :3], depth, alpha, feat


class _RasterizeSubsets(torch.autograd.Function):
    """GaussianRasterizer.forward_subsets_grad: ogs_raster_forward_subsets_state, and ogs_raster_backward_subsets for
    the gradients of every slot's colour, feature, depth and alpha images at once."""

    @staticmethod
    def forward(ctx, means3D, opacities, shs, colors_precomp, scales, rotations, cov3D_precomp, extra, subset, S, rs,
                extra_bg):
        return _forward_subsets(ctx, rs, subset, S, means3D, opacities, shs, colors_precomp, scales, rotations,
                                cov3D_precomp, extra, extra_bg)

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_color, grad_depth, grad_alpha, grad_feat):
        means3D, opacities, shs, colors_precomp, scales, rotations, cov3D_precomp, extra = ctx.saved_tensors
        rs, S, n_extra = ctx.rs, ctx.S, ctx.n_extra
        dev = means3D.device
        P = means3D.shape[0]
        H, W = int(rs.image_height), int(rs.image_width)
        need = ctx.needs_input_grad   # means3D, opacities, shs, colors_precomp, scales, rotations, cov3D, extra

        gc, gf = _grad_planes(grad_color, grad_feat, n_extra, (S, H, W), dev)
        gd, ga = _f32c(grad_depth), _f32c(grad_alpha)

        def out(flag, t, *shape):
            return torch.empty(*(shape or t.shape), dtype=torch.float32, device=dev) if flag and t is not None else None

        g_means3D, g_opac, g_sh = out(need[0], means3D), out(need[1], opacities), out(need[2], shs)
        g_colors, g_scales, g_rot = out(need[3], colors_precomp), out(need[4], scales), out(need[5], rotations)
        g_cov, g_extra = out(need[6], cov3D_precomp), out(need[7], extra)
        scratch = torch.empty(_lib.lib().ogs_raster_backward_scratch_floats(P, n_extra), dtype=torch.float32,
                              device=dev)
        ri = _fill_inputs(rs, ctx.bg, means3D, opacities, shs, colors_precomp, scales, rotations, cov3D_precomp, extra,
                          n_extra)
        gi = _lib.RasterGradsIn(_lib.ptr(gc), _lib.ptr(gd), _lib.ptr(ga), _lib.ptr(gf))
        go = _lib.RasterGradsOut(_lib.ptr(g_means3D), None, _lib.ptr(g_opac), _lib.ptr(g_sh), _lib.ptr(g_colors),
                                 _lib.ptr(g_scales), _lib.ptr(g_rot), _lib.ptr(g_cov), _lib.ptr(g_extra), None,
                                 _lib.ptr(scratch), 0, 0)
        _lib.launch("ogs_raster_backward_subsets", dev, C.byref(ri), S, C.byref(ctx.state), C.byref(gi), C.byref(go))
        if g_extra is not None and n_extra != ctx.n_extra_user:
            g_extra = g_extra[:, :ctx.n_extra_user].contiguous()
        return g_means3D, g_opac, g_sh, g_colors, g_scales, g_rot, g_cov, g_extra, None, None, None, None


def rasterize_gaussians(means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp,
                        raster_settings, extra_feats=None, extra_bg=None, sh_rest=None, act_flags=0):
    return _RasterizeGaussians.apply(means3D, means2D, sh, colors_precomp, opacities, scales, rotations,
                                     cov3Ds_precomp, extra_feats, raster_settings, extra_bg, sh_rest, act_flags)


class GaussianRasterizer(nn.Module):
    def __init__(self, raster_settings: GaussianRasterizationSettings):
        super().__init__()
        self.raster_settings = raster_settings

    def markVisible(self, positions: torch.Tensor) -> torch.Tensor:
        """Near-plane frustum test (upstream markVisible): bool [P]."""
        with torch.no_grad():
            pos = _f32c(positions)
            view = _f32c(self.raster_settings.viewmatrix)
            out = torch.empty(pos.shape[0], dtype=torch.uint8, device=pos.device)
            _lib.launch("ogs_mark_visible", pos.device, pos.shape[0], _lib.ptr(pos), _lib.ptr(view), _lib.ptr(out))
        return out.bool()

    def forward_raw(self, means3D, means2D, opacity_logits, features_dc, features_rest, log_scales, raw_rotations,
                    raw_ins_feat=None, extra_bg=None):
        """Raw-parameter entry (SURVEY.md 8a9): takes GaussianModel's PARAMETERS (`_xyz, _opacity, _features_dc,
        _features_rest, _scaling, _rotation, _ins_feat`) and folds the getters of scene/gaussian_model.py:122-169
        -- exp, normalize, sigmoid, the get_features cat, and render()'s (normalize(ins_feat) + 1) / 2 -- into the
        preprocess kernels, forward and backward.  Same return tuple as forward()."""
        flags = _lib.ACT_SCALE_EXP | _lib.ACT_ROT_NORMALIZE | _lib.ACT_OPACITY_SIGMOID
        if raw_ins_feat is not None:
            flags |= _lib.ACT_EXTRA_UNIT_HALF
        color, radii, depth, alpha, feat = rasterize_gaussians(
            means3D, means2D, features_dc, None, opacity_logits, log_scales, raw_rotations, None, self.raster_settings,
            raw_ins_feat, extra_bg, features_rest, flags)
        if raw_ins_feat is None:
            return color, radii, depth, alpha
        return color, radii, depth, alpha, feat

    def forward(self, means3D, means2D, opacities, shs=None, colors_precomp=None, scales=None, rotations=None,
                cov3D_precomp=None, extra_feats=None, extra_bg=None):
        """Reference signature (gaussian_renderer/__init__.py:104-112) + ``extra_feats [P,F]`` /
        ``extra_bg [F]``: F extra channels composited in the same pass (background ``extra_bg``,
        default 0).  Returns ``(color, radii, depth, alpha)`` or, with extra_feats, a fifth
        ``feats [F,H,W]``."""
        shs, colors_precomp, scales, rotations, cov3D_precomp = _check_inputs(
            means3D, shs, colors_precomp, scales, rotations, cov3D_precomp)
        color, radii, depth, alpha, feat = rasterize_gaussians(
            means3D, means2D, shs, colors_precomp, opacities, scales, rotations, cov3D_precomp, self.raster_settings,
            extra_feats, extra_bg)
        if extra_feats is None:
            return color, radii, depth, alpha
        return color, radii, depth, alpha, feat

    def forward_subsets(self, means3D, opacities, subset, num_subsets, shs=None, colors_precomp=None, scales=None,
                        rotations=None, cov3D_precomp=None, extra_feats=None, extra_bg=None):
        """Renders ``num_subsets`` disjoint subsets of the Gaussians in one call (C ABI ogs_raster_forward_subsets):
        ``subset [P]`` holds each Gaussian's slot in ``[0, num_subsets)`` or -1 (not rendered).  Slot k's images equal,
        bit for bit, ``forward()`` on the rows with ``subset == k``.  Activated inputs as for ``forward()``; forward
        only (no backward, no radii: ``forward_subsets_grad`` is the differentiable form) and outside the view cache.
        Returns ``(color [S,3,H,W], depth [S,1,H,W], alpha [S,1,H,W], feats [S,F,H,W] or None)``."""
        shs, colors_precomp, scales, rotations, cov3D_precomp = _check_inputs(
            means3D, shs, colors_precomp, scales, rotations, cov3D_precomp)
        inputs = (means3D, opacities, shs, colors_precomp, scales, rotations, cov3D_precomp, extra_feats)
        if torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in inputs):
            raise _lib.OgsError("forward_subsets has no backward: call it under torch.no_grad() or with inputs that "
                                "do not require grad")
        color, depth, alpha, feats = _forward_subsets(None, self.raster_settings, subset, num_subsets, *inputs, extra_bg)
        return color, depth, alpha, (feats if feats.shape[1] > 0 else None)

    def forward_subsets_grad(self, means3D, opacities, subset, num_subsets, shs=None, colors_precomp=None, scales=None,
                             rotations=None, cov3D_precomp=None, extra_feats=None, extra_bg=None):
        """``forward_subsets`` with a backward (C ABI ogs_raster_forward_subsets_state / ogs_raster_backward_subsets):
        the same arguments, checks and bit-identical images, returned as autograd outputs.  Gradients of every slot's
        colour, features, depth and alpha flow to ``means3D, opacities, shs, colors_precomp, scales, rotations,
        cov3D_precomp, extra_feats`` in one backward; each Gaussian's gradient is that of its own slot's images (those
        of no slot get zero), as ``forward()`` + backward on each slot's rows would give.  There is no ``means2D``
        input, hence no screen-space gradient: a caller that needs one renders each slot with ``forward()``.  Plain
        gradient tensors (no gradient arena, no fused accumulation), outside the view cache; no double backward."""
        shs, colors_precomp, scales, rotations, cov3D_precomp = _check_inputs(
            means3D, shs, colors_precomp, scales, rotations, cov3D_precomp)
        color, depth, alpha, feats = _RasterizeSubsets.apply(means3D, opacities, shs, colors_precomp, scales, rotations,
                                                             cov3D_precomp, extra_feats, subset, num_subsets,
                                                             self.raster_settings, extra_bg)
        return color, depth, alpha, (feats if feats.shape[1] > 0 else None)
