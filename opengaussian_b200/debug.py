"""Parity/inspection helper: one forward through the C ABI + ogs_raster_export of every
intermediate (geometry records, tiles_touched, sorted keys, point list, tile ranges, final_T,
n_contrib).  Used by tests/ and bench.py's workload statistics; not on the product path."""
import ctypes as C

import torch

from . import _lib
from .rasterizer import GaussianRasterizationSettings, _Alloc, _f32c, _fill_inputs


def forward_with_state(rs: GaussianRasterizationSettings, means3D, opacities, shs=None, colors_precomp=None,
                       scales=None, rotations=None, cov3D_precomp=None, extra=None, export=True):
    dev = means3D.device
    means3D, opacities, shs, colors_precomp = _f32c(means3D), _f32c(opacities), _f32c(shs), _f32c(colors_precomp)
    scales, rotations, cov3D_precomp, extra = _f32c(scales), _f32c(rotations), _f32c(cov3D_precomp), _f32c(extra)
    P = means3D.shape[0]
    H, W = int(rs.image_height), int(rs.image_width)
    n_extra = 0 if extra is None else extra.shape[1]
    bg = _f32c(rs.bg).reshape(-1)
    bg_full = bg if n_extra == 0 else torch.cat([bg, bg.new_zeros(n_extra)])
    rs = rs._replace(viewmatrix=_f32c(rs.viewmatrix), projmatrix=_f32c(rs.projmatrix), campos=_f32c(rs.campos))
    color = torch.empty(3 + n_extra, H, W, device=dev)
    depth = torch.empty(H, W, device=dev)
    alpha = torch.empty(H, W, device=dev)
    radii = torch.empty(P, dtype=torch.int32, device=dev)
    ri = _fill_inputs(rs, bg_full, means3D, opacities, shs, colors_precomp, scales, rotations, cov3D_precomp, extra,
                      n_extra)
    ro = _lib.RasterOutputs(_lib.ptr(color), _lib.ptr(depth), _lib.ptr(alpha), _lib.ptr(radii))
    st = _lib.RasterState()
    alloc = _Alloc(dev)
    _lib.launch("ogs_raster_forward", dev, C.byref(ri), C.byref(ro), alloc.fn, alloc.user, C.byref(st))
    N = int(st.num_rendered)
    out = dict(color=color, depth=depth, alpha=alpha, radii=radii, N=N, _bufs=alloc.bufs, _state=st, _inputs=ri,
               _keep=(means3D, opacities, shs, colors_precomp, scales, rotations, cov3D_precomp, extra, bg_full, rs))
    if export:
        tiles = ((W + 15) // 16) * ((H + 15) // 16)
        keys = torch.zeros(max(N, 1), dtype=torch.int64, device=dev)
        plist = torch.zeros(max(N, 1), dtype=torch.int32, device=dev)
        ranges = torch.zeros(tiles, 2, dtype=torch.int32, device=dev)
        xy = torch.zeros(P, 2, device=dev)
        dep = torch.zeros(P, device=dev)
        co = torch.zeros(P, 4, device=dev)
        rgb = torch.zeros(P, 3, device=dev)
        tt = torch.zeros(P, dtype=torch.int32, device=dev)
        fT = torch.zeros(H, W, device=dev)
        nc = torch.zeros(H, W, dtype=torch.int32, device=dev)
        _lib.launch("ogs_raster_export", dev, C.byref(ri), C.byref(st), _lib.ptr(keys), _lib.ptr(plist), _lib.ptr(ranges),
                    _lib.ptr(xy), _lib.ptr(dep), _lib.ptr(co), _lib.ptr(rgb), _lib.ptr(tt), _lib.ptr(fT), _lib.ptr(nc))
        out.update(keys=keys[:N], point_list=plist[:N], ranges=ranges, xy=xy, geom_depth=dep, conic_opacity=co,
                   rgb=rgb, tiles_touched=tt, final_T=fT, n_contrib=nc)
    return out
