"""ctypes binding of libogs_b200.so (the C ABI declared in include/ogs_b200.h).

There is NO fallback: if the shared library is missing or a call fails this module raises.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("OGS_LIB_PATH") or os.path.join(_HERE, "csrc", "libogs_b200.so")   # env: developer A/B builds

ALLOC_FN = C.CFUNCTYPE(C.c_void_p, C.c_void_p, C.c_size_t, C.c_char_p)
_fp = C.c_void_p


class RasterInputs(C.Structure):
    _fields_ = [
        ("P", C.c_int32), ("sh_degree", C.c_int32), ("M", C.c_int32), ("n_extra", C.c_int32),
        ("W", C.c_int32), ("H", C.c_int32),
        ("tanfovx", C.c_float), ("tanfovy", C.c_float), ("scale_modifier", C.c_float),
        ("prefiltered", C.c_int32), ("debug", C.c_int32),
        ("bg", _fp), ("viewmatrix", _fp), ("projmatrix", _fp), ("campos", _fp),
        ("means3D", _fp), ("opacities", _fp), ("shs", _fp), ("colors_precomp", _fp),
        ("scales", _fp), ("rotations", _fp), ("cov3D_precomp", _fp), ("extra", _fp),
        ("act_flags", C.c_int32), ("defer_capacity_check", C.c_int32), ("shs_rest", _fp),
    ]


ACT_SCALE_EXP, ACT_ROT_NORMALIZE, ACT_OPACITY_SIGMOID, ACT_EXTRA_UNIT_HALF = 1, 2, 4, 8


class RasterOutputs(C.Structure):
    _fields_ = [("color", _fp), ("depth", _fp), ("alpha", _fp), ("radii", _fp)]


class RasterState(C.Structure):
    _fields_ = [("geom", _fp), ("binning", _fp), ("image", _fp), ("num_rendered", C.c_int64),
                ("geom_bytes", C.c_int64), ("binning_bytes", C.c_int64), ("image_bytes", C.c_int64), ("feat", _fp)]


class RasterGradsIn(C.Structure):
    _fields_ = [("dL_dcolor", _fp), ("dL_ddepth", _fp), ("dL_dalpha", _fp), ("dL_dfeat", _fp)]


class RasterGradsOut(C.Structure):
    _fields_ = [("dL_dmeans3D", _fp), ("dL_dmeans2D", _fp), ("dL_dopacities", _fp), ("dL_dshs", _fp),
                ("dL_dcolors_precomp", _fp), ("dL_dscales", _fp), ("dL_drotations", _fp),
                ("dL_dcov3D", _fp), ("dL_dextra", _fp), ("dL_dshs_rest", _fp), ("scratch", _fp),
                ("accumulate", C.c_int32), ("reserved_", C.c_int32)]


class FootprintInputs(C.Structure):
    _fields_ = [("P", C.c_int32), ("W", C.c_int32), ("H", C.c_int32), ("act_flags", C.c_int32),
                ("means3D", _fp), ("opacities", _fp), ("scales", _fp), ("rotations", _fp),
                ("scale_modifier", C.c_float), ("tanfovx", C.c_float), ("tanfovy", C.c_float), ("color", C.c_float),
                ("viewmatrix", _fp), ("projmatrix", _fp), ("sam_ids", _fp), ("empty_id", C.c_int32), ("reserved_", C.c_int32)]


class AdamTensor(C.Structure):
    _fields_ = [("param", _fp), ("grad", _fp), ("exp_avg", _fp), ("exp_avg_sq", _fp), ("n", C.c_int64),
                ("step_size", C.c_float), ("bias_correction2_sqrt", C.c_float), ("beta1", C.c_float),
                ("beta2", C.c_float), ("one_minus_beta1", C.c_float), ("one_minus_beta2", C.c_float), ("eps", C.c_float),
                ("reserved_", C.c_float)]


EXPORTS = {
    "ogs_abi_version": (C.c_int, []),
    "ogs_last_error": (C.c_char_p, []),
    "ogs_profile_enable": (None, [C.c_int]),
    "ogs_profile_read": (C.c_int, [C.POINTER(C.c_float), C.POINTER(C.c_int32), C.c_int32]),
    "ogs_raster_forward": (C.c_int, [C.POINTER(RasterInputs), C.POINTER(RasterOutputs), ALLOC_FN, C.c_void_p,
                                     C.POINTER(RasterState), C.c_void_p]),
    "ogs_raster_backward": (C.c_int, [C.POINTER(RasterInputs), C.POINTER(RasterState), C.POINTER(RasterGradsIn),
                                      C.POINTER(RasterGradsOut), C.c_void_p]),
    "ogs_raster_forward_cached": (C.c_int, [C.POINTER(RasterInputs), C.POINTER(RasterOutputs), ALLOC_FN, C.c_void_p,
                                            C.POINTER(RasterState), C.POINTER(RasterState), C.c_void_p]),
    "ogs_raster_cached_bytes": (C.c_int, [C.POINTER(RasterInputs), C.c_int64, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "ogs_raster_capacity_check": (C.c_int, []),
    "ogs_raster_capacity_hint": (C.c_int64, [C.c_int64]),
    "ogs_raster_backward_scratch_floats": (C.c_size_t, [C.c_int32, C.c_int32]),
    "ogs_mark_visible": (C.c_int, [C.c_int32, _fp, _fp, _fp, C.c_void_p]),
    "ogs_raster_export": (C.c_int, [C.POINTER(RasterInputs), C.POINTER(RasterState)] + [_fp] * 10 + [C.c_void_p]),
    "ogs_kmeans_assign": (C.c_int, [C.c_int64, _fp, C.c_int32, _fp, C.c_int32, C.c_float, _fp, C.c_int32, _fp,
                                    C.c_int64, C.c_int64, _fp, _fp, _fp, C.c_void_p]),
    "ogs_kmeans_gather_st": (C.c_int, [C.c_int64, _fp, C.c_int32, _fp, C.c_int32, _fp, _fp, C.c_void_p]),
    "ogs_kmeans_assign_segmented": (C.c_int, [C.c_int64, _fp, C.c_int32, _fp, _fp, _fp, C.c_int32, C.c_int32, _fp, _fp,
                                              C.c_int32, C.c_void_p]),
    "ogs_kmeans_finalize_fixed": (C.c_int, [C.c_int32, C.c_int32, _fp, C.c_int32, C.c_float, _fp, _fp, C.c_void_p]),
    "ogs_kmeans_lloyd_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32]),
    "ogs_kmeans_lloyd_pass": (C.c_int, [C.c_int64, _fp, C.c_int32, _fp, C.c_int32, C.c_float, _fp, C.c_int32, C.c_int32, _fp,
                                        C.c_int64, C.c_int64, _fp, _fp, C.c_float, C.c_void_p, _fp, C.c_void_p]),
    "ogs_kmeans_lloyd_segmented_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32]),
    "ogs_kmeans_lloyd_pass_segmented": (C.c_int, [C.c_int64, _fp, C.c_int32, _fp, _fp, _fp, C.c_int32, C.c_int32, _fp, C.c_int32,
                                                  _fp, C.c_float, C.c_void_p, _fp, C.c_void_p]),
    "ogs_multimem_allreduce_f32": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p]),
    "ogs_peer_comm_create": (C.c_int, [C.c_int32, C.c_int32, C.c_int64, C.POINTER(C.c_void_p), C.c_void_p]),
    "ogs_peer_comm_connect": (C.c_int, [C.c_void_p, C.c_void_p]),
    "ogs_peer_allreduce": (C.c_int, [C.c_void_p, _fp, C.c_int64, C.c_int32, C.c_void_p]),
    "ogs_peer_comm_error": (C.c_int, [C.c_void_p, C.c_void_p]),
    "ogs_peer_comm_destroy": (C.c_int, [C.c_void_p]),
    "ogs_mask_mean_forward": (C.c_int, [C.c_int32, C.c_int32, C.c_int64, _fp, _fp, _fp, _fp, _fp, _fp, _fp, C.c_void_p]),
    "ogs_mask_mean_backward": (C.c_int, [C.c_int32, C.c_int32, C.c_int64, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, C.c_void_p]),
    "ogs_mask_var_forward": (C.c_int, [C.c_int32, C.c_int32, C.c_int64, _fp, _fp, _fp, _fp, _fp, _fp, _fp, C.c_void_p]),
    "ogs_cohesion_forward": (C.c_int, [C.c_int32, C.c_int32, C.c_int64, _fp, _fp, _fp, _fp, _fp, _fp, _fp, C.c_void_p]),
    "ogs_cohesion_backward": (C.c_int, [C.c_int32, C.c_int32, C.c_int64, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, C.c_void_p]),
    "ogs_sam_masks": (C.c_int, [C.c_int32, C.c_int64, _fp, C.c_int32, _fp, _fp, _fp, _fp, C.c_void_p]),
    "ogs_mask_id_map": (C.c_int, [C.c_int32, C.c_int64, _fp, _fp, _fp, C.c_void_p]),
    "ogs_separation_loss": (C.c_int, [C.c_int32, C.c_int32, _fp, C.c_int32, _fp, _fp, _fp, C.c_void_p]),
    "ogs_splat_footprint_votes": (C.c_int, [C.POINTER(FootprintInputs), _fp, _fp, _fp, _fp, _fp, C.POINTER(C.c_int32),
                                            C.c_void_p]),
    "ogs_adam_step": (C.c_int, [C.c_int32, C.c_void_p, C.c_float, C.c_void_p]),
    "ogs_mask_iou_scratch_bytes": (C.c_int64, [C.c_int32, C.c_int32, C.c_int64]),
    "ogs_mask_pair_counts": (C.c_int, [C.c_int32, C.c_int32, C.c_int64, _fp, _fp, _fp, _fp, _fp, C.c_void_p]),
}

_LIB = None


class OgsError(RuntimeError):
    pass


def lib() -> C.CDLL:
    """Loads the CUDA library; raises (never falls back) when it has not been built."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise OgsError(f"{LIB_PATH} not found: run `python -m opengaussian_b200.build` "
                           "(the sm_100a CUDA extension is mandatory; there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in EXPORTS.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        if L.ogs_abi_version() != 7:
            raise OgsError("libogs_b200.so ABI version mismatch")
        _LIB = L
    return _LIB


def check(rc: int, what: str):
    if rc != 0:
        msg = lib().ogs_last_error().decode("utf-8", "replace")
        if rc == -2:
            raise Exception(msg)          # same exception type/message as the reference Python layer
        raise OgsError(f"{what} failed (rc={rc}): {msg}")


def launch(name: str, device, *args) -> None:
    """Calls the C-ABI entry point `name` with `args` followed by the current stream of `device`, with `device` the
    current CUDA device for the duration of the call (the library keys its per-device state on cudaGetDevice, and CUDA
    refuses a launch into another device's stream); raises as check() does on a non-zero return."""
    with torch.cuda.device(device):
        rc = getattr(lib(), name)(*args, C.c_void_p(torch.cuda.current_stream(device).cuda_stream))
    check(rc, name)


PROFILE_FAMILIES = ("preprocess_fwd", "depth_sort_scan", "emit", "tile_sort", "tile_ranges", "blend_fwd",
                    "blend_bwd", "preprocess_bwd", "kmeans_assign", "mask_stats", "adam", "footprint")


def profile_enable(on: bool):
    lib().ogs_profile_enable(int(on))


def profile_read():
    """{family: (total_ms, launches)} since the last read (synchronises the recorded events)."""
    n = len(PROFILE_FAMILIES)
    ms = (C.c_float * n)()
    cnt = (C.c_int32 * n)()
    check(lib().ogs_profile_read(ms, cnt, n), "ogs_profile_read")
    return {PROFILE_FAMILIES[i]: (float(ms[i]), int(cnt[i])) for i in range(n)}


def ptr(t):
    """Device pointer of a (contiguous) tensor or None."""
    return None if t is None else t.data_ptr()
