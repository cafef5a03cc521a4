"""CPU tests (no GPU): the C-ABI library builds for sm_100a, loads, and exports every symbol that
include/ogs_b200.h declares; argument validation works without touching a device."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from opengaussian_b200 import build, _lib
    build.build()
    return _lib.lib()


def test_header_symbols_exported(lib):
    hdr = open(os.path.join(ROOT, "include", "ogs_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = set(re.findall(r"\b(ogs_[a-z0-9_]+)\s*\(", hdr))
    names -= {"ogs_alloc_fn"}
    assert len(names) >= 10
    from opengaussian_b200 import _lib
    assert names == set(_lib.EXPORTS), names ^ set(_lib.EXPORTS)
    for n in names:
        assert hasattr(lib, n), n


def test_abi_version_7_and_sass_target(lib):
    assert lib.ogs_abi_version() == 7
    import subprocess
    from opengaussian_b200 import _lib
    out = subprocess.run(["cuobjdump", "-lelf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out and "sm_90" not in out and "sm_80" not in out


def test_argument_validation_without_device(lib):
    from opengaussian_b200 import _lib
    ri = _lib.RasterInputs()
    ri.P, ri.W, ri.H = 4, 0, 16
    st = _lib.RasterState()
    ro = _lib.RasterOutputs()
    cb = _lib.ALLOC_FN(lambda u, n, t: None)
    rc = lib.ogs_raster_forward(C.byref(ri), C.byref(ro), cb, None, C.byref(st), None)
    assert rc == -1 and b"bad sizes" in lib.ogs_last_error()
    ri.W = 16
    rc = lib.ogs_raster_forward(C.byref(ri), C.byref(ro), cb, None, C.byref(st), None)
    assert rc == -2 and b"excatly one of either SHs or precomputed colors" in lib.ogs_last_error()
    rc = lib.ogs_kmeans_assign(10, None, 6, None, 0, 1.0, None, 4, None, -1, 0, None, None, None, None)
    assert rc == -1
    assert lib.ogs_raster_backward_scratch_floats(100, 6) == 100 * 16


def test_missing_library_fails_loudly(monkeypatch):
    from opengaussian_b200 import _lib
    monkeypatch.setattr(_lib, "_LIB", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libogs_b200.so")
    with pytest.raises(_lib.OgsError, match="no CPU fallback"):
        _lib.lib()


def test_cpu_tensors_rejected():
    import torch
    from opengaussian_b200.rasterizer import GaussianRasterizationSettings, GaussianRasterizer
    from opengaussian_b200._lib import OgsError
    rs = GaussianRasterizationSettings(16, 16, 0.5, 0.5, torch.zeros(3), 1.0, torch.eye(4), torch.eye(4), 0,
                                       torch.zeros(3), False, False)
    x = torch.zeros(4, 3)
    with pytest.raises(OgsError, match="no CPU fallback"):
        GaussianRasterizer(rs)(means3D=x, means2D=x, opacities=torch.ones(4, 1), colors_precomp=x,
                               scales=x + 1, rotations=torch.ones(4, 4))
