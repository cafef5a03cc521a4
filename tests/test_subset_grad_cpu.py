"""CPU tests (no GPU) of the differentiable subset path: argument validation of ogs_raster_forward_subsets_state and
ogs_raster_backward_subsets before any device work, and render()'s rule for how a cluster / leaf pass is rendered."""
import ctypes as C

import pytest

from opengaussian_b200 import renderer


@pytest.fixture(scope="module")
def lib():
    from opengaussian_b200 import _lib, build
    build.build()
    return _lib.lib()


def _inputs():
    from opengaussian_b200 import _lib
    ri = _lib.RasterInputs()
    ri.P, ri.W, ri.H = 4, 16, 16
    fake = C.c_void_p(256)             # never dereferenced: every call below fails validation first
    ri.colors_precomp = ri.means3D = ri.opacities = ri.scales = ri.rotations = fake
    ri.bg = ri.viewmatrix = ri.projmatrix = ri.campos = fake
    return ri


def test_forward_subsets_state_validation_without_device(lib):
    from opengaussian_b200 import _lib
    ri = _inputs()
    so = _lib.SubsetOutputs(C.c_void_p(256), None, C.c_void_p(256))
    cb = _lib.ALLOC_FN(lambda u, n, t: None)
    st = _lib.RasterState()
    subset = C.c_void_p(256)
    rc = lib.ogs_raster_forward_subsets_state(C.byref(ri), subset, 2, C.byref(so), cb, None, None, None)
    assert rc == -1 and b"state is NULL" in lib.ogs_last_error()
    for S in (0, _lib.MAX_SUBSETS + 1):
        rc = lib.ogs_raster_forward_subsets_state(C.byref(ri), subset, S, C.byref(so), cb, None, C.byref(st), None)
        assert rc == -1 and b"out of range" in lib.ogs_last_error()
    ri.act_flags = _lib.ACT_SCALE_EXP
    rc = lib.ogs_raster_forward_subsets_state(C.byref(ri), subset, 2, C.byref(so), cb, None, C.byref(st), None)
    assert rc == -1 and b"act_flags == 0" in lib.ogs_last_error()
    ri.act_flags = 0
    rc = lib.ogs_raster_forward_subsets_state(C.byref(ri), None, 2, C.byref(so), cb, None, C.byref(st), None)
    assert rc == -1 and b"subset is NULL" in lib.ogs_last_error()


def test_backward_subsets_validation_without_device(lib):
    from opengaussian_b200 import _lib
    ri = _inputs()
    fake = C.c_void_p(256)
    st = _lib.RasterState()
    gi = _lib.RasterGradsIn(fake, None, None, None)
    go = _lib.RasterGradsOut()
    go.scratch = fake

    def call(S=2, state=C.byref(st), gin=C.byref(gi)):
        return lib.ogs_raster_backward_subsets(C.byref(ri), S, state, gin, C.byref(go), None)

    assert call(state=None) == -1 and b"state/grads/scratch must be set" in lib.ogs_last_error()
    for S in (0, -3, _lib.MAX_SUBSETS + 1):
        assert call(S=S) == -1 and b"out of range" in lib.ogs_last_error()
    no_image = _lib.RasterGradsIn(None, fake, fake, None)      # depth / alpha gradients but no colour or feature image
    assert call(gin=C.byref(no_image)) == -1 and b"state/grads/scratch must be set" in lib.ogs_last_error()
    ri.act_flags = _lib.ACT_OPACITY_SIGMOID
    assert call() == -1 and b"act_flags == 0" in lib.ogs_last_error()
    ri.act_flags = 0
    go.accumulate = 1
    assert call() == -1 and b"accumulate" in lib.ogs_last_error()
    go.accumulate = 0
    # a state that is empty, or whose buffer sizes belong to other sizes, is refused before any device work
    assert call() == -1 and b"state does not belong" in lib.ogs_last_error()
    st.geom = st.binning = st.image = fake
    st.num_rendered, st.geom_bytes, st.binning_bytes, st.image_bytes = 0, 1 << 20, 1 << 20, 1 << 20
    assert call() == -1 and b"state does not belong" in lib.ogs_last_error()


def test_subset_route():
    route = renderer._subset_route
    # no gradient: one forward_subsets call; fused=False and pipe.batched_subsets = False keep the loop
    assert route(True, True, False, False) == "batched"
    assert route(True, True, False, True) == "batched"       # means2D requiring grad matters only when grad flows
    assert route(False, True, False, False) == "loop"
    assert route(True, False, False, False) == "loop"
    # gradient: one forward_subsets_grad call unless the screen-space points need their gradient
    assert route(True, True, True, False) == "batched_grad"
    assert route(True, True, True, True) == "loop"
    assert route(False, True, True, False) == "loop"
    assert route(True, False, True, False) == "loop"


def test_slot_route_reads_grad_mode():
    import torch
    x = torch.zeros(3, 3)
    feat = torch.zeros(3, 6, requires_grad=True)
    sink = torch.zeros(3, 3, requires_grad=True)
    route = renderer._slot_route
    assert route(True, True, x, x, feat) == "batched_grad"               # grad flows to feat: forward_subsets_grad
    assert route(True, True, sink, x, feat) == "loop"                    # trainable screen-space points: the loop
    assert route(True, False, x, x, feat) == "loop"                      # pipe.batched_subsets = False
    with torch.no_grad():
        assert route(True, True, sink, x, feat) == "batched"             # no gradient at all: forward_subsets
        assert route(False, True, x, x, feat) == "loop"
