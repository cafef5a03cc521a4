"""Host logic of the frozen-geometry view cache (opengaussian_b200.rasterizer.ViewCache): what counts as "the same
geometry" (storage + shape + version counter), one entry per camera, least-recently-used eviction under a byte budget.
The GPU behaviour is in tests/test_view_cache_gpu.py."""
import types

import torch

from opengaussian_b200.rasterizer import GaussianRasterizationSettings, ViewCache, _sig, _ViewEntry, camera_inputs


def _rs(view, proj, campos, sh_degree=3):
    return GaussianRasterizationSettings(48, 64, 0.5, 0.4, torch.zeros(3), 1.0, view, proj, sh_degree, campos, False, False)


def _geo(P=10):
    g = types.SimpleNamespace()
    g.means3D, g.opacities, g.scales, g.rotations = torch.rand(P, 3), torch.rand(P, 1), torch.rand(P, 3), torch.rand(P, 4)
    g.sh, g.sh_rest = torch.rand(P, 1, 3), torch.rand(P, 15, 3)
    return g


def _keys(rs, g, act=7, n_feat=6):
    return ViewCache.keys(rs, g.means3D, g.opacities, g.sh, g.sh_rest, None, g.scales, g.rotations, None, act, n_feat)


def _entry(geom_key, nbytes):
    e = _ViewEntry()
    e.geom_key, e.nbytes = geom_key, nbytes
    e.state = e.geom = e.binning = e.radii = e.keep = None
    return e


def test_signature_follows_torch_version_counter():
    x = torch.zeros(4, 3)
    s0 = _sig(x)
    assert _sig(x.detach()) == s0                  # train.py:431-436: a new tensor object per iteration, same contents
    x.add_(1)
    assert _sig(x) != s0                           # optimizer steps and every other in-place op bump the version
    s1 = _sig(x)
    x.detach().mul_(2)                             # ... also through a detached alias
    assert _sig(x) != s1
    assert _sig(x.clone()) != _sig(x)              # new storage (densification, load_ply)
    assert _sig(None) is None


def test_keys_separate_camera_from_geometry():
    view, proj, pos = torch.eye(4), torch.eye(4), torch.zeros(3)
    g = _geo()
    cam, geom = _keys(_rs(view, proj, pos), g)
    cam_b, geom_b = _keys(_rs(view, proj, pos), g)
    assert cam == cam_b and geom == geom_b
    assert _keys(_rs(view.clone(), proj, pos), g)[0] != cam            # another camera tensor
    assert _keys(_rs(view, proj, pos, sh_degree=2), g)[0] != cam       # oneupSHdegree changes the colours
    g.opacities.mul_(0.5)
    cam_c, geom_c = _keys(_rs(view, proj, pos), g)
    assert cam_c == cam and geom_c != geom
    # the trained feature tensor is not part of either key; only whether it is activated in the kernel matters
    assert _keys(_rs(view, proj, pos), g, act=7 | 8)[1] == geom_c
    assert _keys(_rs(view, proj, pos), g, n_feat=0)[1] != geom_c


def test_lookup_insert_supersede_and_lru():
    vc = ViewCache()
    vc.max_bytes = 250
    assert vc.lookup("camA", "g0") is None and vc.misses == 1
    assert vc.insert("camA", _entry("g0", 100))
    assert vc.lookup("camA", "g0") is not None and vc.hits == 1
    assert vc.lookup("camA", "g1") is None                              # same camera, geometry moved on
    assert vc.insert("camA", _entry("g1", 100)) and len(vc) == 1 and vc.bytes == 100   # superseded, not duplicated
    assert vc.insert("camB", _entry("g1", 100)) and vc.bytes == 200
    assert vc.lookup("camA", "g1") is not None                          # camA is now the most recently used
    assert vc.insert("camC", _entry("g1", 100))                         # over budget: camB goes
    assert len(vc) == 2 and vc.bytes == 200 and vc.evictions == 1
    assert vc.lookup("camB", "g1") is None and vc.lookup("camA", "g1") is not None
    assert not vc.insert("camD", _entry("g1", 1000)) and len(vc) == 2   # larger than the whole budget: not kept
    vc.clear()
    assert len(vc) == 0 and vc.bytes == 0
    assert set(vc.stats()) >= {"entries", "bytes", "hits", "misses", "evictions", "max_bytes"}


def test_activated_tensors_are_admitted_on_their_second_sighting_only():
    vc = ViewCache()
    t1, t2 = torch.zeros(3), torch.zeros(3)
    assert not vc.second_sighting(0, ("cam", _sig(t1)), (t1,))          # first time: remembered, not admitted
    assert vc.second_sighting(0, ("cam", _sig(t1)), (t1,))              # the same tensors again: admitted
    assert not vc.second_sighting(0, ("cam", _sig(t2)), (t2,))          # other tensors (a getter's new result): not admitted
    assert not vc.second_sighting(0, ("cam", _sig(t1)), (t1,))          # ... and the alternation never is
    assert not vc.second_sighting(1, ("cam", _sig(t1)), (t1,))          # records are per device
    vc.clear()
    assert not vc.second_sighting(0, ("cam", _sig(t1)), (t1,))
    # raw-parameter and activated forwards of one camera are different entries (the flag is part of the camera key)
    view, proj, pos = torch.eye(4), torch.eye(4), torch.zeros(3)
    g = _geo()
    assert _keys(_rs(view, proj, pos), g, act=7)[0] != _keys(_rs(view, proj, pos), g, act=0)[0]
    assert _keys(_rs(view, proj, pos), g, act=7)[0] == _keys(_rs(view, proj, pos), g, act=7 | 8)[0]


def _reference_camera(seed=0):
    """Camera tensors as scene/cameras.py:71-73 builds them: transposed (non-contiguous) view and projection, their
    product, the centre row of the inverse."""
    g = torch.Generator().manual_seed(seed)
    w2v = torch.eye(4)
    w2v[:3, :3] = torch.linalg.qr(torch.randn(3, 3, generator=g))[0]
    w2v[:3, 3] = torch.randn(3, generator=g)
    view = torch.tensor(w2v.numpy()).transpose(0, 1)
    proj = torch.rand(4, 4, generator=g).transpose(0, 1)
    full = view.unsqueeze(0).bmm(proj.unsqueeze(0)).squeeze(0)
    return view, full, view.inverse()[3, :3]


def test_reference_camera_key_repeats_and_its_copy_is_reused():
    view, full, centre = _reference_camera()
    assert not view.is_contiguous() and not centre.is_contiguous()     # inverse() returns a column-major matrix
    key, (v, p, c) = camera_inputs(view, full, centre)
    assert v.is_contiguous() and v.dtype == torch.float32 and torch.equal(v, view)
    assert c.is_contiguous() and torch.equal(c, centre)
    assert p is full                                   # already what the C ABI takes: no copy
    for _ in range(3):
        key2, (v2, p2, c2) = camera_inputs(view, full, centre)
        assert key2 == key and v2 is v and p2 is p and c2 is c
    assert camera_inputs(view.detach(), full, centre)[0] == key   # another tensor object over the same contents
    # the key is the one ViewCache.keys takes from the caller's settings, not from the copy
    g = _geo()
    assert _keys(_rs(view, full, centre), g)[0] == ViewCache.keys(
        _rs(v, p, c), g.means3D, g.opacities, g.sh, g.sh_rest, None, g.scales, g.rotations, None, 7, 6, cam_key=key)[0]
    assert _keys(_rs(v, p, c), g)[0] != _keys(_rs(view, full, centre), g)[0]
    # a float64 camera: one float32 copy, reused
    d = view.double()
    k64, (v64, _, _) = camera_inputs(d, full, centre)
    assert v64.dtype == torch.float32 and camera_inputs(d, full, centre)[1][0] is v64 and k64 != key


def test_in_place_camera_edit_gives_a_new_key_and_a_fresh_copy():
    view, full, centre = _reference_camera(1)
    key, (v, _, _) = camera_inputs(view, full, centre)
    before = v.clone()
    view.mul_(2.0)                                      # through the transposed tensor
    key2, (v2, _, _) = camera_inputs(view, full, centre)
    assert key2 != key and v2 is not v and torch.equal(v2, view) and torch.equal(v, before)
    view._base.add_(1.0)                                 # through its base: the version counter is shared
    key3, (v3, _, _) = camera_inputs(view, full, centre)
    assert key3 not in (key, key2) and torch.equal(v3, view)
    full.sub_(0.5)                                      # a contiguous matrix is keyed the same way
    key4, (_, p4, _) = camera_inputs(view, full, centre)
    assert key4 != key3 and p4 is full and camera_inputs(view, full, centre)[0] == key4


def test_equal_values_in_a_new_camera_tensor_are_a_new_key():
    view, full, centre = _reference_camera(2)
    key, (v, _, _) = camera_inputs(view, full, centre)
    twin = view._base.clone().transpose(0, 1)            # same values, new storage (a re-created Camera)
    key2, (v2, _, _) = camera_inputs(twin, full, centre)
    assert key2 != key and v2 is not v and torch.equal(v2, v)
    assert camera_inputs(view, full, centre)[0] == key and camera_inputs(view, full, centre)[1][0] is v
