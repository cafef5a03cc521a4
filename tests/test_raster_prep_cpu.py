"""Host-side preparation shared by the frame and subset rasterizer calls (opengaussian_b200.rasterizer): extra channels
padded to a compiled width, the [bg | extra_bg | 0] background, the image-gradient planes a backward hands the C ABI,
and the CUDA requirement of every entry point."""
import pytest
import torch

from opengaussian_b200 import _lib
from opengaussian_b200.rasterizer import (_SUPPORTED_C, GaussianRasterizationSettings, GaussianRasterizer, _bg_full,
                                          _grad_planes, _pad_extra)


@pytest.mark.parametrize("F", range(1, _SUPPORTED_C[-1] - 2))
def test_pad_extra_to_each_compiled_width(F):
    extra = torch.rand(5, F)
    padded, n = _pad_extra(extra)
    assert 3 + n == min(c for c in _SUPPORTED_C if c >= 3 + F)
    assert padded.shape == (5, n) and padded.is_contiguous()
    assert torch.equal(padded[:, :F], extra) and not padded[:, F:].any()
    if n == F:
        assert padded is extra


def test_pad_extra_without_channels_and_beyond_the_widest():
    assert _pad_extra(None) == (None, 0)
    with pytest.raises(_lib.OgsError, match="at most 13 channels"):
        _pad_extra(torch.rand(5, _SUPPORTED_C[-1] - 2))


def test_raw_extra_channels_need_a_compiled_width():
    with pytest.raises(_lib.OgsError, match=r"raw extra_feats need 3 \+ F in"):
        _pad_extra(torch.rand(5, 2), _lib.ACT_EXTRA_UNIT_HALF)
    extra = torch.rand(5, 3)
    assert _pad_extra(extra, _lib.ACT_EXTRA_UNIT_HALF) == (extra, 3)


def test_bg_full():
    bg = torch.tensor([0.1, 0.2, 0.3])
    assert torch.equal(_bg_full(bg, None, 0), bg)
    assert torch.equal(_bg_full(bg, None, 3), torch.tensor([0.1, 0.2, 0.3, 0, 0, 0]))
    ebg = torch.tensor([0.4, 0.5])
    six = _bg_full(bg, ebg, 6)
    assert torch.equal(six, torch.tensor([0.1, 0.2, 0.3, 0.4, 0.5, 0, 0, 0, 0]))
    # cached per width: another width does not evict it, an in-place edit of a source rebuilds it
    assert torch.equal(_bg_full(bg, ebg, 3), torch.tensor([0.1, 0.2, 0.3, 0.4, 0.5, 0]))
    assert _bg_full(bg, ebg, 6) is six
    ebg.mul_(2)
    assert torch.equal(_bg_full(bg, ebg, 6), torch.tensor([0.1, 0.2, 0.3, 0.8, 1.0, 0, 0, 0, 0]))


@pytest.mark.parametrize("lead", [(), (4,)], ids=["CHW", "SCHW"])
def test_grad_planes(lead):
    H, W = 5, 7
    shape = lead + (H, W)

    def planes(c):
        return torch.rand(*lead, c, H, W)

    gc = planes(3)
    # no extra channels: the colour gradient as given, or zero colour planes when the loss reads no image
    assert _grad_planes(gc, None, 0, shape, "cpu") == (gc, None)
    c, f = _grad_planes(None, None, 0, shape, "cpu")
    assert f is None and c.shape == (*lead, 3, H, W) and not c.any()
    # feature gradient absent (or an empty feature image): zero feature planes, the colour gradient may be None
    for gf in (None, planes(0)):
        c, f = _grad_planes(None, gf, 6, shape, "cpu")
        assert c is None and f.shape == (*lead, 6, H, W) and not f.any()
    # present at the padded width: passed as is
    gf = planes(6)
    c, f = _grad_planes(gc, gf, 6, shape, "cpu")
    assert c is gc and f is gf
    # present for fewer channels than were rendered: zero planes for the padding channels
    gf = planes(4)
    c, f = _grad_planes(gc, gf, 6, shape, "cpu")
    assert f.shape == (*lead, 6, H, W)
    assert torch.equal(f[..., :4, :, :], gf) and not f[..., 4:, :, :].any()


def test_subset_calls_reject_cpu_tensors():
    rs = GaussianRasterizationSettings(16, 16, 0.5, 0.5, torch.zeros(3), 1.0, torch.eye(4), torch.eye(4), 0,
                                       torch.zeros(3), False, False)
    x = torch.zeros(4, 3)
    kw = dict(colors_precomp=x, scales=x + 1, rotations=torch.ones(4, 4))
    subset = torch.zeros(4, dtype=torch.int32)
    rast = GaussianRasterizer(rs)
    with pytest.raises(_lib.OgsError, match="no CPU fallback"):
        rast.forward_subsets(x, torch.ones(4, 1), subset, 1, **kw)
    with pytest.raises(_lib.OgsError, match="no CPU fallback"):
        rast.forward_subsets_grad(x, torch.ones(4, 1), subset, 1, **kw)
