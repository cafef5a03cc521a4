"""CPU tests (no GPU) of `_lib.launch`, the one call path into the C ABI for every entry point that takes a stream:
it makes the tensors' device current for the call, appends that device's current stream, and turns a non-zero
return into the same exceptions `_lib.check` raises.  The library and the torch.cuda device / stream calls are
replaced by recording fakes."""
import ctypes as C

import pytest
import torch

from opengaussian_b200 import _lib


class _FakeLib:
    def __init__(self, rc):
        self.rc = rc
        self.calls = []
        self.current = [0]          # the fake "current device" stack

    def ogs_last_error(self):
        return b"the library's message"

    def __getattr__(self, name):
        def fn(*args):
            self.calls.append((name, self.current[-1], args))
            return self.rc
        return fn


class _FakeStream:
    def __init__(self, device):
        self.cuda_stream = 0x1000 + torch.device(device).index


@pytest.fixture
def fake(monkeypatch):
    def make(rc):
        lib = _FakeLib(rc)

        class device:
            def __init__(self, d):
                self.index = torch.device(d).index

            def __enter__(self):
                lib.current.append(self.index)

            def __exit__(self, *exc):
                lib.current.pop()
                return False

        monkeypatch.setattr(_lib, "_LIB", lib)
        monkeypatch.setattr(torch.cuda, "device", device)
        monkeypatch.setattr(torch.cuda, "current_stream", lambda d=None: _FakeStream(d))
        return lib
    return make


def test_launch_enters_the_device_and_appends_its_stream(fake):
    lib = fake(0)
    assert _lib.launch("ogs_mask_mean_forward", torch.device("cuda", 1), 3, 6, None) is None
    (name, current, args), = lib.calls
    assert name == "ogs_mask_mean_forward"
    assert current == 1                                     # called with the tensors' device current
    assert args[:3] == (3, 6, None)
    assert isinstance(args[3], C.c_void_p) and args[3].value == 0x1001     # that device's current stream, last
    assert lib.current == [0]                               # the previous device is current again


@pytest.mark.parametrize("rc", [1, 700, -1, -5])
def test_launch_raises_ogs_error_naming_the_entry_point(fake, rc):
    fake(rc)
    with pytest.raises(_lib.OgsError) as e:
        _lib.launch("ogs_kmeans_assign", torch.device("cuda", 0), 1, 2)
    assert "ogs_kmeans_assign" in str(e.value) and f"rc={rc}" in str(e.value)
    assert "the library's message" in str(e.value)


def test_launch_raises_plain_exception_on_minus_two(fake):
    lib = fake(-2)
    with pytest.raises(Exception) as e:
        _lib.launch("ogs_raster_forward", torch.device("cuda", 2))
    assert type(e.value) is Exception and str(e.value) == "the library's message"
    assert lib.current == [0]
