"""Argument checks of the grid_sample-mode warp (vsrb_flow_warp_ex / _ex_bwd and the drop-in flow_warp) that run
without a GPU: bad enum values are refused with a message before anything reaches the device."""
import ctypes as C

import pytest
import torch


@pytest.fixture(scope="module")
def lib():
    from vsrlab_b200 import build, _lib
    build.build()
    return _lib.load()


# fake device addresses: every call below must fail its argument checks before a kernel could touch them
X, FLOW, OUT = C.c_void_p(1 << 20), C.c_void_p(2 << 20), C.c_void_p(3 << 20)


def _fwd(lib, interp, pad, align, dtype=0, c=64):
    return lib.vsrb_flow_warp_ex(X, 0, FLOW, 0, OUT, 1, 4, 4, c, dtype, interp, pad, align, None)


def _bwd(lib, interp, pad, align, dtype=0, c=64):
    return lib.vsrb_flow_warp_ex_bwd(X, FLOW, OUT, C.c_void_p(4 << 20), C.c_void_p(5 << 20), 1, 4, 4, c, dtype, interp, pad, align,
                                     None)


@pytest.mark.parametrize("call", [_fwd, _bwd])
def test_bad_modes_are_refused(lib, call):
    from vsrlab_b200 import _lib
    assert call(lib, 3, _lib.PAD_ZEROS, 1) == -1
    assert b"interpolation" in lib.vsrb_last_error()
    assert call(lib, -1, _lib.PAD_ZEROS, 1) == -1
    assert call(lib, _lib.INTERP_BICUBIC, 3, 1) == -1
    assert b"padding" in lib.vsrb_last_error()
    assert call(lib, _lib.INTERP_NEAREST, _lib.PAD_REFLECTION, 2) == -1
    assert b"align_corners" in lib.vsrb_last_error()


def test_bad_channels_and_dtype_are_refused(lib):
    from vsrlab_b200 import _lib
    assert _fwd(lib, _lib.INTERP_BICUBIC, _lib.PAD_ZEROS, 1, dtype=_lib.BF16, c=12) == -1
    assert b"c % 8" in lib.vsrb_last_error()
    assert _fwd(lib, _lib.INTERP_NEAREST, _lib.PAD_ZEROS, 0, dtype=_lib.F32, c=6) == -1
    assert _fwd(lib, _lib.INTERP_NEAREST, _lib.PAD_ZEROS, 1, dtype=_lib.BF16X2, c=32) == -1     # split-bf16: default mode only
    assert _bwd(lib, _lib.INTERP_BICUBIC, _lib.PAD_ZEROS, 1, dtype=_lib.BF16X2) == -1


def test_default_entry_point_still_refuses_reflection(lib):
    from vsrlab_b200 import _lib
    assert lib.vsrb_flow_warp(X, 0, FLOW, 0, OUT, 1, 4, 4, 64, _lib.BF16, _lib.PAD_REFLECTION, None) == -1
    assert b"padding" in lib.vsrb_last_error()


def test_dropin_mode_strings():
    from vsrlab.vsr.models.RealBasicVSR.modules.spynet import flow_warp
    from vsrlab_b200 import VsrbError
    x, fl = torch.rand(1, 8, 4, 4), torch.zeros(1, 4, 4, 2)
    with pytest.raises(ValueError):
        flow_warp(x, fl, interpolation="area")
    with pytest.raises(ValueError):
        flow_warp(x, fl, padding_mode="circular")
    with pytest.raises(ValueError):
        flow_warp(x, fl, "nearest4")
    # valid modes: still no CPU fallback
    for interp, pad, align in (("nearest", "zeros", True), ("bicubic", "reflection", False), ("bilinear", "border", False)):
        with pytest.raises(VsrbError):
            flow_warp(x, fl, interp, pad, align)
