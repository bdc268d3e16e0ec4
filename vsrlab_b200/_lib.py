"""ctypes binding of libvsrb200.so (the C-ABI declared in include/vsrb200.h).

The library is built in-tree by ``python -m vsrlab_b200.build`` (nvcc, sm_100a).
There is no fallback: if the shared object is missing or a call fails, the
caller gets an exception.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

HERE = Path(__file__).resolve().parent
LIB_PATH = HERE / "csrc" / "libvsrb200.so"

BF16, F32, BF16X2 = 0, 1, 2
ACT_NONE, ACT_RELU, ACT_LRELU = 0, 1, 2
PAD_ZEROS, PAD_BORDER, PAD_REFLECTION = 0, 1, 2
INTERP_BILINEAR, INTERP_NEAREST, INTERP_BICUBIC = 0, 1, 2
EPI_NHWC, EPI_CLEAN, EPI_FLOW, EPI_SR = 0, 1, 2, 3
CONV_PDL = 1
CONV_SR_U8, CONV_SR_F16 = 2, 4


class ConvGeom(C.Structure):
    _fields_ = [
        ("kh", C.c_int32), ("kw", C.c_int32),
        ("n_seg", C.c_int32),
        ("seg_c", C.c_int32 * 4),
        ("seg_off", C.c_int32 * 4),
        ("cout", C.c_int32),
        ("pixshuf", C.c_int32),
        ("groups", C.c_int32),
        ("dtype", C.c_int32),
        ("transpose", C.c_int32),
    ]


class ConvArgs(C.Structure):
    _fields_ = [
        ("geom", ConvGeom),
        ("n_in", C.c_int32),
        ("inp", C.c_void_p * 6),
        ("in_c", C.c_int32 * 6),
        ("in_c0", C.c_int32 * 6),
        ("in_wseg", C.c_int32 * 6),
        ("batch", C.c_int32), ("h", C.c_int32), ("w", C.c_int32),
        ("imgs_per_group", C.c_int32),
        ("packed", C.c_void_p),
        ("act", C.c_int32),
        ("slope", C.c_float),
        ("epilogue", C.c_int32),
        ("out", C.c_void_p),
        ("out_c", C.c_int32),
        ("out_img_stride", C.c_int64),
        ("out_group_stride", C.c_int64),
        ("residual", C.c_void_p),
        ("res_c", C.c_int32),
        ("f32_io", C.c_void_p),
        ("f32_in", C.c_void_p),
        ("aux_h", C.c_int32), ("aux_w", C.c_int32),
        ("max_ctas", C.c_int32),
        ("flags", C.c_int32),
        ("split", C.c_int32),
        ("patch", C.c_void_p),
        ("patch_img_stride", C.c_int64), ("patch_group_stride", C.c_int64),
    ]


# every symbol include/vsrb200.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "vsrb_version": (C.c_int, []),
    "vsrb_last_error": (C.c_char_p, []),
    "vsrb_device_info": (C.c_int, [C.POINTER(C.c_int32)] * 3),
    "vsrb_launch_count": (C.c_int64, []),
    "vsrb_debug_status": (C.c_int, [C.c_void_p]),
    "vsrb_debug_trace": (C.c_int, [C.c_void_p, C.c_int32]),
    "vsrb_ring_debug_stats": (C.c_int, [C.c_void_p, C.c_int32]),
    "vsrb_im2col3x3_c3": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "vsrb_pixel_unshuffle2": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "vsrb_packed_weight_bytes": (C.c_size_t, [C.POINTER(ConvGeom)]),
    "vsrb_pack_conv_weight": (C.c_int, [C.POINTER(ConvGeom), C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "vsrb_conv2d_fwd": (C.c_int, [C.POINTER(ConvArgs), C.c_void_p]),
    "vsrb_conv_plan_info": (C.c_int, [C.POINTER(ConvGeom), C.POINTER(C.c_int32)]),
    "vsrb_conv2d_wgrad_multi": (C.c_int, [C.POINTER(ConvGeom), C.c_int32, C.POINTER(C.c_void_p), C.POINTER(C.c_int32),
                                          C.POINTER(C.c_void_p), C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                          C.c_void_p, C.c_void_p]),
    "vsrb_conv2d_wgrad": (C.c_int, [C.POINTER(ConvGeom), C.POINTER(C.c_void_p), C.POINTER(C.c_int32), C.c_void_p, C.c_int32,
                                    C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "vsrb_flow_warp_bwd": (C.c_int, [C.c_void_p] * 5 + [C.c_int32] * 6 + [C.c_void_p]),
    "vsrb_flow_warp": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                 C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "vsrb_flow_warp_groups": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p] + [C.c_int32] * 7 +
                              [C.c_void_p]),
    "vsrb_flow_warp_ex": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p] + [C.c_int32] * 8 + [C.c_void_p]),
    "vsrb_flow_warp_ex_bwd": (C.c_int, [C.c_void_p] * 5 + [C.c_int32] * 8 + [C.c_void_p]),
    "vsrb_nchw_to_nhwc": (C.c_int, [C.c_void_p, C.c_void_p] + [C.c_int32] * 6 + [C.c_void_p]),
    "vsrb_nhwc_to_nchw": (C.c_int, [C.c_void_p, C.c_void_p] + [C.c_int32] * 6 + [C.c_void_p]),
    "vsrb_spynet_pyramid_base": (C.c_int, [C.c_void_p, C.c_void_p] + [C.c_int32] * 5 +
                                 [C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_void_p]),
    "vsrb_avgpool2_c4": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "vsrb_spynet_level_input": (C.c_int, [C.c_void_p] * 6 + [C.c_int32] * 5 + [C.c_void_p]),
    "vsrb_flow_resize": (C.c_int, [C.c_void_p, C.c_void_p] + [C.c_int32] * 5 + [C.c_void_p]),
    "vsrb_charbonnier": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p]),
    "vsrb_charbonnier_resized": (C.c_int, [C.c_void_p, C.c_void_p] + [C.c_int32] * 5 + [C.c_float, C.c_void_p, C.c_void_p, C.c_void_p,
                                                                                       C.c_float, C.c_void_p]),
    "vsrb_psnr_sums": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p]),
    "vsrb_ssim_sums": (C.c_int, [C.c_void_p, C.c_void_p] + [C.c_int32] * 5 + [C.c_void_p, C.c_void_p]),
    # deterministic variants: the arguments above + (workspace, workspace_bytes) before the stream
    "vsrb_conv2d_wgrad_det_workspace_bytes": (C.c_size_t, [C.POINTER(ConvGeom)] + [C.c_int32] * 5),
    "vsrb_conv2d_wgrad_det": (C.c_int, [C.POINTER(ConvGeom), C.POINTER(C.c_void_p), C.POINTER(C.c_int32), C.c_void_p, C.c_int32,
                                        C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_size_t, C.c_void_p]),
    "vsrb_conv2d_wgrad_multi_det": (C.c_int, [C.POINTER(ConvGeom), C.c_int32, C.POINTER(C.c_void_p), C.POINTER(C.c_int32),
                                              C.POINTER(C.c_void_p), C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                              C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "vsrb_flow_warp_bwd_det_workspace_bytes": (C.c_size_t, [C.c_int32] * 4),
    "vsrb_flow_warp_bwd_det": (C.c_int, [C.c_void_p] * 5 + [C.c_int32] * 6 + [C.c_void_p, C.c_size_t, C.c_void_p]),
    "vsrb_charbonnier_det_workspace_bytes": (C.c_size_t, [C.c_int64]),
    "vsrb_charbonnier_resized_det_workspace_bytes": (C.c_size_t, [C.c_int32] * 3),
    "vsrb_psnr_sums_det_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int64]),
    "vsrb_ssim_sums_det_workspace_bytes": (C.c_size_t, [C.c_int32] * 4),
    "vsrb_charbonnier_det": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float,
                                       C.c_void_p, C.c_size_t, C.c_void_p]),
    "vsrb_charbonnier_resized_det": (C.c_int, [C.c_void_p, C.c_void_p] + [C.c_int32] * 5 + [C.c_float, C.c_void_p, C.c_void_p,
                                                                                           C.c_void_p, C.c_float, C.c_void_p,
                                                                                           C.c_size_t, C.c_void_p]),
    "vsrb_psnr_sums_det": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "vsrb_ssim_sums_det": (C.c_int, [C.c_void_p, C.c_void_p] + [C.c_int32] * 5 + [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
}

_lib = None


class VsrbError(RuntimeError):
    pass


def load() -> C.CDLL:
    """dlopen the kernel library once; raise if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("VSRB200_LIB", LIB_PATH))
    if not path.exists() and "VSRB200_LIB" not in os.environ:
        # not built yet (fresh checkout): compile the kernels in-tree with nvcc; there is still no non-CUDA path
        try:
            from . import build as _build
            _build.build()
        except Exception as e:  # noqa: BLE001
            raise VsrbError(f"{path} is missing and building it failed: {e}") from e
    if not path.exists():
        raise VsrbError(
            f"{path} not found: build the sm_100a kernels first (python -m vsrlab_b200.build). "
            "vsrlab_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(str(path))
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().vsrb_last_error()
        raise VsrbError(f"{what} failed ({rc}): {msg.decode() if msg else '?'}")
