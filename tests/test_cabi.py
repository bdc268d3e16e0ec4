"""The C-ABI library loads without a GPU and exports every symbol include/vsrb200.h declares."""
import ctypes as C
import re
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]


@pytest.fixture(scope="module")
def lib():
    from vsrlab_b200 import build, _lib
    build.build()
    return _lib.load()


def header_symbols():
    text = (ROOT / "include" / "vsrb200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(vsrb_[a-z0-9_]+)\s*\(", text)))


def test_header_and_binding_agree(lib):
    from vsrlab_b200 import _lib
    names = header_symbols()
    assert len(names) >= 14
    assert sorted(_lib.SYMBOLS.keys()) == names
    for n in names:
        assert getattr(lib, n) is not None


def test_version_and_geometry_helpers_run_on_cpu(lib):
    from vsrlab_b200 import _lib
    assert lib.vsrb_version() == 101
    g = _lib.ConvGeom()
    g.kh = g.kw = 3
    g.n_seg = 1
    g.seg_c[0] = 64
    g.cout = 64
    g.groups = 1
    g.dtype = _lib.BF16
    # bias header + classic image (9 taps x 64 x 64 bf16) + the ring-walk image: 2 CTA ranks x (3 filter columns x 96 rows x 128 B
    # + the 32 x 64 B im2col tile of a 3-channel segment)
    assert lib.vsrb_packed_weight_bytes(C.byref(g)) == 1024 + 9 * 64 * 64 * 2 + 2 * (3 * 96 * 128 + 32 * 64)
    g.dtype = _lib.F32
    assert lib.vsrb_packed_weight_bytes(C.byref(g)) == 1024 + 9 * 64 * 64 * 4
    g.kh = 4                                            # even kernels are rejected with a message, not a crash
    assert lib.vsrb_packed_weight_bytes(C.byref(g)) == 0
    assert b"unsupported" in lib.vsrb_last_error()


def test_struct_layout_matches_header(lib):
    """ctypes mirrors of the C structs: sizes follow the C layout rules of the header."""
    from vsrlab_b200 import _lib
    assert C.sizeof(_lib.ConvGeom) == 16 * 4          # kh kw n_seg seg_c[4] seg_off[4] cout pixshuf groups dtype transpose
    assert C.sizeof(_lib.ConvArgs) % 8 == 0
    assert _lib.ConvArgs.packed.offset % 8 == 0 and _lib.ConvArgs.out_img_stride.offset % 8 == 0


def test_conv_plan_selection(lib):
    """The tiling the library picks per geometry (DESIGN.md 4.1 cost model): the hot 3x3 64->64 conv and the
    SPyNet 7x7 convs use the stacked layout, stems with 3 input channels and 1x1 / pixel-shuffle convs the classic one."""
    from vsrlab_b200 import _lib

    def plan(k, segs, cout, pixshuf=0):
        g = _lib.ConvGeom()
        g.kh = g.kw = k
        g.n_seg = len(segs)
        for i, c in enumerate(segs):
            g.seg_c[i] = c
        g.cout, g.groups, g.dtype, g.pixshuf = cout, 1, _lib.BF16, pixshuf
        info = (C.c_int32 * 8)()
        assert lib.vsrb_conv_plan_info(C.byref(g), info) == 0
        return list(info)
    stacked, n_tile, n_blocks, mma_n = plan(3, [64], 64)[:4]
    assert (stacked, n_tile, n_blocks, mma_n) == (1, 64, 1, 192)
    assert plan(3, [64, 3], 64)[:4] == [1, 64, 1, 192]          # cat([lr_i, feat]) stem: two K segments
    assert plan(3, [3], 64)[0] == 0                              # 16-channel (32-byte-row) stem stays classic
    assert plan(1, [64, 64], 64)[:4] == [0, 64, 1, 64]           # 1x1 fusion conv
    assert plan(3, [64], 256, pixshuf=2)[:4] == [0, 128, 2, 128]  # upsampling conv: N = 128, two blocks
    for segs, cout in (([8], 32), ([32], 64), ([64], 32), ([32], 16), ([16], 2)):
        info = plan(7, segs, cout)
        # stacked, N <= 256; a block's weights either stream (<= 128 KiB) or half of them stays resident per CTA of a pair
        assert info[0] == 1 and info[3] <= 256 and info[7] <= 200
    assert plan(7, [64], 32)[4] == 32 and plan(7, [32], 64)[4] == 32      # CTA-pair plans keep 64-byte K rows for 7x7


# Split-bf16 stores move 16 channels (two 16-byte vectors) at channel c0 and at c0 + out_c/2, and the 16-channel EPI_CLEAN
# store is two 16-byte vectors: vsrb_conv2d_fwd refuses every channel stride or alignment those stores cannot honour before
# it touches the device.  Only refused configurations are called here, with placeholder addresses that are never read;
# the accepted boundaries run on real tensors on the GPU: the EPI_CLEAN split shadow (out_c = 32) in
# test_gpu_image_epilogues.py, EPI_NHWC split outputs and residuals (out_c = 32, 64, 128) in test_gpu_parity.py.
E_ARG = -1
FAKE = 1 << 20                                          # non-null, 16-byte aligned placeholder address


def conv_args(epilogue, cout, out_c, split, out=FAKE, res_c=0):
    from vsrlab_b200 import _lib
    g = _lib.ConvGeom()
    g.kh = g.kw = 3
    g.n_seg = 1
    g.seg_c[0] = 64
    g.cout, g.groups, g.dtype = cout, 1, _lib.BF16
    a = _lib.ConvArgs()
    a.geom = g
    a.inp[0], a.in_c[0] = FAKE, 64
    a.batch, a.h, a.w, a.imgs_per_group = 1, 8, 8, 1
    a.packed, a.epilogue, a.out, a.out_c, a.split = FAKE, epilogue, out, out_c, split
    a.f32_io = FAKE
    if res_c:
        a.residual, a.res_c = FAKE, res_c
    return a


REFUSED = [
    # (epilogue, cout, out_c, split, out offset in bytes, res_c, message fragment)
    *[("clean", 3, oc, 1, 0, 0, b"out_c must be 32") for oc in (3, 8, 16, 17, 24, 31, 33, 48, 64)],
    ("clean", 3, 32, 1, 2, 0, b"16-byte aligned"),
    ("clean", 3, 32, 1, 8, 0, b"16-byte aligned"),
    ("clean", 3, 16, 0, 2, 0, b"16-byte aligned"),
    ("clean", 3, 16, 0, 8, 0, b"16-byte aligned"),
    *[("nhwc", 16, oc, 1, 0, 0, b"multiples of 16") for oc in (40, 56, 72)],
    ("nhwc", 16, 32, 1, 0, 40, b"multiples of 16"),
    ("nhwc", 16, 64, 1, 0, 72, b"multiples of 16"),
]


@pytest.mark.parametrize("epi,cout,out_c,split,off,res_c,msg", REFUSED)
def test_conv_refuses_unstorable_split_and_clean_layouts(lib, epi, cout, out_c, split, off, res_c, msg):
    from vsrlab_b200 import _lib
    a = conv_args({"clean": _lib.EPI_CLEAN, "nhwc": _lib.EPI_NHWC}[epi], cout, out_c, split, FAKE + off, res_c)
    assert lib.vsrb_conv2d_fwd(C.byref(a), None) == E_ARG
    assert msg in lib.vsrb_last_error()


# vsrb_conv2d_wgrad refuses, before it touches the device, every call its kernels cannot honour: grouped weights, tensors
# the 16-byte vector loads cannot read, channel strides that are not a multiple of 8, a dz with fewer channels than cout,
# element types other than bf16 and fp32, and filters no kernel takes.  Placeholder addresses as above: only refused
# calls are made.
def wgrad_call(lib, kh=3, kw=3, segs=(64,), cout=64, dtype="bf16", groups=1, ipg=2, in_off=(0, 0), in_c=None, dz_off=0, dz_c=64):
    from vsrlab_b200 import _lib
    g = _lib.ConvGeom()
    g.kh, g.kw, g.n_seg = kh, kw, len(segs)
    off = 0
    for i, c in enumerate(segs):
        g.seg_off[i], g.seg_c[i] = off, c
        off += c
    g.cout, g.groups, g.dtype = cout, groups, {"bf16": _lib.BF16, "fp32": _lib.F32, "bf16x2": _lib.BF16X2}[dtype]
    ins = (C.c_void_p * 2)(*[FAKE + (i + 1) * (1 << 16) + in_off[i] for i in range(2)])
    cs = (C.c_int32 * 2)(*(in_c or (*segs, 0)[:2]))
    return lib.vsrb_conv2d_wgrad(C.byref(g), ins, cs, C.c_void_p(FAKE + dz_off), dz_c, 2, 8, 8, ipg, off,
                                 C.c_void_p(FAKE + (1 << 18)), None, None)


WGRAD_REFUSED = {
    "groups2": (dict(groups=2, ipg=1), b"grouped"),
    "imgs_per_group": (dict(ipg=1), b"grouped"),
    "in_unaligned": (dict(in_off=(2, 0)), b"16-byte aligned"),
    "in1_unaligned": (dict(segs=(64, 64), in_off=(0, 8)), b"16-byte aligned"),
    "dz_unaligned": (dict(dz_off=4), b"16-byte aligned"),
    "in_c": (dict(segs=(60,), in_c=(60, 0)), b"multiple of 8"),
    "dz_c": (dict(cout=60, dz_c=60), b"multiple of 8"),
    "dz_c_below_cout": (dict(dz_c=56), b">= cout"),
    "bf16_3x5": (dict(kw=5), b"no kernel for a 3x5"),
    "bf16_1x5": (dict(kh=1, kw=5), b"no kernel for a 1x5"),
    "fp32_5x5": (dict(kh=5, kw=5, dtype="fp32"), b"no kernel for a 5x5"),
    "even_4x4": (dict(kh=4, kw=4), b"odd sizes"),
    "9x9": (dict(kh=9, kw=9), b"odd sizes"),
    "split_bf16": (dict(dtype="bf16x2"), b"bf16 or fp32"),
}


@pytest.mark.parametrize("case", list(WGRAD_REFUSED))
def test_wgrad_refuses_before_launch(lib, case):
    kw, msg = WGRAD_REFUSED[case]
    assert wgrad_call(lib, **kw) == E_ARG
    assert msg in lib.vsrb_last_error(), lib.vsrb_last_error()
