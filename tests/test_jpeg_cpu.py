"""pysp_jpeg_encode_ycc420 without a GPU.  The NumPy restatement (tests/jpeg_ref.py) is pinned to libjpeg through Pillow, byte
for byte: across qualities, contents (random, smooth, flat with long zero runs, extreme values, 0xFF-dense output) and sizes of
every residue mod 16, down to 2x2; and against Pillow's JPEG of the 8-bit sRGB image when W is a multiple of 16.  The kernels'
phases run serially through the host emulation (tests/host_emu/jpeg_emu.cpp): their coefficients, bit counts, offsets and file equal the
restatement, and they write nothing past the file.  The quantisation's reciprocal division is checked exhaustively, the
library rejects invalid arguments before touching a device, and the size helpers hold."""
import ctypes as C
import io
import os
import subprocess

import numpy as np
import pytest

import jpeg_ref as J
from pysp_b200 import _capi
from ycc420_ref import upsample2x2, ycc420

QUALITIES = (1, 2, 10, 25, 50, 51, 75, 90, 95, 99, 100)
CONTENTS = ("random", "smooth", "flat", "extreme", "ffdense")
SENTINEL = 0xA5


def _pil():
    Image = pytest.importorskip("PIL.Image")
    from PIL import features
    if not features.check("jpg"):
        pytest.skip("Pillow was built without JPEG support")
    return Image


def pillow_planes(Y, Cb, Cr, quality):
    """libjpeg's JPEG of the planes (chroma repeated 2x2: its h2v2 downsample gives the planes back)"""
    Image = _pil()
    b = io.BytesIO()
    Image.merge("YCbCr", [Image.fromarray(np.ascontiguousarray(p)) for p in (Y, upsample2x2(Cb), upsample2x2(Cr))]).save(
        b, format="JPEG", quality=quality, subsampling=2)
    return b.getvalue()


def pillow_rgb(S, quality):
    Image = _pil()
    b = io.BytesIO()
    Image.fromarray(np.ascontiguousarray(S)).save(b, format="JPEG", quality=quality, subsampling=2)
    return b.getvalue()


def content(kind, H, W, seed=0):
    """(Y, Cb, Cr) uint8 planes of an H x W frame"""
    rng = np.random.default_rng(seed)
    h, w = H // 2, W // 2
    if kind == "random":
        return tuple(rng.integers(0, 256, s, dtype=np.uint8) for s in ((H, W), (h, w), (h, w)))
    if kind == "smooth":
        yy, xx = np.mgrid[0:H, 0:W]
        Y = (128 + 100 * np.sin(xx / 13.0 + seed) * np.cos(yy / 9.0)).astype(np.uint8)
        return Y, Y[::2, ::2] // 2 + 64, 255 - Y[::2, ::2]
    if kind == "flat":
        # constant planes with a few isolated specks: long zero runs (ZRL), and the dummy blocks' DC
        planes = [np.full(s, v, dtype=np.uint8) for s, v in (((H, W), 90), ((h, w), 140), ((h, w), 100))]
        for p in planes:
            n = max(1, p.size // 97)
            p.reshape(-1)[rng.integers(0, p.size, n)] = rng.integers(0, 256, n, dtype=np.uint8)
        return tuple(planes)
    if kind == "extreme":
        # 0/255 checkerboards inside 8x8 blocks that alternate with flat black / white blocks: the largest AC magnitudes and,
        # at quality 100, DC differences of category 11
        yy, xx = np.mgrid[0:H, 0:W]
        blk = ((yy // 8) + (xx // 8)) % 3
        Y = np.where(blk == 0, ((yy + xx) & 1) * 255, np.where(blk == 1, 0, 255)).astype(np.uint8)
        return Y, 255 - Y[::2, ::2], Y[1::2, 1::2]
    if kind == "ffdense":
        # a +-2 checkerboard: at quality 90 about a fifth of the entropy-coded bytes are 0xFF
        yy, xx = np.mgrid[0:H, 0:W]
        Y = (128 + 2 * (((yy + xx) & 1) * 2 - 1)).astype(np.uint8)
        return Y, Y[::2, ::2], 255 - Y[::2, ::2]
    raise ValueError(kind)


def check_restatement(Y, Cb, Cr, q, what):
    got, want = J.encode(Y, Cb, Cr, q), pillow_planes(Y, Cb, Cr, q)
    if got != want:
        first = next((i for i in range(min(len(got), len(want))) if got[i] != want[i]), min(len(got), len(want)))
        raise AssertionError("%s: restatement differs from libjpeg (%d vs %d bytes, first difference at %d)" % (
            what, len(got), len(want), first))
    assert len(got) <= J.max_bytes(*Y.shape)
    return got


@pytest.mark.parametrize("kind", CONTENTS)
@pytest.mark.parametrize("q", QUALITIES)
def test_restatement_equals_pillow(q, kind):
    for H, W in ((48, 64), (34, 50)):
        check_restatement(*content(kind, H, W, q), q, "%s %dx%d q=%d" % (kind, H, W, q))


def test_contents_reach_their_cases():
    """the special contents do what they are there for: DC category 11 and 10-bit AC magnitudes, ZRL, dense 0xFF bytes"""
    zz = J.coefficients(*content("extreme", 48, 64), 100)
    assert J._nbits(J.dc_differences(zz)).max() == 11 and J._nbits(zz[:, 1:]).max() == 10
    zz = J.coefficients(*content("flat", 48, 64), 50)
    nz = zz[:, 1:] != 0
    last = np.maximum.accumulate(np.where(nz, np.arange(1, 64), 0), axis=1)
    prev = np.concatenate([np.zeros((len(zz), 1), dtype=np.int64), last[:, :-1]], axis=1)
    assert ((np.arange(1, 64) - prev - 1 >= 16) & nz).any(), "no zero run of 16 or more before a coefficient"
    data = J.encode(*content("ffdense", 48, 64), 90)[J.HEADER_BYTES:-2]
    assert data.count(b"\xff\x00") >= len(data) // 6


@pytest.mark.parametrize("hm", range(0, 16, 2))
@pytest.mark.parametrize("wm", range(0, 16, 2))
def test_restatement_sizes(hm, wm):
    """every residue of H and W mod 16 (partial MCUs, dummy blocks, edge replication), one quality and content each"""
    i = hm * 8 + wm
    H, W = 32 + hm, 48 + wm
    q, kind = QUALITIES[i % len(QUALITIES)], CONTENTS[i % len(CONTENTS)]
    check_restatement(*content(kind, H, W, i), q, "%s %dx%d q=%d" % (kind, H, W, q))
    if hm and wm:
        check_restatement(*content(kind, hm, wm, i), q, "%s %dx%d q=%d" % (kind, hm, wm, q))


@pytest.mark.parametrize("shape", [(2, 2), (2, 4), (4, 2), (2, 18), (18, 2), (6, 6), (8, 8), (10, 16)])
def test_restatement_tiny(shape):
    for q in (1, 75, 100):
        check_restatement(*content("random", *shape, q), q, "%s q=%d" % (shape, q))


@pytest.mark.parametrize("H", [20, 34, 66])
@pytest.mark.parametrize("W", [32, 48, 96, 128])
def test_restatement_equals_pillow_rgb(H, W):
    """W % 16 == 0: the file of the ycc420 planes of an 8-bit sRGB image is libjpeg's JPEG of that image"""
    S = np.random.default_rng(H * W).integers(0, 256, (H, W, 3), dtype=np.uint8)
    for q in (50, 75, 95):
        assert J.encode(*ycc420(S), q) == pillow_rgb(S, q), "%dx%d q=%d" % (H, W, q)


def test_restatement_equals_pillow_rgb_all_colours():
    from test_ycc420_cpu import all_colours
    S = all_colours()
    assert J.encode(*ycc420(S), 90) == pillow_rgb(S, 90)


# ---- the kernels' phases through the host emulation --------------------------------------------------------------------
@pytest.fixture(scope="module")
def jemu(tmp_path_factory):
    """tests/host_emu/jpeg_emu.cpp, compiled with g++ into a temporary directory (the tree is left as it is)"""
    if not os.path.exists("/usr/bin/g++"):
        pytest.skip("g++ not available")
    src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_emu", "jpeg_emu.cpp")
    so = str(tmp_path_factory.mktemp("jpeg_emu") / "libpysp_jpeg_emu.so")
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-o", so,
                           src])
    lib = C.CDLL(so)
    u8, i64 = C.c_void_p, C.c_int64
    lib.emu_jpeg_encode.argtypes = [u8, i64, u8, u8, i64, C.c_int, C.c_int, C.c_int, u8, i64, u8, u8, i64]
    lib.emu_jpeg_layout.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    lib.emu_jpeg_check_reciprocals.restype = C.c_int64
    lib.emu_jpeg_last_error.restype = C.c_char_p
    return lib


def padded(p, pad):
    """p in the top-left corner of a sentinel array `pad` columns wider (a row pitch above the width)"""
    a = np.full((p.shape[0], p.shape[1] + pad), SENTINEL, dtype=np.uint8)
    a[:, :p.shape[1]] = p
    return a


def emu_encode(lib, Y, Cb, Cr, q, pad=(0, 0)):
    """(file, workspace) from the emulation; the output and workspace buffers are sized exactly and must keep their tails"""
    H, W = Y.shape
    y, cb, cr = padded(Y, pad[0]), padded(Cb, pad[1]), padded(Cr, pad[1])
    cap = int(_capi.lib().pysp_jpeg_max_bytes(H, W))
    nws = int(_capi.lib().pysp_jpeg_workspace_bytes(H, W))
    out = np.full(cap + 64, SENTINEL, dtype=np.uint8)
    ws = np.full(nws + 64, SENTINEL, dtype=np.uint8)
    n = np.zeros(1, dtype=np.int64)
    rc = lib.emu_jpeg_encode(y.ctypes.data, y.strides[0], cb.ctypes.data, cr.ctypes.data, cb.strides[0], H, W, q, out.ctypes.data,
                             cap, n.ctypes.data, ws.ctypes.data, nws)
    assert rc == 0, lib.emu_jpeg_last_error()
    n = int(n[0])
    assert (out[n:] == SENTINEL).all(), "bytes past the file were written"
    assert (ws[nws:] == SENTINEL).all(), "the workspace was overrun"
    return out[:n].tobytes(), ws


EMU_CASES = [((48, 64), "random", 75, (0, 0)), ((34, 50), "smooth", 90, (3, 1)), ((18, 18), "flat", 50, (0, 5)),
             ((66, 130), "extreme", 100, (8, 2)), ((30, 46), "ffdense", 90, (1, 0)), ((2, 2), "random", 1, (0, 0)),
             ((20, 28), "random", 95, (5, 7)), ((40, 24), "smooth", 10, (0, 0))]


@pytest.mark.parametrize("case", range(len(EMU_CASES)))
def test_emulated_kernels_equal_restatement(jemu, case):
    (H, W), kind, q, pad = EMU_CASES[case]
    Y, Cb, Cr = content(kind, H, W, case)
    data, ws = emu_encode(jemu, Y, Cb, Cr, q, pad)
    zz = J.coefficients(Y, Cb, Cr, q)
    counts, _ = J.entropy_bits(zz)
    o = [C.c_int64() for _ in range(3)]
    jemu.emu_jpeg_layout(H, W, *[C.byref(v) for v in o])
    nb = len(zz)
    coef = ws[o[0].value:o[0].value + nb * 128].view(np.int16).reshape(nb, 64)
    bits = ws[o[1].value:o[1].value + nb * 4].view(np.uint32)
    boff = ws[o[2].value:o[2].value + nb * 8].view(np.int64)
    assert np.array_equal(coef, zz), "quantised coefficients"
    assert np.array_equal(bits, counts), "block bit counts"
    assert np.array_equal(boff, np.cumsum(counts) - counts), "block bit offsets"
    assert data == J.encode(Y, Cb, Cr, q)


def test_reciprocal_division_exhaustive(jemu):
    """the kernels' quantisation (multiply by ceil(2^32 / d), shift) equals (|c| + d/2) / d for every divisor d = 8 * (1..255)
    and every |c| < 2^15"""
    assert jemu.emu_jpeg_check_reciprocals() == 0


def _encode_args(H=16, W=16, q=75, **over):
    """arguments of pysp_jpeg_encode_ycc420 with host buffers (the library checks them before any CUDA call)"""
    keep = [np.zeros((max(H, 2), max(W, 2)), dtype=np.uint8), np.zeros(1 << 16, dtype=np.uint8), np.zeros(1, dtype=np.int64)]
    L = _capi.lib()
    cap = int(L.pysp_jpeg_max_bytes(H, W)) if H > 0 and W > 0 else 0
    nws = int(L.pysp_jpeg_workspace_bytes(H, W)) if H > 0 and W > 0 else 0
    a = dict(y=keep[0].ctypes.data, y_pitch=W, cb=keep[0].ctypes.data, cr=keep[0].ctypes.data, c_pitch=W // 2, H=H, W=W, q=q,
             out=keep[1].ctypes.data, cap=cap, out_len=keep[2].ctypes.data, ws=keep[1].ctypes.data, nws=nws, stream=None)
    a.update(over)
    return list(a.values()), keep


@pytest.mark.parametrize("over", [dict(q=0), dict(q=101), dict(H=15), dict(W=7), dict(H=0), dict(W=65536, cap=1 << 40, nws=1 << 40),
                                  dict(y_pitch=15), dict(c_pitch=7), dict(cap=1000), dict(nws=100), dict(y=None), dict(cb=None),
                                  dict(cr=None), dict(out=None), dict(out_len=None), dict(ws=None)])
def test_invalid_arguments(jemu, over):
    """bad size, quality, pitches, capacity, workspace or a null pointer: PYSP_ERR_INVALID from the library (no GPU is touched:
    the plan runs first) and from the emulation"""
    args, keep = _encode_args(**over)
    L = _capi.lib()
    assert L.pysp_jpeg_encode_ycc420(*args) == _capi.ERR_INVALID
    assert len(L.pysp_last_error()) > 0
    assert jemu.emu_jpeg_encode(*args[:-1]) == _capi.ERR_INVALID
    ok, keep2 = _encode_args()
    assert jemu.emu_jpeg_encode(*ok[:-1]) == _capi.OK


def test_size_helpers():
    """pysp_jpeg_max_bytes is the documented bound (and the restatement's); both helpers are 0 for invalid sizes; the
    workspace grows with the frame and holds at least the coefficients"""
    L = _capi.lib()
    for H, W in ((2, 2), (16, 16), (34, 50), (4000, 6000), (65534, 65534), (8660, 11548)):
        mcus = -(-H // 16) * -(-W // 16)
        assert L.pysp_jpeg_max_bytes(H, W) == 623 + 2 * -(-6 * mcus * 1660 // 8) + 2 == J.max_bytes(H, W)
        assert L.pysp_jpeg_workspace_bytes(H, W) >= 6 * mcus * 128
    assert L.pysp_jpeg_workspace_bytes(64, 64) > L.pysp_jpeg_workspace_bytes(32, 32) > 0
    for H, W in ((0, 16), (16, 0), (3, 16), (16, 5), (65536, 16), (-2, 16)):
        assert L.pysp_jpeg_max_bytes(H, W) == 0 and L.pysp_jpeg_workspace_bytes(H, W) == 0
    for kind in CONTENTS:                  # the bound holds for the largest files this suite makes
        Y, Cb, Cr = content(kind, 48, 64)
        assert len(J.encode(Y, Cb, Cr, 100)) <= J.max_bytes(48, 64)
