"""pysp_jpeg_encode_rgb without a GPU.  The NumPy restatement (tests/jpeg_rgb_ref.py) is pinned to libjpeg through Pillow, byte
for byte, at 4:4:4, 4:2:2 and 4:2:0: across qualities 1..100, contents (random, smooth, flat with long zero runs, extreme
values, 0xFF-dense output), every residue of H and W mod 16 (odd ones included), 1x1, 1xN and Nx1, and all 2^24 colours in one
4096x4096 image.  The kernels' phases run serially through the host emulation (tests/host_emu/jpeg_rgb_emu.cpp): the converted
planes, coefficients, bit counts, offsets and file equal the restatement, from padded pitches of any residue, and nothing is
written past the file or the workspace; the 4:2:0 planes path on the same generalised geometry still equals tests/jpeg_ref.py.
The library rejects invalid arguments before touching a device, and the size helpers hold."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import jpeg_ref as J
import jpeg_rgb_ref as R
from pysp_b200 import _capi
from test_jpeg_cpu import CONTENTS, QUALITIES, content

SENTINEL = 0xA5


@pytest.fixture(scope="module", autouse=True)
def _pil():
    pytest.importorskip("PIL.Image")
    from PIL import features
    if not features.check("jpg"):
        pytest.skip("Pillow was built without JPEG support")


def check_restatement(S, q, s, what):
    got, want = R.encode(S, q, s), R.pillow_rgb(S, q, s)
    if got != want:
        first = next((i for i in range(min(len(got), len(want))) if got[i] != want[i]), min(len(got), len(want)))
        raise AssertionError("%s %s: restatement differs from libjpeg (%d vs %d bytes, first difference at %d)" % (
            what, R.NAMES[s], len(got), len(want), first))
    assert len(got) <= R.max_bytes(S.shape[0], S.shape[1], s)
    return got


@pytest.mark.parametrize("kind", CONTENTS)
@pytest.mark.parametrize("q", QUALITIES)
@pytest.mark.parametrize("s", R.SUBSAMPLINGS)
def test_restatement_equals_pillow(s, q, kind):
    for H, W in ((48, 64), (35, 51)):
        check_restatement(R.rgb_content(kind, H, W, q), q, s, "%s %dx%d q=%d" % (kind, H, W, q))


def test_restatement_every_quality():
    """qualities 1..100 at each subsampling (smooth content: every quantisation table entry matters)"""
    for q in range(1, 101):
        check_restatement(R.rgb_content("smooth", 24, 40, q), q, q % 3, "smooth 24x40 q=%d" % q)


@pytest.mark.parametrize("hm", range(16))
@pytest.mark.parametrize("s", R.SUBSAMPLINGS)
def test_restatement_sizes(s, hm):
    """every residue of H and W mod 16, odd ones included (partial MCUs, dummy blocks, the chroma edge rule)"""
    for wm in range(16):
        i = hm * 16 + wm
        H, W = 32 + hm, 48 + wm
        q, kind = QUALITIES[i % len(QUALITIES)], CONTENTS[i % len(CONTENTS)]
        check_restatement(R.rgb_content(kind, H, W, i), q, s, "%s %dx%d q=%d" % (kind, H, W, q))
        if hm and wm:
            check_restatement(R.rgb_content(kind, hm, wm, i), q, s, "%s %dx%d q=%d" % (kind, hm, wm, q))


@pytest.mark.parametrize("shape", [(1, 1), (1, 2), (2, 1), (1, 17), (17, 1), (1, 100), (100, 1), (3, 3), (7, 9)])
def test_restatement_tiny(shape):
    for s in R.SUBSAMPLINGS:
        for q in (1, 75, 100):
            check_restatement(R.rgb_content("random", *shape, q), q, s, "%s q=%d" % (shape, q))


@pytest.mark.parametrize("s", R.SUBSAMPLINGS)
def test_restatement_all_colours(s):
    """all 2^24 colours in one 4096x4096 image"""
    from test_ycc420_cpu import all_colours
    check_restatement(all_colours(), 90, s, "all colours")


def test_restatement_420_planes_agree_when_w_is_a_multiple_of_16():
    """at 4:2:0 with W % 16 == 0 the convert phase's planes are the ycc420 planes and the files agree with jpeg_ref's"""
    from ycc420_ref import ycc420
    for H, W in ((20, 32), (33, 48), (66, 96)):
        S = R.rgb_content("random", H, W, H)
        Y, Cb, Cr = R.planes(S, 2)
        y0, cb0, cr0 = ycc420(S[:H - H % 2])
        assert np.array_equal(Y[:H - H % 2], y0) and np.array_equal(Cb[:H // 2], cb0) and np.array_equal(Cr[:H // 2], cr0)
        if H % 2 == 0:
            assert R.encode(S, 75, 2) == J.encode(y0, cb0, cr0, 75)


# ---- the kernels' phases through the host emulation --------------------------------------------------------------------
@pytest.fixture(scope="module")
def remu(tmp_path_factory):
    """tests/host_emu/jpeg_rgb_emu.cpp, compiled with g++ into a temporary directory (the tree is left as it is)"""
    if not os.path.exists("/usr/bin/g++"):
        pytest.skip("g++ not available")
    src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_emu", "jpeg_rgb_emu.cpp")
    so = str(tmp_path_factory.mktemp("jpeg_rgb_emu") / "libpysp_jpeg_rgb_emu.so")
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-o", so,
                           src])
    lib = C.CDLL(so)
    p, i64, i32 = C.c_void_p, C.c_int64, C.c_int
    lib.emu_jpeg_rgb_encode.argtypes = [p, i64, i32, i32, i32, i32, p, i64, p, p, i64]
    lib.emu_jpeg_rgb_layout.argtypes = [i32, i32, i32, C.POINTER(C.c_int64)]
    lib.emu_jpeg_encode.argtypes = [p, i64, p, p, i64, i32, i32, i32, p, i64, p, p, i64]
    lib.emu_jpeg_last_error.restype = C.c_char_p
    return lib


def padded_rgb(S, pad):
    """S in the top-left corner of a sentinel byte array whose rows are `pad` bytes longer than 3W (any residue)"""
    H, W = S.shape[:2]
    a = np.full((H, 3 * W + pad), SENTINEL, dtype=np.uint8)
    a[:, :3 * W] = S.reshape(H, 3 * W)
    return a


def emu_rgb_encode(lib, S, q, s, pad=0):
    """(file, workspace) from the emulation; the output and workspace buffers are sized exactly and must keep their tails"""
    H, W = S.shape[:2]
    a = padded_rgb(S, pad)
    cap = int(_capi.lib().pysp_jpeg_rgb_max_bytes(H, W, s))
    nws = int(_capi.lib().pysp_jpeg_rgb_workspace_bytes(H, W, s))
    out = np.full(cap + 64, SENTINEL, dtype=np.uint8)
    ws = np.full(nws + 64, SENTINEL, dtype=np.uint8)
    n = np.zeros(1, dtype=np.int64)
    rc = lib.emu_jpeg_rgb_encode(a.ctypes.data, a.strides[0], H, W, q, s, out.ctypes.data, cap, n.ctypes.data, ws.ctypes.data, nws)
    assert rc == 0, lib.emu_jpeg_last_error()
    n = int(n[0])
    assert (out[n:] == SENTINEL).all(), "bytes past the file were written"
    assert (ws[nws:] == SENTINEL).all(), "the workspace was overrun"
    return out[:n].tobytes(), ws


EMU_CASES = [((48, 64), "random", 75, 0), ((35, 51), "smooth", 90, 1), ((17, 18), "flat", 50, 5), ((66, 131), "extreme", 100, 2),
             ((31, 45), "ffdense", 90, 7), ((1, 1), "random", 1, 0), ((1, 29), "random", 95, 3), ((29, 1), "smooth", 10, 4),
             ((9, 23), "random", 60, 11)]


@pytest.mark.parametrize("s", R.SUBSAMPLINGS)
@pytest.mark.parametrize("case", range(len(EMU_CASES)))
def test_emulated_kernels_equal_restatement(remu, case, s):
    (H, W), kind, q, pad = EMU_CASES[case]
    S = R.rgb_content(kind, H, W, case)
    data, ws = emu_rgb_encode(remu, S, q, s, pad)
    planes = R.planes(S, s)
    zz = R.coefficients(*planes, q, s)
    counts, _ = R.entropy_bits(zz, s)
    o = (C.c_int64 * 6)()
    remu.emu_jpeg_rgb_layout(H, W, s, o)
    nb = len(zz)
    for k, (P, name) in enumerate(zip(planes, ("Y", "Cb", "Cr"))):
        got = ws[o[3 + k]:o[3 + k] + P.size].reshape(P.shape)
        assert np.array_equal(got, P), "converted %s plane" % name
    assert np.array_equal(ws[o[0]:o[0] + nb * 128].view(np.int16).reshape(nb, 64), zz), "quantised coefficients"
    assert np.array_equal(ws[o[1]:o[1] + nb * 4].view(np.uint32), counts), "block bit counts"
    assert np.array_equal(ws[o[2]:o[2] + nb * 8].view(np.int64), np.cumsum(counts) - counts), "block bit offsets"
    assert data == R.encode(S, q, s)
    assert data == R.pillow_rgb(S, q, s)


@pytest.mark.parametrize("case", range(4))
def test_emulated_ycc420_planes_on_the_generalised_geometry(remu, case):
    """pysp_jpeg_encode_ycc420's phases, now reading the MCU shape from the parameters, still give jpeg_ref's file"""
    (H, W), kind, q = [((48, 64), "random", 75), ((34, 50), "smooth", 90), ((2, 2), "flat", 1), ((66, 130), "extreme", 100)][case]
    Y, Cb, Cr = (np.ascontiguousarray(P) for P in content(kind, H, W, case))
    cap = int(_capi.lib().pysp_jpeg_max_bytes(H, W))
    nws = int(_capi.lib().pysp_jpeg_workspace_bytes(H, W))
    out = np.full(cap + 64, SENTINEL, dtype=np.uint8)
    ws = np.zeros(nws, dtype=np.uint8)
    n = np.zeros(1, dtype=np.int64)
    assert remu.emu_jpeg_encode(Y.ctypes.data, W, Cb.ctypes.data, Cr.ctypes.data, W // 2, H, W, q, out.ctypes.data, cap,
                                n.ctypes.data, ws.ctypes.data, nws) == 0
    assert out[:int(n[0])].tobytes() == J.encode(Y, Cb, Cr, q)
    assert (out[int(n[0]):] == SENTINEL).all()


@pytest.mark.parametrize("s", R.SUBSAMPLINGS)
def test_random_noise_q100_within_max_bytes(remu, s):
    """the bound holds for the largest files: random noise at quality 100 (odd sizes too)"""
    for H, W in ((64, 64), (33, 47)):
        S = R.rgb_content("random", H, W, 7)
        data, _ = emu_rgb_encode(remu, S, 100, s)
        assert len(data) <= int(_capi.lib().pysp_jpeg_rgb_max_bytes(H, W, s)) == R.max_bytes(H, W, s)
        assert len(data) > R.max_bytes(H, W, s) // 8


def _rgb_args(H=16, W=16, q=75, s=2, **over):
    """arguments of pysp_jpeg_encode_rgb with host buffers (the library checks them before any CUDA call)"""
    keep = [np.zeros(3 * 64 * 64, dtype=np.uint8), np.zeros(1 << 17, dtype=np.uint8), np.zeros(1, dtype=np.int64)]
    L = _capi.lib()
    ok = 0 <= s <= 2 and H > 0 and W > 0
    cap = int(L.pysp_jpeg_rgb_max_bytes(H, W, s)) if ok else 1 << 40
    nws = int(L.pysp_jpeg_rgb_workspace_bytes(H, W, s)) if ok else 1 << 40
    a = dict(rgb=keep[0].ctypes.data, pitch=3 * W, H=H, W=W, q=q, s=s, out=keep[1].ctypes.data, cap=cap,
             out_len=keep[2].ctypes.data, ws=keep[1].ctypes.data, nws=nws, stream=None)
    a.update(over)
    return list(a.values()), keep


@pytest.mark.parametrize("over", [dict(s=-1), dict(s=3), dict(q=0), dict(q=101), dict(H=0), dict(W=0), dict(H=65536),
                                  dict(W=65536), dict(H=-1), dict(pitch=47), dict(pitch=0), dict(cap=1000), dict(nws=100),
                                  dict(rgb=None), dict(out=None), dict(out_len=None), dict(ws=None)])
def test_invalid_arguments(remu, over):
    """bad subsampling, size, quality, pitch, capacity, workspace or a null pointer: PYSP_ERR_INVALID from the library (no GPU
    is touched: the plan runs first) and from the emulation"""
    args, keep = _rgb_args(**over)
    L = _capi.lib()
    assert L.pysp_jpeg_encode_rgb(*args) == _capi.ERR_INVALID
    assert len(L.pysp_last_error()) > 0
    assert remu.emu_jpeg_rgb_encode(*args[:-1]) == _capi.ERR_INVALID
    ok, keep2 = _rgb_args()
    assert remu.emu_jpeg_rgb_encode(*ok[:-1]) == _capi.OK


def test_mcu_of_block_by_reciprocal():
    """the block phases find block b's MCU as (b * ceil(2^32 / slots)) >> 32: exact for every b < 2^31 (more than any frame
    has blocks) because m * slots - 2^32 <= 2 for the 3, 4 and 6 slots of 4:4:4, 4:2:2 and 4:2:0"""
    for slots in (3, 4, 6):
        m = -(-(1 << 32) // slots)
        assert m * slots - (1 << 32) <= 2
        rng = np.random.default_rng(slots)
        b = np.concatenate([np.arange(1 << 16), (1 << 31) - 1 - np.arange(1 << 16), rng.integers(0, 1 << 31, 1 << 16)])
        assert np.array_equal((b.astype(np.uint64) * np.uint64(m)) >> np.uint64(32), (b // slots).astype(np.uint64))
    assert 3 * 8192 * 8192 < 1 << 31 and 4 * 4096 * 8192 < 1 << 31 and 6 * 4096 * 4096 < 1 << 31


def test_size_helpers():
    """pysp_jpeg_rgb_max_bytes is the documented bound (and the restatement's); both helpers are 0 for invalid arguments; the
    workspace holds at least the coefficients and the converted planes; 4:2:0 needs no more than pysp_jpeg_max_bytes"""
    L = _capi.lib()
    for H, W in ((1, 1), (16, 16), (35, 51), (4000, 6000), (65535, 65535), (8660, 11548)):
        for s in R.SUBSAMPLINGS:
            (h, v), (my, mx) = R.SAMPLING[s], R.mcus(H, W, s)
            nb = (h * v + 2) * my * mx
            assert L.pysp_jpeg_rgb_max_bytes(H, W, s) == 623 + 2 * -(-nb * 1660 // 8) + 2 == R.max_bytes(H, W, s)
            assert L.pysp_jpeg_rgb_workspace_bytes(H, W, s) >= nb * 128 + H * W + 2 * 8 * mx * -(-H // v)
        if H % 2 == 0 and W % 2 == 0:
            assert L.pysp_jpeg_rgb_max_bytes(H, W, 2) == L.pysp_jpeg_max_bytes(H, W)
    for H, W, s in ((0, 16, 0), (16, 0, 1), (65536, 16, 2), (16, 65536, 0), (-2, 16, 1), (16, 16, 3), (16, 16, -1)):
        assert L.pysp_jpeg_rgb_max_bytes(H, W, s) == 0 and L.pysp_jpeg_rgb_workspace_bytes(H, W, s) == 0
    assert _capi.JPEG_444 == 0 and _capi.JPEG_422 == 1 and _capi.JPEG_420 == 2
