"""PYSP_OUT_YCC420_U8 without a GPU.  The NumPy restatement (tests/ycc420_ref.py) is pinned to libjpeg through Pillow: a JPEG
written from the restated planes is byte-identical to the one libjpeg writes from the 8-bit sRGB image.  The store of the
develop kernels runs through the host emulation (tests/host_emu) on the seeded cases of test_tile_logic_matrix: the planes
are the restatement of the same case's srgb_u8 output, every row band writes exactly its rows, and the plan rejects bad
chroma arguments."""
import ctypes as C
import io

import numpy as np
import pytest

from pysp_b200 import _capi
from test_tile_logic import LUT, M, WB, emu, emu_develop  # noqa: F401  (emu is a fixture)
from test_tile_logic_matrix import N_CASES, TILES, describe, halo_rows, matrix_case
from ycc420_ref import upsample2x2, ycc420, ycc_full

SENTINEL = 0xA5


def _jpeg(img, subsampling):
    buf = io.BytesIO()
    img.save(buf, format="JPEG", quality=95, subsampling=subsampling)
    return buf.getvalue()


def _pil():
    Image = pytest.importorskip("PIL.Image")
    from PIL import features
    if not features.check("jpg"):
        pytest.skip("Pillow was built without JPEG support")
    return Image


def assert_jpeg_identical(Image, S, planes, subsampling, what):
    """JPEG of the RGB image S against the JPEG of the YCbCr planes (full-resolution planes as libjpeg receives them)"""
    rgb = _jpeg(Image.fromarray(np.ascontiguousarray(S)), subsampling)
    ycc = _jpeg(Image.merge("YCbCr", [Image.fromarray(np.ascontiguousarray(p)) for p in planes]), subsampling)
    assert rgb == ycc, "%s: the JPEG written from the planes differs from libjpeg's own conversion" % what


def all_colours():
    i = np.arange(1 << 24, dtype=np.uint32).reshape(4096, 4096)
    return np.stack([(i >> 16) & 255, (i >> 8) & 255, i & 255], axis=-1).astype(np.uint8)


def test_restatement_is_libjpeg_444_all_colours():
    Image = _pil()
    S = all_colours()
    assert_jpeg_identical(Image, S, [p.astype(np.uint8) for p in ycc_full(S)], 0, "all 2^24 colours, 4:4:4")


def test_restatement_is_libjpeg_420_all_colours():
    Image = _pil()
    S = all_colours()
    Y, Cb, Cr = ycc420(S)
    assert_jpeg_identical(Image, S, [Y, upsample2x2(Cb), upsample2x2(Cr)], 2, "all 2^24 colours, 4:2:0")


@pytest.mark.parametrize("shape", [(64, 96), (128, 208), (48, 160), (256, 336), (16, 16), (112, 400)])
def test_restatement_is_libjpeg_420_random(shape):
    """random images of multiple-of-16 sizes (libjpeg pads partial MCUs from full-resolution chroma, so other sizes differ
    outside the image)"""
    Image = _pil()
    S = np.random.default_rng(shape[0] * 1000 + shape[1]).integers(0, 256, shape + (3,), dtype=np.uint8)
    Y, Cb, Cr = ycc420(S)
    assert_jpeg_identical(Image, S, [Y, upsample2x2(Cb), upsample2x2(Cr)], 2, "random %dx%d" % shape)


def test_restatement_ranges():
    """libjpeg's chroma rounding constant (ONE_HALF - 1) keeps every value of every colour in 0..255"""
    for p in ycc_full(all_colours()):
        assert p.min() >= 0 and p.max() <= 255


def planes_buffers(rows, W, pad):
    """sentinel-filled Y [rows, W + pad[0]] and Cb, Cr [rows/2, W/2 + pad[1]] (the row pitch includes the padding), each
    with as many sentinel guard rows above and below: a row stored in the wrong place changes a guard instead of memory
    outside the test's arrays.  Returns the whole arrays; `inner` gives the planes the develop writes."""
    y = np.full((3 * rows, W + pad[0]), SENTINEL, dtype=np.uint8)
    cb = np.full((3 * (rows // 2), W // 2 + pad[1]), SENTINEL, dtype=np.uint8)
    cr = np.full((3 * (rows // 2), W // 2 + pad[1]), SENTINEL, dtype=np.uint8)
    return y, cb, cr


def inner(bufs):
    return tuple(b[b.shape[0] // 3:2 * b.shape[0] // 3] for b in bufs)


def ycc_args(src, stages, y, cb, cr, pattern="RGGB", black=None, white=None, hdr=False, quality=0, band=None, held=None,
             out_row0=0, **over):
    H, W = src.shape
    rb, re = band or (0, H)
    nscr = (2 if stages >= 2 else 1) * ((re - rb) + 8 * max(stages, 0)) * W * 3
    scratch = np.full(max(nscr, 1), np.nan, dtype=np.float32)
    r0, nr = held or (0, H)
    part = np.ascontiguousarray(src[r0:r0 + nr])
    kw = dict(height=H, width=W, pattern=pattern, in_kind=_capi.IN_U16 if src.dtype == np.uint16 else _capi.IN_F32,
              in_ptr=part.ctypes.data, in_pitch=part.strides[0], in_row0=r0, in_rows=nr, black=black, white=white, wb=WB,
              cam_to_srgb=M, stages=stages, is_hdr=hdr, gamma=False, out_kind=_capi.OUT_YCC420_U8, out_ptr=y.ctypes.data,
              out_pitch=y.strides[0], out_row0=out_row0, row_begin=rb, row_end=re, scratch_ptr=scratch.ctypes.data,
              scratch_bytes=scratch.nbytes, lut_ptr=LUT.ctypes.data, quality=quality, out_cb_ptr=cb.ctypes.data,
              out_cr_ptr=cr.ctypes.data, out_chroma_pitch=cb.strides[0])
    kw.update(over)
    return _capi.fill_develop_args(**kw), (part, scratch)


def emu_ycc(lib, src, stages, bufs, tile, **kw):
    a, keep = ycc_args(src, stages, *inner(bufs), **kw)
    rc = lib.emu_develop(C.byref(a), tile[0], tile[1])
    assert rc == 0, lib.emu_last_error()


def expected_buffers(planes, rows, W, pad, rb, re):
    """sentinel buffers of planes_buffers(rows, W, pad) with Y rows [rb, re) and chroma rows [rb/2, re/2) of `planes`"""
    bufs = planes_buffers(rows, W, pad)
    y, cb, cr = inner(bufs)
    y[rb:re, :W] = planes[0][rb:re]
    cb[rb // 2:re // 2, :W // 2] = planes[1][rb // 2:re // 2]
    cr[rb // 2:re // 2, :W // 2] = planes[2][rb // 2:re // 2]
    return bufs


def assert_planes_equal(got, want, what):
    for name, g, w in zip(("Y", "Cb", "Cr"), got, want):
        if not np.array_equal(g, w):
            bad = np.argwhere(g != w)
            raise AssertionError("%s %s: %d bytes differ; first at %s: %d vs %d" % (
                what, name, len(bad), bad[0].tolist(), g[tuple(bad[0])], w[tuple(bad[0])]))


# row paddings of the planes (bytes): none, word-aligned, and odd pitches that force the byte-by-byte store
PADS = ((0, 0), (4, 2), (3, 1), (8, 5))


@pytest.mark.parametrize("seed", range(N_CASES))
def test_ycc420_matrix_through_emulation(emu, seed):
    """The planes equal the restatement of the emulation's own srgb_u8 output of the same case, byte for byte (padding
    untouched); every band of the case's split, developed from its rows + halo into sentinel-filled full-frame planes,
    writes exactly its rows, equal to the whole frame."""
    c = matrix_case(seed)
    tile = TILES[int(np.random.default_rng(seed).integers(0, len(TILES)))]
    pad = PADS[seed % len(PADS)]
    kw = dict(pattern=c.pattern, hdr=c.hdr, quality=int(c.quality == "fast"))
    if c.kind == "u16":
        kw.update(black=c.black, white=c.white)
    what = describe(c) + " tile=%s pad=%s" % (tile, pad)
    s8 = emu_develop(emu, c.src, c.stages, out_kind=_capi.OUT_SRGB_U8, tile=tile, **kw)
    ref = ycc420(s8)
    got = planes_buffers(c.H, c.W, pad)
    emu_ycc(emu, c.src, c.stages, got, tile, **kw)
    assert_planes_equal(got, expected_buffers(ref, c.H, c.W, pad, 0, c.H), what)
    halo = halo_rows(c)
    for rb, re in zip(c.cuts[:-1], c.cuts[1:]):
        r0, r1 = max(0, rb - halo), min(c.H, re + halo)
        got = planes_buffers(c.H, c.W, pad)
        emu_ycc(emu, c.src, c.stages, got, tile, band=(rb, re), held=(r0, r1 - r0), **kw)
        assert_planes_equal(got, expected_buffers(ref, c.H, c.W, pad, rb, re), "%s band [%d,%d)" % (what, rb, re))


def test_ycc420_band_with_own_rows(emu):
    """a band into planes that start at the band (out_row0 = row_begin), on a flipped frame"""
    c = matrix_case(1)
    src = c.src
    kw = dict(pattern="BGGR", black=c.black, white=c.white) if c.kind == "u16" else dict(pattern="BGGR")
    whole = planes_buffers(c.H, c.W, (0, 0))
    emu_ycc(emu, src, 1, whole, (60, 60), **kw)
    whole = inner(whole)
    rb, re = c.cuts[1], c.H
    got = planes_buffers(re - rb, c.W, (0, 0))
    emu_ycc(emu, src, 1, got, (60, 60), band=(rb, re), out_row0=rb, **kw)
    want = planes_buffers(re - rb, c.W, (0, 0))
    for w, p, r in zip(inner(want), whole, (rb, rb // 2, rb // 2)):
        w[:] = p[r:]
    assert_planes_equal(got, want, "band [%d,%d) out_row0=%d" % (rb, re, rb))


@pytest.mark.parametrize("over", [dict(out_cb_ptr=None), dict(out_cr_ptr=None), dict(out_chroma_pitch=7),
                                  dict(out_row0=1, row_begin=2), dict(out_pitch=15)])
def test_ycc420_invalid_arguments(emu, over):
    """null Cb / Cr plane, chroma pitch below W/2, odd out_row0, Y pitch below W: PYSP_ERR_INVALID from the plan, both in
    the emulation and in the library (the plan runs before any CUDA call)"""
    src = np.zeros((16, 16), dtype=np.float32)
    y, cb, cr = inner(planes_buffers(16, 16, (0, 0)))
    a, keep = ycc_args(src, 0, y, cb, cr, **over)
    assert emu.emu_develop(C.byref(a), 16, 8) == _capi.ERR_INVALID
    assert len(emu.emu_last_error()) > 0
    assert _capi.lib().pysp_develop(C.byref(a), None) == _capi.ERR_INVALID
    ok, keep = ycc_args(src, 0, y, cb, cr)
    assert emu.emu_develop(C.byref(ok), 16, 8) == _capi.OK


def test_other_kinds_ignore_chroma_fields(emu):
    """the appended fields are read for the YCbCr kind only: garbage there changes nothing for srgb_u8"""
    src = np.random.default_rng(3).random((20, 28), dtype=np.float32)
    want = emu_develop(emu, src, 1, out_kind=_capi.OUT_SRGB_U8)
    out = np.zeros((20, 28, 3), dtype=np.uint8)
    y, cb, cr = inner(planes_buffers(20, 28, (0, 0)))
    a, keep = ycc_args(src, 1, y, cb, cr, out_kind=_capi.OUT_SRGB_U8, out_ptr=out.ctypes.data, out_pitch=out.strides[0],
                       out_cb_ptr=None, out_cr_ptr=8, out_chroma_pitch=-5)
    assert emu.emu_develop(C.byref(a), 16, 8) == _capi.OK
    assert np.array_equal(out, want)
