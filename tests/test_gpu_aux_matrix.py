"""The steps either side of the develop path and the normalisation, through the C ABI, across the shapes, pitches, alignments,
aliasing, NULL pointers and edge values where their kernels switch code paths: flat-field correction (vector / scalar
path, plane means above 2^24 sites), hot-pixel detection (aligned / unaligned interior loads, word / byte mask stores),
camera-space fusion (whole / partial work items), raw-space fusion (both fuse_kernel instantiations) and bayer_normalize.
Bit for bit against the oracle (NaN at the same places where it can occur); every seeded case names its parameters when it
fails."""
import ctypes as C
import itertools

import numpy as np
import pytest
import torch

from conftest import assert_bit_equal, assert_bit_equal_nan
from oracle import ahd_spec as sp
from oracle import aux_spec as ax
from pysp_b200 import synthetic as syn

pytestmark = pytest.mark.gpu
f32 = np.float32
SENTINEL = -12345.0           # float32 value of every byte a call must not write


@pytest.fixture(scope="module")
def L():
    from pysp_b200 import _capi
    assert torch.cuda.is_available(), "these tests need the GPU"
    return _capi.lib()


def stream():
    return torch.cuda.current_stream().cuda_stream


class Buf:
    """A 2-D array in device memory at a chosen pitch (elements) and base offset (elements) inside a larger allocation
    filled with a sentinel: `ptr`, `pitch` (bytes); `read()` returns the [rows, cols] view, `untouched()` checks that
    nothing outside it was written."""

    def __init__(self, a, pitch=None, offset=0, fill=SENTINEL):
        a = np.ascontiguousarray(a)
        self.rows, self.cols = a.shape
        self.pitch_elems = self.cols if pitch is None else pitch
        assert self.pitch_elems >= self.cols
        dt = {np.dtype(np.float32): torch.float32, np.dtype(np.int32): torch.int32, np.dtype(np.uint8): torch.uint8,
              np.dtype(np.uint16): torch.int16}[a.dtype]
        n = offset + self.rows * self.pitch_elems + 8
        self.base = torch.full((n,), fill, dtype=dt, device="cuda")
        self.view = self.base[offset:offset + self.rows * self.pitch_elems].view(self.rows, self.pitch_elems)[:, :self.cols]
        src = a.view(np.int16) if a.dtype == np.uint16 else a
        self.view.copy_(torch.from_numpy(src))
        self.before = self.base.clone()
        self.mask = torch.ones(n, dtype=torch.bool, device="cuda")
        self.mask[offset:offset + self.rows * self.pitch_elems].view(self.rows, self.pitch_elems)[:, :self.cols] = False
        self.ptr = self.view.data_ptr()
        self.pitch = self.pitch_elems * self.base.element_size()
        self.dtype = a.dtype

    def read(self):
        v = self.view.cpu().numpy()
        return v.view(np.uint16) if self.dtype == np.uint16 else v

    def untouched(self):
        return torch.equal(self.base[self.mask], self.before[self.mask])


def f32ptr(vals):
    vals = [float(v) for v in vals]
    return (C.c_float * len(vals))(*vals)


# ---------------------------------------------------------------------------------------------------------------------
# plane means and flat field
# ---------------------------------------------------------------------------------------------------------------------
def call_flat(L, s, f, o, H, W, clamp, ws_bytes=None):
    nws = int(L.pysp_flat_workspace_bytes(H, W)) if ws_bytes is None else ws_bytes
    ws = torch.empty(max(nws, 1), dtype=torch.uint8, device="cuda")
    rc = L.pysp_flat_frame_correction(s.ptr, s.pitch, f.ptr, f.pitch, o.ptr, o.pitch, H, W, int(clamp), ws.data_ptr(), nws,
                                      stream())
    torch.cuda.synchronize()
    return rc


def test_flat_frame_correction_100mp(L):
    """8662 x 11550: 25 011 525 sites per plane, above 2^24, where float32(n) != n.  The means must be np.mean's."""
    from pysp_b200 import engine
    flat = np.random.default_rng(0).random((8662, 11550), dtype=f32)
    sensor = np.random.default_rng(1).random((8662, 11550), dtype=f32)
    got = engine.flat_frame_correction(engine.to_device(sensor), engine.to_device(flat)).cpu().numpy()
    assert_bit_equal_nan(got, ax.flat_frame_correction(sensor, flat), "100 MP flat-field correction")


FLAT_LAYOUTS = ["contig", "pad16", "pad_odd", "unaligned", "alias"]
FLAT_CASES = list(itertools.product([0, 2], FLAT_LAYOUTS, [0, 1]))


@pytest.mark.parametrize("wmod,layout,clamp", FLAT_CASES)
def test_flat_frame_correction_matrix(L, wmod, layout, clamp):
    seed = FLAT_CASES.index((wmod, layout, clamp))
    rng = np.random.default_rng(100 + seed)
    H = 2 * int(rng.integers(1, 40))
    W = 4 * int(rng.integers(1, 40)) + wmod
    what = "flat seed=%d H=%d W=%d layout=%s clamp=%d" % (seed, H, W, layout, clamp)
    sensor = rng.uniform(-0.1, 1.2, size=(H, W)).astype(f32)
    flat = rng.uniform(0.3, 1.0, size=(H, W)).astype(f32)
    pick = lambda p: rng.random((H, W)) < p                          # noqa: E731
    flat[pick(0.05)] = 0.0                                           # x / 0 = +-inf, 0 / 0 = NaN
    flat[pick(0.03)] *= -1.0                                         # negative quotients -> 0
    sensor[pick(0.03)] = 0.0
    if seed % 5 == 4:
        flat[pick(0.01)] = np.nan                                    # the plane's mean becomes NaN
    else:
        sensor[pick(0.02)] = np.nan
    # one special plane.  A flat plane of zeros has mean 0, so every quotient is 0 / 0 = NaN (variant 3); +-inf quotients
    # everywhere need a non-zero mean: a few flat sites of 1 under +inf photosites, zeros elsewhere (variant 1: all
    # infinite, copied unchanged); NaN photosites over those sites and zero photosites among the rest mix NaN = 0 / 0 and
    # x / 0 = +inf without any finite quotient (variant 2: +inf becomes NaN)
    variant = seed % 4
    if variant:
        py, px = [(0, 0), (0, 1), (1, 1), (1, 0)][(seed // 4) % 4]     # R, G1, B, G2
        fp, sp_ = flat[py::2, px::2], sensor[py::2, px::2]
        fp[...] = 0.0
        sp_[...] = rng.uniform(0.1, 1.0, size=sp_.shape).astype(f32)
        sp_[0, 0] = -0.5                                             # -inf
        if variant in (1, 2):
            few = rng.random(fp.shape) < 0.1
            few.flat[-1] = True
            fp[few] = 1.0
            sp_[few] = np.inf if variant == 1 else np.nan
        if variant == 2:
            sp_[(rng.random(fp.shape) < 0.3) & ~few] = 0.0
    want = ax.flat_frame_correction(sensor, flat, bool(clamp))
    pads = {"contig": (0, 0, 0), "pad16": (4, 8, 12), "pad_odd": (1, 3, 2), "unaligned": (0, 0, 0), "alias": (4, 4, 4)}[layout]
    off = 1 if layout == "unaligned" else 0
    s = Buf(sensor, W + pads[0], off)
    f = Buf(flat, W + pads[1], off)
    o = s if layout == "alias" else Buf(np.zeros((H, W), f32), W + pads[2], off)
    assert call_flat(L, s, f, o, H, W, clamp) == 0, what
    assert_bit_equal_nan(o.read(), want, what)
    assert s.untouched() and f.untouched() and o.untouched(), what + ": wrote outside the image"
    if layout != "alias":
        assert_bit_equal(s.read(), sensor, what + ": sensor changed")
    assert_bit_equal(f.read(), flat, what + ": flat changed")


def test_flat_workspace_one_byte_short(L):
    from pysp_b200 import _capi
    H, W = 34, 50
    a = np.random.default_rng(7).random((H, W), dtype=f32)
    s, f, o = Buf(a), Buf(a + f32(0.5)), Buf(np.zeros((H, W), f32))
    nws = int(L.pysp_flat_workspace_bytes(H, W))
    assert call_flat(L, s, f, o, H, W, 0, nws - 1) == _capi.ERR_INVALID
    ws = torch.empty(nws, dtype=torch.uint8, device="cuda")
    means = torch.empty(4, dtype=torch.float32, device="cuda")
    assert L.pysp_bayer_plane_means(s.ptr, s.pitch, H, W, means.data_ptr(), ws.data_ptr(), nws - 1, stream()) == _capi.ERR_INVALID
    assert L.pysp_bayer_plane_means(s.ptr, s.pitch, H, W, means.data_ptr(), ws.data_ptr(), nws, stream()) == 0
    evens, odds = a[0::2].astype(f32), a[1::2].astype(f32)
    want = [np.mean(evens[:, 0::2]), np.mean(evens[:, 1::2]), np.mean(odds[:, 1::2]), np.mean(odds[:, 0::2])]
    assert_bit_equal(means.cpu().numpy(), np.array(want, f32), "plane means after a refused call")


def test_plane_means_padded_unaligned(L):
    """pysp_bayer_plane_means on a padded, unaligned mosaic (odd pitch in floats, base 4 bytes off)"""
    for seed, (H, W) in enumerate([(2, 2), (2, 258), (6, 10), (130, 70), (1000, 1502)]):
        a = np.random.default_rng(200 + seed).random((H, W), dtype=f32)
        b = Buf(a, W + 3, 1)
        nws = int(L.pysp_flat_workspace_bytes(H, W))
        ws = torch.empty(nws, dtype=torch.uint8, device="cuda")
        means = torch.empty(4, dtype=torch.float32, device="cuda")
        assert L.pysp_bayer_plane_means(b.ptr, b.pitch, H, W, means.data_ptr(), ws.data_ptr(), nws, stream()) == 0
        evens, odds = a[0::2].astype(f32), a[1::2].astype(f32)
        want = [np.mean(evens[:, 0::2]), np.mean(evens[:, 1::2]), np.mean(odds[:, 1::2]), np.mean(odds[:, 0::2])]
        assert_bit_equal(means.cpu().numpy(), np.array(want, f32), "plane means %dx%d, padded and unaligned" % (H, W))


# ---------------------------------------------------------------------------------------------------------------------
# hot pixels
# ---------------------------------------------------------------------------------------------------------------------
HOT_LAYOUTS = ["contig", "pitch8_4", "row_offset", "mask_offset"]
HOT_CASES = list(itertools.product(["h2", "h3", "big"], [0, 1, 2, 3], HOT_LAYOUTS))


@pytest.mark.parametrize("hkind,wmod,layout", HOT_CASES)
def test_hot_pixels_matrix(L, hkind, wmod, layout):
    seed = HOT_CASES.index((hkind, wmod, layout))
    rng = np.random.default_rng(300 + seed)
    h = {"h2": 2, "h3": 3, "big": int(rng.integers(3, 24))}[hkind]
    w = 4 * int(rng.integers(1 if wmod else 2, 10)) + wmod          # w >= 2; interior items need w >= 9
    H, W = 2 * h, 2 * w
    min_count = [-1, 0, 4, 7, 8][seed % 5]
    min_delta = [-0.1, 0.0, 0.01][seed % 3]
    what = "hot seed=%d H=%d W=%d layout=%s min_count=%d min_delta=%g" % (seed, H, W, layout, min_count, min_delta)
    sensor = (rng.integers(0, 6, size=(H, W)) / 8.0).astype(f32)     # coarse levels: ties with the neighbours
    sensor[rng.random((H, W)) < 0.08] = f32(1.5)                     # hot
    sensor[rng.random((H, W)) < 0.03] = np.nan
    sensor[rng.random((H, W)) < 0.02] = np.inf
    sensor[rng.random((H, W)) < 0.02] = -np.inf
    want = np.stack(ax.find_erroneous_pixels_threshold(sensor, min_delta, min_count)).astype(np.uint8)
    pitch = W + 1 if layout == "pitch8_4" else W                     # pitch % 8 == 4 bytes
    s = Buf(sensor, pitch, 1 if layout == "row_offset" else 0)
    m = Buf(np.zeros((4 * h, w), np.uint8), None, 1 if layout == "mask_offset" else 0, fill=0xAB)
    rc = L.pysp_find_hot_pixels_threshold(s.ptr, s.pitch, H, W, C.c_float(min_delta), min_count, m.ptr, stream())
    torch.cuda.synchronize()
    assert rc == 0, what
    got = m.read().reshape(4, h, w)
    bad = np.argwhere(got != want)
    assert bad.size == 0, "%s: %d masks differ, first (plane, qy, qx) %s" % (what, len(bad), bad[:3].tolist())
    assert m.untouched() and s.untouched(), what + ": wrote outside the masks"


# ---------------------------------------------------------------------------------------------------------------------
# camera-space fusion
# ---------------------------------------------------------------------------------------------------------------------
CAM_LAYOUTS = ["aligned", "img_off", "out_off", "count_off", "count_null"]
CAM_CASES = list(itertools.product([1, 2, 5, 16], [0, 1, 2, 3], CAM_LAYOUTS))


def cam_exposures(rng, n, npx, wb):
    evs = [float(e) for e in np.round(rng.uniform(8.0, 13.0, size=n), 2)]
    if n >= 2:                                          # equal top EVs, different images: the last one is the brightest
        top = max(evs)
        evs[int(rng.integers(0, n - 1))] = top
        evs[n - 1] = top
    base = rng.uniform(0.0, 1.2, size=(npx, 3)).astype(f32)
    imgs = []
    for i in range(n):
        im = np.minimum(base * f32(2.0 ** (10.0 - evs[i])) * wb * f32(1.0 + 0.1 * i), wb).astype(f32)
        r = rng.random(npx)
        im[r < 0.05] = 0.0
        im[(r >= 0.05) & (r < 0.1)] = wb                # saturated (weight 0)
        im[(r >= 0.1) & (r < 0.13)] *= -1.0
        im[(r >= 0.13) & (r < 0.15), int(rng.integers(0, 3))] = np.nan
        k = min(3, npx)
        im[:k] = np.where(rng.random((k, 1)) < 0.5, wb, 0.0)   # every weight 0 in every exposure: the brightest fallback
        imgs.append(im)
    return evs, imgs


@pytest.mark.parametrize("n,pmod,layout", CAM_CASES)
def test_fuse_from_debayer_matrix(L, n, pmod, layout):
    seed = CAM_CASES.index((n, pmod, layout))
    rng = np.random.default_rng(400 + seed)
    npx = 4 * int(rng.integers(1, 60)) + pmod
    write_back = seed % 2
    wb = syn.wb_multipliers().astype(f32)
    norm = [bool(v) for v in rng.random(n) < 0.5]
    m = sp.cam_to_lin_srgb_matrix(syn.MAT_XYZ_TO_CAM, syn.WHITE_XYZ)
    evs, imgs = cam_exposures(rng, n, npx, wb)
    what = "fuse_cam seed=%d n=%d n_px=%d layout=%s write_back=%d normalized=%s" % (seed, n, npx, layout, write_back, norm)
    # normalised exposures are stored divided by max(wb) (image_base.py:56-57 multiplies them back)
    stored = [(im / np.max(wb)).astype(f32) if nz else im for im, nz in zip(imgs, norm)]
    want_lin, want_cnt, left = ax.fuse_exposures_from_debayer([s.copy() for s in stored], evs, wb, m, norm)
    tgt = sum(evs) / n
    offs = [2 ** (e - tgt) for e in evs]
    off_max = float(np.max(offs))
    brightest = max(i for i, o in enumerate(offs) if o == off_max)
    bufs = [Buf(s.reshape(-1, 3).reshape(1, -1), None, 3 if (layout == "img_off" and i == n - 1) else 0)
            for i, s in enumerate(stored)]
    out = Buf(np.zeros((1, 3 * npx), f32), None, 3 if layout == "out_off" else 0)
    cnt = None if layout == "count_null" else Buf(np.zeros((1, 3 * npx), np.int32), None, 3 if layout == "count_off" else 0,
                                                   fill=-7)
    ptrs = (C.c_void_p * n)(*[b.ptr for b in bufs])
    md = (C.c_double * 9)(*[float(v) for v in np.asarray(m, np.float64).reshape(-1)])
    rc = L.pysp_fuse_exposures_from_debayer(ptrs, n, npx, f32ptr(wb), C.c_float(float(np.max(wb))),
                                            (C.c_int32 * n)(*[int(v) for v in norm]), f32ptr([f32(o) for o in offs]),
                                            f32ptr([f32(1.6 ** (-0.1 * o)) for o in offs]), brightest, off_max, md, out.ptr,
                                            cnt.ptr if cnt else None, write_back, stream())
    torch.cuda.synchronize()
    assert rc == 0, what
    assert_bit_equal_nan(out.read().reshape(npx, 3), want_lin, what + ": linear sRGB")
    assert out.untouched(), what + ": wrote outside the output"
    if cnt is not None:
        got_cnt = cnt.read().reshape(npx, 3)
        assert np.array_equal(got_cnt, want_cnt), "%s: counts differ at %s" % (what, np.argwhere(got_cnt != want_cnt)[:3].tolist())
        assert cnt.untouched(), what + ": wrote outside the counts"
    for i, b in enumerate(bufs):
        img = b.read().reshape(npx, 3)
        if write_back:
            assert_bit_equal_nan(img, left[i], what + ": exposure %d after the round trip" % i)
        else:
            assert_bit_equal(img, stored[i], what + ": exposure %d changed without write_back" % i)
        assert b.untouched(), what + ": wrote outside exposure %d" % i


def test_fuse_from_debayer_rejects_17(L):
    from pysp_b200 import _capi
    n = 17
    bufs = [torch.zeros(12, dtype=torch.float32, device="cuda") for _ in range(n)]
    out = torch.zeros(12, dtype=torch.float32, device="cuda")
    ptrs = (C.c_void_p * n)(*[b.data_ptr() for b in bufs])
    md = (C.c_double * 9)(*([1.0, 0, 0, 0, 1.0, 0, 0, 0, 1.0]))
    rc = L.pysp_fuse_exposures_from_debayer(ptrs, n, 4, f32ptr([2.0, 1.0, 1.5]), C.c_float(2.0), None, f32ptr([1.0] * n),
                                            f32ptr([1.0] * n), 0, 1.0, md, out.data_ptr(), None, 1, stream())
    assert rc == _capi.ERR_INVALID


# ---------------------------------------------------------------------------------------------------------------------
# raw-space fusion
# ---------------------------------------------------------------------------------------------------------------------
RAW_LAYOUTS = ["contig", "pad16", "pad_odd"]
RAW_CASES = list(itertools.product([1, 3, 16], [0, 2], RAW_LAYOUTS, [True, False]))


@pytest.mark.parametrize("n,wmod,layout,with_count", RAW_CASES)
def test_fuse_raw_matrix(L, n, wmod, layout, with_count):
    from pysp_b200.raw_hdr import fusion_constants
    seed = RAW_CASES.index((n, wmod, layout, with_count))
    rng = np.random.default_rng(500 + seed)
    H = 2 * int(rng.integers(1, 30))
    W = 4 * int(rng.integers(1, 30)) + wmod
    what = "fuse_raw seed=%d n=%d H=%d W=%d layout=%s count=%s" % (seed, n, H, W, layout, with_count)
    wb = syn.wb_multipliers()
    evs = [float(e) for e in np.round(rng.uniform(8.0, 13.0, size=n), 2)]
    base = rng.uniform(0.0, 1.3, size=(H, W)).astype(f32)
    brackets = []
    for i in range(n):
        b = np.clip(base * f32(2.0 ** (10.0 - evs[i])) + rng.normal(0, 0.01, (H, W)).astype(f32), 0, 1).astype(f32)
        r = rng.random((H, W))
        b[r < 0.05] = 1.0                               # clipped
        b[(r >= 0.05) & (r < 0.1)] = 0.0
        b[(r >= 0.1) & (r < 0.12)] = np.nan
        b[:2, :2] = 1.0 if i % 2 else 0.0               # weight 0 in every bracket: the brightest fallback
        brackets.append(b)
    want, want_cnt, _, _ = sp.fuse_exposures(brackets, evs, wb)
    _, offs, bias = fusion_constants(evs, wb)
    pads = {"contig": (0, 0, 0), "pad16": (4, 8, 12), "pad_odd": (1, 3, 5)}[layout]
    ins = [Buf(b, W + pads[0]) for b in brackets]
    out = Buf(np.zeros((H, W), f32), W + pads[1])
    cnt = Buf(np.zeros((H, W), np.int32), W + pads[2], fill=-7) if with_count else None
    ptrs = (C.c_void_p * n)(*[b.ptr for b in ins])
    rc = L.pysp_fuse_exposures(ptrs, n, ins[0].pitch, H, W, f32ptr(offs), f32ptr(np.asarray(bias, f32).reshape(-1)),
                               int(np.argmax(offs)), out.ptr, out.pitch, cnt.ptr if cnt else None, cnt.pitch if cnt else 0,
                               stream())
    torch.cuda.synchronize()
    assert rc == 0, what
    assert_bit_equal_nan(out.read(), want, what)
    assert out.untouched(), what + ": wrote outside the output"
    if cnt is not None:
        assert np.array_equal(cnt.read(), want_cnt), what + ": counts"
        assert cnt.untouched(), what + ": wrote outside the counts"


def test_fuse_raw_rejects_17(L):
    from pysp_b200 import _capi
    n = 17
    bufs = [torch.zeros((4, 4), dtype=torch.float32, device="cuda") for _ in range(n)]
    out = torch.zeros((4, 4), dtype=torch.float32, device="cuda")
    ptrs = (C.c_void_p * n)(*[b.data_ptr() for b in bufs])
    rc = L.pysp_fuse_exposures(ptrs, n, 16, 4, 4, f32ptr([1.0] * n), f32ptr([1.0] * 3 * n), 0, out.data_ptr(), 16, None, 0,
                               stream())
    assert rc == _capi.ERR_INVALID


# ---------------------------------------------------------------------------------------------------------------------
# normalisation
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("W,in_off,out_pad", [(512, 0, 0), (514, 0, 0), (512, 1, 0), (514, 1, 3), (512, 0, 4)])
def test_normalize_all_codes(L, W, in_off, out_pad):
    """every 16-bit code at every CFA site, four distinct black / white levels; W % 8 in {0, 2}; base 2 bytes off"""
    H = 512
    rng = np.random.default_rng(600 + W + in_off + out_pad)
    raw = np.empty((H, W), np.uint16)
    for py, px in ((0, 0), (0, 1), (1, 1), (1, 0)):
        n = (H // 2) * (W // 2)
        codes = np.concatenate([np.arange(65536), rng.integers(0, 65536, n - 65536)]).astype(np.uint16)
        raw[py::2, px::2] = rng.permutation(codes).reshape(H // 2, W // 2)
    black = [512.0, 1023.5, 64.0, 2048.0]                       # R, G1, B, G2
    white = [16383.0, 15000.0, 65535.0, 4095.0]
    what = "normalize W=%d in_off=%d out_pad=%d" % (W, in_off, out_pad)
    s = Buf(raw, None, in_off, fill=0x5A5A)
    o = Buf(np.zeros((H, W), f32), W + out_pad)
    rc = L.pysp_normalize_u16(s.ptr, s.pitch, o.ptr, o.pitch, H, W, f32ptr(black), f32ptr(white), stream())
    torch.cuda.synchronize()
    assert rc == 0, what
    assert_bit_equal(o.read(), sp.normalize(raw, black, white), what)
    assert o.untouched(), what + ": wrote outside the output"
