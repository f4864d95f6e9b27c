"""The input matrix of the develop kernels through the host emulation (tests/host_emu) against the oracle: float32, HDR and
u16 mosaics, QualityDemosaic.Best at 0-3 stages and Fast, on every CFA pattern, ragged frame sizes (widths 0 and 2 mod 4),
random tile sizes and random row bands.  Also the wire formats: srgb_u8 / srgb_u16 are the float32 gamma output of the
same case rounded to nearest (the emulation has no half conversion; lin_f16 is checked on the GPU only).

`matrix_case` / `matrix_reference` also feed tests/test_gpu_develop_matrix.py, which runs the same cases on the device."""
import collections

import numpy as np
import pytest

from oracle import ahd_spec as sp
from pysp_b200 import _capi
from pysp_b200 import synthetic as syn
from conftest import assert_bit_equal
from test_tile_logic import M, WB, emu, emu_develop  # noqa: F401  (emu is a fixture)

PATTERNS = ("RGGB", "BGGR", "GRBG", "GBRG")
KINDS = ("u16", "f32", "hdr")
ALGOS = ((0, "best"), (1, "best"), (2, "best"), (3, "best"), (0, "fast"))     # (stages, quality)
N_CASES = 32
TILES = ((16, 8), (20, 8), (60, 28), (60, 60), (56, 30), (60, 44))
QUANT = ((_capi.OUT_SRGB_U8, 255.0, np.uint8), (_capi.OUT_SRGB_U16, 65535.0, np.uint16))

Case = collections.namedtuple("Case", "seed H W pattern kind stages quality src black white hdr cuts")


def matrix_case(seed, max_side=300):
    """Seeded case: pattern, input kind, algorithm and width mod 4 follow the seed so that, over the N_CASES seeds, every
    pair of them occurs; the sizes (even, 4 .. max_side, a quarter of them below 24) and the band cuts are random."""
    rng = np.random.default_rng(700 + seed)
    pattern = PATTERNS[seed % 4]
    kind = KINDS[(seed // 4) % 3]
    stages, quality = ALGOS[seed % 5]
    side = lambda: 24 if rng.random() < 0.25 else max_side
    H = 2 * int(rng.integers(2, side() // 2 + 1))
    W = 4 * int(rng.integers(1, side() // 4 + 1)) + 2 * ((seed // 3) % 2)
    black = white = None
    if kind == "u16":
        black = tuple(int(v) for v in rng.integers(400, 600, 4))
        white = tuple(int(v) for v in rng.integers(15000, 16384, 4))
        src = syn.random_mosaic(H, W, 800 + seed) if seed % 3 == 0 else syn.scene(H, W, 800 + seed)
    else:
        src = syn.scene(H, W, 800 + seed).astype(np.float32) / np.float32(16383.0)
        if kind == "hdr":                     # about 20 % of the sites above 1, as a fused HDR mosaic has them
            src = (src * np.where(rng.random((H, W)) < 0.2, np.float32(3.0), np.float32(1.0))).astype(np.float32)
    cuts = sorted(set([0, H] + [2 * int(v) for v in rng.integers(1, H // 2, size=min(3, H // 2 - 1))])) if H > 4 else [0, H]
    return Case(seed, H, W, pattern, kind, stages, quality, src, black, white, kind == "hdr", cuts)


def matrix_reference(c):
    """(cam, lin, pick_h) of the oracle; pick_h (the AHD direction map, stored orientation) is None for Fast."""
    if c.kind == "u16":
        if c.quality == "fast":
            lin, cam = sp.develop_fast(c.src, c.black, c.white, WB, syn.MAT_XYZ_TO_CAM, syn.WHITE_XYZ, c.pattern)
            return cam, lin, None
        lin, cam, ex = sp.develop(c.src, c.black, c.white, WB, syn.MAT_XYZ_TO_CAM, syn.WHITE_XYZ, c.stages, c.pattern, keep=True)
        return cam, lin, np.ascontiguousarray(sp.to_rggb(ex["pick_h"], c.pattern))
    s = sp.to_rggb(c.src, c.pattern)
    pick = None
    if c.quality == "fast":
        cam = sp.eag_demosaic(s, WB)
    else:
        cam, ex = sp.ahd_demosaic(s, WB, M, c.stages, hdr=c.hdr, keep=True)
        pick = np.ascontiguousarray(sp.to_rggb(ex["pick_h"], c.pattern))
    cam = np.ascontiguousarray(sp.to_rggb(cam, c.pattern))
    return cam, sp.to_lin_srgb(cam, M), pick


def halo_rows(c):
    return 6 + 4 * (c.stages if c.quality == "best" else 0)


def quantised(g, scale, dtype):
    """the wire formats' rounding: round half to even of clip(g, 0, 1) * scale (exact in float64), NaN -> 0"""
    g = np.asarray(g, dtype=np.float32).astype(np.float64)
    return np.rint(np.clip(np.where(np.isnan(g), 0.0, g), 0.0, 1.0) * scale).astype(dtype)


def describe(c):
    return "case %d: %dx%d %s %s %s stages=%d" % (c.seed, c.H, c.W, c.pattern, c.kind, c.quality, c.stages)


@pytest.mark.parametrize("seed", range(N_CASES))
def test_matrix_through_emulation(emu, seed):
    """Whole frame against the oracle (camera RGB and linear sRGB), every band (its rows + halo only) against the whole
    frame; srgb_u8 / srgb_u16 exactly the quantised float32 gamma output, on the whole frame and on every band."""
    c = matrix_case(seed)
    cam, lin, _ = matrix_reference(c)
    tile = TILES[int(np.random.default_rng(seed).integers(0, len(TILES)))]
    kw = dict(pattern=c.pattern, tile=tile, hdr=c.hdr, quality=int(c.quality == "fast"))
    if c.kind == "u16":
        kw.update(black=c.black, white=c.white)
    what = describe(c) + " tile=%s" % (tile,)
    assert_bit_equal(emu_develop(emu, c.src, c.stages, out_kind=_capi.OUT_CAM_F32, **kw), cam, what + " cam")
    whole = emu_develop(emu, c.src, c.stages, **kw)
    assert_bit_equal(whole, lin, what + " lin")
    g = emu_develop(emu, c.src, c.stages, gamma=True, **kw)
    for kind, scale, dt in QUANT:
        assert np.array_equal(emu_develop(emu, c.src, c.stages, out_kind=kind, **kw), quantised(g, scale, dt)), what + " kind %d" % kind
    halo = halo_rows(c)
    for rb, re in zip(c.cuts[:-1], c.cuts[1:]):
        r0, r1 = max(0, rb - halo), min(c.H, re + halo)
        bk = dict(kw, band=(rb, re), held=(r0, r1 - r0))
        band = "%s band [%d,%d)" % (what, rb, re)
        assert_bit_equal(emu_develop(emu, c.src, c.stages, **bk), whole[rb:re], band + " lin")
        for kind, scale, dt in QUANT:
            assert np.array_equal(emu_develop(emu, c.src, c.stages, out_kind=kind, **bk), quantised(g[rb:re], scale, dt)), \
                band + " kind %d" % kind
