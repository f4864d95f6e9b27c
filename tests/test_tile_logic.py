"""Tile logic of the CUDA kernels, run through the host emulation (tests/host_emu) against the oracle:
tiling, halos, the six border rules, partial tiles, CFA flips, row bands, HDR.  The emulation compiles the
very same tile functions as the CUDA build (see tests/host_emu/emu.cpp); it is test infrastructure only."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, assert_bit_equal
from oracle import ahd_spec as sp
from pysp_b200 import _capi
from pysp_b200 import synthetic as syn

EMU_DIR = os.path.join(ROOT, "tests", "host_emu")
WB = syn.wb_multipliers()
M = sp.cam_to_lin_srgb_matrix(syn.MAT_XYZ_TO_CAM, syn.WHITE_XYZ)


@pytest.fixture(scope="module")
def emu():
    so = os.path.join(EMU_DIR, "libpysp_emu.so")
    srcs = [os.path.join(EMU_DIR, "emu.cpp")] + [os.path.join(ROOT, "pysp_b200", "csrc", f)
                                                 for f in os.listdir(os.path.join(ROOT, "pysp_b200", "csrc"))]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        if not os.path.exists("/usr/bin/g++"):
            pytest.skip("g++ not available")
        subprocess.check_call([os.path.join(EMU_DIR, "build.sh")])
    lib = C.CDLL(so)
    lib.emu_develop.argtypes = [C.POINTER(_capi.DevelopArgs), C.c_int, C.c_int]
    lib.emu_last_error.restype = C.c_char_p
    return lib


def packed_lut():
    """the device layout of the Lab table, produced by the library's own (host-side) packer"""
    from pysp_b200 import build
    build.build()
    L = _capi.lib()
    lut = np.ascontiguousarray(np.load(os.path.join(ROOT, "pysp_b200", "data", "lab_lut33_i16.npy")).astype(np.int16))
    p = np.zeros(int(L.pysp_lab_lut_bytes()), dtype=np.uint8)
    assert L.pysp_lab_lut_pack_host(lut.ctypes.data, p.ctypes.data) == 0
    return p


LUT = packed_lut()


OUT_DTYPES = {_capi.OUT_CAM_F32: np.float32, _capi.OUT_LIN_F32: np.float32, _capi.OUT_LIN_F16: np.float16,
              _capi.OUT_SRGB_U8: np.uint8, _capi.OUT_SRGB_U16: np.uint16}


def emu_develop(lib, src, stages, pattern="RGGB", tile=(16, 8), black=syn.BLACK, white=syn.WHITE,
                out_kind=_capi.OUT_LIN_F32, band=None, hdr=False, held=None, quality=0, gamma=False):
    """src: uint16 counts or float32 sensor; `held` = (row0, rows) keeps only that slice of the frame."""
    H, W = src.shape
    rb, re = band or (0, H)
    dt = OUT_DTYPES[out_kind]
    out = np.full((re - rb, W, 3), np.nan if dt == np.float32 else 0xA5, dtype=dt)
    nscr = (2 if stages >= 2 else 1) * ((re - rb) + 8 * max(stages, 0)) * W * 3
    scratch = np.full(max(nscr, 1), np.nan, dtype=np.float32)
    r0, nr = held or (0, H)
    part = np.ascontiguousarray(src[r0:r0 + nr])
    a = _capi.fill_develop_args(H, W, pattern, _capi.IN_U16 if src.dtype == np.uint16 else _capi.IN_F32,
                                part.ctypes.data, part.strides[0], r0, nr, black, white, WB, M, stages, hdr, gamma,
                                out_kind, out.ctypes.data, out.strides[0], rb, rb, re, scratch.ctypes.data,
                                scratch.nbytes, LUT.ctypes.data, quality=quality)
    rc = lib.emu_develop(C.byref(a), tile[0], tile[1])
    assert rc == 0, lib.emu_last_error()
    return out


@pytest.mark.parametrize("shape", [(4, 6), (8, 8), (10, 14), (34, 50), (40, 130)])
@pytest.mark.parametrize("stages", [0, 1, 2])
def test_frames(emu, shape, stages):
    raw = syn.scene(shape[0], shape[1], 3) if shape[0] > 10 else syn.random_mosaic(shape[0], shape[1], 3)
    lin, cam = sp.develop(raw, syn.BLACK, syn.WHITE, WB, syn.MAT_XYZ_TO_CAM, syn.WHITE_XYZ, stages)
    for tile in ((16, 8), (20, 8), (60, 28), (60, 60)):
        assert_bit_equal(emu_develop(emu, raw, stages, tile=tile), lin, "lin %s" % (tile,))
        assert_bit_equal(emu_develop(emu, raw, stages, tile=tile, out_kind=_capi.OUT_CAM_F32), cam, "cam %s" % (tile,))


@pytest.mark.parametrize("pattern", ["RGGB", "BGGR", "GRBG", "GBRG"])
def test_patterns_and_levels(emu, pattern):
    raw = syn.scene(36, 52, 6)
    black, white = (500, 510, 520, 530), (16383, 16000, 15800, 16100)
    lin, _ = sp.develop(raw, black, white, WB, syn.MAT_XYZ_TO_CAM, syn.WHITE_XYZ, 1, pattern)
    assert_bit_equal(emu_develop(emu, raw, 1, pattern, black=black, white=white), lin, pattern)


@pytest.mark.parametrize("pattern", ["RGGB", "GRBG"])
@pytest.mark.parametrize("stages", [0, 1, 2])
def test_row_bands_equal_whole_frame(emu, stages, pattern):
    """A band developed from only its rows + halo is bit-identical to the same rows of the whole frame."""
    raw = syn.scene(64, 40, 7)
    whole = emu_develop(emu, raw, stages, pattern)
    halo = 6 + 4 * stages
    for rb, re in ((0, 20), (20, 44), (44, 64)):
        r0, r1 = max(0, rb - halo), min(64, re + halo)
        band = emu_develop(emu, raw, stages, pattern, band=(rb, re), held=(r0, r1 - r0))
        assert_bit_equal(band, whole[rb:re], "band [%d,%d)" % (rb, re))


@pytest.mark.parametrize("seed", range(12))
def test_ragged_frames_and_bands(emu, seed):
    """Seeded random cases: ragged even frame sizes (down to 4x4, widths that are 2 mod 4, not multiples of any tile size),
    every CFA pattern, per-site levels, 0-3 stages, random tile size and a random split into row bands -- whole frame
    against the oracle, every band against the whole frame."""
    rng = np.random.default_rng(100 + seed)
    H, W = 2 * int(rng.integers(2, 50)), 2 * int(rng.integers(2, 60))
    stages = int(rng.integers(0, 4))
    pattern = ("RGGB", "BGGR", "GRBG", "GBRG")[int(rng.integers(0, 4))]
    black = tuple(int(v) for v in rng.integers(400, 600, 4))
    white = tuple(int(v) for v in rng.integers(15000, 16384, 4))
    tile = ((16, 8), (20, 8), (60, 28), (60, 60), (56, 30))[int(rng.integers(0, 5))]
    raw = syn.random_mosaic(H, W, 200 + seed) if seed % 3 == 0 else syn.scene(H, W, 200 + seed)
    lin, _ = sp.develop(raw, black, white, WB, syn.MAT_XYZ_TO_CAM, syn.WHITE_XYZ, stages, pattern)
    whole = emu_develop(emu, raw, stages, pattern, tile=tile, black=black, white=white)
    assert_bit_equal(whole, lin, "%dx%d %s stages=%d tile=%s" % (H, W, pattern, stages, tile))
    cuts = sorted(set([0, H] + [2 * int(v) for v in rng.integers(1, H // 2, size=min(3, H // 2 - 1))])) if H > 4 else [0, H]
    halo = 6 + 4 * stages
    for rb, re in zip(cuts[:-1], cuts[1:]):
        r0, r1 = max(0, rb - halo), min(H, re + halo)
        band = emu_develop(emu, raw, stages, pattern, tile=tile, black=black, white=white, band=(rb, re), held=(r0, r1 - r0))
        assert_bit_equal(band, whole[rb:re], "band [%d,%d) of %dx%d" % (rb, re, H, W))


def test_hdr_and_f32_input(emu):
    rng = np.random.default_rng(9)
    sensor = (syn.scene(32, 44, 9).astype(np.float32) / 16383.0) * np.where(rng.random((32, 44)) < 0.2, 3.0, 1.0)
    sensor = sensor.astype(np.float32)
    for stages in (0, 1):
        cam = sp.ahd_demosaic(sensor, WB, M, stages, hdr=True)
        assert_bit_equal(emu_develop(emu, sensor, stages, hdr=True, out_kind=_capi.OUT_CAM_F32), cam, "hdr cam")
        assert_bit_equal(emu_develop(emu, sensor, stages, hdr=True), sp.to_lin_srgb(cam, M), "hdr lin")


def test_nonfinite_photosites(emu):
    """the tile functions reproduce the reference on +inf / -inf / NaN photosites (multiplicative blend, NaN-keeping clip)"""
    from conftest import assert_bit_equal_nan, golden
    d = golden("nonfinite48x64_s0")
    assert_bit_equal_nan(emu_develop(emu, d["sensor"], 0, out_kind=_capi.OUT_CAM_F32), d["cam"], "non-finite cam")
    assert_bit_equal_nan(emu_develop(emu, d["sensor"], 0), d["lin"], "non-finite lin")


def test_golden_through_emulation(emu):
    from conftest import golden
    d = golden("scene64x96_BGGR")
    out = emu_develop(emu, d["raw"], int(d["stages"]), "BGGR", black=d["black"], white=d["white"])
    assert_bit_equal(out, d["lin"], "golden BGGR")


@pytest.mark.parametrize("name", ["fast_rand8x8", "fast_scene34x50", "fast_scene64x96_GBRG", "fast_flat20x28", "fast_rand66x130"])
def test_fast_quality_golden(emu, name):
    """QualityDemosaic.Fast (edge-assisted Gaussian) against the reference's golden outputs."""
    from conftest import golden
    d = golden(name)
    for tile in ((16, 8), (20, 8), (60, 28), (60, 60), (60, 44)):
        cam = emu_develop(emu, d["raw"], 3, str(d["pattern"]), tile=tile, out_kind=_capi.OUT_CAM_F32, quality=1)
        assert_bit_equal(cam, d["cam"], "Fast camera RGB %s" % (tile,))
        assert_bit_equal(emu_develop(emu, d["raw"], 0, str(d["pattern"]), tile=tile, quality=1), d["lin"], "Fast linear sRGB")


def test_fast_quality_bands(emu):
    raw = syn.scene(48, 72, 12)
    whole = emu_develop(emu, raw, 0, quality=1)
    lin, _ = sp.develop_fast(raw, syn.BLACK, syn.WHITE, WB, syn.MAT_XYZ_TO_CAM, syn.WHITE_XYZ)
    assert_bit_equal(whole, lin, "Fast vs oracle")
    for rb, re in ((0, 20), (20, 48)):
        r0, r1 = max(0, rb - 6), min(48, re + 6)
        assert_bit_equal(emu_develop(emu, raw, 0, band=(rb, re), held=(r0, r1 - r0), quality=1), whole[rb:re], "Fast band")
