"""oracle/aux_spec.py (flat-field correction, hot-pixel detection, camera-space HDR fusion) against the fixtures
produced by the unmodified reference (tests/golden/make_golden_aux.py).  Bit-exact."""
import numpy as np
import pytest

from conftest import assert_bit_equal, golden
from oracle import ahd_spec as sp
from oracle import aux_spec as ax
from pysp_b200 import synthetic as syn

FLAT = ["aux_flat34x50", "aux_flat130x70_zeros", "aux_flat64x96_clamp_dead", "aux_flat200x304"]
HOT = ["aux_hot34x50", "aux_hot66x130", "aux_hot8x8"]
FUSE = ["aux_fusecam24x40", "aux_fusecam16x12_norm", "aux_fusecam20x28_nondyadic"]


def assert_same_float_bits(a, b, what):
    """bit equality with NaN == NaN (payloads are not compared)"""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    nan = np.isnan(a) & np.isnan(b)
    assert_bit_equal(np.where(nan, 0, a), np.where(nan, 0, b), what)


def reference_planes(m):
    """the four CFA planes as the reference takes them: strided views of the row-split copies (bayer_chan_mixer.py:13-21)"""
    evens, odds = m[0::2, :].astype(np.float32), m[1::2, :].astype(np.float32)
    return evens[:, 0::2], evens[:, 1::2], odds[:, 1::2], odds[:, 0::2]


# mosaic shapes whose planes hold 1, 127, 128, 129, 8191, 8192, 8193 sites, 2^24 (8192 x 8192), 4097^2 = 2^24 + 8193 and
# 4331 x 5775 = 25 011 525 (a 100 MP mosaic; float32(n) = 25 011 524): above 2^24 sites np.mean's float64 division by the
# integer count differs from a division by float32(n)
PLANE_MEAN_SHAPES = [(2, 2), (2, 254), (2, 256), (2, 258), (2, 16382), (2, 16384), (2, 16386), (8192, 8192), (8194, 8194),
                     (8662, 11550)]


def test_pairwise_sum_is_numpys():
    rng = np.random.default_rng(5)
    for n in (1, 7, 8, 9, 127, 128, 129, 1000, 30000, 123457):
        a = rng.random(n).astype(np.float32)
        assert ax.pairwise_sum(a) == np.add.reduce(a), n
    m = rng.random((200, 300)).astype(np.float32)
    plane = m[0::2, :].astype(np.float32)[:, 1::2]          # bayer_to_rgbg's strided view (bayer_chan_mixer.py:13-21)
    assert ax.plane_mean(plane) == np.mean(plane)
    # one 100 MP mosaic (seed 0); every other shape is its top-left corner
    big = np.random.default_rng(0).random((8662, 11550), dtype=np.float32)
    for shape in PLANE_MEAN_SHAPES:
        for i, p in enumerate(reference_planes(big[:shape[0], :shape[1]])):
            got, want = ax.plane_mean(p), np.mean(p)
            assert got.dtype == np.float32 and got.view(np.uint32) == want.view(np.uint32), (shape, i, got, want)


@pytest.mark.parametrize("name", FLAT)
def test_flat_frame_correction(name):
    d = golden(name)
    assert_same_float_bits(ax.flat_frame_correction(d["sensor"], d["flat"], bool(d["clamp"])), d["out"], name)


@pytest.mark.parametrize("name", HOT)
def test_hot_pixel_threshold(name):
    d = golden(name)
    masks = ax.find_erroneous_pixels_threshold(d["sensor"], float(d["min_delta"]), int(d["min_neighbour_count"]))
    assert np.array_equal(np.stack(masks), d["masks"])


@pytest.mark.parametrize("name", FUSE)
def test_fuse_exposures_from_debayer(name):
    d = golden(name)
    m = sp.cam_to_lin_srgb_matrix(syn.MAT_XYZ_TO_CAM, syn.WHITE_XYZ)
    n = len(d["evs"])
    lin, cnt, left = ax.fuse_exposures_from_debayer(list(d["images"]), list(d["evs"]), d["wb"], m, [bool(d["norm"])] * n)
    assert_bit_equal(lin, d["lin"], "fused linear sRGB")
    assert np.array_equal(cnt, d["count"])
    assert_bit_equal(np.stack(left), d["left"], "images after the wb_undo/wb_apply round trip")
