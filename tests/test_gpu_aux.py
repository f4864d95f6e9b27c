"""GPU parity of the steps either side of the develop path (SURVEY.md section 8f) through the C ABI / drop-in layer:
flat-field correction (incl. NumPy-ordered plane means), hot-pixel detection, camera-space HDR fusion.  Bit-exact against
the fixtures of the unmodified reference and against the oracle on larger seeded inputs."""
import numpy as np
import pytest
import torch

from conftest import assert_bit_equal, golden
from oracle import ahd_spec as sp
from oracle import aux_spec as ax
from pysp_b200 import synthetic as syn
from test_oracle_aux import FLAT, FUSE, HOT, assert_same_float_bits

pytestmark = pytest.mark.gpu


class Holder:
    def __init__(self, sensor):
        self.sensor_scaled = sensor


@pytest.fixture(scope="module")
def eng():
    from pysp_b200 import engine, _capi
    assert torch.cuda.is_available(), "these tests need the GPU"
    _capi.lib()
    return engine


@pytest.mark.parametrize("shape", [(4, 6), (16, 16), (34, 50), (400, 600), (2000, 3000), (2, 2), (2, 258), (8194, 8194),
                                   (8662, 11550)])
def test_plane_means_are_numpys(eng, shape):
    """(2, 258): 129 sites, one 128-element leaf and a tail.  8194 x 8194 (4097^2 = 2^24 + 8193 sites) and 8662 x 11550
    (25 011 525): planes above 2^24 sites, where np.mean's float64 division by the count differs from a division by
    float32(n); their wide tree levels run in tree_level_kernel."""
    if shape[0] * shape[1] > 2 ** 26:
        m = np.random.default_rng(0).random(shape, dtype=np.float32)
    else:
        rng = np.random.default_rng(shape[0])
        m = (rng.random(shape) * rng.choice([1e-3, 1.0, 50.0], size=shape)).astype(np.float32)
    got = eng.bayer_plane_means(eng.to_device(m)).cpu().numpy()
    evens, odds = m[0::2, :].astype(np.float32), m[1::2, :].astype(np.float32)      # bayer_chan_mixer.py:13-21
    want = np.array([np.mean(evens[:, 0::2]), np.mean(evens[:, 1::2]), np.mean(odds[:, 1::2]), np.mean(odds[:, 0::2])], np.float32)
    assert_bit_equal(got, want, "np.mean of the CFA planes %s" % (shape,))


@pytest.mark.parametrize("name", FLAT)
def test_flat_frame_correction_fixtures(eng, name):
    from pysp_b200 import flat_frame_correction
    d = golden(name)
    img = Holder(d["sensor"].copy())
    flat_frame_correction(img, Holder(d["flat"]), clamp_high=bool(d["clamp"]))
    assert isinstance(img.sensor_scaled, np.ndarray)
    assert_same_float_bits(img.sensor_scaled, d["out"], name)


def test_flat_frame_correction_24mp(eng):
    rng = np.random.default_rng(3)
    H, W = 4000, 6000
    sensor = rng.random((H, W), dtype=np.float32)
    y, x = np.mgrid[0:H, 0:W].astype(np.float32)
    flat = (0.9 - 0.5 * (((y - H / 2) / H) ** 2 + ((x - W / 2) / W) ** 2) + rng.normal(0, 0.01, (H, W))).astype(np.float32)
    flat[rng.integers(0, H, 50), rng.integers(0, W, 50)] = 0.0
    got = eng.flat_frame_correction(eng.to_device(sensor), eng.to_device(flat)).cpu().numpy()
    assert_same_float_bits(got, ax.flat_frame_correction(sensor, flat), "24 MP flat-field correction")


def test_plane_means_and_flat_field_are_graph_capturable(eng):
    """include/pysp_b200.h: pysp_bayer_plane_means and pysp_flat_frame_correction only launch kernels (the summation tree
    is derived on the device, the flat-field statistics are reset there), so both can be captured into one CUDA graph and
    replayed on new inputs.  2050 x 2050: 1025^2 sites, leaves on two depths and a wide tree level; the flat fields
    have zeros (+inf quotients replaced by the plane's maximum) and different maxima, so statistics left over from the
    previous replay would show."""
    H, W = 2050, 2050
    rng = np.random.default_rng(9)
    sens, flats = [], []
    for k in range(2):
        sens.append(eng.to_device(rng.random((H, W), dtype=np.float32)))
        f = (0.5 + (1.5 - k) * rng.random((H, W), dtype=np.float32)).astype(np.float32)
        f[rng.integers(0, H, 40), rng.integers(0, W, 40)] = 0.0
        flats.append(eng.to_device(f))
    want = [(eng.bayer_plane_means(f), eng.flat_frame_correction(s, f)) for s, f in zip(sens, flats)]
    src_s, src_f = sens[0].clone(), flats[0].clone()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        means = eng.bayer_plane_means(src_f)
        out = eng.flat_frame_correction(src_s, src_f)
    for k in range(2):
        src_s.copy_(sens[k])                # new inputs in the captured buffers, same graph
        src_f.copy_(flats[k])
        means.zero_()
        out.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(means.view(torch.int32), want[k][0].view(torch.int32)), k
        assert torch.equal(out.view(torch.int32), want[k][1].view(torch.int32)), k


@pytest.mark.parametrize("name", HOT)
def test_hot_pixels_fixtures(eng, name):
    from pysp_b200 import find_erroneous_pixels_threshold
    d = golden(name)
    masks = find_erroneous_pixels_threshold(Holder(d["sensor"]), float(d["min_delta"]), int(d["min_neighbour_count"]))
    assert len(masks) == 4 and masks[0].dtype == np.bool_
    assert np.array_equal(np.stack(masks), d["masks"])


def test_hot_pixels_large(eng):
    sensor = (syn.scene(1000, 1504, 4, noise=80.0).astype(np.float32) / np.float32(16383.0)).astype(np.float32)
    got = eng.find_hot_pixels_threshold(eng.to_device(sensor), 0.01, 5).cpu().numpy()
    assert np.array_equal(got, np.stack(ax.find_erroneous_pixels_threshold(sensor, 0.01, 5)))


@pytest.mark.parametrize("name", FUSE)
def test_fuse_from_debayer_fixtures(eng, name):
    import pysp_b200 as P
    d = golden(name)
    wbc = P.CameraWhiteBalance(syn.MAT_XYZ_TO_CAM, syn.WHITE_XYZ)
    objs = []
    for img, ev in zip(d["images"], d["evs"]):
        o = P.RawDemosaicData(img.copy(), d["wb"].copy(), wb_norm=bool(d["norm"]))
        o.mat_xyz = wbc.get_matrix()
        o.current_ev = float(ev)
        objs.append(o)
    lin, cnt = P.fuse_exposures_from_debayer(objs)
    assert_bit_equal(lin, d["lin"], "fused linear sRGB")
    assert np.array_equal(cnt, d["count"]) and cnt.dtype == np.int32
    assert_bit_equal(np.stack([o.image for o in objs]), d["left"], "exposures after the round trip")
    assert P.fuse_exposures_from_debayer([]) is None


def test_fuse_from_debayer_non_power_of_two_offsets(eng):
    """EV spacing that makes the offsets non-dyadic: the brightest-frame fallback is a float64 product (raw_hdr.py:75)."""
    rng = np.random.default_rng(8)
    wb = syn.wb_multipliers()
    m = sp.cam_to_lin_srgb_matrix(syn.MAT_XYZ_TO_CAM, syn.WHITE_XYZ)
    evs = [9.3, 10.1, 11.45]
    base = rng.uniform(0, 1.2, size=(60, 90, 3)).astype(np.float32)
    imgs = [np.minimum(base * np.float32(2.0 ** (10 - e)) * wb, wb).astype(np.float32) for e in evs]
    for im in imgs:
        im[:7, :9] = 0.0
        im[7:9, :9] = wb                      # saturated in every exposure: weight 0 -> fallback with a non-zero value
    want_lin, want_cnt, _ = ax.fuse_exposures_from_debayer(imgs, evs, wb, m)
    tgt = sum(evs) / 3
    offs = [2 ** (e - tgt) for e in evs]
    lin, cnt = eng.fuse_exposures_from_debayer([eng.to_device(i) for i in imgs], wb, float(max(wb)), [False] * 3,
                                               [np.float32(o) for o in offs], [np.float32(1.6 ** (-0.1 * o)) for o in offs],
                                               int(np.argmax(offs)), float(np.max(offs)), m)
    assert_bit_equal(lin.cpu().numpy(), want_lin, "fused linear sRGB (non-dyadic offsets)")
    assert np.array_equal(cnt.cpu().numpy(), want_cnt)
