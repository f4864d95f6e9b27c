"""DNG WarpRectilinear resampling on the GPU pinned bit for bit.  The coordinate table is the device's own (so the 2-ulp
tolerance of the table against the reference's libm powf does not enter); with it, clipped as apply_opcode_3_warp clips it,
every plane of pysp_warp_rectilinear_apply and of pysp_remap_lanczos4 must equal warp_spec.remap_lanczos4 -- cv2.remap's
INTER_LANCZOS4 restated -- exactly: 1 to 4 planes, with and without a prior, frames under 8 px, ragged tiles, a frame whose
blocks loop over more than one tile, launches in which some blocks stage a shared-memory patch and others gather from
global memory, and the two-step form with an interleaved destination and padded pitches."""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import assert_bit_equal
from oracle import warp_spec as ws

pytestmark = pytest.mark.gpu
f32 = np.float32
PW, PH = 56, 28                # PYSP_WARP_PW / PYSP_WARP_PH of warp.cuh: the shared-memory patch of one 32 x 8 block


@pytest.fixture(scope="module")
def eng():
    from pysp_b200 import engine, _capi
    assert torch.cuda.is_available()
    _capi.lib()
    return engine


def clipped(table, H, W):
    return np.clip(table[..., 0], 0, W - 1), np.clip(table[..., 1], 0, H - 1)


def blocks_fitting(tables, H, W):
    """per 32 x 8 block of warp_apply_kernel: whether the bounding box of the 8 x 8 windows of all its pixels and planes fits
    the shared-memory patch (else the block gathers from global memory)"""
    ox, oy = [], []
    for t in tables:
        mx, my = clipped(t, H, W)
        ox.append((np.rint(mx * f32(32)).astype(np.int64) >> 5) - 3)
        oy.append((np.rint(my * f32(32)).astype(np.int64) >> 5) - 3)
    ox, oy = np.stack(ox), np.stack(oy)
    fit = []
    for y0 in range(0, H, 8):
        for x0 in range(0, W, 32):
            bx, by = ox[:, y0:y0 + 8, x0:x0 + 32], oy[:, y0:y0 + 8, x0:x0 + 32]
            fit.append(bx.max() + 8 - bx.min() <= PW and by.max() + 8 - by.min() <= PH)
    return np.array(fit)


def check_warp(eng, img, coeffs, centre, scale, prior, what):
    """fused kernel and two-step form against the oracle on the device's tables; returns the tables"""
    H, W, n = img.shape
    src = torch.from_numpy(img).cuda()
    pr = None if prior is None else torch.from_numpy(prior).cuda()
    fused = eng.warp_rectilinear(src, coeffs, centre, scale, prior=pr).cpu().numpy()
    tables = []
    for c in range(n):
        seed = None if pr is None else pr[:, :, c, :].contiguous()
        tab = eng.warp_table(H, W, coeffs[c], centre, scale, seed=seed)
        t = tab.cpu().numpy()
        tables.append(t)
        want = ws.remap_lanczos4(img[:, :, c], *clipped(t, H, W))
        assert_bit_equal(fused[:, :, c], want, "%s: warp_rectilinear plane %d" % (what, c))
        two = eng.remap_lanczos4(src, c, tab).cpu().numpy()
        assert_bit_equal(two, want, "%s: remap_lanczos4 plane %d" % (what, c))
    return tables


def random_coeffs(rng, n):
    return [(1.0 + rng.uniform(-0.01, 0.01), rng.uniform(-0.06, 0.02), rng.uniform(-0.01, 0.02), rng.uniform(-0.004, 0.004),
             rng.uniform(-0.002, 0.002), rng.uniform(-0.002, 0.002)) for _ in range(n)]


SHAPES = [(1, 40), (40, 1), (6, 5), (7, 9), (37, 61), (8, 32), (45, 100)]


@pytest.mark.parametrize("with_prior", [False, True])
@pytest.mark.parametrize("planes", [1, 2, 3, 4])
@pytest.mark.parametrize("shape", SHAPES)
def test_warp_matrix(eng, shape, planes, with_prior):
    seed = 1000 + 16 * SHAPES.index(shape) + 2 * planes + int(with_prior)
    rng = np.random.default_rng(seed)
    H, W = shape
    img = rng.uniform(-0.2, 1.5, size=(H, W, planes)).astype(f32)
    coeffs = random_coeffs(rng, planes)
    centre = (float(rng.uniform(0.3, 0.7)), float(rng.uniform(0.3, 0.7)))
    scale = float(rng.choice([1.0, 0.7, 1.3]))
    prior = None
    if with_prior:
        yy, xx = np.mgrid[0:H, 0:W].astype(f32)
        prior = np.empty((H, W, planes, 2), f32)
        for c in range(planes):
            prior[:, :, c, 0] = xx + rng.uniform(-1.5, 1.5, size=(H, W)).astype(f32)
            prior[:, :, c, 1] = yy + rng.uniform(-1.5, 1.5, size=(H, W)).astype(f32)
    what = "warp seed=%d %dx%d planes=%d prior=%s centre=%s scale=%g" % (seed, H, W, planes, with_prior, centre, scale)
    check_warp(eng, img, coeffs, centre, scale, prior, what)


def test_warp_blocks_loop(eng):
    """808 x 1504: 101 x 47 = 4747 blocks of 32 x 8, more than the 148 * 32 of the grid, so blocks take a second tile and the
    second of the two alternating bounding boxes"""
    rng = np.random.default_rng(1100)
    H, W = 808, 1504
    assert ((H + 7) // 8) * ((W + 31) // 32) > 148 * 32
    img = rng.random((H, W, 2), dtype=f32)
    coeffs = [(1.002, -0.041, 0.013, -0.002, 0.0006, -0.0003), (0.999, -0.035, 0.009, -0.001, 0.0002, -0.0005)]
    tables = check_warp(eng, img, coeffs, (0.5012, 0.4979), 1.0, None, "808x1504, 2 planes")
    assert blocks_fitting(tables, H, W).all()


@pytest.mark.parametrize("k", [(2.2, -0.3, 0.1, 0.0, 0.05, -0.04), (1.01, -0.02, 0.0, 0.0, 0.3, 0.25), (1.3, 0.5, 0.0, 0.0, 0.0, 0.0)])
def test_warp_smem_and_fallback_in_one_launch(eng, k):
    """strong distortion: blocks near the centre stage the shared-memory patch, blocks further out do not fit it and gather
    from global memory; both in the same launch, both bit-exact"""
    rng = np.random.default_rng(1200)
    H, W = 200, 328
    img = rng.random((H, W, 3), dtype=f32)
    tables = check_warp(eng, img, [k] * 3, (0.47, 0.52), 1.0, None, "200x328 k=%s" % (k,))
    fit = blocks_fitting(tables, H, W)
    assert fit.any() and not fit.all(), (k, int(fit.sum()), fit.size)


def test_remap_interleaved_padded(eng):
    """pysp_remap_lanczos4 on plane c of an interleaved image with a padded source pitch, into every second float of a
    padded destination (dst_step 2), through a map with a padded pitch; nothing else of the destination is written"""
    from pysp_b200 import _capi
    L = _capi.lib()
    rng = np.random.default_rng(1300)
    H, W, n = 37, 61, 3
    img = rng.random((H, W, n), dtype=f32)
    spitch, dpitch, mpitch = W * n + 5, 2 * W + 3, W + 3                   # floats, floats, float pairs
    src = torch.zeros((H, spitch), dtype=torch.float32, device="cuda")
    src[:, :W * n] = torch.from_numpy(img.reshape(H, W * n)).cuda()
    tab_t = eng.warp_table(H, W, (1.01, -0.05, 0.01, 0.0, 0.001, -0.002), (0.45, 0.55), 1.0)
    tab = tab_t.cpu().numpy()
    mp = torch.full((H, mpitch, 2), 1e9, dtype=torch.float32, device="cuda")
    mp[:, :W] = tab_t
    lt = eng.lanczos_tab(torch.device("cuda"))
    for c in range(n):
        dst = torch.full((H, dpitch), -7.0, dtype=torch.float32, device="cuda")
        rc = L.pysp_remap_lanczos4(src.data_ptr() + 4 * c, spitch * 4, n, dst.data_ptr() + 4, dpitch * 4, 2, H, W,
                                   mp.data_ptr(), mpitch * 8, lt.data_ptr(), torch.cuda.current_stream().cuda_stream)
        assert rc == 0
        d = dst.cpu().numpy()
        assert_bit_equal(d[:, 1:2 * W:2], ws.remap_lanczos4(img[:, :, c], *clipped(tab, H, W)), "interleaved remap plane %d" % c)
        untouched = np.ones_like(d, dtype=bool)
        untouched[:, 1:2 * W:2] = False
        assert np.all(d[untouched] == -7.0), "remap wrote outside its plane (plane %d)" % c
