"""DNG WarpRectilinear on the GPU (SURVEY.md section 8f-4) through the C ABI: coordinate tables within 2 ulp of the
reference (its generated C calls libm's powf, which is not correctly rounded), Lanczos-4 resampling within 1e-4 relative
of cv2.remap outside pixels whose 1/32-px phase differs (their count is reported)."""
import numpy as np
import pytest
import torch

from conftest import golden
from oracle import warp_spec as ws

pytestmark = pytest.mark.gpu
CASES = ["warp_96x128", "warp_70x50_scale"]


@pytest.fixture(scope="module")
def eng():
    from pysp_b200 import engine, _capi
    assert torch.cuda.is_available()
    _capi.lib()
    return engine


def ulp_distance(a, b):
    a = np.ascontiguousarray(a, dtype=np.float32).view(np.int32).astype(np.int64)
    b = np.ascontiguousarray(b, dtype=np.float32).view(np.int32).astype(np.int64)
    a = np.where(a < 0, -(a & 0x7FFFFFFF), a)
    b = np.where(b < 0, -(b & 0x7FFFFFFF), b)
    return np.abs(a - b)


def phases(table, W, H):
    x = np.clip(table[..., 0], 0, W - 1)
    y = np.clip(table[..., 1], 0, H - 1)
    return np.rint(x * np.float32(32)).astype(np.int64), np.rint(y * np.float32(32)).astype(np.int64)


def check_warped(got, want, table_got, table_ref, W, H, what):
    px, py = phases(table_got, W, H)
    qx, qy = phases(table_ref, W, H)
    same = (px == qx) & (py == qy)
    err = np.abs(got.astype(np.float64) - want) / np.maximum(np.abs(want), 1e-3)
    print("%s: %d of %d pixels sample a different 1/32-px phase; max relative error elsewhere %.3g, there %.3g" % (
        what, int((~same).sum()), same.size, float(err[same].max()), float(err[~same].max()) if (~same).any() else 0.0))
    assert err[same].max() <= 1e-4, what
    assert (~same).mean() < 0.01, what


@pytest.mark.parametrize("name", CASES)
def test_tables(eng, name):
    from pysp_b200.dng_warp_corr import compute_offset_remapping_table, compute_remapping_table
    d = golden(name)
    H, W, _ = d["image"].shape
    for i in range(3):
        k = [float(v) for v in d["coeffs"][i]]
        t = compute_remapping_table(*k, W, H, float(d["centre"][0]), float(d["centre"][1]), float(d["scale"]))
        assert isinstance(t, np.ndarray) and t.dtype == np.float32 and t.shape == (H, W, 2)
        u = ulp_distance(t, d["tables"][i])
        print(name, "plane", i, "table: max ulp distance", int(u.max()), "; values differing", int((u > 0).sum()), "of", u.size)
        # positions near 0 (first row / column) have huge relative ulp counts for tiny absolute errors: absolute floor
        assert np.all((u <= 2) | (np.abs(t - d["tables"][i]) <= 2e-6))
        tp = compute_offset_remapping_table(d["prior"][..., i, :], *k, W, H, float(d["centre"][0]), float(d["centre"][1]),
                                            float(d["scale"]))
        up = ulp_distance(tp, d["tables_prior"][i])
        assert np.all((up <= 2) | (np.abs(tp - d["tables_prior"][i]) <= 2e-6))


@pytest.mark.parametrize("name", CASES)
def test_apply_opcode_3_warp(eng, name):
    from pysp_b200.dng_warp_corr import apply_opcode_3_warp
    d = golden(name)
    H, W, _ = d["image"].shape
    tabs = [eng.warp_table(H, W, d["coeffs"][i], d["centre"], float(d["scale"])).cpu().numpy() for i in range(3)]
    img = np.array(d["image"], copy=True)
    apply_opcode_3_warp(img, d["opcode"].tobytes(), float(d["scale"]))
    for i in range(3):
        check_warped(img[..., i], d["warped"][..., i], tabs[i], d["tables"][i], W, H, "%s plane %d" % (name, i))
    # CUDA tensor in place, with a prior
    t = torch.from_numpy(np.array(d["image"], copy=True)).cuda()
    apply_opcode_3_warp(t, d["opcode"].tobytes(), float(d["scale"]), prior=d["prior"])
    tabs_p = [eng.warp_table(H, W, d["coeffs"][i], d["centre"], float(d["scale"]),
                             seed=torch.from_numpy(np.ascontiguousarray(d["prior"][..., i, :])).cuda()).cpu().numpy() for i in range(3)]
    for i in range(3):
        check_warped(t.cpu().numpy()[..., i], d["warped_prior"][..., i], tabs_p[i], d["tables_prior"][i], W, H,
                     "%s plane %d with prior" % (name, i))
    # the two-step form (table in HBM, then remap) gives the same bits as the fused kernel
    src = torch.from_numpy(np.array(d["image"], copy=True)).cuda()
    fused = eng.warp_rectilinear(src, d["coeffs"], d["centre"], float(d["scale"]))
    for i in range(3):
        two = eng.remap_lanczos4(src, i, eng.warp_table(H, W, d["coeffs"][i], d["centre"], float(d["scale"])))
        assert torch.equal(two.view(torch.int32), fused[..., i].contiguous().view(torch.int32))


def test_warp_against_oracle_24mp_crop(eng):
    """a 2000x3000 linear-sRGB-like image: GPU against the oracle (tables by the C restatement, remap restated from cv2)"""
    H, W = 1000, 1504
    rng = np.random.default_rng(5)
    img = rng.random((H, W, 3), dtype=np.float32)
    coeffs = [(1.002, -0.041, 0.013, -0.002, 0.0006, -0.0003), (0.999, -0.035, 0.009, -0.001, 0.0002, -0.0005),
              (1.001, -0.038, 0.011, -0.003, 0.0004, -0.0001)]
    centre = (0.5012, 0.4979)
    want = ws.apply_warp_rectilinear(img, coeffs, centre, 1.0)
    got = eng.warp_rectilinear(torch.from_numpy(img).cuda(), coeffs, centre, 1.0).cpu().numpy()
    for i in range(3):
        tg = eng.warp_table(H, W, coeffs[i], centre, 1.0).cpu().numpy()
        tr = ws.remapping_table(coeffs[i], W, H, centre, 1.0)
        check_warped(got[..., i], want[..., i], tg, tr, W, H, "1.5 MP plane %d" % i)


def test_identity_and_errors(eng):
    """kr0 = 1, everything else 0: the table is the pixel grid and the warp is the identity; bad arguments raise ValueError"""
    H, W = 64, 80
    t = eng.warp_table(H, W, (1, 0, 0, 0, 0, 0), (0.5, 0.5), 1.0).cpu().numpy()
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float32)
    assert np.abs(t[..., 0] - xx).max() <= 1e-4 and np.abs(t[..., 1] - yy).max() <= 1e-4
    img = torch.rand((H, W, 3), device="cuda")
    out = eng.warp_rectilinear(img, [(1, 0, 0, 0, 0, 0)] * 3, (0.5, 0.5), 0.0)     # scale 0: exactly the pixel grid
    assert torch.equal(out, img)
    # strong magnification / shear: the source windows of a block no longer fit the shared-memory patch and the kernel
    # gathers from global memory instead -- same bits as the two-step form (table in HBM, then remap) either way
    big = torch.rand((200, 328, 3), device="cuda")
    for k in ((2.2, -0.3, 0.1, 0.0, 0.05, -0.04), (0.45, 0.2, 0.0, 0.0, 0.0, 0.0), (1.01, -0.02, 0.0, 0.0, 0.3, 0.25),
              (1.3, 0.5, 0.0, 0.0, 0.0, 0.0)):
        fused = eng.warp_rectilinear(big, [k] * 3, (0.47, 0.52), 1.0)
        for i in range(3):
            two = eng.remap_lanczos4(big, i, eng.warp_table(200, 328, k, (0.47, 0.52), 1.0))
            assert torch.equal(two.view(torch.int32), fused[..., i].contiguous().view(torch.int32)), k
    with pytest.raises(ValueError):
        eng.warp_rectilinear(img, [(1, 0, 0, 0, 0, 0)] * 2, (0.5, 0.5))
    with pytest.raises(ValueError):
        eng.warp_table(1, 1, (1, 0, 0, 0, 0, 0), (0.5, 0.5))                        # the reference: ZeroDivisionError
