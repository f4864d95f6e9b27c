"""The develop kernels on the GPU away from the u16 / AHD / float32-output corner: float32 and HDR mosaics and
QualityDemosaic.Fast on every CFA pattern, ragged sizes, padded pitches and row bands, against the oracle; every output kind
(lin_f16, the float32 gamma, srgb_u8 / srgb_u16) through the K1, K2 and Fast epilogues; non-finite photosites under flips;
the generic (non-TMA) loads and stores on those branches; the point-wise matrix and gamma kernels.

The seeded cases are those of tests/test_tile_logic_matrix.py, which runs them through the host emulation.  On the device
they also reach what the emulation cannot: TMA boxes of float32 mosaics under flips, the word-packed stores of the narrow
kinds, the float -> half conversion and the hardware gamma."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, assert_bit_equal, assert_bit_equal_nan, golden
from oracle import ahd_spec as sp
from pysp_b200 import synthetic as syn
from test_tile_logic import M, WB
from test_tile_logic_matrix import N_CASES, Case, describe, halo_rows, matrix_case, matrix_reference, quantised

pytestmark = pytest.mark.gpu

NARROW = (("srgb_u8", 255.0, np.uint8), ("srgb_u16", 65535.0, np.uint16))
OUT_DTYPES = {"cam": torch.float32, "lin": torch.float32, "lin_f16": torch.float16, "srgb_u8": torch.uint8,
              "srgb_u16": torch.uint16}
SENTINEL = 0xA5                               # every byte of an output buffer before the develop


@pytest.fixture(scope="module")
def eng():
    from pysp_b200 import engine, _capi
    assert torch.cuda.is_available(), "these tests need the GPU"
    _capi.lib()
    return engine


def host(t):
    torch.cuda.synchronize()
    return t.cpu().numpy()


def assert_half_equal(a, b, what=""):
    """float16 bit equality; NaN must sit at the same places, with any payload"""
    a, b = np.asarray(a), np.asarray(b)
    assert a.dtype == np.float16 and b.dtype == np.float16 and a.shape == b.shape, (what, a.dtype, b.dtype, a.shape, b.shape)
    na, nb = np.isnan(a), np.isnan(b)
    assert np.array_equal(na, nb), "%s: NaN at different places (%d vs %d)" % (what, int(na.sum()), int(nb.sum()))
    bad = (a.view(np.uint16) != b.view(np.uint16)) & ~na
    if bad.any():
        idx = np.argwhere(bad)[0]
        raise AssertionError("%s: %d of %d halves differ; first at %s: %s vs %s" % (
            what, int(bad.sum()), bad.size, idx.tolist(), a[tuple(idx)], b[tuple(idx)]))


def assert_gamma_close(g, lin, what=""):
    """the gamma contract: within 1e-4 * max(|ref|, 1e-3) of the oracle's lin_srgb_to_srgb, NaN where the input is NaN"""
    ref = sp.lin_srgb_to_srgb(lin)
    nan = np.isnan(ref)
    assert np.array_equal(np.isnan(g), nan), "%s: NaN at different places" % what
    err = np.abs(g[~nan].astype(np.float64) - ref[~nan])
    lim = 1e-4 * np.maximum(np.abs(ref[~nan].astype(np.float64)), 1e-3)
    assert np.all(err <= lim), "%s: gamma off by %.3g (%d values over the tolerance)" % (what, float(err.max()), int((err > lim).sum()))


def develop_kw(c):
    kw = dict(stages=c.stages, pattern=c.pattern, hdr=c.hdr, quality=c.quality)
    if c.kind == "u16":
        kw.update(black=c.black, white=c.white)
    return kw


def sentinel_buffer(rows, W, out):
    """an output tensor of kind `out` [rows, W, 3] whose bytes all hold SENTINEL, and its byte view"""
    esz = torch.empty((), dtype=OUT_DTYPES[out]).element_size()
    buf = torch.full((rows, W, 3 * esz), SENTINEL, dtype=torch.uint8, device="cuda")
    return buf.view(OUT_DTYPES[out]), buf


def develop_band(eng, c, src, r0, rb, re, out_row0, out="lin", gamma=False, dir_map=None):
    """rows [rb, re) developed from `src` (frame rows [r0, r0 + len(src))) into rows [rb - out_row0, re - out_row0) of a
    taller output tensor; the rows above the band must keep their sentinel bytes"""
    t, buf = sentinel_buffer(re - out_row0, c.W, out)
    eng.develop(src, WB, M, out=out, gamma=gamma, out_tensor=t, rows=(rb, re), frame_height=c.H, in_row0=r0,
                out_row0=out_row0, dir_map=dir_map, **develop_kw(c))
    assert (host(buf[:rb - out_row0]) == SENTINEL).all(), "%s: rows above band [%d,%d) were written" % (describe(c), rb, re)
    return host(t[rb - out_row0:])


@pytest.mark.parametrize("seed", range(N_CASES))
def test_develop_matrix(eng, seed):
    """One seeded case (u16 with per-site levels, float32 or HDR float32; Best at 0-3 stages or Fast; any CFA pattern;
    ragged size, width 0 or 2 mod 4).  Camera RGB, linear sRGB and the AHD direction map equal the oracle bit for bit on the
    whole frame and from a row-padded upload.  Every output kind: lin_f16 is the float32 result cast to half, the float32
    gamma is within the gamma contract, srgb_u8 / srgb_u16 are that gamma output rounded to nearest, exactly.  Every band
    of a random split, developed from its rows + halo only (odd-numbered bands into a taller output tensor whose rows
    above the band must stay untouched), equals the whole frame in every output kind."""
    c = matrix_case(seed)
    what = describe(c)
    cam, lin, pick = matrix_reference(c)
    kw = develop_kw(c)
    best = c.quality == "best"
    t = eng.to_device(c.src)

    def run(src=t, **extra):
        return host(eng.develop(src, WB, M, **kw, **extra))

    assert_bit_equal(run(out="cam"), cam, what + " cam")
    dm = torch.full((c.H, c.W), SENTINEL, dtype=torch.uint8, device="cuda") if best else None
    assert_bit_equal(run(out="lin", dir_map=dm), lin, what + " lin")
    if best:
        whole_map = host(dm)
        assert np.array_equal(whole_map, pick.astype(np.uint8)), what + " direction map"
    padded = eng.to_device(c.src, pad_pitch=True)
    assert_bit_equal(run(padded, out="cam"), cam, what + " cam (padded pitch)")
    assert_bit_equal(run(padded, out="lin"), lin, what + " lin (padded pitch)")

    g = run(gamma=True)
    assert_gamma_close(g, lin, what + " gamma")
    for kind, scale, dt in NARROW:
        q = run(out=kind)
        assert q.dtype == dt and np.array_equal(q, quantised(g, scale, dt)), "%s %s" % (what, kind)
    assert_half_equal(run(out="lin_f16"), lin.astype(np.float16), what + " lin_f16")
    assert_half_equal(run(out="lin_f16", gamma=True), g.astype(np.float16), what + " lin_f16 with gamma")

    halo = halo_rows(c)
    for i, (rb, re) in enumerate(zip(c.cuts[:-1], c.cuts[1:])):
        r0, r1 = max(0, rb - halo), min(c.H, re + halo)
        src = eng.to_device(np.ascontiguousarray(c.src[r0:r1]))
        out_row0 = 0 if i % 2 else rb
        band = "%s band [%d,%d) out_row0=%d" % (what, rb, re, out_row0)
        args = (eng, c, src, r0, rb, re, out_row0)
        assert_bit_equal(develop_band(*args, out="cam"), cam[rb:re], band + " cam")
        bm = torch.full((re - out_row0, c.W), SENTINEL, dtype=torch.uint8, device="cuda") if best else None
        assert_bit_equal(develop_band(*args, dir_map=bm), lin[rb:re], band + " lin")
        if best:
            got = host(bm)
            assert (got[:rb - out_row0] == SENTINEL).all() and np.array_equal(got[rb - out_row0:], whole_map[rb:re]), \
                band + " direction map"
        assert_bit_equal(develop_band(*args, gamma=True), g[rb:re], band + " gamma")
        for kind, scale, dt in NARROW:
            assert np.array_equal(develop_band(*args, out=kind), quantised(g[rb:re], scale, dt)), "%s %s" % (band, kind)
        assert_half_equal(develop_band(*args, out="lin_f16"), lin[rb:re].astype(np.float16), band + " lin_f16")
        assert_half_equal(develop_band(*args, out="lin_f16", gamma=True), g[rb:re].astype(np.float16), band + " lin_f16 with gamma")


@pytest.mark.parametrize("pattern", ["BGGR", "GRBG", "GBRG"])
def test_nonfinite_photosites_mirrored(eng, pattern):
    """+inf / -inf / NaN photosites of a float32 mosaic stored under a mirrored pattern: the mirrored golden camera RGB,
    linear sRGB and direction map (NaN-aware; a float32 mosaic has no per-site levels, so this is exact).  The wire
    formats give 0 and lin_f16 a NaN half where linear sRGB is NaN."""
    d = golden("nonfinite48x64_s0")
    t = eng.to_device(np.ascontiguousarray(sp.to_rggb(d["sensor"], pattern)))
    cam, lin = sp.to_rggb(d["cam"], pattern), np.ascontiguousarray(sp.to_rggb(d["lin"], pattern))
    kw = dict(stages=0, pattern=pattern)
    dm = torch.zeros(lin.shape[:2], dtype=torch.uint8, device="cuda")
    assert_bit_equal_nan(host(eng.develop(t, WB, M, out="cam", dir_map=dm, **kw)), cam, pattern + " cam")
    assert np.array_equal(host(dm).astype(bool), sp.to_rggb(d["pick_h"], pattern)), pattern + " direction map"
    assert_bit_equal_nan(host(eng.develop(t, WB, M, **kw)), lin, pattern + " lin")
    nan = np.isnan(lin)
    assert nan.any()
    g = host(eng.develop(t, WB, M, gamma=True, **kw))
    assert_gamma_close(g, lin, pattern + " gamma")
    for kind, scale, dt in NARROW:
        q = host(eng.develop(t, WB, M, out=kind, **kw))
        assert np.array_equal(q, quantised(g, scale, dt)) and not q[nan].any(), "%s %s" % (pattern, kind)
    assert_half_equal(host(eng.develop(t, WB, M, out="lin_f16", **kw)), lin.astype(np.float16), pattern + " lin_f16")


def generic_path_cases():
    """Run in a child process by test_generic_paths_new_branches, with PYSP_DISABLE_TMA set."""
    from pysp_b200 import engine as eng
    H, W = 128, 184                      # float32 rows of 16-byte multiples: these take TMA unless the hook disables it
    f32 = syn.scene(H, W, 41).astype(np.float32) / np.float32(16383.0)
    hdr = (f32 * np.where(np.random.default_rng(41).random((H, W)) < 0.2, np.float32(3.0), np.float32(1.0))).astype(np.float32)
    for src, pattern, stages, quality, kind in ((f32, "BGGR", 1, "best", "f32"), (hdr, "GRBG", 2, "best", "hdr"),
                                                (f32, "GBRG", 0, "fast", "f32")):
        c = Case(0, H, W, pattern, kind, stages, quality, src, None, None, kind == "hdr", [0, H])
        cam, lin, _ = matrix_reference(c)
        t = eng.to_device(src)
        assert_bit_equal(host(eng.develop(t, WB, M, out="cam", **develop_kw(c))), cam, describe(c) + " cam")
        assert_bit_equal(host(eng.develop(t, WB, M, **develop_kw(c))), lin, describe(c) + " lin")
    H, W = 126, 182                      # W = 2 mod 4: the srgb_u8 rows are not whole 32-bit words
    raw = syn.scene(H, W, 42)
    c = Case(0, H, W, "GBRG", "u16", 0, "best", raw, syn.BLACK, syn.WHITE, False, [0, H])
    _, lin, _ = matrix_reference(c)
    t = eng.to_device(raw, pad_pitch=True)
    g = host(eng.develop(t, WB, M, gamma=True, **develop_kw(c)))
    assert_gamma_close(g, lin, describe(c) + " gamma")
    for kind, scale, dt in NARROW:
        assert np.array_equal(host(eng.develop(t, WB, M, out=kind, **develop_kw(c))), quantised(g, scale, dt)), kind


@pytest.mark.parametrize("mode", ["1", "2", "3"])
def test_generic_paths_new_branches(mode):
    """float32 / HDR / Fast inputs and the narrow kinds through the generic loads (1), stores (2) or both (3), forced
    through the library's test hook, which is read once per process: hence a fresh process per mode."""
    code = "import sys\nsys.path[:0] = [%r, %r]\nimport test_gpu_develop_matrix as t\nt.generic_path_cases()\nprint('ok')\n" % (
        ROOT, os.path.join(ROOT, "tests"))
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, PYSP_DISABLE_TMA=mode), capture_output=True, text=True)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-3000:]


def test_pointwise_matrix_and_gamma(eng):
    """cam_to_rgb with gamma equals the develop's fused gamma, its half output the develop's lin_f16; srgb_gamma on a view
    one element in with an odd count (the scalar path) equals the aligned call (vector path + tail); edge inputs of the
    gamma stay within the contract of the oracle, NaN stays NaN."""
    t = eng.to_device(syn.scene(150, 206, 51))
    kw = dict(stages=1, pattern="GRBG", black=syn.BLACK, white=syn.WHITE)
    cam = eng.develop(t, WB, M, out="cam", **kw)
    g = eng.develop(t, WB, M, gamma=True, **kw)
    assert_bit_equal(host(eng.cam_to_rgb(cam, M, clip=True, gamma=True)), host(g), "cam_to_rgb with gamma")
    half = eng.cam_to_rgb(cam, M, clip=True, half=True)
    assert half.dtype == torch.float16
    assert_half_equal(host(half), host(eng.develop(t, WB, M, out="lin_f16", **kw)), "cam_to_rgb half")

    lin = eng.develop(t, WB, M, **kw).reshape(-1)
    n = lin.numel() - 1 if lin.numel() % 2 == 0 else lin.numel() - 2
    view = lin[1:1 + n]
    assert n % 2 == 1 and view.data_ptr() % 16 != 0
    assert_bit_equal(host(eng.srgb_gamma(view)), host(eng.srgb_gamma(view.clone())), "srgb_gamma, unaligned view")

    f = np.float32
    knee, one = f(0.0031308), f(1.0)
    edges = np.array([0.0, -0.0, 1e-45, -1e-45, 1.1754942e-38, 1.1754944e-38, np.nextafter(knee, f(0)), knee,
                      np.nextafter(knee, one), 0.04045, 0.5, np.nextafter(one, f(0)), one, np.nextafter(one, f(2)), 1.5,
                      3.4e38, np.inf, -np.inf, np.nan, -0.25, 0.75], dtype=f)
    assert edges.size % 4 != 0
    x = torch.from_numpy(np.concatenate([edges[:1], edges])).cuda()
    aligned = host(eng.srgb_gamma(x[1:].clone()))          # vector path + tail
    unaligned = host(eng.srgb_gamma(x[1:]))                # one element in: scalar path
    assert_gamma_close(aligned, edges, "gamma on edge inputs")
    assert_bit_equal_nan(unaligned, aligned, "gamma on edge inputs, unaligned")
