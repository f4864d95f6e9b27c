"""PYSP_OUT_YCC420_U8 on the device: the planes of every K1 / K2 / Fast epilogue equal the NumPy restatement
(tests/ycc420_ref.py, pinned to libjpeg) of the GPU's own srgb_u8 output of the same call, on the seeded cases of
test_tile_logic_matrix (whole frame, row-padded upload, row bands into taller padded planes), through the generic loads,
on non-finite photosites under every pattern, and on a 24 MP frame, where a JPEG written from the planes is byte-identical
to the one libjpeg writes from srgb_u8.  FramePipeline(out="ycc420") delivers the same bytes to host memory."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, golden
from oracle import ahd_spec as sp
from pysp_b200 import synthetic as syn
from test_gpu_develop_matrix import develop_kw
from test_tile_logic import M, WB
from test_tile_logic_matrix import N_CASES, Case, describe, halo_rows, matrix_case
from test_ycc420_cpu import PADS, assert_planes_equal, expected_buffers, inner, planes_buffers
from ycc420_ref import upsample2x2, ycc420

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    from pysp_b200 import engine, _capi
    assert torch.cuda.is_available(), "these tests need the GPU"
    _capi.lib()
    return engine


def host(t):
    torch.cuda.synchronize()
    return t.cpu().numpy()


def develop_planes(eng, t, **kw):
    """engine.develop(out="ycc420") -> host planes; the three views lie back to back in one I420 buffer"""
    y, cb, cr = eng.develop(t, WB, M, out="ycc420", **kw)
    n, W = y.shape
    assert cb.shape == cr.shape == (n // 2, W // 2)
    assert cb.data_ptr() == y.data_ptr() + n * W and cr.data_ptr() == cb.data_ptr() + (n // 2) * (W // 2)
    assert y.untyped_storage().nbytes() >= n * W * 3 // 2
    return host(y), host(cb), host(cr)


def ycc_into_buffers(eng, t, n_rows, W, pad, **kw):
    """develop into sentinel planes of n_rows rows with padded pitches and guard rows (test_ycc420_cpu.planes_buffers);
    host copies of the whole buffers"""
    bufs = tuple(torch.from_numpy(b).cuda() for b in planes_buffers(n_rows, W, pad))
    y, cb, cr = inner(bufs)                                    # [n_rows, W] views whose row pitch includes the padding
    eng.develop(t, WB, M, out="ycc420", out_tensor=(y[:, :W], cb[:, :W // 2], cr[:, :W // 2]), **kw)
    return tuple(host(b) for b in bufs)


@pytest.mark.parametrize("seed", range(N_CASES))
def test_ycc420_matrix(eng, seed):
    """Whole frame (contiguous and row-padded upload) equals the restatement of srgb_u8 of the same call; every band of a
    random split from its rows + halo writes exactly its rows into padded planes, odd-numbered bands into planes that start
    above the band (out_row0 < row_begin)."""
    c = matrix_case(seed)
    what = describe(c)
    kw = develop_kw(c)
    t = eng.to_device(c.src)
    ref = ycc420(host(eng.develop(t, WB, M, out="srgb_u8", **kw)))
    assert_planes_equal(develop_planes(eng, t, **kw), ref, what)
    padded = eng.to_device(c.src, pad_pitch=True)
    assert_planes_equal(develop_planes(eng, padded, **kw), ref, what + " (padded upload)")
    pad = PADS[seed % len(PADS)]
    halo = halo_rows(c)
    for i, (rb, re) in enumerate(zip(c.cuts[:-1], c.cuts[1:])):
        r0, r1 = max(0, rb - halo), min(c.H, re + halo)
        src = eng.to_device(np.ascontiguousarray(c.src[r0:r1]))
        out_row0 = (rb // 4) * 2 if i % 2 else rb             # even, below row_begin for odd-numbered bands
        got = ycc_into_buffers(eng, src, re - out_row0, c.W, pad, rows=(rb, re), frame_height=c.H, in_row0=r0,
                               out_row0=out_row0, **kw)
        from_row0 = (ref[0][out_row0:], ref[1][out_row0 // 2:], ref[2][out_row0 // 2:])     # plane row 0 = out_row0
        want = expected_buffers(from_row0, re - out_row0, c.W, pad, rb - out_row0, re - out_row0)
        assert_planes_equal(got, want, "%s band [%d,%d) out_row0=%d pad=%s" % (what, rb, re, out_row0, pad))


def generic_path_cases():
    """Run in a child process by test_ycc420_generic_paths, with PYSP_DISABLE_TMA set."""
    from pysp_b200 import engine as eng
    H, W = 128, 184
    f32 = syn.scene(H, W, 41).astype(np.float32) / np.float32(16383.0)
    hdr = (f32 * np.where(np.random.default_rng(41).random((H, W)) < 0.2, np.float32(3.0), np.float32(1.0))).astype(np.float32)
    raw = syn.scene(126, 182, 42)                        # W = 2 mod 4: the flipped planes take the byte-by-byte store
    for src, pattern, stages, quality, kind in ((f32, "BGGR", 1, "best", "f32"), (hdr, "GRBG", 2, "best", "hdr"),
                                                (f32, "GBRG", 0, "fast", "f32"), (raw, "GBRG", 0, "best", "u16")):
        c = Case(0, src.shape[0], src.shape[1], pattern, kind, stages, quality, src, syn.BLACK, syn.WHITE, kind == "hdr",
                 [0, src.shape[0]])
        t = eng.to_device(src, pad_pitch=True)
        ref = ycc420(host(eng.develop(t, WB, M, out="srgb_u8", **develop_kw(c))))
        assert_planes_equal(develop_planes(eng, t, **develop_kw(c)), ref, describe(c))


@pytest.mark.parametrize("mode", ["1", "2", "3"])
def test_ycc420_generic_paths(mode):
    """the YCbCr planes through the generic loads (1), stores (2) or both (3), forced through the library's test hook,
    which is read once per process: hence a fresh process per mode"""
    code = "import sys\nsys.path[:0] = [%r, %r]\nimport test_gpu_ycc420 as t\nt.generic_path_cases()\nprint('ok')\n" % (
        ROOT, os.path.join(ROOT, "tests"))
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, PYSP_DISABLE_TMA=mode), capture_output=True, text=True)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-3000:]


@pytest.mark.parametrize("pattern", ["RGGB", "BGGR", "GRBG", "GBRG"])
def test_ycc420_nonfinite(eng, pattern):
    """+inf / -inf / NaN photosites: NaN quantises to 0 in srgb_u8, and the planes are the restatement of that"""
    d = golden("nonfinite48x64_s0")
    t = eng.to_device(np.ascontiguousarray(sp.to_rggb(d["sensor"], pattern)))
    s8 = host(eng.develop(t, WB, M, out="srgb_u8", stages=0, pattern=pattern))
    assert np.isnan(d["lin"]).any()
    assert_planes_equal(develop_planes(eng, t, stages=0, pattern=pattern), ycc420(s8), pattern)


def test_ycc420_config2_frame_and_jpeg(eng):
    """6000x4000, stages = 1 (the benchmark's frame): planes equal the restatement, and the JPEG Pillow writes from them
    is byte-identical to the one it writes from srgb_u8 (4:2:0, quality 95)"""
    from test_ycc420_cpu import _pil, assert_jpeg_identical
    from pysp_b200.colour import cam_to_rgb_matrix
    from pysp_b200.wb_cct import CameraWhiteBalance
    Image = _pil()
    cam_wb = CameraWhiteBalance(syn.MAT_XYZ_TO_CAM, syn.WHITE_XYZ)
    kw = dict(stages=1, black=syn.BLACK, white=syn.WHITE)
    wb, m = cam_wb.get_reciprocal_multipliers(), cam_to_rgb_matrix(cam_wb.get_matrix())
    t = eng.to_device(syn.scene(4000, 6000, 0))
    s8 = host(eng.develop(t, wb, m, out="srgb_u8", **kw))
    planes = tuple(host(p) for p in eng.develop(t, wb, m, out="ycc420", **kw))
    ref = ycc420(s8)
    assert_planes_equal(planes, ref, "6000x4000")
    assert_jpeg_identical(Image, s8, [planes[0], upsample2x2(planes[1]), upsample2x2(planes[2])], 2, "6000x4000")


def test_ycc420_frame_pipeline(eng):
    """FramePipeline(out="ycc420"): flat I420 host outputs of H*W*3/2 bytes, equal to engine.develop's planes"""
    from pysp_b200.pipeline import FramePipeline
    H, W = 500, 760
    kw = dict(stages=1, black=syn.BLACK, white=syn.WHITE)
    pipe = FramePipeline(H, W, WB, M, out="ycc420", **kw)
    assert pipe.d2h_bytes() == H * W * 3 // 2
    raws = [syn.scene(H, W, 60 + i) for i in range(5)]
    src = [torch.from_numpy(r.view(np.int16)).pin_memory() for r in raws]
    dst = [pipe.pinned_output() for _ in raws]
    assert dst[0].shape == (H * W * 3 // 2,) and dst[0].dtype == torch.uint8
    pipe.run(src, dst)
    for i, r in enumerate(raws):
        want = np.concatenate([p.reshape(-1) for p in develop_planes(eng, eng.to_device(r), **kw)])
        assert np.array_equal(dst[i].numpy(), want), "frame %d" % i
