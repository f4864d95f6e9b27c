"""pysp_jpeg_encode_rgb on the device at 4:4:4, 4:2:2 and 4:2:0: the file equals the NumPy restatement (tests/jpeg_rgb_ref.py)
and Pillow's JPEG of the RGB image byte for byte on the CPU suite's matrix of qualities, contents and sizes (every residue of H
and W mod 16, odd ones included, down to 1x1), from images with padded row pitches of any residue, and writes nothing past its
length; develop(out="srgb_u8") + encode_jpeg_rgb of the benchmark's 6000x4000 frame and of an odd-sized crop of it equals Pillow;
at 4:2:0 with W % 16 == 0 it equals encode_jpeg of the ycc420 planes of the same develop; a 100 MP frame at 4:4:4 equals Pillow;
a side stream and a CUDA graph replay give the same bytes; FramePipeline(out="jpeg") delivers the engine's files at every
jpeg_subsampling; invalid input raises ValueError."""
import numpy as np
import pytest
import torch

import jpeg_rgb_ref as R
from pysp_b200 import synthetic as syn
from test_jpeg_cpu import CONTENTS, QUALITIES
from test_tile_logic import M, WB

pytestmark = pytest.mark.gpu
SENTINEL = 0xA5


@pytest.fixture(scope="module")
def eng():
    from pysp_b200 import engine, _capi
    assert torch.cuda.is_available(), "these tests need the GPU"
    _capi.lib()
    return engine


def device_rgb(S, pad=0):
    """a CUDA [H, W, 3] view with strides (3W + pad, 3, 1) over a sentinel buffer holding S"""
    H, W = S.shape[:2]
    buf = torch.full((H, 3 * W + pad), SENTINEL, dtype=torch.uint8, device="cuda")
    buf[:, :3 * W] = torch.from_numpy(np.ascontiguousarray(S).reshape(H, 3 * W)).cuda()
    return buf.as_strided((H, W, 3), (3 * W + pad, 3, 1))


def encode_on_device(eng, rgb, q, s, stream=None):
    """the file as bytes; the output buffer has 64 sentinel bytes past the capacity, and none past the file may change"""
    H, W = rgb.shape[:2]
    cap = eng.jpeg_rgb_max_bytes(H, W, s)
    buf = torch.full((cap + 64,), SENTINEL, dtype=torch.uint8, device=rgb.device)
    out, n = eng.encode_jpeg_rgb(rgb, q, s, out_tensor=buf, stream=stream)
    assert out.data_ptr() == buf.data_ptr()
    torch.cuda.synchronize()
    n = int(n.item())
    host = buf.cpu().numpy()
    assert 0 < n <= cap and (host[n:] == SENTINEL).all(), "bytes past the file were written"
    return host[:n].tobytes()


def matrix_cases():
    cases = [((48, 64), kind, q) for q in QUALITIES for kind in CONTENTS]
    for i, (hm, wm) in enumerate((h, w) for h in range(16) for w in range(16)):
        cases.append(((32 + hm, 48 + wm), CONTENTS[i % len(CONTENTS)], QUALITIES[i % len(QUALITIES)]))
    tiny = ((1, 1), (1, 2), (2, 1), (1, 17), (17, 1), (1, 100), (100, 1), (7, 9))
    cases += [(sh, "random", q) for sh in tiny for q in (1, 75, 100)]
    return cases


@pytest.mark.parametrize("s", R.SUBSAMPLINGS)
def test_matrix_equals_restatement_and_pillow(eng, s):
    pads = (0, 1, 5, 64, 7, 2)                  # row pitches 3W + pad: multiples of 3 or 4 and neither
    for i, ((H, W), kind, q) in enumerate(matrix_cases()):
        S = R.rgb_content(kind, H, W, i)
        pad = pads[i % len(pads)]
        got = encode_on_device(eng, device_rgb(S, pad), q, s)
        what = "%s %s %dx%d q=%d pitch=%d" % (R.NAMES[s], kind, H, W, q, 3 * W + pad)
        assert got == R.encode(S, q, s), what + ": differs from the restatement"
        assert got == R.pillow_rgb(S, q, s), what + ": differs from Pillow"


@pytest.fixture(scope="module")
def bench_frame(eng):
    """the benchmark's 6000x4000 frame, stages = 1: (srgb_u8 CUDA tensor, ycc420 planes) of one develop each"""
    from pysp_b200.colour import cam_to_rgb_matrix
    from pysp_b200.wb_cct import CameraWhiteBalance
    cam_wb = CameraWhiteBalance(syn.MAT_XYZ_TO_CAM, syn.WHITE_XYZ)
    kw = dict(stages=1, black=syn.BLACK, white=syn.WHITE)
    wb, m = cam_wb.get_reciprocal_multipliers(), cam_to_rgb_matrix(cam_wb.get_matrix())
    t = eng.to_device(syn.scene(4000, 6000, 0))
    return eng.develop(t, wb, m, out="srgb_u8", **kw), eng.develop(t, wb, m, out="ycc420", **kw)


def test_bench_frame_equals_pillow(eng, bench_frame):
    """develop(out="srgb_u8") + encode_jpeg_rgb is Pillow's JPEG of the image at qualities 75 / 90 / 95 and every subsampling"""
    s8 = bench_frame[0]
    host = s8.cpu().numpy()
    for s in R.SUBSAMPLINGS:
        for q in (75, 90, 95):
            assert encode_on_device(eng, s8, q, s) == R.pillow_rgb(host, q, s), "%s q=%d" % (R.NAMES[s], q)


def test_odd_crop_equals_pillow(eng, bench_frame):
    """a 3999x5997 crop (a view with the frame's pitch): odd H and W, partial MCUs, the chroma edge rule at both edges"""
    crop = bench_frame[0][1:4000, 2:5999]
    assert crop.shape[:2] == (3999, 5997) and crop.stride() == (18000, 3, 1)
    host = crop.cpu().numpy()
    for s in R.SUBSAMPLINGS:
        assert encode_on_device(eng, crop, 90, s) == R.pillow_rgb(host, 90, s), R.NAMES[s]


def test_420_equals_planes_route(eng, bench_frame):
    """W = 6000 is a multiple of 16: at 4:2:0 the RGB route and encode_jpeg of the ycc420 planes write the same file"""
    s8, planes = bench_frame
    for q in (75, 95):
        buf, n = eng.encode_jpeg(planes, q)
        torch.cuda.synchronize()
        assert encode_on_device(eng, s8, q, "4:2:0") == bytes(buf[:int(n.item())].cpu().numpy()), "q=%d" % q


def test_100mp_frame_444_equals_pillow(eng):
    """11548 x 8660 at 4:4:4 (W % 8 = 4: partial blocks along the right edge), smooth content with noise"""
    H, W = 8660, 11548
    g = torch.Generator(device="cuda").manual_seed(5)
    yy = torch.arange(H, device="cuda", dtype=torch.float32)[:, None, None]
    xx = torch.arange(W, device="cuda", dtype=torch.float32)[None, :, None]
    ph = torch.tensor([0.0, 1.0, 2.0], device="cuda")[None, None, :]
    S = 128 + 90 * torch.sin(xx / 97 + ph) * torch.cos(yy / 61) + torch.randint(-6, 7, (H, W, 3), device="cuda", generator=g)
    S = S.clamp(0, 255).to(torch.uint8)
    assert encode_on_device(eng, S, 90, "4:4:4") == R.pillow_rgb(S.cpu().numpy(), 90, 0)


def test_side_stream_and_graph_replay(eng):
    S = R.rgb_content("random", 67, 131, 3)
    rgb = device_rgb(S, 5)
    for s in R.SUBSAMPLINGS:
        want = R.encode(S, 85, s)
        st = torch.cuda.Stream()
        st.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(st):
            buf, n = eng.encode_jpeg_rgb(rgb, 85, s, stream=st)
        st.synchronize()
        assert bytes(buf[:int(n.item())].cpu().numpy()) == want, "side stream %s" % R.NAMES[s]

        gbuf = torch.empty(eng.jpeg_rgb_max_bytes(67, 131, s), dtype=torch.uint8, device="cuda")
        eng.encode_jpeg_rgb(rgb, 85, s, out_tensor=gbuf)          # warm-up outside the capture
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            _, gn = eng.encode_jpeg_rgb(rgb, 85, s, out_tensor=gbuf)
        gbuf.fill_(0)
        g.replay()
        torch.cuda.synchronize()
        assert bytes(gbuf[:int(gn.item())].cpu().numpy()) == want, "graph replay %s" % R.NAMES[s]
        S2 = R.rgb_content("smooth", 67, 131, 4 + s)               # new content in the same image, same graph
        rgb.copy_(torch.from_numpy(S2).cuda())
        g.replay()
        torch.cuda.synchronize()
        assert bytes(gbuf[:int(gn.item())].cpu().numpy()) == R.encode(S2, 85, s), "graph replay on a new image %s" % R.NAMES[s]
        rgb.copy_(torch.from_numpy(S).cuda())


def test_invalid_input_raises(eng):
    rgb = device_rgb(R.rgb_content("random", 16, 16), 0)
    bad = [dict(rgb=rgb.cpu()), dict(rgb=rgb[..., :2]), dict(rgb=rgb.to(torch.int16)), dict(rgb=rgb.permute(1, 0, 2)),
           dict(rgb=rgb[:, ::2]), dict(subsampling="4:1:1"), dict(subsampling=3), dict(subsampling=True), dict(quality=0),
           dict(quality=101), dict(out_tensor=torch.empty(100, dtype=torch.uint8, device="cuda")),
           dict(out_tensor=torch.empty(1 << 20, dtype=torch.int32, device="cuda"))]
    for over in bad:
        a = dict(rgb=rgb, quality=75, subsampling="4:2:0", out_tensor=None)
        a.update(over)
        with pytest.raises(ValueError):
            eng.encode_jpeg_rgb(a["rgb"], a["quality"], a["subsampling"], out_tensor=a["out_tensor"])
    with pytest.raises(ValueError):
        eng.jpeg_rgb_max_bytes(0, 16, 0)


@pytest.mark.parametrize("subsampling", ["4:4:4", "4:2:2", "4:2:0", 0, 1])
def test_frame_pipeline_jpeg_subsampling(eng, subsampling):
    """FramePipeline(out="jpeg", jpeg_subsampling=...): each host output holds develop(out="srgb_u8") + encode_jpeg_rgb (4:4:4,
    4:2:2), or develop(out="ycc420") + encode_jpeg as before (4:2:0); the outputs are sized by the matching max-bytes helper"""
    from pysp_b200.pipeline import FramePipeline
    H, W = 500, 760
    s = eng.jpeg_subsampling(subsampling)
    kw = dict(stages=1, black=syn.BLACK, white=syn.WHITE)
    for depth in (3, 1):
        pipe = FramePipeline(H, W, WB, M, out="jpeg", jpeg_quality=90, jpeg_subsampling=subsampling, depth=depth, **kw)
        raws = [syn.scene(H, W, 70 + i) for i in range(4)]
        src = [torch.from_numpy(r.view(np.int16)).pin_memory() for r in raws]
        dst = [pipe.pinned_output() for _ in raws]
        assert dst[0].numel() == (eng.jpeg_max_bytes(H, W) if s == 2 else eng.jpeg_rgb_max_bytes(H, W, s))
        lens = pipe.run(src, dst)
        for i, r in enumerate(raws):
            t = eng.to_device(r)
            if s == 2:
                buf, n = eng.encode_jpeg(eng.develop(t, WB, M, out="ycc420", **kw), 90)
            else:
                buf, n = eng.encode_jpeg_rgb(eng.develop(t, WB, M, out="srgb_u8", **kw), 90, s)
            want = bytes(buf[:int(n.item())].cpu().numpy())
            assert lens[i] == len(want) and bytes(dst[i][:lens[i]].numpy()) == want, "depth %d frame %d" % (depth, i)
