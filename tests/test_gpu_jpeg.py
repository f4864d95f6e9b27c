"""pysp_jpeg_encode_ycc420 on the device: the file equals the NumPy restatement (tests/jpeg_ref.py) and Pillow's JPEG of the
planes byte for byte on the CPU suite's matrix of qualities, contents and sizes, from planes with padded pitches, and writes
nothing past its length; develop(out="ycc420") + encode of the benchmark's 6000x4000 frame equals Pillow's JPEG of
develop(out="srgb_u8"); a 100 MP frame equals Pillow's JPEG of its planes; a frame of more than 2^32 bits of entropy-coded data
is exact (64-bit offsets); a side stream and a CUDA graph replay give the same bytes; FramePipeline(out="jpeg") delivers the
engine's files."""
import numpy as np
import pytest
import torch

import jpeg_ref as J
from pysp_b200 import synthetic as syn
from test_jpeg_cpu import CONTENTS, QUALITIES, content, pillow_planes, pillow_rgb
from test_tile_logic import M, WB

pytestmark = pytest.mark.gpu
SENTINEL = 0xA5


@pytest.fixture(scope="module")
def eng():
    from pysp_b200 import engine, _capi
    assert torch.cuda.is_available(), "these tests need the GPU"
    _capi.lib()
    return engine


def device_planes(Y, Cb, Cr, pad=(0, 0)):
    """CUDA views of the planes inside buffers `pad` bytes wider than each plane row (row pitch above the width)"""
    out = []
    for p, k in ((Y, 0), (Cb, 1), (Cr, 1)):
        buf = torch.full((p.shape[0], p.shape[1] + pad[k]), SENTINEL, dtype=torch.uint8, device="cuda")
        buf[:, :p.shape[1]] = torch.from_numpy(np.ascontiguousarray(p)).cuda()
        out.append(buf[:, :p.shape[1]])
    return tuple(out)


def encode_on_device(eng, planes, q, stream=None):
    """the file as bytes; the output buffer has 64 sentinel bytes past the capacity, and none past the file may change"""
    H, W = planes[0].shape
    cap = eng.jpeg_max_bytes(H, W)
    buf = torch.full((cap + 64,), SENTINEL, dtype=torch.uint8, device=planes[0].device)
    out, n = eng.encode_jpeg(planes, q, out_tensor=buf, stream=stream)
    assert out.data_ptr() == buf.data_ptr()
    torch.cuda.synchronize()
    n = int(n.item())
    host = buf.cpu().numpy()
    assert 0 < n <= cap and (host[n:] == SENTINEL).all(), "bytes past the file were written"
    return host[:n].tobytes()


def matrix_cases():
    cases = [((48, 64), kind, q) for q in QUALITIES for kind in CONTENTS]
    for i, (hm, wm) in enumerate((h, w) for h in range(0, 16, 2) for w in range(0, 16, 2)):
        cases.append(((32 + hm, 48 + wm), CONTENTS[i % len(CONTENTS)], QUALITIES[i % len(QUALITIES)]))
    cases += [(s, "random", q) for s in ((2, 2), (2, 4), (4, 2), (2, 18), (18, 2), (6, 6), (10, 16)) for q in (1, 75, 100)]
    return cases


def test_matrix_equals_restatement_and_pillow(eng):
    pads = ((0, 0), (4, 2), (3, 1), (64, 33))
    for i, ((H, W), kind, q) in enumerate(matrix_cases()):
        Y, Cb, Cr = content(kind, H, W, i)
        got = encode_on_device(eng, device_planes(Y, Cb, Cr, pads[i % len(pads)]), q)
        what = "%s %dx%d q=%d pad=%s" % (kind, H, W, q, pads[i % len(pads)])
        assert got == J.encode(Y, Cb, Cr, q), what + ": differs from the restatement"
        assert got == pillow_planes(Y, Cb, Cr, q), what + ": differs from Pillow"


def test_bench_frame_equals_pillow_of_srgb(eng):
    """6000x4000, stages = 1 (the benchmark's frame): develop(out="ycc420") + encode_jpeg is Pillow's JPEG of the srgb_u8
    image of the same develop, at qualities 75, 90 and 95"""
    from pysp_b200.colour import cam_to_rgb_matrix
    from pysp_b200.wb_cct import CameraWhiteBalance
    cam_wb = CameraWhiteBalance(syn.MAT_XYZ_TO_CAM, syn.WHITE_XYZ)
    kw = dict(stages=1, black=syn.BLACK, white=syn.WHITE)
    wb, m = cam_wb.get_reciprocal_multipliers(), cam_to_rgb_matrix(cam_wb.get_matrix())
    t = eng.to_device(syn.scene(4000, 6000, 0))
    s8 = eng.develop(t, wb, m, out="srgb_u8", **kw).cpu().numpy()
    planes = eng.develop(t, wb, m, out="ycc420", **kw)
    for q in (75, 90, 95):
        assert encode_on_device(eng, planes, q) == pillow_rgb(s8, q), "q=%d" % q


def test_100mp_frame_equals_pillow_of_planes(eng):
    """11548 x 8660 (W % 16 = 12: partial MCUs and dummy blocks along the right edge), smooth content with noise"""
    H, W = 8660, 11548
    g = torch.Generator(device="cuda").manual_seed(5)
    yy = torch.arange(H, device="cuda", dtype=torch.float32)[:, None]
    xx = torch.arange(W, device="cuda", dtype=torch.float32)[None, :]
    Y = (128 + 90 * torch.sin(xx / 97) * torch.cos(yy / 61) + torch.randint(-6, 7, (H, W), device="cuda", generator=g)).clamp(0, 255)
    Y = Y.to(torch.uint8)
    Cb = (Y[::2, ::2] // 2 + 64).contiguous()
    Cr = (255 - Y[1::2, 1::2]).contiguous()
    got = encode_on_device(eng, (Y, Cb, Cr), 90)
    assert got == pillow_planes(Y.cpu().numpy(), Cb.cpu().numpy(), Cr.cpu().numpy(), 90)


def test_more_than_2_to_32_bits(eng):
    """Every MCU of the frame is one random 16x16 tile, so the entropy-coded data is the first MCU's bits followed by the same
    bits B2 for every later MCU.  The frame is sized so that their total exceeds 2^32; the stuffed bytes are undone on the
    device and compared with the periodic continuation of the restatement of a 17-MCU strip."""
    q = 100
    rng = np.random.default_rng(9)
    tY = rng.integers(0, 256, (16, 16), dtype=np.uint8)
    tC = [rng.integers(0, 256, (8, 8), dtype=np.uint8) for _ in range(2)]
    strip = (np.tile(tY, (1, 17)), np.tile(tC[0], (1, 17)), np.tile(tC[1], (1, 17)))
    counts, bits = J.entropy_bits(J.coefficients(*strip, q))
    mcu = counts.reshape(-1, 6).sum(axis=1)
    b1, b2 = int(mcu[0]), int(mcu[1])
    assert (mcu[1:] == b2).all()
    cols = 1024
    rows = -(-((1 << 32) + (1 << 28) - b1) // (b2 * cols)) + 1
    H, W = 16 * rows, 16 * cols
    n_mcu = rows * cols
    total = b1 + (n_mcu - 1) * b2
    assert total > 1 << 32
    Y = torch.from_numpy(tY).cuda().repeat(rows, cols)
    Cb, Cr = (torch.from_numpy(t).cuda().repeat(rows, cols) for t in tC)
    out, n = eng.encode_jpeg((Y, Cb, Cr), q)
    torch.cuda.synchronize()
    n = int(n.item())
    assert bytes(out[:J.HEADER_BYTES].cpu().numpy()) == J.header(H, W, q)
    assert bytes(out[n - 2:n].cpu().numpy()) == b"\xff\xd9"
    data = out[J.HEADER_BYTES:n - 2]
    stuffed = torch.zeros_like(data, dtype=torch.bool)
    stuffed[1:] = (data[1:] == 0) & (data[:-1] == 0xFF)
    data = data[~stuffed]
    N = (total + 7) // 8
    assert data.numel() == N, "stream length"
    small = np.packbits(bits)                    # b1 + 16 * b2 bits: whole bytes cover one byte period b2 after j0
    j0, period = -(-b1 // 8), b2
    assert j0 + period <= len(small) - 1
    head = torch.from_numpy(small[:j0].copy()).cuda()
    cyc = torch.from_numpy(small[j0:j0 + period].copy()).cuda()
    assert torch.equal(data[:j0], head)
    body = data[j0:N - 1].view(-1)
    reps = -(-body.numel() // period)
    want = cyc.repeat(reps)[:body.numel()]
    assert torch.equal(body, want), "periodic part"
    pad = 8 * N - total
    last = int(cyc[(N - 1 - j0) % period]) | ((1 << pad) - 1)
    assert int(data[N - 1]) == last


def test_side_stream_and_graph_replay(eng):
    Y, Cb, Cr = content("random", 66, 130, 3)
    planes = device_planes(Y, Cb, Cr, (5, 3))
    want = J.encode(Y, Cb, Cr, 85)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        buf, n = eng.encode_jpeg(planes, 85, stream=s)
    s.synchronize()
    assert bytes(buf[:int(n.item())].cpu().numpy()) == want, "side stream"

    cap = eng.jpeg_max_bytes(66, 130)
    gbuf = torch.empty(cap, dtype=torch.uint8, device="cuda")
    eng.encode_jpeg(planes, 85, out_tensor=gbuf)             # warm-up outside the capture
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        _, gn = eng.encode_jpeg(planes, 85, out_tensor=gbuf)
    gbuf.fill_(0)
    g.replay()
    torch.cuda.synchronize()
    assert bytes(gbuf[:int(gn.item())].cpu().numpy()) == want, "graph replay"
    Y2, Cb2, Cr2 = content("smooth", 66, 130, 4)               # new content in the same planes, same graph
    for dst, src in zip(planes, (Y2, Cb2, Cr2)):
        dst.copy_(torch.from_numpy(src).cuda())
    g.replay()
    torch.cuda.synchronize()
    assert bytes(gbuf[:int(gn.item())].cpu().numpy()) == J.encode(Y2, Cb2, Cr2, 85), "graph replay on new planes"


def test_frame_pipeline_jpeg(eng):
    """FramePipeline(out="jpeg"): run returns the lengths, and each host output holds develop(out="ycc420") + encode_jpeg"""
    from pysp_b200.pipeline import FramePipeline
    H, W = 500, 760
    kw = dict(stages=1, black=syn.BLACK, white=syn.WHITE)
    for depth in (3, 1):
        pipe = FramePipeline(H, W, WB, M, out="jpeg", jpeg_quality=90, depth=depth, **kw)
        raws = [syn.scene(H, W, 70 + i) for i in range(5)]
        src = [torch.from_numpy(r.view(np.int16)).pin_memory() for r in raws]
        dst = [pipe.pinned_output() for _ in raws]
        assert dst[0].numel() == eng.jpeg_max_bytes(H, W)
        lens = pipe.run(src, dst)
        for i, r in enumerate(raws):
            planes = eng.develop(eng.to_device(r), WB, M, out="ycc420", **kw)
            buf, n = eng.encode_jpeg(planes, 90)
            want = bytes(buf[:int(n.item())].cpu().numpy())
            assert lens[i] == len(want) and bytes(dst[i][:lens[i]].numpy()) == want, "depth %d frame %d" % (depth, i)
