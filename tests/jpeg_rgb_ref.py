"""NumPy restatement of pysp_jpeg_encode_rgb (include/pysp_b200.h): the baseline JPEG libjpeg-turbo writes from an 8-bit RGB
image of any size at 4:4:4, 4:2:2 or 4:2:0 with its defaults.  Built on tests/jpeg_ref.py (tables, DCT, quantisation, Huffman
symbols, stuffing) and tests/ycc420_ref.py (colour conversion); tests/test_jpeg_rgb_cpu.py pins it to Pillow byte for byte.
Also the RGB test images and Pillow's encode of them."""
import io

import numpy as np

import jpeg_ref as J
from ycc420_ref import h2v2, ycc_full

SUBSAMPLINGS = (0, 1, 2)                        # Pillow's integers: 4:4:4, 4:2:2, 4:2:0
SAMPLING = {0: (1, 1), 1: (2, 1), 2: (2, 2)}    # (h, v): Y blocks per MCU across / down
NAMES = {0: "4:4:4", 1: "4:2:2", 2: "4:2:0"}


def mcus(H, W, s):
    h, v = SAMPLING[s]
    return -(-H // (8 * v)), -(-W // (8 * h))


def planes(S, s):
    """(Y [H, W], Cb, Cr [ceil(H/v), 8 * mx]) uint8: what the convert phase stores.  Full-resolution chroma with its last
    column repeated out to 8h * mx columns and its last row out to a multiple of v rows, then downsampled (jcsample.c)."""
    h, v = SAMPLING[s]
    H, W = S.shape[:2]
    _, mx = mcus(H, W, s)
    Y, cb, cr = ycc_full(S)

    def down(c):
        c = np.pad(c, ((0, -H % v), (0, 8 * h * mx - W)), mode="edge")
        if h == 1:
            return c
        if v == 1:                              # h2v1_downsample: bias 0, 1, 0, 1, ...
            t = c[:, 0::2] + c[:, 1::2]
            return (t + (np.arange(t.shape[1]) & 1)) >> 1
        return h2v2(c)

    return Y.astype(np.uint8), down(cb).astype(np.uint8), down(cr).astype(np.uint8)


def coefficients(Y, Cb, Cr, quality, s):
    """quantised coefficients [n_blocks, 64] in zigzag order, MCU order (h*v Y slots in raster order, Cb, Cr); dummy Y slots
    carry the DC of the slot before them and zero AC.  Cb / Cr are the convert phase's planes: the block loader repeats their
    last row out to 8 * my rows."""
    h, v = SAMPLING[s]
    H, W = Y.shape
    my, mx = mcus(H, W, s)
    ny = h * v
    d = 8 * J.quant_tables(quality)

    def q(P, t):
        b = J._blocks(P)
        c = J.fdct_islow(b.reshape(-1, 8, 8)).reshape(b.shape[0], b.shape[1], 64)
        return J.quantize(c, d[t])[..., J.ZIGZAG]

    zy = q(Y, 0)
    out = np.zeros((my, mx, ny + 2, 64), dtype=np.int64)
    real = np.zeros((my, mx, ny), dtype=bool)
    for k in range(ny):
        part = zy[k // h::v, k % h::h]
        out[:part.shape[0], :part.shape[1], k] = part
        real[:part.shape[0], :part.shape[1], k] = True
    for k in range(1, ny):
        out[..., k, 0] = np.where(real[..., k], out[..., k, 0], out[..., k - 1, 0])
    out[..., ny, :] = q(Cb, 1)
    out[..., ny + 1, :] = q(Cr, 1)
    return out.reshape(-1, 64)


def dc_differences(zz, s):
    """DC difference of each block against the previous block of its component (MCU order)"""
    h, v = SAMPLING[s]
    ny = h * v
    dc = zz[:, 0].reshape(-1, ny + 2)
    diff = np.empty_like(dc)
    diff[:, :ny] = np.diff(dc[:, :ny].reshape(-1), prepend=0).reshape(-1, ny)
    for k in (ny, ny + 1):
        diff[:, k] = np.diff(dc[:, k], prepend=0)
    return diff.reshape(-1)


def entropy_bits(zz, s, chunk=16384):
    """(bits per block, the scan's bit string as uint8 0/1), as jpeg_ref.entropy_bits for an MCU of h*v + 2 blocks"""
    h, v = SAMPLING[s]
    diff = dc_differences(zz, s)
    table = (np.arange(zz.shape[0]) % (h * v + 2) >= h * v).astype(np.int64)
    counts = np.zeros(zz.shape[0], dtype=np.int64)
    parts = []
    for b0 in range(0, zz.shape[0], chunk):
        sl = slice(b0, b0 + chunk)
        vals = np.zeros((len(zz[sl]), 65), dtype=np.uint64)
        lens = np.zeros((len(zz[sl]), 65), dtype=np.int64)
        for t in (0, 1):
            m = table[sl] == t
            vals[m], lens[m] = J._block_items(zz[sl][m], diff[sl][m], t)
        counts[sl] = lens.sum(axis=1)
        keep = lens.reshape(-1) > 0
        val, ln = vals.reshape(-1)[keep], lens.reshape(-1)[keep]
        rep = np.repeat(np.arange(len(val)), ln)
        start = np.cumsum(ln) - ln
        shift = (ln[rep] - 1 - (np.arange(len(rep)) - start[rep])).astype(np.uint64)
        parts.append(((val[rep] >> shift) & np.uint64(1)).astype(np.uint8))
    return counts, np.concatenate(parts)


def header(H, W, quality, s):
    """jpeg_ref.header with the Y sampling byte of SOF0 (offset 169) set to (h << 4) | v"""
    h, v = SAMPLING[s]
    b = bytearray(J.header(H, W, quality))
    b[169] = (h << 4) | v
    return bytes(b)


def encode(S, quality, s):
    """the JFIF file of a uint8 [H, W, 3] RGB image"""
    H, W = S.shape[:2]
    _, bits = entropy_bits(coefficients(*planes(S, s), quality, s), s)
    return header(H, W, quality, s) + J.stuff(bits) + b"\xff\xd9"


def max_bytes(H, W, s):
    """pysp_jpeg_rgb_max_bytes"""
    h, v = SAMPLING[s]
    my, mx = mcus(H, W, s)
    return J.HEADER_BYTES + 2 * -(-(h * v + 2) * my * mx * (11 + 11 + 63 * (16 + 10)) // 8) + 2


def pillow_rgb(S, quality, s):
    """libjpeg's JPEG of the RGB image through Pillow"""
    from PIL import Image
    b = io.BytesIO()
    Image.fromarray(np.ascontiguousarray(S), "RGB").save(b, format="JPEG", quality=quality, subsampling=s)
    return b.getvalue()


def rgb_content(kind, H, W, seed=0):
    """uint8 [H, W, 3] test image of any size: the content kinds of tests/test_jpeg_cpu.py, in RGB"""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:H, 0:W]
    if kind == "random":
        return rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    if kind == "smooth":
        a = 128 + 100 * np.sin(xx / 13.0 + seed) * np.cos(yy / 9.0)
        return np.stack([a, 255 - a, (a + 64) % 256], axis=-1).astype(np.uint8)
    if kind == "flat":
        # a constant colour with a few isolated specks: long zero runs (ZRL), and the dummy blocks' DC
        S = np.empty((H, W, 3), dtype=np.uint8)
        S[...] = (90, 140, 100)
        n = max(1, H * W // 97)
        S.reshape(-1, 3)[rng.integers(0, H * W, n)] = rng.integers(0, 256, (n, 3), dtype=np.uint8)
        return S
    if kind == "extreme":
        # 0/255 checkerboards inside 8x8 blocks alternating with flat black / white blocks, with opposite colours in the
        # chroma: the largest AC magnitudes and DC differences
        blk = ((yy // 8) + (xx // 8)) % 3
        a = np.where(blk == 0, ((yy + xx) & 1) * 255, np.where(blk == 1, 0, 255))
        return np.stack([a, 255 - a, a], axis=-1).astype(np.uint8)
    if kind == "ffdense":
        # a +-2 checkerboard in grey: many 0xFF bytes in the entropy-coded data at quality 90
        a = 128 + 2 * (((yy + xx) & 1) * 2 - 1)
        return np.stack([a, a, a], axis=-1).astype(np.uint8)
    raise ValueError(kind)
