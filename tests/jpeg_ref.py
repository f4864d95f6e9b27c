"""NumPy restatement of pysp_jpeg_encode_ycc420 (include/pysp_b200.h): the baseline JPEG libjpeg-turbo writes from YCbCr 4:2:0
planes with its defaults (ISLOW DCT, Annex K tables, no restart markers, JFIF 1.01).  It builds its own header and tables;
tests/test_jpeg_cpu.py pins it to Pillow byte for byte.  Vectorised over blocks: a 24 MP frame takes seconds."""
import numpy as np

# Annex K.1, natural order
STD_QUANT = np.array([
    [16, 11, 10, 16, 24, 40, 51, 61, 12, 12, 14, 19, 26, 58, 60, 55, 14, 13, 16, 24, 40, 57, 69, 56,
     14, 17, 22, 29, 51, 87, 80, 62, 18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55, 64, 81, 104, 113, 92,
     49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99],
    [17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99, 99, 99,
     47, 66, 99, 99] + [99] * 36], dtype=np.int64)

# zigzag position -> natural index
ZIGZAG = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14,
                   21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53,
                   60, 61, 54, 47, 55, 62, 63])

# Annex K.3: (BITS, HUFFVAL) of DC luma, AC luma, DC chroma, AC chroma (the DHT order)
_AC_LUMA_VALS = bytes.fromhex(
    "01020300041105122131410613516107227114328191a1082342b1c11552d1f02433627282090a161718191a25262728292a3435363738393a"
    "434445464748494a535455565758595a636465666768696a737475767778797a838485868788898a92939495969798999aa2a3a4a5a6a7a8a9"
    "aab2b3b4b5b6b7b8b9bac2c3c4c5c6c7c8c9cad2d3d4d5d6d7d8d9dae1e2e3e4e5e6e7e8e9eaf1f2f3f4f5f6f7f8f9fa")
_AC_CHROMA_VALS = bytes.fromhex(
    "000102031104052131061241510761711322328108144291a1b1c109233352f0156272d10a162434e125f11718191a262728292a35363738"
    "393a434445464748494a535455565758595a636465666768696a737475767778797a82838485868788898a92939495969798999aa2a3a4a5a6"
    "a7a8a9aab2b3b4b5b6b7b8b9bac2c3c4c5c6c7c8c9cad2d3d4d5d6d7d8d9dae2e3e4e5e6e7e8e9eaf2f3f4f5f6f7f8f9fa")
HUFF_SPECS = [
    ([0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0], list(range(12))),
    ([0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 125], list(_AC_LUMA_VALS)),
    ([0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0], list(range(12))),
    ([0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 119], list(_AC_CHROMA_VALS)),
]
HEADER_BYTES = 623


def huffman_codes(bits, vals):
    """canonical codes (Annex C): (code[256], length[256]) by symbol, length 0 where the table has no code"""
    code, length = np.zeros(256, dtype=np.uint64), np.zeros(256, dtype=np.int64)
    c, k = 0, 0
    for n in range(1, 17):
        for _ in range(bits[n - 1]):
            code[vals[k]], length[vals[k]] = c, n
            c += 1
            k += 1
        c <<= 1
    return code, length


_CODES = [huffman_codes(*s) for s in HUFF_SPECS]          # DC0, AC0, DC1, AC1


def quant_tables(quality):
    """[2, 64] natural order (jcparam.c, force_baseline)"""
    scale = 5000 // quality if quality < 50 else 200 - 2 * quality
    return np.clip((STD_QUANT * scale + 50) // 100, 1, 255)


def header(H, W, quality):
    q = quant_tables(quality)
    h = bytearray(b"\xff\xd8\xff\xe0\x00\x10JFIF\x00\x01\x01\x00\x00\x01\x00\x01\x00\x00")
    for t in range(2):
        h += bytes([0xFF, 0xDB, 0, 67, t]) + bytes(q[t][ZIGZAG].astype(np.uint8))
    h += bytes([0xFF, 0xC0, 0, 17, 8, H >> 8, H & 255, W >> 8, W & 255, 3, 1, 0x22, 0, 2, 0x11, 1, 3, 0x11, 1])
    for t, (bits, vals) in enumerate(HUFF_SPECS):
        h += bytes([0xFF, 0xC4, 0, 3 + 16 + len(vals), ((t & 1) << 4) | (t >> 1)]) + bytes(bits) + bytes(vals)
    h += bytes([0xFF, 0xDA, 0, 12, 3, 1, 0x00, 2, 0x11, 3, 0x11, 0, 63, 0])
    assert len(h) == HEADER_BYTES
    return bytes(h)


def _descale(x, n):
    return (x + (1 << (n - 1))) >> n


def _fdct_1d(d, first):
    """jfdctint.c (ISLOW) along the last axis of an int64 array"""
    cb, p1 = 13, 2
    sh = cb - p1 if first else cb + p1
    d = [d[..., i] for i in range(8)]
    t0, t7, t1, t6 = d[0] + d[7], d[0] - d[7], d[1] + d[6], d[1] - d[6]
    t2, t5, t3, t4 = d[2] + d[5], d[2] - d[5], d[3] + d[4], d[3] - d[4]
    t10, t13, t11, t12 = t0 + t3, t0 - t3, t1 + t2, t1 - t2
    o = [None] * 8
    o[0] = (t10 + t11) << p1 if first else _descale(t10 + t11, p1)
    o[4] = (t10 - t11) << p1 if first else _descale(t10 - t11, p1)
    z1 = (t12 + t13) * 4433
    o[2] = _descale(z1 + t13 * 6270, sh)
    o[6] = _descale(z1 - t12 * 15137, sh)
    z1, z2, z3, z4 = t4 + t7, t5 + t6, t4 + t6, t5 + t7
    z5 = (z3 + z4) * 9633
    t4, t5, t6, t7 = t4 * 2446, t5 * 16819, t6 * 25172, t7 * 12299
    z1, z2, z3, z4 = z1 * -7373, z2 * -20995, z3 * -16069 + z5, z4 * -3196 + z5
    o[7], o[5] = _descale(t4 + z1 + z3, sh), _descale(t5 + z2 + z4, sh)
    o[3], o[1] = _descale(t6 + z2 + z3, sh), _descale(t7 + z1 + z4, sh)
    return np.stack(o, axis=-1)


def fdct_islow(blocks):
    """[n, 8, 8] samples - 128 (int64) -> [n, 8, 8] ISLOW coefficients (scaled by 8)"""
    rows = _fdct_1d(blocks, True)
    return np.swapaxes(_fdct_1d(np.swapaxes(rows, 1, 2), False), 1, 2)


def quantize(c, d):
    r = (np.abs(c) + d // 2) // d
    return np.where(c < 0, -r, r)


def _blocks(P):
    """edge-padded [by, bx, 8, 8] int64 blocks of a plane"""
    h, w = P.shape
    P = np.pad(np.asarray(P), ((0, -h % 8), (0, -w % 8)), mode="edge").astype(np.int64) - 128
    return P.reshape(P.shape[0] // 8, 8, P.shape[1] // 8, 8).swapaxes(1, 2)


def coefficients(Y, Cb, Cr, quality):
    """quantised coefficients [n_blocks, 64] in zigzag order, blocks in MCU order (Y00 Y01 Y10 Y11 Cb Cr); dummy Y slots
    carry the DC of the slot before them and zero AC"""
    H, W = Y.shape
    my, mx = -(-H // 16), -(-W // 16)
    d = 8 * quant_tables(quality)

    def q(P, t):
        b = _blocks(P)
        c = fdct_islow(b.reshape(-1, 8, 8)).reshape(b.shape[0], b.shape[1], 64)
        return quantize(c, d[t])[..., ZIGZAG]

    zy = q(Y, 0)
    out = np.zeros((my, mx, 6, 64), dtype=np.int64)
    real = np.zeros((my, mx, 4), dtype=bool)
    for s in range(4):
        dy, dx = s >> 1, s & 1
        part = zy[dy::2, dx::2]
        out[:part.shape[0], :part.shape[1], s] = part
        real[:part.shape[0], :part.shape[1], s] = True
    for s in range(1, 4):
        out[..., s, 0] = np.where(real[..., s], out[..., s, 0], out[..., s - 1, 0])
    out[..., 4, :] = q(Cb, 1)
    out[..., 5, :] = q(Cr, 1)
    return out.reshape(-1, 64)


def dc_differences(zz):
    """DC difference of each block against the previous block of its component (MCU order)"""
    dc = zz[:, 0].reshape(-1, 6)
    diff = np.empty_like(dc)
    y = dc[:, :4].reshape(-1)
    diff[:, :4] = np.diff(y, prepend=0).reshape(-1, 4)
    for s in (4, 5):
        diff[:, s] = np.diff(dc[:, s], prepend=0)
    return diff.reshape(-1)


def _nbits(v):
    a = np.abs(v)
    n = np.zeros(a.shape, dtype=np.int64)
    while True:
        m = a >> n > 0
        if not m.any():
            return n
        n += m


def _mag(v, n):
    return (np.where(v < 0, v - 1, v) & ((np.int64(1) << n) - 1)).astype(np.uint64)


def _block_items(zz, diff, table):
    """values [n, 65] (uint64) and lengths [n, 65] of the symbols of each block: DC, one per AC position (with the ZRLs before
    it and its magnitude bits), EOB; length 0 where there is none"""
    n = zz.shape[0]
    dcc, dcl = _CODES[2 * table]
    acc, acl = _CODES[2 * table + 1]
    vals = np.zeros((n, 65), dtype=np.uint64)
    lens = np.zeros((n, 65), dtype=np.int64)
    s = _nbits(diff)
    vals[:, 0] = (dcc[s] << s.astype(np.uint64)) | _mag(diff, s)
    lens[:, 0] = dcl[s] + s
    ac = zz[:, 1:]
    nz = ac != 0
    k = np.arange(1, 64)
    last = np.maximum.accumulate(np.where(nz, k, 0), axis=1)
    prev = np.concatenate([np.zeros((n, 1), dtype=np.int64), last[:, :-1]], axis=1)
    run = k - prev - 1
    zrl, r = run >> 4, run & 15
    s = _nbits(ac)
    sym = (r << 4) | s
    pre = np.zeros(ac.shape, dtype=np.uint64)
    for i in range(3):
        pre = np.where(zrl > i, (pre << np.uint64(acl[0xF0])) | acc[0xF0], pre)
    v = (((pre << acl[sym].astype(np.uint64)) | acc[sym]) << s.astype(np.uint64)) | _mag(ac, s)
    vals[:, 1:64] = np.where(nz, v, 0)
    lens[:, 1:64] = np.where(nz, zrl * acl[0xF0] + acl[sym] + s, 0)
    eob = last[:, -1] < 63
    vals[:, 64] = np.where(eob, acc[0], 0)
    lens[:, 64] = np.where(eob, acl[0], 0)
    return vals, lens


def entropy_bits(zz, chunk=16384):
    """(bits per block, the scan's bit string as uint8 0/1) of quantised zigzag coefficients in MCU order"""
    diff = dc_differences(zz)
    table = (np.arange(zz.shape[0]) % 6 >= 4).astype(np.int64)
    counts = np.zeros(zz.shape[0], dtype=np.int64)
    parts = []
    for b0 in range(0, zz.shape[0], chunk):
        sl = slice(b0, b0 + chunk)
        vals = np.zeros((len(zz[sl]), 65), dtype=np.uint64)
        lens = np.zeros((len(zz[sl]), 65), dtype=np.int64)
        for t in (0, 1):
            m = table[sl] == t
            vals[m], lens[m] = _block_items(zz[sl][m], diff[sl][m], t)
        counts[sl] = lens.sum(axis=1)
        keep = lens.reshape(-1) > 0
        v, ln = vals.reshape(-1)[keep], lens.reshape(-1)[keep]
        rep = np.repeat(np.arange(len(v)), ln)
        start = np.cumsum(ln) - ln
        shift = (ln[rep] - 1 - (np.arange(len(rep)) - start[rep])).astype(np.uint64)
        parts.append(((v[rep] >> shift) & np.uint64(1)).astype(np.uint8))
    return counts, np.concatenate(parts)


def stuff(bitstring):
    """pad with 1-bits to whole bytes, then a 0x00 after every 0xFF"""
    pad = -len(bitstring) % 8
    data = np.packbits(np.concatenate([bitstring, np.ones(pad, dtype=np.uint8)]))
    ff = np.flatnonzero(data == 0xFF)
    return np.insert(data, ff + 1, 0).tobytes()


def encode(Y, Cb, Cr, quality):
    """the JFIF file of Y [H, W] and Cb, Cr [H/2, W/2] uint8 planes"""
    H, W = Y.shape
    assert H % 2 == 0 and W % 2 == 0 and Cb.shape == Cr.shape == (H // 2, W // 2)
    _, bits = entropy_bits(coefficients(Y, Cb, Cr, quality))
    return header(H, W, quality) + stuff(bits) + b"\xff\xd9"


def max_bytes(H, W):
    """pysp_jpeg_max_bytes"""
    blocks = 6 * (-(-H // 16)) * (-(-W // 16))
    return HEADER_BYTES + 2 * -(-blocks * (11 + 11 + 63 * (16 + 10)) // 8) + 2
