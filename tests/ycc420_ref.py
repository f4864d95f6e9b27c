"""NumPy restatement of PYSP_OUT_YCC420_U8 (include/pysp_b200.h): libjpeg's integer R'G'B' -> full-range YCbCr
(jccolor.c rgb_ycc_convert) and 4:2:0 chroma average (jcsample.c h2v2_downsample) of the 8-bit sRGB result.  Shared by the
tests and tools/ycc_bench.py; pinned to libjpeg itself by tests/test_ycc420_cpu.py."""
import numpy as np


def ycc_full(S):
    """uint8 [..., 3] R'G'B' -> (Y, cb, cr) int64 arrays of the same shape (no subsampling)"""
    S = np.asarray(S).astype(np.int64)
    R, G, B = S[..., 0], S[..., 1], S[..., 2]
    Y = (19595 * R + 38470 * G + 7471 * B + 32768) >> 16
    cb = (-11059 * R - 21709 * G + 32768 * B + (128 << 16) + 32767) >> 16
    cr = (32768 * R - 27439 * G - 5329 * B + (128 << 16) + 32767) >> 16
    return Y, cb, cr


def h2v2(c):
    """2x2 average of an even-sized [rows, W] plane whose column 0 is stored column 0: bias 1, 2, 1, 2, ... along a row"""
    s = c[0::2, 0::2] + c[0::2, 1::2] + c[1::2, 0::2] + c[1::2, 1::2]
    return (s + 1 + (np.arange(s.shape[1]) & 1)) >> 2


def ycc420(S):
    """uint8 [rows, W, 3] (whole stored rows starting at an even row) -> uint8 planes Y [rows, W], Cb, Cr [rows/2, W/2]"""
    Y, cb, cr = ycc_full(S)
    return Y.astype(np.uint8), h2v2(cb).astype(np.uint8), h2v2(cr).astype(np.uint8)


def upsample2x2(c):
    """each chroma sample repeated 2x2: libjpeg's h2v2 average of the result gives the plane back exactly"""
    return np.repeat(np.repeat(c, 2, axis=0), 2, axis=1)
