// pysp_b200 -- baseline JPEG encode, byte-identical to libjpeg-turbo's encode with its defaults (ISLOW DCT, Annex K
// quantisation and Huffman tables, no restart markers, JFIF 1.01 header), of YCbCr 4:2:0 planes (pysp_jpeg_encode_ycc420) or of
// an 8-bit RGB image at 4:4:4, 4:2:2 or 4:2:0 (pysp_jpeg_encode_rgb).  The contracts are restated in NumPy by tests/jpeg_ref.py
// and tests/jpeg_rgb_ref.py.
//
// An MCU holds h x v Y blocks (h, v = the luma sampling factors: 2x2 for 4:2:0, 2x1 for 4:2:2, 1x1 for 4:4:4), then one Cb and
// one Cr block: `slots` = h*v + 2 blocks.  The chroma planes are read as planes of cw x ch samples.
//
// Phases, each a kernel whose work items are independent (tests/host_emu/jpeg_emu.cpp and jpeg_rgb_emu.cpp run them serially on
// the CPU):
//   header   one item per header byte (623 bytes: SOI APP0 DQT DQT SOF0 DHT x4 SOS) and per quantisation divisor;
//   convert  (RGB input only) one item per chroma sample: libjpeg's YCbCr of the h x v pixels it covers, the Y samples and the
//            downsampled Cb / Cr stored as planes in the workspace; from there on the two entry points run the same phases;
//   block    one item per 8x8 block in MCU order (Y slots in raster order, Cb, Cr): load with edge replication, ISLOW DCT,
//            quantise, store the zigzag coefficients, and count the block's Huffman bits.  The DC predictor is the quantised DC of the
//            block before it in the component; the ISLOW DC is exactly the sum of (x - 128) over the block, so it is
//            recomputed from the pixels rather than waited for;
//   scan     exclusive prefix sum of the block bit counts (64-bit offsets);
//   zero     clears the words of the entropy-coded stream the frame uses;
//   pack     one item per block: its codes, big-endian, at its bit offset; the words it shares with its neighbours are
//            combined with atomicOr (order-independent), the words inside it are stored;
//   count    one item per 64 stream bytes: how many are 0xFF (the last byte padded with 1-bits first);
//   scan     exclusive prefix sum of those counts;
//   emit     one item per 64 stream bytes: the bytes, each 0xFF followed by 0x00, at their stuffed offset; the last item
//            appends EOI and stores the file length.
#pragma once
#include <stdio.h>

#include "pysp_common.cuh"

#ifdef PYSP_HOST_EMU
#define PYSP_JPEG_CONST static const
static inline int pysp_clz32(uint32_t v) { return v ? __builtin_clz(v) : 32; }
#else
#define PYSP_JPEG_CONST static __constant__ const
__device__ __forceinline__ int pysp_clz32(uint32_t v) { return __clz((int)v); }
#endif

namespace pysp {

constexpr int JPEG_HEADER_BYTES = 623;
constexpr int JPEG_HUFF_WORDS = 12 + 12 + 256 + 256;
constexpr int JPEG_MAX_BLOCK_BITS = 11 + 11 + 63 * (16 + 10);   // see pysp_jpeg_max_bytes
constexpr int JPEG_EMIT_BYTES = 64;                             // stream bytes per count / emit item
constexpr int JPEG_SCAN_CHUNK = 1024;                           // items per CTA of the scan kernels

// zigzag position -> natural (row-major) index
PYSP_HOSTDEV constexpr int jpeg_zigzag(int k) {
    const unsigned char z[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                 41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
    return z[k];
}

// Annex K.1 quantisation tables, natural order (luminance, chrominance)
PYSP_JPEG_CONST uint8_t kJpegStdQuant[2][64] = {
    {16, 11, 10, 16, 24,  40,  51,  61,  12, 12, 14, 19, 26,  58,  60,  55,  14, 13, 16, 24, 40,  57,  69,  56,
     14, 17, 22, 29, 51,  87,  80,  62,  18, 22, 37, 56, 68,  109, 103, 77,  24, 35, 55, 64, 81,  104, 113, 92,
     49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99},
    {17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99, 99, 99, 47, 66, 99, 99,
     99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99,
     99, 99, 99, 99, 99, 99, 99, 99}};

// Annex K.3 tables in the order of the DHT markers (DC luma, AC luma, DC chroma, AC chroma): BITS, the number of codes of
// each length 1..16, then HUFFVAL (the DC tables use the first 12)
PYSP_JPEG_CONST uint8_t kJpegDhtBits[4][16] = {
    {0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0},
    {0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 125},
    {0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0},
    {0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 119},
};
PYSP_JPEG_CONST uint8_t kJpegDhtVals[4][162] = {
    {0x00, 0x01, 0x02, 0x03, 0x04, 0x05, 0x06, 0x07, 0x08, 0x09, 0x0a, 0x0b, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00,
     0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00,
     0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00,
     0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00,
     0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00,
     0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00,
     0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00,
     0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00,
     0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00},
    {0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71,
     0x14, 0x32, 0x81, 0x91, 0xa1, 0x08, 0x23, 0x42, 0xb1, 0xc1, 0x15, 0x52, 0xd1, 0xf0, 0x24, 0x33, 0x62, 0x72,
     0x82, 0x09, 0x0a, 0x16, 0x17, 0x18, 0x19, 0x1a, 0x25, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x34, 0x35, 0x36, 0x37,
     0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59,
     0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x83,
     0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3,
     0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3,
     0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe1, 0xe2,
     0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf1, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa},
    {0x00, 0x01, 0x02, 0x03, 0x04, 0x05, 0x06, 0x07, 0x08, 0x09, 0x0a, 0x0b, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00,
     0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00,
     0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00,
     0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00,
     0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00,
     0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00,
     0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00,
     0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00,
     0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00},
    {0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22,
     0x32, 0x81, 0x08, 0x14, 0x42, 0x91, 0xa1, 0xb1, 0xc1, 0x09, 0x23, 0x33, 0x52, 0xf0, 0x15, 0x62, 0x72, 0xd1,
     0x0a, 0x16, 0x24, 0x34, 0xe1, 0x25, 0xf1, 0x17, 0x18, 0x19, 0x1a, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x35, 0x36,
     0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58,
     0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a,
     0x82, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a,
     0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba,
     0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda,
     0xe2, 0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa},
};
// The same tables as encoder codes (the canonical codes of BITS / HUFFVAL, Annex C): (length << 16) | code, length 0 for
// symbols a table lacks.  [0, 12) DC luma, [12, 24) DC chroma, [24, 280) AC luma, [280, 536) AC chroma, by symbol.
PYSP_JPEG_CONST uint32_t kJpegHuff[JPEG_HUFF_WORDS] = {
    0x020000, 0x030002, 0x030003, 0x030004, 0x030005, 0x030006, 0x04000e, 0x05001e, 0x06003e, 0x07007e,
    0x0800fe, 0x0901fe,
    0x020000, 0x020001, 0x020002, 0x030006, 0x04000e, 0x05001e, 0x06003e, 0x07007e, 0x0800fe, 0x0901fe,
    0x0a03fe, 0x0b07fe,
    0x04000a, 0x020000, 0x020001, 0x030004, 0x04000b, 0x05001a, 0x070078, 0x0800f8, 0x0a03f6, 0x10ff82,
    0x10ff83, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x04000c, 0x05001b, 0x070079,
    0x0901f6, 0x0b07f6, 0x10ff84, 0x10ff85, 0x10ff86, 0x10ff87, 0x10ff88, 0x000000, 0x000000, 0x000000,
    0x000000, 0x000000, 0x000000, 0x05001c, 0x0800f9, 0x0a03f7, 0x0c0ff4, 0x10ff89, 0x10ff8a, 0x10ff8b,
    0x10ff8c, 0x10ff8d, 0x10ff8e, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x06003a,
    0x0901f7, 0x0c0ff5, 0x10ff8f, 0x10ff90, 0x10ff91, 0x10ff92, 0x10ff93, 0x10ff94, 0x10ff95, 0x000000,
    0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x06003b, 0x0a03f8, 0x10ff96, 0x10ff97, 0x10ff98,
    0x10ff99, 0x10ff9a, 0x10ff9b, 0x10ff9c, 0x10ff9d, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000,
    0x000000, 0x07007a, 0x0b07f7, 0x10ff9e, 0x10ff9f, 0x10ffa0, 0x10ffa1, 0x10ffa2, 0x10ffa3, 0x10ffa4,
    0x10ffa5, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x07007b, 0x0c0ff6, 0x10ffa6,
    0x10ffa7, 0x10ffa8, 0x10ffa9, 0x10ffaa, 0x10ffab, 0x10ffac, 0x10ffad, 0x000000, 0x000000, 0x000000,
    0x000000, 0x000000, 0x000000, 0x0800fa, 0x0c0ff7, 0x10ffae, 0x10ffaf, 0x10ffb0, 0x10ffb1, 0x10ffb2,
    0x10ffb3, 0x10ffb4, 0x10ffb5, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x0901f8,
    0x0f7fc0, 0x10ffb6, 0x10ffb7, 0x10ffb8, 0x10ffb9, 0x10ffba, 0x10ffbb, 0x10ffbc, 0x10ffbd, 0x000000,
    0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x0901f9, 0x10ffbe, 0x10ffbf, 0x10ffc0, 0x10ffc1,
    0x10ffc2, 0x10ffc3, 0x10ffc4, 0x10ffc5, 0x10ffc6, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000,
    0x000000, 0x0901fa, 0x10ffc7, 0x10ffc8, 0x10ffc9, 0x10ffca, 0x10ffcb, 0x10ffcc, 0x10ffcd, 0x10ffce,
    0x10ffcf, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x0a03f9, 0x10ffd0, 0x10ffd1,
    0x10ffd2, 0x10ffd3, 0x10ffd4, 0x10ffd5, 0x10ffd6, 0x10ffd7, 0x10ffd8, 0x000000, 0x000000, 0x000000,
    0x000000, 0x000000, 0x000000, 0x0a03fa, 0x10ffd9, 0x10ffda, 0x10ffdb, 0x10ffdc, 0x10ffdd, 0x10ffde,
    0x10ffdf, 0x10ffe0, 0x10ffe1, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x0b07f8,
    0x10ffe2, 0x10ffe3, 0x10ffe4, 0x10ffe5, 0x10ffe6, 0x10ffe7, 0x10ffe8, 0x10ffe9, 0x10ffea, 0x000000,
    0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x10ffeb, 0x10ffec, 0x10ffed, 0x10ffee, 0x10ffef,
    0x10fff0, 0x10fff1, 0x10fff2, 0x10fff3, 0x10fff4, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000,
    0x0b07f9, 0x10fff5, 0x10fff6, 0x10fff7, 0x10fff8, 0x10fff9, 0x10fffa, 0x10fffb, 0x10fffc, 0x10fffd,
    0x10fffe, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000,
    0x020000, 0x020001, 0x030004, 0x04000a, 0x050018, 0x050019, 0x060038, 0x070078, 0x0901f4, 0x0a03f6,
    0x0c0ff4, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x04000b, 0x060039, 0x0800f6,
    0x0901f5, 0x0b07f6, 0x0c0ff5, 0x10ff88, 0x10ff89, 0x10ff8a, 0x10ff8b, 0x000000, 0x000000, 0x000000,
    0x000000, 0x000000, 0x000000, 0x05001a, 0x0800f7, 0x0a03f7, 0x0c0ff6, 0x0f7fc2, 0x10ff8c, 0x10ff8d,
    0x10ff8e, 0x10ff8f, 0x10ff90, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x05001b,
    0x0800f8, 0x0a03f8, 0x0c0ff7, 0x10ff91, 0x10ff92, 0x10ff93, 0x10ff94, 0x10ff95, 0x10ff96, 0x000000,
    0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x06003a, 0x0901f6, 0x10ff97, 0x10ff98, 0x10ff99,
    0x10ff9a, 0x10ff9b, 0x10ff9c, 0x10ff9d, 0x10ff9e, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000,
    0x000000, 0x06003b, 0x0a03f9, 0x10ff9f, 0x10ffa0, 0x10ffa1, 0x10ffa2, 0x10ffa3, 0x10ffa4, 0x10ffa5,
    0x10ffa6, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x070079, 0x0b07f7, 0x10ffa7,
    0x10ffa8, 0x10ffa9, 0x10ffaa, 0x10ffab, 0x10ffac, 0x10ffad, 0x10ffae, 0x000000, 0x000000, 0x000000,
    0x000000, 0x000000, 0x000000, 0x07007a, 0x0b07f8, 0x10ffaf, 0x10ffb0, 0x10ffb1, 0x10ffb2, 0x10ffb3,
    0x10ffb4, 0x10ffb5, 0x10ffb6, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x0800f9,
    0x10ffb7, 0x10ffb8, 0x10ffb9, 0x10ffba, 0x10ffbb, 0x10ffbc, 0x10ffbd, 0x10ffbe, 0x10ffbf, 0x000000,
    0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x0901f7, 0x10ffc0, 0x10ffc1, 0x10ffc2, 0x10ffc3,
    0x10ffc4, 0x10ffc5, 0x10ffc6, 0x10ffc7, 0x10ffc8, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000,
    0x000000, 0x0901f8, 0x10ffc9, 0x10ffca, 0x10ffcb, 0x10ffcc, 0x10ffcd, 0x10ffce, 0x10ffcf, 0x10ffd0,
    0x10ffd1, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x0901f9, 0x10ffd2, 0x10ffd3,
    0x10ffd4, 0x10ffd5, 0x10ffd6, 0x10ffd7, 0x10ffd8, 0x10ffd9, 0x10ffda, 0x000000, 0x000000, 0x000000,
    0x000000, 0x000000, 0x000000, 0x0901fa, 0x10ffdb, 0x10ffdc, 0x10ffdd, 0x10ffde, 0x10ffdf, 0x10ffe0,
    0x10ffe1, 0x10ffe2, 0x10ffe3, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x0b07f9,
    0x10ffe4, 0x10ffe5, 0x10ffe6, 0x10ffe7, 0x10ffe8, 0x10ffe9, 0x10ffea, 0x10ffeb, 0x10ffec, 0x000000,
    0x000000, 0x000000, 0x000000, 0x000000, 0x000000, 0x0e3fe0, 0x10ffed, 0x10ffee, 0x10ffef, 0x10fff0,
    0x10fff1, 0x10fff2, 0x10fff3, 0x10fff4, 0x10fff5, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000,
    0x0a03fa, 0x0f7fc3, 0x10fff6, 0x10fff7, 0x10fff8, 0x10fff9, 0x10fffa, 0x10fffb, 0x10fffc, 0x10fffd,
    0x10fffe, 0x000000, 0x000000, 0x000000, 0x000000, 0x000000,
};

// quality scaling of jcparam.c (jpeg_quality_scaling + jpeg_add_quant_table with force_baseline): natural order
PYSP_HD int jpeg_quant_value(int table, int k, int quality) {
    const int scale = quality < 50 ? 5000 / quality : 200 - 2 * quality;
    const int v = (kJpegStdQuant[table][k] * scale + 50) / 100;
    return v < 1 ? 1 : (v > 255 ? 255 : v);
}

// Quantisation divides |c| + d/2 by d = 8 * qtab (the ISLOW output is scaled by 8), d in 8..2040, |c| < 2^15.  The division is
// a multiply by m = ceil(2^32 / d) and a shift: with e = m*d - 2^32 < d, n*m / 2^32 = n/d + n*e / (d * 2^32), and n*e < 2^32
// for n < 2^21 keeps the floor exact.  tests/test_jpeg_cpu.py checks every divisor and numerator exhaustively.
PYSP_HOSTDEV inline uint32_t jpeg_recip(uint32_t d) { return (uint32_t)((0x100000000ull + d - 1) / d); }
PYSP_HOSTDEV inline uint32_t jpeg_div(uint32_t n, uint32_t m) { return (uint32_t)(((uint64_t)n * m) >> 32); }
PYSP_HOSTDEV inline int jpeg_quantize(int c, uint32_t d, uint32_t m) {
    const uint32_t r = jpeg_div((uint32_t)(c < 0 ? -c : c) + (d >> 1), m);
    return c < 0 ? -(int)r : (int)r;
}

struct JpegParams {
    const uint8_t* y;
    const uint8_t* cb;
    const uint8_t* cr;
    int64_t y_pitch, c_pitch;
    int H, W, quality;
    int h, v;                  // Y blocks per MCU across / down (the luma sampling factors, 1 or 2; chroma is 1x1)
    int slots;                 // blocks per MCU: h*v Y slots, Cb, Cr
    uint32_t slots_m;          // jpeg_recip(slots): block b < 2^31 is in MCU jpeg_div(b, slots_m) (exact: m * slots - 2^32 <= 2)
    int cw, ch;                // chroma plane width / height in samples
    int ybw, ybh;              // Y blocks across / down: ceil(W/8), ceil(H/8)
    int mcux, mcuy;            // MCUs across / down: ceil(W/8h), ceil(H/8v) (= chroma blocks across / down)
    int64_t n_blocks;          // slots per MCU; below 2^31 for every size (at most 3 * 8192 * 8192 at 4:4:4)
    int64_t max_items;         // count / emit items of the largest possible stream
    uint8_t* out;
    int64_t* out_len;
    // workspace (pysp_jpeg_workspace_bytes)
    uint32_t* qt;              // [0, 128): divisors d = 8 * qtab (luma, chroma; natural order); [128, 256): their jpeg_recip
    int64_t* totals;           // [0] stream bits, [1] 0xFF bytes in the stream
    int16_t* coef;             // [n_blocks][64] quantised coefficients, zigzag order; dummy blocks: DC only
    uint32_t* bits;            // [n_blocks] Huffman bits of each block
    int64_t* boff;             // [n_blocks] bit offset of each block (exclusive scan of bits)
    int64_t* bchunk;           // [ceil(n_blocks / JPEG_SCAN_CHUNK)] scan partials
    uint32_t* words;           // entropy-coded stream, big-endian within each 32-bit word
    uint32_t* ffcnt;           // [max_items] 0xFF bytes per item
    int64_t* foff;             // [max_items] 0xFF bytes before each item (exclusive scan of ffcnt)
    int64_t* fchunk;           // [ceil(max_items / JPEG_SCAN_CHUNK)] scan partials
    // RGB input (pysp_jpeg_encode_rgb): the convert phase writes the planes y / cb / cr then read, in the workspace:
    // Y [H][W], Cb and Cr [ch][cw] with cw = 8 * mcux, ch = ceil(H/v)
    const uint8_t* rgb;        // [H][W][3], row pitch rgb_pitch bytes; nullptr for pysp_jpeg_encode_ycc420
    int64_t rgb_pitch;
    uint8_t* conv_y;
    uint8_t* conv_cb;
    uint8_t* conv_cr;
};

// luma sampling factors of Pillow's `subsampling` (PYSP_JPEG_444 / 422 / 420)
static inline int jpeg_h(int subsampling) { return subsampling == 0 ? 1 : 2; }
static inline int jpeg_v(int subsampling) { return subsampling == 2 ? 2 : 1; }

static inline int64_t jpeg_align(int64_t v) { return (v + 255) / 256 * 256; }

// The workspace layout of an MCU of h x v Y blocks, plus the convert phase's planes when `planes`; with base == nullptr only the
// size is computed.  Returns the total bytes.
static inline int64_t jpeg_layout(int H, int W, int h, int v, bool planes, char* base, JpegParams* p) {
    const int mcux = (W + 8 * h - 1) / (8 * h), mcuy = (H + 8 * v - 1) / (8 * v);
    const int64_t mcus = (int64_t)mcux * mcuy, nb = (h * v + 2) * mcus;
    const int64_t max_bits = nb * JPEG_MAX_BLOCK_BITS;
    const int64_t max_items = ((max_bits + 7) / 8 + JPEG_EMIT_BYTES - 1) / JPEG_EMIT_BYTES;
    int64_t o = 0;
    auto take = [&](int64_t bytes) { char* q = base ? base + o : nullptr; o = jpeg_align(o + bytes); return q; };
    JpegParams t;
    t.qt = (uint32_t*)take(256 * 4);
    t.totals = (int64_t*)take(2 * 8);
    t.coef = (int16_t*)take(nb * 128);
    t.bits = (uint32_t*)take(nb * 4);
    t.boff = (int64_t*)take(nb * 8);
    t.bchunk = (int64_t*)take((nb + JPEG_SCAN_CHUNK - 1) / JPEG_SCAN_CHUNK * 8);
    t.words = (uint32_t*)take((max_bits / 32 + 2) * 4);
    t.ffcnt = (uint32_t*)take(max_items * 4);
    t.foff = (int64_t*)take(max_items * 8);
    t.fchunk = (int64_t*)take((max_items + JPEG_SCAN_CHUNK - 1) / JPEG_SCAN_CHUNK * 8);
    t.conv_y = t.conv_cb = t.conv_cr = nullptr;
    if (planes) {
        const int64_t nc = (int64_t)8 * mcux * ((H + v - 1) / v);
        t.conv_y = (uint8_t*)take((int64_t)H * W);
        t.conv_cb = (uint8_t*)take(nc);
        t.conv_cr = (uint8_t*)take(nc);
    }
    if (p) {
        p->qt = t.qt; p->totals = t.totals; p->coef = t.coef; p->bits = t.bits; p->boff = t.boff; p->bchunk = t.bchunk;
        p->words = t.words; p->ffcnt = t.ffcnt; p->foff = t.foff; p->fchunk = t.fchunk;
        p->conv_y = t.conv_y; p->conv_cb = t.conv_cb; p->conv_cr = t.conv_cr;
        p->n_blocks = nb; p->max_items = max_items;
    }
    return o;
}

// the layout of pysp_jpeg_encode_ycc420 (4:2:0 planes)
static inline int64_t jpeg_layout(int H, int W, char* base, JpegParams* p) { return jpeg_layout(H, W, 2, 2, false, base, p); }

// Worst case of the file (see pysp_jpeg_max_bytes and pysp_jpeg_rgb_max_bytes in include/pysp_b200.h)
static inline int64_t jpeg_max_bytes(int H, int W, int h, int v) {
    const int64_t nb = (h * v + 2) * (int64_t)((W + 8 * h - 1) / (8 * h)) * ((H + 8 * v - 1) / (8 * v));
    return JPEG_HEADER_BYTES + 2 * ((nb * JPEG_MAX_BLOCK_BITS + 7) / 8) + 2;
}

static inline bool jpeg_size_ok(int H, int W) { return H >= 2 && W >= 2 && H <= 65535 && W <= 65535 && !(H & 1) && !(W & 1); }
static inline bool jpeg_rgb_size_ok(int H, int W, int subsampling) {
    return H >= 1 && W >= 1 && H <= 65535 && W <= 65535 && subsampling >= 0 && subsampling <= 2;
}

// geometry of an MCU of h x v Y blocks and cw x ch chroma planes
static inline void jpeg_geometry(JpegParams* p, int H, int W, int h, int v, int cw, int ch, int quality, uint8_t* out,
                                 int64_t* out_len) {
    p->H = H; p->W = W; p->quality = quality;
    p->h = h; p->v = v; p->slots = h * v + 2; p->slots_m = jpeg_recip(h * v + 2); p->cw = cw; p->ch = ch;
    p->ybw = (W + 7) / 8; p->ybh = (H + 7) / 8; p->mcux = (W + 8 * h - 1) / (8 * h); p->mcuy = (H + 8 * v - 1) / (8 * v);
    p->out = out; p->out_len = out_len;
    p->rgb = nullptr; p->rgb_pitch = 0;
}

// Checks every argument before anything runs; fills *p.  err gets the reason of a PYSP_ERR_INVALID.
static inline int plan_jpeg(const uint8_t* y, int64_t y_pitch, const uint8_t* cb, const uint8_t* cr, int64_t c_pitch, int H, int W,
                            int quality, uint8_t* out, int64_t out_capacity, int64_t* out_len, void* ws, int64_t ws_bytes,
                            JpegParams* p, char* err, size_t err_len) {
    if (!y || !cb || !cr || !out || !out_len || !ws) { snprintf(err, err_len, "pysp_jpeg_encode_ycc420: null pointer"); return -1; }
    if (!jpeg_size_ok(H, W)) { snprintf(err, err_len, "pysp_jpeg_encode_ycc420: %dx%d: height and width must be even, 2..65535", H, W); return -1; }
    if (quality < 1 || quality > 100) { snprintf(err, err_len, "pysp_jpeg_encode_ycc420: quality %d outside 1..100", quality); return -1; }
    if (y_pitch < W || c_pitch < W / 2) { snprintf(err, err_len, "pysp_jpeg_encode_ycc420: pitch below the plane width"); return -1; }
    if (out_capacity < jpeg_max_bytes(H, W, 2, 2)) {
        snprintf(err, err_len, "pysp_jpeg_encode_ycc420: out_capacity %lld < pysp_jpeg_max_bytes = %lld", (long long)out_capacity,
                 (long long)jpeg_max_bytes(H, W, 2, 2));
        return -1;
    }
    const int64_t need = jpeg_layout(H, W, nullptr, nullptr);
    if (ws_bytes < need) {
        snprintf(err, err_len, "pysp_jpeg_encode_ycc420: workspace %lld < pysp_jpeg_workspace_bytes = %lld", (long long)ws_bytes, (long long)need);
        return -1;
    }
    jpeg_layout(H, W, (char*)ws, p);
    jpeg_geometry(p, H, W, 2, 2, W / 2, H / 2, quality, out, out_len);
    p->y = y; p->cb = cb; p->cr = cr; p->y_pitch = y_pitch; p->c_pitch = c_pitch;
    return 0;
}

// The same for pysp_jpeg_encode_rgb: the block phases read the convert phase's planes in the workspace.
static inline int plan_jpeg_rgb(const uint8_t* rgb, int64_t pitch, int H, int W, int quality, int subsampling, uint8_t* out,
                                int64_t out_capacity, int64_t* out_len, void* ws, int64_t ws_bytes, JpegParams* p, char* err,
                                size_t err_len) {
    if (!rgb || !out || !out_len || !ws) { snprintf(err, err_len, "pysp_jpeg_encode_rgb: null pointer"); return -1; }
    if (subsampling < 0 || subsampling > 2) {
        snprintf(err, err_len, "pysp_jpeg_encode_rgb: subsampling %d is not PYSP_JPEG_444 / 422 / 420 (0 / 1 / 2)", subsampling);
        return -1;
    }
    if (!jpeg_rgb_size_ok(H, W, subsampling)) { snprintf(err, err_len, "pysp_jpeg_encode_rgb: %dx%d: height and width must be 1..65535", H, W); return -1; }
    if (quality < 1 || quality > 100) { snprintf(err, err_len, "pysp_jpeg_encode_rgb: quality %d outside 1..100", quality); return -1; }
    if (pitch < 3 * (int64_t)W) { snprintf(err, err_len, "pysp_jpeg_encode_rgb: pitch %lld below 3 * width", (long long)pitch); return -1; }
    const int h = jpeg_h(subsampling), v = jpeg_v(subsampling);
    if (out_capacity < jpeg_max_bytes(H, W, h, v)) {
        snprintf(err, err_len, "pysp_jpeg_encode_rgb: out_capacity %lld < pysp_jpeg_rgb_max_bytes = %lld", (long long)out_capacity,
                 (long long)jpeg_max_bytes(H, W, h, v));
        return -1;
    }
    const int64_t need = jpeg_layout(H, W, h, v, true, nullptr, nullptr);
    if (ws_bytes < need) {
        snprintf(err, err_len, "pysp_jpeg_encode_rgb: workspace %lld < pysp_jpeg_rgb_workspace_bytes = %lld", (long long)ws_bytes,
                 (long long)need);
        return -1;
    }
    jpeg_layout(H, W, h, v, true, (char*)ws, p);
    const int mcux = (W + 8 * h - 1) / (8 * h);
    jpeg_geometry(p, H, W, h, v, 8 * mcux, (H + v - 1) / v, quality, out, out_len);
    p->rgb = rgb; p->rgb_pitch = pitch;
    p->y = p->conv_y; p->cb = p->conv_cb; p->cr = p->conv_cr; p->y_pitch = W; p->c_pitch = p->cw;
    return 0;
}

// ---- header ---------------------------------------------------------------------------------------------------------
// byte i of SOI, APP0 (JFIF 1.01, no units, density 1:1), DQT luma, DQT chroma (8-bit, zigzag order), SOF0 (3 components,
// Y h x v (`hv` = h << 4 | v), Cb and Cr 1x1), DHT DC0, AC0, DC1, AC1, SOS (Y: tables 0/0, Cb and Cr: 1/1, Ss 0, Se 63, Ah Al 0)
PYSP_HD uint8_t jpeg_header_byte(int i, int H, int W, int quality, int hv) {
    if (i < 20) {
        const uint8_t a[20] = {0xFF, 0xD8, 0xFF, 0xE0, 0, 16, 'J', 'F', 'I', 'F', 0, 1, 1, 0, 0, 1, 0, 1, 0, 0};
        return a[i];
    }
    if (i < 158) {                                     // two DQT markers of 69 bytes
        const int t = (i - 20) / 69, j = (i - 20) - 69 * t;
        if (j < 5) { const uint8_t a[5] = {0xFF, 0xDB, 0, 67, 0}; return j == 4 ? (uint8_t)t : a[j]; }
        return (uint8_t)jpeg_quant_value(t, jpeg_zigzag(j - 5), quality);
    }
    if (i < 177) {                                     // SOF0
        const uint8_t a[19] = {0xFF, 0xC0, 0, 17, 8, (uint8_t)(H >> 8), (uint8_t)H, (uint8_t)(W >> 8), (uint8_t)W, 3,
                               1, 0, 0, 2, 0x11, 1, 3, 0x11, 1};
        return i == 169 ? (uint8_t)hv : a[i - 158];
    }
    if (i < 609) {                                     // DHT: DC (33 bytes), AC (183 bytes), DC, AC
        int j = i - 177, t = 0;
        for (;;) {
            const int n = (t & 1) ? 162 : 12, len = 5 + 16 + n;
            if (j < len) break;
            j -= len;
            ++t;
        }
        const int n = (t & 1) ? 162 : 12;
        if (j == 0) return 0xFF;
        if (j == 1) return 0xC4;
        if (j == 2) return 0;
        if (j == 3) return (uint8_t)(3 + 16 + n);
        if (j == 4) return (uint8_t)(((t & 1) << 4) | (t >> 1));
        if (j < 21) return kJpegDhtBits[t][j - 5];
        return kJpegDhtVals[t][j - 21];
    }
    const uint8_t a[14] = {0xFF, 0xDA, 0, 12, 3, 1, 0x00, 2, 0x11, 3, 0x11, 0, 63, 0};
    return a[i - 609];
}

// header item i (i < JPEG_HEADER_BYTES) and divisor item i (i < 128)
PYSP_HD void jpeg_header_item(const JpegParams& p, int i) {
    if (i < JPEG_HEADER_BYTES) p.out[i] = jpeg_header_byte(i, p.H, p.W, p.quality, (p.h << 4) | p.v);
    if (i < 128) {
        const uint32_t d = 8u * (uint32_t)jpeg_quant_value(i >> 6, i & 63, p.quality);
        p.qt[i] = d;
        p.qt[128 + i] = jpeg_recip(d);
    }
}

// ---- conversion of RGB input ----------------------------------------------------------------------------------------
// convert item (cx, cy), cx < cw, cy < ch: chroma sample (cx, cy) and the Y samples of the h x v pixels it covers
// (jccolor.c rgb_ycc_convert, as PYSP_OUT_YCC420_U8 states it).  Full-resolution chroma is taken with the last column and row
// of the image repeated past its edges, then downsampled (jcsample.c): 4:2:2 (a + b + (cx & 1)) >> 1 (h2v1_downsample),
// 4:2:0 (a + b + c + d + 1 + (cx & 1)) >> 2 (h2v2_downsample), 4:4:4 a copy.  The block loader repeats the last chroma row.
PYSP_HD void jpeg_convert_item(const JpegParams& p, int cx, int cy) {
    int sb = 0, sr = 0;
    for (int dy = 0; dy < p.v; ++dy) {
        const int y = cy * p.v + dy, yy = y < p.H ? y : p.H - 1;
        const uint8_t* row = p.rgb + yy * p.rgb_pitch;
        for (int dx = 0; dx < p.h; ++dx) {
            const int x = cx * p.h + dx, xx = x < p.W ? x : p.W - 1;
            const int R = row[3 * xx], G = row[3 * xx + 1], B = row[3 * xx + 2];
            if (x < p.W && y < p.H) p.conv_y[(int64_t)y * p.W + x] = (uint8_t)((19595 * R + 38470 * G + 7471 * B + 32768) >> 16);
            sb += (-11059 * R - 21709 * G + 32768 * B + (128 << 16) + 32767) >> 16;
            sr += (32768 * R - 27439 * G - 5329 * B + (128 << 16) + 32767) >> 16;
        }
    }
    const int n = p.h * p.v, bias = n == 1 ? 0 : (cx & 1) + (n >> 2), sh = n >> 1;
    const int64_t o = (int64_t)cy * p.cw + cx;
    p.conv_cb[o] = (uint8_t)((sb + bias) >> sh);
    p.conv_cr[o] = (uint8_t)((sr + bias) >> sh);
}

// ---- blocks ---------------------------------------------------------------------------------------------------------
struct JpegBlock { const uint8_t* plane; int64_t pitch; int h, w, by, bx, comp; bool real; };

// block b in MCU order: slots 0 .. h*v-1 are Y (h x v, raster order), then Cb, Cr.  A Y slot outside the Y blocks is a dummy.
PYSP_HD JpegBlock jpeg_block_at(const JpegParams& p, int64_t mcu, int slot) {
    JpegBlock k;
    const int my = (int)(mcu / p.mcux), mx = (int)(mcu - (int64_t)my * p.mcux), ny = p.slots - 2;
    if (slot < ny) {
        k.plane = p.y; k.pitch = p.y_pitch; k.h = p.H; k.w = p.W; k.comp = 0;
        k.by = p.v * my + (slot >> (p.h - 1)); k.bx = p.h * mx + (slot & (p.h - 1));     // h is 1 or 2
        k.real = k.by < p.ybh && k.bx < p.ybw;
    } else {
        k.plane = slot == ny ? p.cb : p.cr; k.pitch = p.c_pitch; k.h = p.ch; k.w = p.cw; k.comp = slot - ny + 1;
        k.by = my; k.bx = mx; k.real = true;
    }
    return k;
}

// x - 128 over the block, the last row and column of the plane repeated past its edge
PYSP_HD void jpeg_load(const JpegBlock& k, int* d) {
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        const int yy = k.by * 8 + r < k.h ? k.by * 8 + r : k.h - 1;
        const uint8_t* row = k.plane + yy * k.pitch;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const int xx = k.bx * 8 + c < k.w ? k.bx * 8 + c : k.w - 1;
            d[r * 8 + c] = (int)row[xx] - 128;
        }
    }
}

// quantised DC of (mcu, slot); a dummy slot takes the DC of the slot before it (slot 0 is always real)
PYSP_HD int jpeg_slot_dc(const JpegParams& p, const uint32_t* qt, int64_t mcu, int slot) {
    JpegBlock k = jpeg_block_at(p, mcu, slot);
    while (!k.real) k = jpeg_block_at(p, mcu, --slot);
    int d[64];
    jpeg_load(k, d);
    int s = 0;
#pragma unroll
    for (int i = 0; i < 64; ++i) s += d[i];
    const int t = k.comp ? 64 : 0;
    return jpeg_quantize(s, qt[t], qt[128 + t]);
}

// DC predictor of block b: the quantised DC of the previous block of the same component (0 for the first)
PYSP_HD int jpeg_dc_pred(const JpegParams& p, const uint32_t* qt, int64_t mcu, int slot) {
    const int ny = p.slots - 2;
    if (slot >= 1 && slot < ny) return jpeg_slot_dc(p, qt, mcu, slot - 1);
    if (mcu == 0) return 0;
    return jpeg_slot_dc(p, qt, mcu - 1, slot == 0 ? ny - 1 : slot);
}

#define PYSP_DESCALE(x, n) (((x) + (1 << ((n) - 1))) >> (n))
// jfdctint.c (ISLOW): CONST_BITS 13, PASS1_BITS 2; `d` is one row (stride 1) or one column (stride 8)
template <bool PASS1>
PYSP_HD void jpeg_fdct_1d(int* d, int s) {
    constexpr int CB = 13, P1 = 2, SH = PASS1 ? CB - P1 : CB + P1;
    const int tmp0 = d[0] + d[7 * s], tmp7 = d[0] - d[7 * s], tmp1 = d[s] + d[6 * s], tmp6 = d[s] - d[6 * s];
    const int tmp2 = d[2 * s] + d[5 * s], tmp5 = d[2 * s] - d[5 * s], tmp3 = d[3 * s] + d[4 * s], tmp4 = d[3 * s] - d[4 * s];
    const int tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
    d[0] = PASS1 ? (tmp10 + tmp11) * (1 << P1) : PYSP_DESCALE(tmp10 + tmp11, P1);
    d[4 * s] = PASS1 ? (tmp10 - tmp11) * (1 << P1) : PYSP_DESCALE(tmp10 - tmp11, P1);
    int z1 = (tmp12 + tmp13) * 4433;
    d[2 * s] = PYSP_DESCALE(z1 + tmp13 * 6270, SH);
    d[6 * s] = PYSP_DESCALE(z1 - tmp12 * 15137, SH);
    z1 = tmp4 + tmp7;
    int z2 = tmp5 + tmp6, z3 = tmp4 + tmp6, z4 = tmp5 + tmp7;
    const int z5 = (z3 + z4) * 9633;
    const int t4 = tmp4 * 2446, t5 = tmp5 * 16819, t6 = tmp6 * 25172, t7 = tmp7 * 12299;
    z1 *= -7373; z2 *= -20995; z3 *= -16069; z4 *= -3196;
    z3 += z5; z4 += z5;
    d[7 * s] = PYSP_DESCALE(t4 + z1 + z3, SH);
    d[5 * s] = PYSP_DESCALE(t5 + z2 + z4, SH);
    d[3 * s] = PYSP_DESCALE(t6 + z2 + z3, SH);
    d[s] = PYSP_DESCALE(t7 + z1 + z4, SH);
}
#undef PYSP_DESCALE

PYSP_HD int jpeg_nbits(int v) { return 32 - pysp_clz32((uint32_t)(v < 0 ? -v : v)); }

// Huffman coding of one block (zz: quantised coefficients in zigzag order, zz[0] unused: `diff` is the DC difference).  Each
// symbol goes to sink.put(value, length) with its magnitude bits appended to the code (at most 16 + 10 bits).
template <class Sink>
PYSP_HD void jpeg_code_block(const int* zz, int diff, const uint32_t* huff, int table, Sink& sink) {
    const uint32_t* dc = huff + 12 * table;
    const uint32_t* ac = huff + 24 + 256 * table;
    int n = jpeg_nbits(diff);
    uint32_t e = dc[n];
    sink.put(((e & 0xFFFF) << n) | ((uint32_t)(diff < 0 ? diff - 1 : diff) & ((1u << n) - 1)), (e >> 16) + n);
    int run = 0;
#pragma unroll
    for (int k = 1; k < 64; ++k) {
        const int v = zz[k];
        if (v == 0) { ++run; continue; }
        for (; run > 15; run -= 16) { e = ac[0xF0]; sink.put(e & 0xFFFF, e >> 16); }
        n = jpeg_nbits(v);
        e = ac[(run << 4) | n];
        sink.put(((e & 0xFFFF) << n) | ((uint32_t)(v < 0 ? v - 1 : v) & ((1u << n) - 1)), (e >> 16) + n);
        run = 0;
    }
    if (run) { e = ac[0]; sink.put(e & 0xFFFF, e >> 16); }
}

struct JpegBitCount {
    uint32_t n = 0;
    PYSP_HD void put(uint32_t, uint32_t len) { n += len; }
};

// block item: DCT, quantisation, zigzag store, bit count.  qt / huff may be shared-memory copies.
PYSP_HD void jpeg_block_item(const JpegParams& p, const uint32_t* qt, const uint32_t* huff, int64_t b) {
    const int64_t mcu = jpeg_div((uint32_t)b, p.slots_m);          // b < n_blocks < 2^31
    const int slot = (int)(b - p.slots * mcu);
    const JpegBlock k = jpeg_block_at(p, mcu, slot);
    const int t = k.comp ? 64 : 0;
    int zz[64];
    if (k.real) {
        int d[64];
        jpeg_load(k, d);
#pragma unroll
        for (int r = 0; r < 8; ++r) jpeg_fdct_1d<true>(d + 8 * r, 1);
#pragma unroll
        for (int c = 0; c < 8; ++c) jpeg_fdct_1d<false>(d + c, 8);
#pragma unroll
        for (int i = 0; i < 64; ++i) {
            const int n = jpeg_zigzag(i);
            zz[i] = jpeg_quantize(d[n], qt[t + n], qt[128 + t + n]);
        }
    } else {
#pragma unroll
        for (int i = 1; i < 64; ++i) zz[i] = 0;
        zz[0] = jpeg_slot_dc(p, qt, mcu, slot);
    }
    const int pred = jpeg_dc_pred(p, qt, mcu, slot);
    JpegBitCount cnt;
    jpeg_code_block(zz, zz[0] - pred, huff, k.comp ? 1 : 0, cnt);
    p.bits[b] = cnt.n;
    uint32_t* dst = (uint32_t*)(p.coef + 64 * b);
#pragma unroll
    for (int i = 0; i < 32; ++i) dst[i] = (uint32_t)(uint16_t)zz[2 * i] | ((uint32_t)(uint16_t)zz[2 * i + 1] << 16);
}

// ---- packing --------------------------------------------------------------------------------------------------------
// Writes bits MSB first from bit offset `pos` of the word stream: the first and the last word of the block may be shared with
// the neighbouring blocks and are OR-ed in atomically; whole words inside the block are stored.
struct JpegBitWriter {
    uint32_t* words;
    int64_t w;        // index of the word being filled
    uint64_t acc;     // pending bits, right-aligned
    int nacc;         // number of pending bits, counting from the start of word w
    bool first;
    PYSP_HD void emit(uint32_t v, bool shared) {
        if (shared) {
#ifdef PYSP_HOST_EMU
            words[w] |= v;
#else
            atomicOr(words + w, v);
#endif
        } else {
            words[w] = v;
        }
    }
    PYSP_HD void put(uint32_t v, uint32_t len) {
        acc = (acc << len) | v;
        nacc += (int)len;
        if (nacc >= 32) {
            nacc -= 32;
            emit((uint32_t)(acc >> nacc), first);
            first = false;
            acc &= (1ull << nacc) - 1;
            ++w;
        }
    }
    PYSP_HD void finish() { if (nacc > 0) emit((uint32_t)(acc << (32 - nacc)), true); }
};

// pack item: block b's codes at its bit offset (the zero phase has cleared the words first)
PYSP_HD void jpeg_pack_item(const JpegParams& p, const uint32_t* huff, int64_t b) {
    const int64_t mcu = jpeg_div((uint32_t)b, p.slots_m);          // b < n_blocks < 2^31
    const int slot = (int)(b - p.slots * mcu), ny = p.slots - 2;
    const int comp = slot < ny ? 0 : slot - ny + 1;
    int zz[64];
    const uint32_t* src = (const uint32_t*)(p.coef + 64 * b);
#pragma unroll
    for (int i = 0; i < 32; ++i) {
        const uint32_t v = src[i];
        zz[2 * i] = (int16_t)(v & 0xFFFF);
        zz[2 * i + 1] = (int16_t)(v >> 16);
    }
    // DC of the previous block of the component, from the stored coefficients
    int pred = 0;
    if (slot >= 1 && slot < ny) pred = p.coef[64 * (b - 1)];
    else if (mcu > 0) pred = p.coef[64 * (slot == 0 ? b - 3 : b - p.slots)];      // slot 0: the last Y slot, 3 blocks back
    const int64_t pos = p.boff[b];
    JpegBitWriter wr;
    wr.words = p.words; wr.w = pos >> 5; wr.acc = 0; wr.nacc = (int)(pos & 31); wr.first = true;
    jpeg_code_block(zz, zz[0] - pred, huff, comp ? 1 : 0, wr);
    wr.finish();
}

// ---- byte stuffing --------------------------------------------------------------------------------------------------
PYSP_HD int64_t jpeg_stream_bytes(int64_t bits) { return (bits + 7) >> 3; }
PYSP_HD int64_t jpeg_emit_items(int64_t bits) { return (jpeg_stream_bytes(bits) + JPEG_EMIT_BYTES - 1) / JPEG_EMIT_BYTES; }

// stream byte j (j < jpeg_stream_bytes(bits)); the bits after the last code are 1s
PYSP_HD uint32_t jpeg_stream_byte(const uint32_t* words, int64_t j, int64_t bits) {
    uint32_t v = (words[j >> 2] >> (24 - 8 * (int)(j & 3))) & 0xFF;
    const int64_t end = 8 * (j + 1);
    if (end > bits) v |= (1u << (int)(end - bits)) - 1;
    return v;
}

PYSP_HD void jpeg_count_item(const JpegParams& p, int64_t bits, int64_t i) {
    const int64_t n = jpeg_stream_bytes(bits), j0 = i * JPEG_EMIT_BYTES;
    const int64_t j1 = j0 + JPEG_EMIT_BYTES < n ? j0 + JPEG_EMIT_BYTES : n;
    uint32_t c = 0;
    for (int64_t j = j0; j < j1; ++j) c += jpeg_stream_byte(p.words, j, bits) == 0xFF;
    p.ffcnt[i] = c;
}

// emit item: bytes [64 i, 64 i + 64) of the stream after the header, each 0xFF followed by a 0x00; the last item ends the file
PYSP_HD void jpeg_emit_item(const JpegParams& p, int64_t bits, int64_t i) {
    const int64_t n = jpeg_stream_bytes(bits), j0 = i * JPEG_EMIT_BYTES;
    const int64_t j1 = j0 + JPEG_EMIT_BYTES < n ? j0 + JPEG_EMIT_BYTES : n;
    int64_t o = JPEG_HEADER_BYTES + j0 + p.foff[i];
    for (int64_t j = j0; j < j1; ++j) {
        const uint32_t v = jpeg_stream_byte(p.words, j, bits);
        p.out[o++] = (uint8_t)v;
        if (v == 0xFF) p.out[o++] = 0;
    }
    if (j1 == n) {
        p.out[o] = 0xFF;
        p.out[o + 1] = 0xD9;
        *p.out_len = o + 2;
    }
}

}  // namespace pysp

#ifndef PYSP_HOST_EMU
namespace pysp {

constexpr int JPEG_THREADS = 256;
constexpr int JPEG_SCAN_PER = JPEG_SCAN_CHUNK / JPEG_THREADS;

__global__ void __launch_bounds__(JPEG_THREADS) jpeg_header_kernel(const JpegParams p) {
    for (int i = threadIdx.x; i < JPEG_HEADER_BYTES; i += blockDim.x) jpeg_header_item(p, i);
}

// one row of chroma samples per blockIdx.y
__global__ void __launch_bounds__(JPEG_THREADS) jpeg_convert_kernel(const JpegParams p) {
    const int cx = blockIdx.x * blockDim.x + threadIdx.x;
    if (cx < p.cw) jpeg_convert_item(p, cx, blockIdx.y);
}

__device__ __forceinline__ void jpeg_tables_to_smem(uint32_t* s_huff, uint32_t* s_qt, const uint32_t* qt) {
    for (int i = threadIdx.x; i < JPEG_HUFF_WORDS; i += blockDim.x) s_huff[i] = kJpegHuff[i];
    if (s_qt)
        for (int i = threadIdx.x; i < 256; i += blockDim.x) s_qt[i] = qt[i];
    __syncthreads();
}

__global__ void __launch_bounds__(JPEG_THREADS) jpeg_block_kernel(const JpegParams p) {
    __shared__ uint32_t s_huff[JPEG_HUFF_WORDS], s_qt[256];
    jpeg_tables_to_smem(s_huff, s_qt, p.qt);
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b < p.n_blocks) jpeg_block_item(p, s_qt, s_huff, b);
}

__global__ void __launch_bounds__(JPEG_THREADS) jpeg_pack_kernel(const JpegParams p) {
    __shared__ uint32_t s_huff[JPEG_HUFF_WORDS];
    jpeg_tables_to_smem(s_huff, nullptr, nullptr);
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b < p.n_blocks) jpeg_pack_item(p, s_huff, b);
}

// the kernels over the stuffed stream learn its length from the scan of the block bits: fixed grids, grid-stride items
__global__ void __launch_bounds__(JPEG_THREADS) jpeg_zero_kernel(const JpegParams p) {
    const int64_t n = p.totals[0] / 32 + 1;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) p.words[i] = 0;
}

__global__ void __launch_bounds__(JPEG_THREADS) jpeg_count_kernel(const JpegParams p) {
    const int64_t bits = p.totals[0], n = jpeg_emit_items(bits);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        jpeg_count_item(p, bits, i);
}

__global__ void __launch_bounds__(JPEG_THREADS) jpeg_emit_kernel(const JpegParams p) {
    const int64_t bits = p.totals[0], n = jpeg_emit_items(bits);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        jpeg_emit_item(p, bits, i);
}

// ---- exclusive scan, uint32 -> int64: per-chunk sums, one CTA over the chunk sums, per-chunk downsweep -----------------
// n items: n_host, or jpeg_emit_items(*n_bits) when n_bits is given (the count of the stuffing items is known on the device only)
struct JpegScan { const uint32_t* in; int64_t* out; int64_t* chunk; int64_t* total; int64_t n_host; const int64_t* n_bits; };

__device__ __forceinline__ int64_t jpeg_scan_n(const JpegScan& s) { return s.n_bits ? jpeg_emit_items(*s.n_bits) : s.n_host; }

// exclusive prefix of v over the CTA; *sum = the CTA's total (shared)
__device__ __forceinline__ int64_t jpeg_block_exclusive(int64_t v, int64_t* sum) {
    __shared__ int64_t s_warp[JPEG_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int64_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int64_t y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) s_warp[warp] = x;
    __syncthreads();
    int64_t before = 0, all = 0;
#pragma unroll
    for (int k = 0; k < JPEG_THREADS / 32; ++k) {
        const int64_t w = s_warp[k];
        if (k < warp) before += w;
        all += w;
    }
    __syncthreads();                                  // s_warp is reused by the next call
    *sum = all;
    return before + x - v;
}

__global__ void __launch_bounds__(JPEG_THREADS) jpeg_scan_reduce_kernel(const JpegScan s) {
    const int64_t n = jpeg_scan_n(s), chunks = (n + JPEG_SCAN_CHUNK - 1) / JPEG_SCAN_CHUNK;
    for (int64_t c = blockIdx.x; c < chunks; c += gridDim.x) {
        int64_t v = 0;
#pragma unroll
        for (int k = 0; k < JPEG_SCAN_PER; ++k) {
            const int64_t i = c * JPEG_SCAN_CHUNK + threadIdx.x * JPEG_SCAN_PER + k;
            if (i < n) v += s.in[i];
        }
        int64_t sum;
        jpeg_block_exclusive(v, &sum);
        if (threadIdx.x == 0) s.chunk[c] = sum;
    }
}

__global__ void __launch_bounds__(JPEG_THREADS) jpeg_scan_top_kernel(const JpegScan s) {
    const int64_t n = jpeg_scan_n(s), chunks = (n + JPEG_SCAN_CHUNK - 1) / JPEG_SCAN_CHUNK;
    int64_t carry = 0;
    for (int64_t c0 = 0; c0 < chunks; c0 += JPEG_THREADS) {
        const int64_t c = c0 + threadIdx.x;
        const int64_t v = c < chunks ? s.chunk[c] : 0;
        int64_t sum;
        const int64_t ex = jpeg_block_exclusive(v, &sum);
        if (c < chunks) s.chunk[c] = carry + ex;
        carry += sum;
    }
    if (threadIdx.x == 0) *s.total = carry;
}

__global__ void __launch_bounds__(JPEG_THREADS) jpeg_scan_down_kernel(const JpegScan s) {
    const int64_t n = jpeg_scan_n(s), chunks = (n + JPEG_SCAN_CHUNK - 1) / JPEG_SCAN_CHUNK;
    for (int64_t c = blockIdx.x; c < chunks; c += gridDim.x) {
        const int64_t i0 = c * JPEG_SCAN_CHUNK + threadIdx.x * JPEG_SCAN_PER;
        uint32_t v[JPEG_SCAN_PER];
        int64_t t = 0;
#pragma unroll
        for (int k = 0; k < JPEG_SCAN_PER; ++k) {
            v[k] = i0 + k < n ? s.in[i0 + k] : 0;
            t += v[k];
        }
        int64_t sum;
        int64_t o = s.chunk[c] + jpeg_block_exclusive(t, &sum);
#pragma unroll
        for (int k = 0; k < JPEG_SCAN_PER; ++k) {
            if (i0 + k < n) s.out[i0 + k] = o;
            o += v[k];
        }
    }
}

}  // namespace pysp
#endif
