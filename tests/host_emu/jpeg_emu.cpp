// TEST INFRASTRUCTURE ONLY -- host emulation of the JPEG encode phases in pysp_b200/csrc/jpeg.cuh.
//
// The encode kernels are written as phases of independent work items (jpeg.cuh), so the same source compiles for the host
// (PYSP_HOST_EMU): a phase runs its items serially and the scans are plain loops.  This lets tests/test_jpeg_cpu.py compare the
// kernels' coefficients, bit counts, offsets and file with the NumPy restatement without a GPU.  It is NOT a CPU fallback: it
// is never built into libpysp_b200.so, never imported by the pysp_b200 package, and its entry points take HOST pointers.
// tests/test_jpeg_cpu.py builds it with g++ into a temporary directory.
#define PYSP_HOST_EMU 1
#include <stdio.h>
#include <stdlib.h>
#include <vector>

struct uint4 { unsigned int x, y, z, w; };

#include "../../include/pysp_b200.h"
#include "../../pysp_b200/csrc/jpeg.cuh"

using namespace pysp;

static char g_err[512];

extern "C" const char* emu_jpeg_last_error(void) { return g_err; }

static void emu_scan(const uint32_t* in, int64_t* out, int64_t n, int64_t* total) {
    int64_t acc = 0;
    for (int64_t i = 0; i < n; ++i) { out[i] = acc; acc += in[i]; }
    *total = acc;
}

// the phases of pysp_jpeg_encode_ycc420 in launch order, same arguments (host pointers, no stream)
extern "C" int emu_jpeg_encode(const uint8_t* y, int64_t y_pitch, const uint8_t* cb, const uint8_t* cr, int64_t c_pitch, int H, int W,
                               int quality, uint8_t* out, int64_t out_capacity, int64_t* out_len, void* ws, int64_t ws_bytes) {
    JpegParams p;
    if (plan_jpeg(y, y_pitch, cb, cr, c_pitch, H, W, quality, out, out_capacity, out_len, ws, ws_bytes, &p, g_err, sizeof(g_err)))
        return PYSP_ERR_INVALID;
    for (int i = 0; i < JPEG_HEADER_BYTES; ++i) jpeg_header_item(p, i);
    for (int64_t b = 0; b < p.n_blocks; ++b) jpeg_block_item(p, p.qt, kJpegHuff, b);
    emu_scan(p.bits, p.boff, p.n_blocks, p.totals);
    const int64_t bits = p.totals[0];
    for (int64_t i = 0; i <= bits / 32; ++i) p.words[i] = 0;
    for (int64_t b = 0; b < p.n_blocks; ++b) jpeg_pack_item(p, kJpegHuff, b);
    const int64_t items = jpeg_emit_items(bits);
    for (int64_t i = 0; i < items; ++i) jpeg_count_item(p, bits, i);
    emu_scan(p.ffcnt, p.foff, items, p.totals + 1);
    for (int64_t i = 0; i < items; ++i) jpeg_emit_item(p, bits, i);
    return PYSP_OK;
}

// byte offsets in the workspace of the quantised coefficients, the block bit counts and the block bit offsets
extern "C" void emu_jpeg_layout(int H, int W, int64_t* coef, int64_t* bits, int64_t* boff) {
    JpegParams p;
    std::vector<char> base(jpeg_layout(H, W, nullptr, nullptr));
    jpeg_layout(H, W, base.data(), &p);
    *coef = (char*)p.coef - base.data(); *bits = (char*)p.bits - base.data(); *boff = (char*)p.boff - base.data();
}

// the quantisation's reciprocal division against integer division: every divisor 8 * (1..255) and every |c| < 2^15;
// returns the number of mismatches
extern "C" int64_t emu_jpeg_check_reciprocals(void) {
    int64_t bad = 0;
    for (uint32_t q = 1; q <= 255; ++q) {
        const uint32_t d = 8 * q, m = jpeg_recip(d);
        for (int c = -32767; c <= 32767; ++c) {
            const int a = c < 0 ? -c : c, want = (a + (int)(d >> 1)) / (int)d;
            bad += jpeg_quantize(c, d, m) != (c < 0 ? -want : want);
        }
    }
    return bad;
}
