// TEST INFRASTRUCTURE ONLY -- host emulation of the RGB JPEG encode phases in pysp_b200/csrc/jpeg.cuh.
//
// jpeg_emu.cpp's entry points (the pysp_jpeg_encode_ycc420 phases, now on the generalised MCU geometry) plus those of
// pysp_jpeg_encode_rgb: the convert phase, then the same block / scan / pack / count / emit phases, each run serially.  Like
// jpeg_emu.cpp it is NOT a CPU fallback: never built into libpysp_b200.so, never imported by the pysp_b200 package, HOST
// pointers only.  tests/test_jpeg_rgb_cpu.py builds it with g++ into a temporary directory.
#include "jpeg_emu.cpp"

// the phases of pysp_jpeg_encode_rgb in launch order, same arguments (host pointers, no stream)
extern "C" int emu_jpeg_rgb_encode(const uint8_t* rgb, int64_t pitch, int H, int W, int quality, int subsampling, uint8_t* out,
                                   int64_t out_capacity, int64_t* out_len, void* ws, int64_t ws_bytes) {
    JpegParams p;
    if (plan_jpeg_rgb(rgb, pitch, H, W, quality, subsampling, out, out_capacity, out_len, ws, ws_bytes, &p, g_err, sizeof(g_err)))
        return PYSP_ERR_INVALID;
    for (int i = 0; i < JPEG_HEADER_BYTES; ++i) jpeg_header_item(p, i);
    for (int cy = 0; cy < p.ch; ++cy)
        for (int cx = 0; cx < p.cw; ++cx) jpeg_convert_item(p, cx, cy);
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

// byte offsets in the workspace of the coefficients, block bit counts, block bit offsets and the converted Y, Cb, Cr planes
extern "C" void emu_jpeg_rgb_layout(int H, int W, int subsampling, int64_t off[6]) {
    JpegParams p;
    const int h = jpeg_h(subsampling), v = jpeg_v(subsampling);
    std::vector<char> base(jpeg_layout(H, W, h, v, true, nullptr, nullptr));
    jpeg_layout(H, W, h, v, true, base.data(), &p);
    const char* q[6] = {(char*)p.coef, (char*)p.bits, (char*)p.boff, (char*)p.conv_y, (char*)p.conv_cb, (char*)p.conv_cr};
    for (int i = 0; i < 6; ++i) off[i] = q[i] - base.data();
}
