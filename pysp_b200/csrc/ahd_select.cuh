// K1: RGGB mosaic tile (+6 px halo) -> AHD direction-selected camera RGB (debayer/ahd.py:69-145).
//
// A persistent CTA develops TW x TH output tiles entirely in shared memory.  The raw mosaic box of the
// NEXT tile is fetched by TMA into a staging buffer while the current tile is computed, and the finished
// tile leaves through a shared-memory staging tile and a TMA store (see pysp_b200.cu for the pipeline).
//   phase 0  staging box -> normalise (normalization.py:20-25) + white balance (ahd.py:77-80) into four
//            quarter-resolution CFA planes (bayer_chan_mixer.py:13-21 becomes index math);
//   phase 1  5-tap H and V green at R/B sites (ahd.py:97-102) and colour differences;
//   phase 2  per 2x2 quad and per direction: green high-pass (ahd.py:120-121), 4-phase Gaussian
//            upsample of (c-g) and g (edge_assisted_gaussian.py:140-143), metric RGB in float64,
//            cv2-Lab through the 33^3 table (ahd.py:45-62); Lab kept for the tile+2 px, the two
//            candidate images for the tile only -- neither ever goes to HBM;
//   phase 3  homogeneity counts (ahd_homogeneity_cython.pyx:36-58) for the tile+1 px;
//   phase 4  3x3 box vote (ahd.py:133-139), select, epilogue -> output staging tile.
// All planes are stored phase-separated ("quarter planes") so that a thread that owns a 2x2 quad
// addresses shared memory with unit stride and compile-time plane offsets.
//
// EDGE=true tiles (touching the frame border, or partial) apply the reference's six border rules by
// index mapping; interior tiles compile to straight-line code.  Band seams are NOT borders: rows
// outside [y_begin,y_end) but inside the frame are read from the buffer like any other halo.
#pragma once
#include "pysp_common.cuh"
#include "tma.cuh"

namespace pysp {

template <int TW_, int TH_>
struct SelectTile {
    static constexpr int TW = TW_, TH = TH_;
    // Raw input box: the stencil needs tile + 6 px.  A TMA tile load needs its inner coordinate to be a multiple of 16
    // bytes (8 u16 / 4 f32), so the box starts box_hx(tile_x) >= 6 px left of the tile: 8 px when the tile origin is a
    // multiple of 8, else 12 px (tiles whose width is 4 mod 8, e.g. 60: every other tile).  The quarter planes keep
    // exactly the 3-quad halo, so only phase 0 sees the variable margin.
    static constexpr int HY = 6;
    static constexpr bool WIDE = (TW % 8) != 0;
    static constexpr int BOXW = TW + (WIDE ? 20 : 16), BOXH = TH + 2 * HY;
    static constexpr int JX = 3, IY = HY / 2;                      // quarter index of the tile's first quad in the planes
    static constexpr int QW = TW / 2 + 2 * JX, QH = BOXH / 2;      // quarter planes incl. the halo quads
    static constexpr int QN = QW * QH;
    PYSP_HD static int box_hx(int tile_x) { return (WIDE && ((tile_x * TW) & 7)) ? 12 : 8; }
    static constexpr int LW = TW + 4, LH = TH + 4;                 // Lab region (tile + 2)
    static constexpr int CW = TW + 2, CH = TH + 2;                 // count region (tile + 1)
    // quarter planes (float): mosaic R,G1,G2,B ; H/V green at R and B ; H/V colour difference at R and B
    enum { P_R = 0, P_G1, P_G2, P_B, P_GHR, P_GHB, P_GVR, P_GVB, P_DHR, P_DHB, P_DVR, P_DVB, NPLANES };
    static constexpr int align128(int v) { return (v + 127) / 128 * 128; }
    // byte offsets into dynamic shared memory
    static constexpr int OFF_BAR = 0;                                            // mbarrier (8 B)
    static constexpr int OFF_STAGE = 128;                                        // raw box, u16 or f32
    static constexpr int OFF_Q = align128(OFF_STAGE + BOXW * BOXH * 4);          // NPLANES x [QH][QW] f32
    static constexpr int OFF_LABL = align128(OFF_Q + NPLANES * QN * 4);          // [2][LH][LW] f32  L
    static constexpr int OFF_LABAB = OFF_LABL + 2 * LH * LW * 4;                 // [2][LH][LW] u32  a|b<<16
    static constexpr int OFF_CAND = align128(OFF_LABAB + 2 * LH * LW * 4);       // [4][TH][TW] f32  RH,BH,RV,BV
    static constexpr int SMEM_BYTES = align128(OFF_CAND + 4 * TH * TW * 4);
    static constexpr int OFF_OUT = OFF_LABL;       // [3][TH][TW] f32 output tile: aliases Lab (dead after phase 3)
    // QualityDemosaic.Fast (eag.cuh) uses the quarter planes and the output tile only
    static constexpr int SMEM_BYTES_EAG = align128(OFF_OUT + 3 * align128(TH * TW * 4));
    static constexpr int OFF_CNT = OFF_Q + P_DHR * QN * 4;   // [CH][CW] u16 (H | V << 8): aliases the D planes (dead after phase 2)
    static_assert(TW % 4 == 0 && TH % 2 == 0 && BOXW % 8 == 0, "tile must be quad aligned and its box 16-byte granular");
    static_assert(3 * ((TH * TW * 4 + 127) / 128 * 128) <= 4 * LH * LW * 4, "output tile must fit in the Lab region");
    static_assert(CH * CW * 2 <= 4 * QN * 4, "count plane must fit in the D planes");
};

// floats between the three planes of an output staging tile in planes mode (TMA sources are 128-byte aligned)
template <int TW, int TH>
struct OutPlane { static constexpr int FLOATS = (TH * TW * 4 + 127) / 128 * 32; };

// stored-orientation origin of the raw input box of a tile, in elements of the held view
template <int TW, int TH>
PYSP_HD void select_input_box(const SelectParams& p, int tile_x, int tile_y, int* bx, int* by) {
    typedef SelectTile<TW, TH> L;
    const int x0 = tile_x * TW - L::box_hx(tile_x), y0 = p.y_begin + tile_y * TH - L::HY;  // logical
    *bx = p.g.flip_x ? p.g.W - (x0 + L::BOXW) : x0;
    *by = (p.g.flip_y ? p.g.H - (y0 + L::BOXH) : y0) - p.in_row0;
}

// origin of the output tile in the destination views; returns the box width in elements
template <int TW, int TH>
PYSP_HD void tile_output_box(const StoreParams& st, const FrameGeom& g, int x0, int y0, int* bx, int* by) {
    if (st.mode == OUT_FINAL) {
        *bx = 3 * (g.flip_x ? g.W - (x0 + TW) : x0);
        *by = (g.flip_y ? g.H - (y0 + TH) : y0) - st.img_row0;
    } else {
        *bx = x0;
        *by = y0 - st.plane_row0;
    }
}

// write one finished pixel into the output staging tile ([TH][3*TW] interleaved in stored orientation, or three
// [TH][TW] planes r-g, b-g, g in logical orientation)
template <int TW, int TH>
PYSP_HD void stage_pixel(float* out, const StoreParams& st, const FrameGeom& g, const ColorParams& c, int ty, int tx, Rgb v) {
    if (st.mode == OUT_FINAL) {
        v = finish_pixel(c, st.kind, v);
        int sy = g.flip_y ? TH - 1 - ty : ty, sx = g.flip_x ? TW - 1 - tx : tx;
        float* o = out + (sy * TW + sx) * 3;
        o[0] = v.r; o[1] = v.g; o[2] = v.b;
    } else {
        int o = ty * TW + tx;
        constexpr int PS = OutPlane<TW, TH>::FLOATS;
        out[o] = v.r - v.g; out[PS + o] = v.b - v.g; out[2 * PS + o] = v.g;
    }
}

// two horizontally adjacent finished pixels (tx even).  Planes leave as 8-byte pair stores (consecutive lanes write
// consecutive pairs: no bank conflicts); the interleaved final layout keeps the per-pixel path (measured: pairs are not faster)
template <int TW, int TH>
PYSP_HD void stage_pixel_pair(float* out, const StoreParams& st, const FrameGeom& g, const ColorParams& c, int ty, int tx, Rgb v0, Rgb v1) {
    if (st.mode == OUT_FINAL) {
        stage_pixel<TW, TH>(out, st, g, c, ty, tx, v0);
        stage_pixel<TW, TH>(out, st, g, c, ty, tx + 1, v1);
    } else {
        const int o = ty * TW + tx;
        constexpr int PS = OutPlane<TW, TH>::FLOATS;
        F2 a, b, d;
        a.x = v0.r - v0.g; a.y = v1.r - v1.g; b.x = v0.b - v0.g; b.y = v1.b - v1.g; d.x = v0.g; d.y = v1.g;
        *(F2*)(out + o) = a; *(F2*)(out + PS + o) = b; *(F2*)(out + 2 * PS + o) = d;
    }
}

// generic (non-TMA) store of the staging tile, clipped to the destination views; converts to half if asked
template <int TW, int TH>
PYSP_HD void store_tile_generic(const float* out, const StoreParams& st, const FrameGeom& g, int x0, int y0) {
    int bx, by;
    tile_output_box<TW, TH>(st, g, x0, y0, &bx, &by);
    if (st.mode == OUT_FINAL) {
        if (st.kind == OUT_YCC420_U8) {
            // JPEG-ready planes: quantise like OUT_SRGB_U8, then libjpeg's integer YCbCr and 4:2:0 average (ycc_block).  A work
            // item is a 2x2 block of the staging tile (2x4 on the word path).  Blocks are 2-aligned in stored coordinates:
            // tile origins, W, H and band bounds are even, also under a flip (the stored origin W - (x0 + TW) is even), so a
            // block lies wholly inside the destination or wholly outside it (partial tiles, negative origins of flipped
            // partial tiles): outside blocks are skipped.  The chroma bias alternates along the STORED chroma column.
            const int sx = bx / 3;                                    // stored column of the tile's first pixel (even)
            auto block = [&](int r, int c, uint32_t bias) {           // staging row r, column c (both even)
                uint32_t R[4], G[4], B[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const float* p = out + (r + (k >> 1)) * (TW * 3) + (c + (k & 1)) * 3;
                    R[k] = quantise(p[0], 255.0f); G[k] = quantise(p[1], 255.0f); B[k] = quantise(p[2], 255.0f);
                }
                return ycc_block(R, G, B, bias);
            };
            char* const yb = (char*)st.img.base;
            char* const cbb = (char*)st.cb.base;
            char* const crb = (char*)st.cr.base;
            const bool words = by >= 0 && by + TH <= st.img.rows && sx >= 0 && sx + TW <= st.img.cols && (sx & 3) == 0 &&
                               st.img.pitch % 4 == 0 && ((uintptr_t)yb % 4) == 0 && st.cb.pitch % 2 == 0 && st.cr.pitch % 2 == 0 &&
                               ((uintptr_t)cbb % 2) == 0 && ((uintptr_t)crb % 2) == 0;
            static_assert(TW % 4 == 0 && TH % 2 == 0, "a tile is a whole number of 2x4 blocks");
            if (words) {
                // 2x4 block: two 32-bit Y words and one 16-bit word per chroma plane; its left chroma column is even
                constexpr int BPR = TW / 4;
                PYSP_ITEMS(i, (TH / 2) * BPR) {
                    const int j = i / BPR, c = 4 * (i - j * BPR), y = by + 2 * j, cy = y >> 1, cx = (sx + c) >> 1;
                    const Ycc2x2 a = block(2 * j, c, 1u), b = block(2 * j, c + 2, 2u);
                    *(uint32_t*)(yb + (long long)y * st.img.pitch + sx + c) = a.y01 | (b.y01 << 16);
                    *(uint32_t*)(yb + (long long)(y + 1) * st.img.pitch + sx + c) = a.y23 | (b.y23 << 16);
                    *(uint16_t*)(cbb + (long long)cy * st.cb.pitch + cx) = (uint16_t)(a.cb | (b.cb << 8));
                    *(uint16_t*)(crb + (long long)cy * st.cr.pitch + cx) = (uint16_t)(a.cr | (b.cr << 8));
                }
            } else {
                constexpr int BPR = TW / 2;
                PYSP_ITEMS(i, (TH / 2) * BPR) {
                    const int j = i / BPR, c = 2 * (i - j * BPR), y = by + 2 * j, x = sx + c;
                    if (y < 0 || y >= st.img.rows || x < 0 || x >= st.img.cols) continue;
                    const int cy = y >> 1, cx = x >> 1;
                    const Ycc2x2 a = block(2 * j, c, 1u + (cx & 1));
                    uint8_t* y0p = (uint8_t*)(yb + (long long)y * st.img.pitch + x);
                    uint8_t* y1p = (uint8_t*)(yb + (long long)(y + 1) * st.img.pitch + x);
                    y0p[0] = (uint8_t)a.y01; y0p[1] = (uint8_t)(a.y01 >> 8);
                    y1p[0] = (uint8_t)a.y23; y1p[1] = (uint8_t)(a.y23 >> 8);
                    ((uint8_t*)(cbb + (long long)cy * st.cb.pitch))[cx] = (uint8_t)a.cb;
                    ((uint8_t*)(crb + (long long)cy * st.cr.pitch))[cx] = (uint8_t)a.cr;
                }
            }
        } else if (st.kind == OUT_LIN_F16 || st.kind >= OUT_SRGB_U8) {
            // narrow outputs: converted on the way out of the float staging tile (consecutive threads write consecutive
            // elements of a tile row).  Quantised sRGB: round-to-nearest of the gamma-encoded value times 255 / 65535.
            // A tile that lies inside the image with 4-byte aligned rows leaves as packed 32-bit words (four u8 or two
            // 16-bit values per store); partial tiles and unaligned rows go element by element.
            const int esz = out_kind_bytes(st.kind);
            const int per = 4 / esz;                                  // elements per 32-bit word
            static_assert((TW * 3) % 4 == 0, "a tile row is a whole number of words for every narrow kind");
            const bool words = by >= 0 && by + TH <= st.img.rows && bx >= 0 && bx + TW * 3 <= st.img.cols &&
                               ((long long)bx * esz) % 4 == 0 && st.img.pitch % 4 == 0 && ((uintptr_t)st.img.base % 4) == 0;
            if (words) {
                const int wpr = TW * 3 / per;                         // words per tile row
                PYSP_ITEMS(i, TH * wpr) {
                    const int r = i / wpr, wc = i - r * wpr;
                    const float* s = out + r * (TW * 3) + wc * per;
                    uint32_t word;
                    if (st.kind == OUT_SRGB_U8)
                        word = quantise(s[0], 255.0f) | (quantise(s[1], 255.0f) << 8) | (quantise(s[2], 255.0f) << 16) | (quantise(s[3], 255.0f) << 24);
                    else if (st.kind == OUT_SRGB_U16)
                        word = quantise(s[0], 65535.0f) | (quantise(s[1], 65535.0f) << 16);
                    else {
#ifndef PYSP_HOST_EMU
                        word = (uint32_t)__half_as_ushort(__float2half_rn(s[0])) | ((uint32_t)__half_as_ushort(__float2half_rn(s[1])) << 16);
#else
                        word = 0;
#endif
                    }
                    *(uint32_t*)((char*)st.img.base + (long long)(by + r) * st.img.pitch + (long long)bx * esz + (long long)wc * 4) = word;
                }
            } else
            PYSP_ITEMS(i, TH * TW * 3) {
                int r = i / (TW * 3), cc = i - r * (TW * 3);
                int gy = by + r, gx = bx + cc;
                if (gy >= 0 && gy < st.img.rows && gx >= 0 && gx < st.img.cols) {
                    char* dst = (char*)st.img.base + (long long)gy * st.img.pitch;
                    if (st.kind == OUT_SRGB_U8) ((uint8_t*)dst)[gx] = (uint8_t)quantise(out[i], 255.0f);
                    else if (st.kind == OUT_SRGB_U16) ((uint16_t*)dst)[gx] = (uint16_t)quantise(out[i], 65535.0f);
#ifndef PYSP_HOST_EMU
                    else ((__half*)dst)[gx] = __float2half_rn(out[i]);
#endif
                }
            }
        } else {
            box_store_generic(out, st.img, bx, by, TW * 3, TH);
        }
    } else {
        for (int k = 0; k < 3; ++k) box_store_generic(out + k * OutPlane<TW, TH>::FLOATS, st.plane[k], bx, by, TW, TH);
    }
}

// 5 taps, strictly left to right (ahd.py:97-102)
PYSP_HD float tap5(float a, float b, float c, float d, float e) {
    return ((((a * PYSP_H0) + (b * PYSP_H1)) + (c * PYSP_H2)) + (d * PYSP_H1)) + (e * PYSP_H0);
}

// correlation accumulators for the four output phases of the 4-phase upsample; v[dy+1][dx+1] are the 3x3
// quarter neighbours.  Taps in raster order; power-of-two weights are exact so fmaf == mul, add.
// base TOP_LEFT (gaussian.py:19-53 with base R): outputs TL,TR,BL,BR of the quad
PYSP_HD void up_tl(const float v[3][3], float o[4]) {
    float a = v[0][0] * 0.015625f;
    a = a + v[0][1] * 0.09375f;
    a = fmaf(v[0][2], 0.015625f, a);
    a = a + v[1][0] * 0.09375f;
    a = a + v[1][1] * 0.5625f;
    a = a + v[1][2] * 0.09375f;
    a = fmaf(v[2][0], 0.015625f, a);
    a = a + v[2][1] * 0.09375f;
    a = fmaf(v[2][2], 0.015625f, a);
    o[0] = a;
    a = v[0][1] * 0.0625f;
    a = fmaf(v[0][2], 0.0625f, a);
    a = a + v[1][1] * 0.375f;
    a = a + v[1][2] * 0.375f;
    a = fmaf(v[2][1], 0.0625f, a);
    a = fmaf(v[2][2], 0.0625f, a);
    o[1] = a;
    a = v[1][0] * 0.0625f;
    a = a + v[1][1] * 0.375f;
    a = fmaf(v[1][2], 0.0625f, a);
    a = fmaf(v[2][0], 0.0625f, a);
    a = a + v[2][1] * 0.375f;
    a = fmaf(v[2][2], 0.0625f, a);
    o[2] = a;
    a = v[1][1] * 0.25f;
    a = fmaf(v[1][2], 0.25f, a);
    a = fmaf(v[2][1], 0.25f, a);
    a = fmaf(v[2][2], 0.25f, a);
    o[3] = a;
}
// base BOTTOM_RIGHT (base B)
PYSP_HD void up_br(const float v[3][3], float o[4]) {
    float a = v[0][0] * 0.25f;
    a = fmaf(v[0][1], 0.25f, a);
    a = fmaf(v[1][0], 0.25f, a);
    a = fmaf(v[1][1], 0.25f, a);
    o[0] = a;
    a = v[0][0] * 0.0625f;
    a = a + v[0][1] * 0.375f;
    a = fmaf(v[0][2], 0.0625f, a);
    a = fmaf(v[1][0], 0.0625f, a);
    a = a + v[1][1] * 0.375f;
    a = fmaf(v[1][2], 0.0625f, a);
    o[1] = a;
    a = v[0][0] * 0.0625f;
    a = fmaf(v[0][1], 0.0625f, a);
    a = a + v[1][0] * 0.375f;
    a = a + v[1][1] * 0.375f;
    a = fmaf(v[2][0], 0.0625f, a);
    a = fmaf(v[2][1], 0.0625f, a);
    o[2] = a;
    a = v[0][0] * 0.015625f;
    a = a + v[0][1] * 0.09375f;
    a = fmaf(v[0][2], 0.015625f, a);
    a = a + v[1][0] * 0.09375f;
    a = a + v[1][1] * 0.5625f;
    a = a + v[1][2] * 0.09375f;
    a = fmaf(v[2][0], 0.015625f, a);
    a = a + v[2][1] * 0.09375f;
    a = fmaf(v[2][2], 0.015625f, a);
    o[3] = a;
}

PYSP_HD float gauss_row(float l, float c, float r) { return (PYSP_GK1 * c) + (PYSP_GK0 * (l + r)); }

// The resample step both demosaics share (edge_assisted_gaussian.py:126-143; AHD runs it per direction, ahd.py:120-127):
// 3x3 Gaussian high-pass of the full-resolution green, 4-phase Gaussian upsample of c - g and g, and their sums, for the
// quad at local quarter index (i, j) of a tile whose quarter planes start at frame quarter index (qy0, qx0).
// GR / GB: green at R / B sites, DR / DB: R - g / B - g, G1 / G2: the balanced native greens.  v gets TL, TR, BL, BR.
template <int TW, int TH, bool EDGE>
PYSP_HD void quad_resample(const float* GR, const float* GB, const float* DR, const float* DB, const float* G1,
                           const float* G2, int i, int j, int qy0, int qx0, int H, int W, Rgb v[4]) {
    constexpr int QW = SelectTile<TW, TH>::QW;
    const int fi = qy0 + i, fj = qx0 + j;              // frame quarter index
    // local quarter row/col of the 3 neighbours under quarter-grid REFLECT_101
    int ri[3], cj[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        ri[d] = EDGE ? reflect101(fi + d - 1, H >> 1) - qy0 : i + d - 1;
        cj[d] = EDGE ? reflect101(fj + d - 1, W >> 1) - qx0 : j + d - 1;
    }
    float gr[3][3], gb[3][3], dr[3][3], db[3][3];
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = 0; b < 3; ++b) {
            int c = ri[a] * QW + cj[b];
            gr[a][b] = GR[c]; gb[a][b] = GB[c]; dr[a][b] = DR[c]; db[a][b] = DB[c];
        }
    // full-res green window rows 2i-1..2i+2, cols 2j-1..2j+2 for the high-pass, with full-res REFLECT_101
    // (ahd.py:120).  Reflection keeps the CFA phase, so the plane of every window cell is static; only its quarter
    // index moves at the frame border.
    float gw[4][4];
    {
        int wr[4], wc[4];
        if (EDGE) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                wr[k] = (reflect101(2 * fi - 1 + k, H) >> 1) - qy0;
                wc[k] = (reflect101(2 * fj - 1 + k, W) >> 1) - qx0;
            }
        } else {
            wr[0] = i - 1; wr[1] = i; wr[2] = i; wr[3] = i + 1;
            wc[0] = j - 1; wc[1] = j; wc[2] = j; wc[3] = j + 1;
        }
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                int c = wr[a] * QW + wc[b];
                const bool oddrow = (a & 1) == 0, oddcol = (b & 1) == 0;   // window starts at -1
                gw[a][b] = oddrow ? (oddcol ? GB[c] : G2[c]) : (oddcol ? G1[c] : GR[c]);
            }
    }
    float hf[4];
    {
        float rp[4][2];
#pragma unroll
        for (int a = 0; a < 4; ++a) {
            rp[a][0] = gauss_row(gw[a][0], gw[a][1], gw[a][2]);
            rp[a][1] = gauss_row(gw[a][1], gw[a][2], gw[a][3]);
        }
#pragma unroll
        for (int a = 0; a < 2; ++a)
#pragma unroll
            for (int b = 0; b < 2; ++b)
                hf[a * 2 + b] = gw[a + 1][b + 1] - gauss_row(rp[a][b], rp[a + 1][b], rp[a + 2][b]);
    }
    float ugr[4], udr[4], ugb[4], udb[4];
    up_tl(gr, ugr); up_tl(dr, udr); up_br(gb, ugb); up_br(db, udb);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        v[k].r = udr[k] + (ugr[k] + hf[k]);          // edge_assisted_gaussian.py:141-143
        v[k].b = udb[k] + (ugb[k] + hf[k]);
        v[k].g = gw[1 + (k >> 1)][1 + (k & 1)];
    }
}

// ---- phase 0: staging box -> normalised, white-balanced quarter planes -------------------------------------
// normalization.py:20-23 on one photosite: clip(raw - black, 0, white) / white.  The IEEE division is replaced,
// when the host has checked it exhaustively for these levels (all 65536 sensor codes, develop_plan.h), by the
// reciprocal + two-FMA correction q = t*r; q' = fma(fma(-q, w, t), r, q), which then gives the same float.
PYSP_HD float normalize_site(const SelectParams& p, uint32_t code, int pos) {
    float raw = pysp_as_float(0x4B000000u | code) - 8388608.0f;          // exact u16 -> float
    float t = fminf(fmaxf(raw - p.black[pos], 0.0f), p.white[pos]);
    if (p.fast_div) {
        float q = t * p.rwhite[pos];
        return fmaf(fmaf(-q, p.white[pos], t), p.rwhite[pos], q);
    }
    return t / p.white[pos];
}

template <int TW, int TH, bool EDGE>
PYSP_D void select_phase0(const SelectParams& p, char* __restrict__ smem, int tile_x, int tile_y) {
    typedef SelectTile<TW, TH> L;
    constexpr int QW = L::QW, QN = L::QN;
    const int H = p.g.H, W = p.g.W;
    const int hx = L::box_hx(tile_x);
    const int bx0 = tile_x * TW - hx, by0 = p.y_begin + tile_y * TH - L::HY;   // logical origin of the box
    const int sh = hx - 2 * L::JX;                            // box column of plane column 0 (2 or 6: even)
    float* Q = (float*)(smem + L::OFF_Q);
    const void* stage = smem + L::OFF_STAGE;
    const int flipmask = (p.g.flip_y << 1) | p.g.flip_x;      // stored CFA position of logical position k is k ^ flipmask
    constexpr int BW2 = L::BOXW / 2;                          // site pairs per box row
    PYSP_ITEMS(it, QN) {
        int qy = it / QW, qx = it - qy * QW;
        // rows beyond the band's last row + halo are never read (a tile that overhangs the end of a row band is an EDGE tile)
        if (EDGE) { if (by0 + 2 * qy >= p.y_end + L::HY) continue; }
        float v[4];
        if (!EDGE) {
            // the two sites of a mosaic row are adjacent in the staging box (also when mirrored): one 32/64-bit load
            const int r0 = p.g.flip_y ? L::BOXH - 1 - 2 * qy : 2 * qy, r1 = p.g.flip_y ? r0 - 1 : r0 + 1;
            const int lp = qx + (sh >> 1);                    // logical pair index in the box row
            const int cp = p.g.flip_x ? BW2 - 1 - lp : lp;
            if (p.in_kind == IN_U16) {
                uint32_t w0 = ((const uint32_t*)stage)[r0 * BW2 + cp], w1 = ((const uint32_t*)stage)[r1 * BW2 + cp];
                if (p.g.flip_x) { w0 = (w0 >> 16) | (w0 << 16); w1 = (w1 >> 16) | (w1 << 16); }
                v[0] = normalize_site(p, w0 & 0xFFFFu, 0 ^ flipmask);
                v[1] = normalize_site(p, w0 >> 16, 1 ^ flipmask);
                v[2] = normalize_site(p, w1 & 0xFFFFu, 2 ^ flipmask);
                v[3] = normalize_site(p, w1 >> 16, 3 ^ flipmask);
            } else {
                const float* sf = (const float*)stage;
                float a0 = sf[(r0 * BW2 + cp) * 2], a1 = sf[(r0 * BW2 + cp) * 2 + 1];
                float b0 = sf[(r1 * BW2 + cp) * 2], b1 = sf[(r1 * BW2 + cp) * 2 + 1];
                v[0] = p.g.flip_x ? a1 : a0; v[1] = p.g.flip_x ? a0 : a1;
                v[2] = p.g.flip_x ? b1 : b0; v[3] = p.g.flip_x ? b0 : b1;
            }
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                // phase-preserving clamp (ahd.py:77-80): the clamped site is always inside the same box
                int y = phase_clamp(by0 + 2 * qy + (k >> 1), H), x = phase_clamp(bx0 + sh + 2 * qx + (k & 1), W);
                int ly = y - by0, lx = x - bx0;
                int si = (p.g.flip_y ? L::BOXH - 1 - ly : ly) * L::BOXW + (p.g.flip_x ? L::BOXW - 1 - lx : lx);
                v[k] = p.in_kind == IN_U16 ? normalize_site(p, ((const uint16_t*)stage)[si], k ^ flipmask)
                                           : ((const float*)stage)[si];
            }
        }
        // the Fast demosaic interpolates the un-balanced greens and balances afterwards (eag.cuh)
        const float wbg = p.algo == ALGO_EAG ? 1.0f : p.c.wb[1];
        Q[L::P_R * QN + it] = v[0] * p.c.wb[0]; Q[L::P_G1 * QN + it] = v[1] * wbg;
        Q[L::P_G2 * QN + it] = v[2] * wbg; Q[L::P_B * QN + it] = v[3] * p.c.wb[2];
    }
}

// ---- phases 1..4 ---------------------------------------------------------------------------------------------
// `before_out` is called by every thread after phase 1 and before the barrier that precedes the first write to the Lab
// planes, whose memory the output staging tile shares (the device pipeline waits there until the previous tile's TMA
// store has read the staging tile).
template <int TW, int TH, bool EDGE, typename BeforeOut>
PYSP_D void select_phases(const SelectParams& p, char* __restrict__ smem, int tile_x, int tile_y, BeforeOut before_out) {
    typedef SelectTile<TW, TH> L;
    constexpr int QW = L::QW, QN = L::QN;
    const int H = p.g.H, W = p.g.W;
    const int hq = H >> 1, wq = W >> 1;
    const int x0 = tile_x * TW, y0 = p.y_begin + tile_y * TH;     // logical origin of the output tile (even)
    constexpr int JX = L::JX, IY = L::IY;                         // local quarter index of the tile's first quad
    const int qx0 = (x0 >> 1) - JX, qy0 = (y0 >> 1) - IY;         // quarter-plane origin
    float* Q = (float*)(smem + L::OFF_Q);
    float* labL = (float*)(smem + L::OFF_LABL);
    uint32_t* labAB = (uint32_t*)(smem + L::OFF_LABAB);
    float* cand = (float*)(smem + L::OFF_CAND);
    uint16_t* cnt = (uint16_t*)(smem + L::OFF_CNT);
    float* out = (float*)(smem + L::OFF_OUT);
    PYSP_PHASE_BEGIN();

    // ---------------- phase 1: directional greens and colour differences at R/B sites ---------------------
    {
        constexpr int GW = TW / 2 + 4, GH = TH / 2 + 4;   // tile quads with a 2-quad halo
        PYSP_ITEMS(it, GW * GH) {
            int gy = it / GW, gx = it - gy * GW;
            int i = gy + IY - 2, j = gx + JX - 2;      // local quarter index
            if (EDGE) {
                int fi = qy0 + i, fj = qx0 + j;
                if (fi < 0 || fi >= hq || fj < 0 || fj >= wq || 2 * fi >= p.y_end + 4) continue;
            }
            int c = i * QW + j;
            const float* R = Q + L::P_R * QN; const float* G1 = Q + L::P_G1 * QN;
            const float* G2 = Q + L::P_G2 * QN; const float* B = Q + L::P_B * QN;
            float r = R[c], b = B[c];
            float ghr = tap5(R[c - 1], G1[c - 1], r, G1[c], R[c + 1]);
            float gvr = tap5(R[c - QW], G2[c - QW], r, G2[c], R[c + QW]);
            float ghb = tap5(B[c - 1], G2[c], b, G2[c + 1], B[c + 1]);
            float gvb = tap5(B[c - QW], G1[c], b, G1[c + QW], B[c + QW]);
            Q[L::P_GHR * QN + c] = ghr; Q[L::P_GVR * QN + c] = gvr;
            Q[L::P_GHB * QN + c] = ghb; Q[L::P_GVB * QN + c] = gvb;
            Q[L::P_DHR * QN + c] = r - ghr; Q[L::P_DVR * QN + c] = r - gvr;
            Q[L::P_DHB * QN + c] = b - ghb; Q[L::P_DVB * QN + c] = b - gvb;
        }
    }
    before_out();
    PYSP_SYNC();
    PYSP_PHASE_MARK(0, 2);

    // ---------------- phase 2: candidates + Lab per quad, both directions ----------------------------------
    {
        constexpr int PW = L::LW / 2, PH = L::LH / 2;  // quads of the Lab region (1-quad halo)
        PYSP_ITEMS(it, PW * PH) {
            int py = it / PW, px = it - py * PW;
            int i = py + IY - 1, j = px + JX - 1;      // local quarter index
            int fi = qy0 + i, fj = qx0 + j;            // frame quarter index
            if (EDGE) { if (fi < 0 || fi >= hq || fj < 0 || fj >= wq || 2 * fi >= p.y_end + 2) continue; }
            const bool inner = py >= 1 && py <= TH / 2 && px >= 1 && px <= TW / 2;
#pragma unroll 1                                       // one copy of the body (measured: unrolling both directions is 2 % slower)
            for (int dir = 0; dir < 2; ++dir) {
                Rgb cv[4];                             // this direction's candidate pixels TL, TR, BL, BR
                quad_resample<TW, TH, EDGE>(Q + (dir ? L::P_GVR : L::P_GHR) * QN, Q + (dir ? L::P_GVB : L::P_GHB) * QN,
                                            Q + (dir ? L::P_DVR : L::P_DHR) * QN, Q + (dir ? L::P_DVB : L::P_DHB) * QN,
                                            Q + L::P_G1 * QN, Q + L::P_G2 * QN, i, j, qy0, qx0, H, W, cv);
                // Lab of the metric image, kept for the tile + 2 px
                float* oL = labL + dir * (L::LH * L::LW);
                uint32_t* oAB = labAB + dir * (L::LH * L::LW);
                // software pipeline over the four pixels: the table loads of pixel k + 1 are issued before pixel k is
                // interpolated (ptxas otherwise runs the pixels strictly one after the other)
                LabQ q[4];
                {
                    float m3[3], luma[4];
                    LabKey key[2];
                    uint4 e[2][4];
                    metric_rgb(p.c, cv[0].r, cv[0].g, cv[0].b, m3, &luma[0]);
                    key[0] = lab_key(p.lut, m3[0], m3[1], m3[2]);
#pragma unroll
                    for (int c = 0; c < 4; ++c) e[0][c] = pysp_ldg(key[0].base + (c >> 1) * PYSP_LUT_NG * PYSP_LUT_NB + (c & 1) * PYSP_LUT_NB);
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        if (k < 3) {
                            metric_rgb(p.c, cv[k + 1].r, cv[k + 1].g, cv[k + 1].b, m3, &luma[k + 1]);
                            key[(k + 1) & 1] = lab_key(p.lut, m3[0], m3[1], m3[2]);
#pragma unroll
                            for (int c = 0; c < 4; ++c)
                                e[(k + 1) & 1][c] = pysp_ldg(key[(k + 1) & 1].base + (c >> 1) * PYSP_LUT_NG * PYSP_LUT_NB + (c & 1) * PYSP_LUT_NB);
                        }
                        q[k] = lab_interp(key[k & 1], e[k & 1][0], e[k & 1][1], e[k & 1][2], e[k & 1][3]);
                        if (p.c.hdr) q[k].L = luma[k];
                    }
                }
                // the two pixels of a row leave as one 8-byte store (a 32-bit store per pixel has lane stride 2: two-way
                // bank conflicts on every store)
#pragma unroll
                for (int a = 0; a < 2; ++a) {
                    const int o = (2 * py + a) * L::LW + 2 * px;
                    F2 l2; l2.x = q[2 * a].L; l2.y = q[2 * a + 1].L;
                    U2 ab2; ab2.x = q[2 * a].ab; ab2.y = q[2 * a + 1].ab;
                    *(F2*)(oL + o) = l2; *(U2*)(oAB + o) = ab2;
                }
                if (inner) {
                    float* oR = cand + (dir * 2 + 0) * (TH * TW);
                    float* oB = cand + (dir * 2 + 1) * (TH * TW);
#pragma unroll
                    for (int a = 0; a < 2; ++a) {
                        const int o = (2 * (py - 1) + a) * TW + 2 * (px - 1);
                        F2 r2; r2.x = cv[2 * a].r; r2.y = cv[2 * a + 1].r;
                        F2 b2; b2.x = cv[2 * a].b; b2.y = cv[2 * a + 1].b;
                        *(F2*)(oR + o) = r2; *(F2*)(oB + o) = b2;
                    }
                }
            }
        }
    }
    PYSP_SYNC();
    PYSP_PHASE_MARK(0, 3);

    // ---------------- phase 3: homogeneity counts for the tile + 1 px ---------------------------------------
    // The centre and the two neighbours along the direction always pass both tests (their distances define
    // eps_l and eps_c), so only the six other window cells are tested: count = 3 + passes.  A work item is a 2x2
    // block of pixels inside its 4x4 Lab window; the distance of a pair of cells is computed once and used from
    // both ends (dL changes sign, dC^2 does not): 26 pair distances per block and direction instead of 32.
    {
        constexpr int BW = L::CW / 2, BH = L::CH / 2;
        static_assert(BW <= 32, "phase 3 maps one row of blocks to a warp");
        PYSP_ROW_ITEMS32(by, bx, BH, BW) {
            int cy = 2 * by, cx = 2 * bx;                 // count-region coords of the block's top-left pixel
            int fy = y0 - 1 + cy, fx = x0 - 1 + cx;       // frame coords
            if (EDGE) { if (fy >= p.y_end + 1) continue; }        // counts are needed for the band's rows + 1 only
            // Lab-region local coords of the 4x4 window (edge-duplicated at the frame border, ahd.py:64)
            int wy[4], wx[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                wy[k] = EDGE ? clampi(fy - 1 + k, H) - (y0 - 2) : cy + k;
                wx[k] = EDGE ? clampi(fx - 1 + k, W) - (x0 - 2) : cx + k;
            }
            uint32_t res[4] = {0, 0, 0, 0};
            // raw window loads of BOTH directions first (L as float, a|b packed), then one direction at a time: the loads
            // of the vertical map are in flight while the horizontal one is evaluated
            float rawl[2][4][4];
            uint32_t rawab[2][4][4];
#pragma unroll
            for (int dir = 0; dir < 2; ++dir) {
                const float* iL = labL + dir * (L::LH * L::LW);
                const uint32_t* iAB = labAB + dir * (L::LH * L::LW);
#pragma unroll
                for (int a = 0; a < 4; ++a) {
                    if (EDGE) {
#pragma unroll
                        for (int b = 0; b < 4; ++b) { int o = wy[a] * L::LW + wx[b]; rawl[dir][a][b] = iL[o]; rawab[dir][a][b] = iAB[o]; }
                    } else {
                        // cx and LW are even: the row is two aligned 8-byte pairs
                        const F2* rl = (const F2*)(iL + (cy + a) * L::LW + cx);
                        const U2* rab = (const U2*)(iAB + (cy + a) * L::LW + cx);
                        F2 l0 = rl[0], l1 = rl[1];
                        U2 q0 = rab[0], q1 = rab[1];
                        rawl[dir][a][0] = l0.x; rawl[dir][a][1] = l0.y; rawl[dir][a][2] = l1.x; rawl[dir][a][3] = l1.y;
                        rawab[dir][a][0] = q0.x; rawab[dir][a][1] = q0.y; rawab[dir][a][2] = q1.x; rawab[dir][a][3] = q1.y;
                    }
                }
            }
#pragma unroll
            for (int dir = 0; dir < 2; ++dir) {
                float wl[4][4], wa[4][4], wb[4][4];
#pragma unroll
                for (int a = 0; a < 4; ++a) {
#pragma unroll
                    for (int b = 0; b < 4; ++b) { wl[a][b] = rawl[dir][a][b]; wa[a][b] = ab_lo(rawab[dir][a][b]); wb[a][b] = ab_hi(rawab[dir][a][b]); }
                }
                // pair distances, first cell = the upper (then left) one: dL = L(second) - L(first)
                float hl[4][3], h2[4][3], vl[3][4], v2[3][4], gl[3][3], g2[3][3], al[3][3], a2[3][3];
#define PYSP_PAIR(DL, D2, y1, x1, y2, x2)                                                \
    {                                                                                   \
        DL = wl[y2][x2] - wl[y1][x1];                                                   \
        float da_ = wa[y2][x2] - wa[y1][x1], db_ = wb[y2][x2] - wb[y1][x1];             \
        D2 = (da_ * da_) + (db_ * db_);                                                 \
    }
#pragma unroll
                for (int a = 1; a < 3; ++a)
#pragma unroll
                    for (int b = 0; b < 3; ++b) PYSP_PAIR(hl[a][b], h2[a][b], a, b, a, b + 1)
#pragma unroll
                for (int a = 0; a < 3; ++a)
#pragma unroll
                    for (int b = 1; b < 3; ++b) PYSP_PAIR(vl[a][b], v2[a][b], a, b, a + 1, b)
#pragma unroll
                for (int a = 0; a < 3; ++a)
#pragma unroll
                    for (int b = 0; b < 3; ++b) {
                        if (!((a == 0 && b == 2) || (a == 2 && b == 0))) PYSP_PAIR(gl[a][b], g2[a][b], a, b, a + 1, b + 1)
                        if (!((a == 0 && b == 0) || (a == 2 && b == 2))) PYSP_PAIR(al[a][b], a2[a][b], a, b + 1, a + 1, b)
                    }
#undef PYSP_PAIR
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int a = 1 + (k >> 1), b = 1 + (k & 1);
                    uint32_t n = 3u;
                    if (dir == 0) {     // horizontal map: eps from the left/right neighbours (pyx:47-51)
                        const float epsl = fmaxf(fabsf(hl[a][b - 1]), fabsf(hl[a][b])), nepsl = -epsl;
                        const float epsc = fmaxf(h2[a][b - 1], h2[a][b]);
                        n = count_ge(n, gl[a - 1][b - 1], nepsl, g2[a - 1][b - 1], epsc);
                        n = count_ge(n, vl[a - 1][b], nepsl, v2[a - 1][b], epsc);
                        n = count_ge(n, al[a - 1][b], nepsl, a2[a - 1][b], epsc);
                        n = count_le(n, al[a][b - 1], epsl, a2[a][b - 1], epsc);
                        n = count_le(n, vl[a][b], epsl, v2[a][b], epsc);
                        n = count_le(n, gl[a][b], epsl, g2[a][b], epsc);
                    } else {            // vertical map: eps from the upper/lower neighbours (pyx:42-46)
                        const float epsl = fmaxf(fabsf(vl[a - 1][b]), fabsf(vl[a][b])), nepsl = -epsl;
                        const float epsc = fmaxf(v2[a - 1][b], v2[a][b]);
                        n = count_ge(n, gl[a - 1][b - 1], nepsl, g2[a - 1][b - 1], epsc);
                        n = count_ge(n, hl[a][b - 1], nepsl, h2[a][b - 1], epsc);
                        n = count_le(n, al[a][b - 1], epsl, a2[a][b - 1], epsc);
                        n = count_ge(n, al[a - 1][b], nepsl, a2[a - 1][b], epsc);
                        n = count_le(n, hl[a][b], epsl, h2[a][b], epsc);
                        n = count_le(n, gl[a][b], epsl, g2[a][b], epsc);
                    }
                    res[k] |= n << (8 * dir);
                }
            }
            // cx and CW are even: one 32-bit store per row of the block
#pragma unroll
            for (int a = 0; a < 2; ++a) *(uint32_t*)(cnt + (cy + a) * L::CW + cx) = res[2 * a] | (res[2 * a + 1] << 16);
        }
    }
    PYSP_SYNC();
    PYSP_PHASE_MARK(0, 4);

    // ---------------- phase 4: 3x3 vote, select, epilogue -> output staging tile ---------------------------
    // A count cell is 16 bits, H count in the low byte and V count in the high byte; two cells per 32-bit word.
    // Window sums stay below 256 per byte (9 x 9), so plain 32-bit adds sum four byte counters at once.
    {
        constexpr int OW = TW / 2, OH = TH / 2;
        static_assert(OW <= 32, "phase 4 maps one row of quads to a warp");
        PYSP_ROW_ITEMS32(oy, ox, OH, OW) {
            int ty = 2 * oy, tx = 2 * ox;                 // tile coords of the quad
            int fy = y0 + ty, fx = x0 + tx;
            if (EDGE) { if (fy >= p.y_end || fx >= W) continue; } // partial tile (even dims: whole quad in or out; y_end <= H)
            uint32_t w0[4], w1[4];                        // per window row: cells (0,1) and (2,3)
            if (EDGE) {
                int wy[4], wx[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    wy[k] = reflect101(fy - 1 + k, H) - (y0 - 1);      // cv2.blur: REFLECT_101
                    wx[k] = reflect101(fx - 1 + k, W) - (x0 - 1);
                }
#pragma unroll
                for (int a = 0; a < 4; ++a) {
                    const uint16_t* r = cnt + wy[a] * L::CW;
                    w0[a] = (uint32_t)r[wx[0]] | ((uint32_t)r[wx[1]] << 16);
                    w1[a] = (uint32_t)r[wx[2]] | ((uint32_t)r[wx[3]] << 16);
                }
            } else {
#pragma unroll
                for (int a = 0; a < 4; ++a) {             // tx and CW are even: aligned 32-bit pairs
                    const uint32_t* r = (const uint32_t*)(cnt + (ty + a) * L::CW + tx);
                    w0[a] = r[0]; w1[a] = r[1];
                }
            }
            int qi = (oy + IY) * QW + ox + JX;
#pragma unroll
            for (int a = 0; a < 2; ++a) {
                const uint32_t v0 = w0[a] + w0[a + 1] + w0[a + 2], v1 = w1[a] + w1[a + 1] + w1[a + 2];   // column sums
                const uint32_t s = v0 + v1;                                    // (c0 + c2, c1 + c3)
                const uint32_t t[2] = {(s & 0xFFFFu) + (v0 >> 16), (s >> 16) + (v1 & 0xFFFFu)};
                const F2* ch = (const F2*)(cand + (ty + a) * TW + tx);         // tx even: one 8-byte load per plane
                const F2 rh = ch[0], bh = ch[TH * TW / 2], rv = ch[TH * TW], bv = ch[3 * TH * TW / 2];
                // ahd.py:139-145 blends h*c + v*(1-c) with c in {0,1}: the chosen candidate plus 0 x the other one, so a
                // non-finite value in the candidate NOT chosen (or in a native green, which both candidates hold) makes
                // the pixel NaN.  For finite candidates the sum is the chosen value, bit for bit.
                Rgb v[2];
#pragma unroll
                for (int b = 0; b < 2; ++b) {
                    const int k = a * 2 + b;
                    const bool pick_h = (t[b] & 0xFFu) < (t[b] >> 8);          // sum_h < sum_v; ties -> V (ahd.py:139)
                    if (p.dir_map) {                                           // optional export of the choice
                        const int sy = p.g.flip_y ? H - 1 - (fy + a) : fy + a, sx = p.g.flip_x ? W - 1 - (fx + b) : fx + b;
                        if (sy >= p.dir_rb && sy < p.dir_re) p.dir_map[(long long)(sy - p.dir_row0) * p.dir_pitch + sx] = pick_h ? 1 : 0;
                    }
                    const float r_h = b ? rh.y : rh.x, r_v = b ? rv.y : rv.x, b_h = b ? bh.y : bh.x, b_v = b ? bv.y : bv.x;
                    float g_h, g_v;
                    if (k == 0) { g_h = Q[L::P_GHR * QN + qi]; g_v = Q[L::P_GVR * QN + qi]; }
                    else if (k == 1) g_h = g_v = Q[L::P_G1 * QN + qi];
                    else if (k == 2) g_h = g_v = Q[L::P_G2 * QN + qi];
                    else { g_h = Q[L::P_GHB * QN + qi]; g_v = Q[L::P_GVB * QN + qi]; }
                    v[b].r = (pick_h ? r_h : r_v) + (pick_h ? r_v : r_h) * 0.0f;
                    v[b].g = (pick_h ? g_h : g_v) + (pick_h ? g_v : g_h) * 0.0f;
                    v[b].b = (pick_h ? b_h : b_v) + (pick_h ? b_v : b_h) * 0.0f;
                }
                stage_pixel_pair<TW, TH>(out, p.st, p.g, p.c, ty + a, tx, v[0], v[1]);
            }
        }
    }
}

template <int TW, int TH>
PYSP_HD bool select_tile_is_edge(const SelectParams& p, int tile_x, int tile_y) {
    const int x0 = tile_x * TW, y0 = p.y_begin + tile_y * TH;
    // frame borders, and tiles that overhang the end of the row range (the EDGE code skips the rows nobody needs)
    return x0 < 6 || y0 < 6 || x0 + TW + 6 > p.g.W || y0 + TH + 6 > p.g.H || y0 + TH > p.y_end;
}

}  // namespace pysp
