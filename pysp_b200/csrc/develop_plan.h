// Host-side planning of one pysp_develop call: argument validation, row ranges of every kernel in the
// chain (K1 select, then one K2 median launch per stage, each shrinking the band by 4 rows per side),
// scratch ping-pong, the 2-D views every kernel loads from / stores to.  Pure C++ (no CUDA calls) so that
// tests/host_emu can drive the same plan.
#pragma once
#include <stdarg.h>
#include <stdio.h>
#include <math.h>
#include <string.h>

#include <mutex>
#include <vector>

#include "../../include/pysp_b200.h"
#include "pysp_common.cuh"

namespace pysp {

struct DevelopPlan {
    SelectParams select;
    int n_stages;
    std::vector<MedianParams> median;      // one launch per postprocess stage (debayer/ahd.py:163-165: no upper limit)
};

static inline int plan_fail(char* err, size_t n, int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(err, n, fmt, ap);
    va_end(ap);
    return code;
}

static inline int64_t develop_scratch_bytes(int32_t width, int32_t rows, int32_t stages) {
    if (stages <= 0) return 0;
    int64_t one = (int64_t)(rows + 8 * stages) * width * 3 * (int64_t)sizeof(float);
    return stages >= 2 ? 2 * one : one;
}

// A view can be moved by TMA when its base and pitch are 16-byte aligned.  Box origins must also land on
// 16-byte columns: tiles start on such columns by construction, a horizontally flipped frame additionally
// needs a row length that is a multiple of 16 bytes (`row_bytes`).
// normalization.py:20-23 divides clip(raw - black, 0, white) by white.  For 16-bit input there are only 65536 sensor
// codes per CFA site, so the host checks exhaustively whether q' = fma(fma(-q, w, t), r, q), q = t*r, r = float(1/w)
// reproduces the IEEE quotient t/w for every code; the kernel then uses that instead of the division sequence.
// The last verdict is cached (levels rarely change between calls).
static inline bool fast_division_is_exact(const float black[4], const float white[4]) {
    static float c_black[4], c_white[4];
    static int c_valid = 0, c_result = 0;
    static std::mutex mu;
    std::lock_guard<std::mutex> lk(mu);
    if (c_valid && !memcmp(c_black, black, 16) && !memcmp(c_white, white, 16)) return c_result != 0;
    bool ok = true;
    for (int pos = 0; pos < 4 && ok; ++pos) {
        const float w = white[pos], b = black[pos];
        if (!(w > 0.0f) || !(w < 1e30f)) { ok = false; break; }
        const float r = 1.0f / w;
        for (int code = 0; code < 65536; ++code) {
            float t = fminf(fmaxf((float)code - b, 0.0f), w);
            volatile float q = t * r;
            float fast = fmaf(fmaf(-q, w, t), r, q);
            volatile float exact = t / w;
            if (!(fast == exact)) { ok = false; break; }
        }
    }
    memcpy(c_black, black, 16); memcpy(c_white, white, 16);
    c_valid = 1; c_result = ok ? 1 : 0;
    return ok;
}

static inline bool tma_ok(const View2D& v, bool flipped_x = false, long long row_bytes = 0) {
    return ((uintptr_t)v.base % 16) == 0 && (v.pitch % 16) == 0 && v.rows > 0 && v.cols > 0 &&
           (!flipped_x || row_bytes % 16 == 0);
}

static inline int plan_develop(const pysp_develop_args* a, int tw1, int th1, int tw2, int th2, DevelopPlan* plan,
                               char* err, size_t errn) {
    if (!a) return plan_fail(err, errn, PYSP_ERR_INVALID, "pysp_develop: null args");
    const int H = a->height, W = a->width;
    if (H < 4 || W < 4 || (H & 1) || (W & 1))
        return plan_fail(err, errn, PYSP_ERR_INVALID, "pysp_develop: frame %dx%d must be even and >= 4x4", H, W);
    int flip_y = 0, flip_x = 0;
    switch (a->cfa_pattern) {                 // image.py:143-152
        case PYSP_CFA_RGGB: break;
        case PYSP_CFA_BGGR: flip_y = flip_x = 1; break;
        case PYSP_CFA_GBRG: flip_x = 1; break;
        case PYSP_CFA_GRBG: flip_y = 1; break;
        default:
            return plan_fail(err, errn, PYSP_ERR_UNSUPPORTED, "pysp_develop: CFA pattern %d not implemented", a->cfa_pattern);
    }
    if (a->in_kind != PYSP_IN_U16 && a->in_kind != PYSP_IN_F32)
        return plan_fail(err, errn, PYSP_ERR_INVALID, "pysp_develop: bad in_kind %d", a->in_kind);
    if (a->out_kind < PYSP_OUT_CAM_F32 || a->out_kind > PYSP_OUT_YCC420_U8)
        return plan_fail(err, errn, PYSP_ERR_INVALID, "pysp_develop: bad out_kind %d", a->out_kind);
    if (!a->in || !a->out || (!a->lab_lut && a->quality == PYSP_QUALITY_BEST))
        return plan_fail(err, errn, PYSP_ERR_INVALID, "pysp_develop: null buffer");
    const int rb = a->row_begin, re = a->row_end;
    if (rb < 0 || re > H || rb >= re || (rb & 1) || (re & 1))
        return plan_fail(err, errn, PYSP_ERR_INVALID, "pysp_develop: row band [%d,%d) must be even and inside the frame", rb, re);
    if (a->out_row0 > rb)
        return plan_fail(err, errn, PYSP_ERR_INVALID, "pysp_develop: out_row0 %d is past row_begin %d", a->out_row0, rb);
    if (a->quality != PYSP_QUALITY_BEST && a->quality != PYSP_QUALITY_FAST)
        return plan_fail(err, errn, PYSP_ERR_UNSUPPORTED, "Quality mode not implemented: %d", a->quality);   // image.py:176
    // postprocess steps are "ignored unless using Best quality" (image.py:163)
    const int S = (a->quality == PYSP_QUALITY_BEST && a->stages > 0) ? a->stages : 0;      // debayer/ahd.py:163
    if ((int64_t)8 * S > 0x3fffffff - H)
        return plan_fail(err, errn, PYSP_ERR_INVALID, "pysp_develop: %d postprocess stages overflow the row arithmetic", S);
    const int64_t esz = a->in_kind == PYSP_IN_U16 ? 2 : 4;
    if (a->in_pitch_bytes < W * esz || (a->in_pitch_bytes % esz) || ((uintptr_t)a->in % esz))
        return plan_fail(err, errn, PYSP_ERR_INVALID, "pysp_develop: bad input pitch/alignment");
    const int64_t osz = out_kind_bytes(a->out_kind);
    const bool ycc = a->out_kind == PYSP_OUT_YCC420_U8;
    const int out_cols = ycc ? W : 3 * W;                 // elements of an output row (YCbCr 4:2:0: of the Y plane)
    if (a->out_pitch_bytes < out_cols * osz || (a->out_pitch_bytes % osz) || ((uintptr_t)a->out % osz))
        return plan_fail(err, errn, PYSP_ERR_INVALID, "pysp_develop: bad output pitch/alignment");
    if (ycc) {                                            // the chroma fields are read for this kind only
        if (!a->out_cb || !a->out_cr)
            return plan_fail(err, errn, PYSP_ERR_INVALID, "pysp_develop: null Cb or Cr plane");
        if (a->out_chroma_pitch_bytes < W / 2)
            return plan_fail(err, errn, PYSP_ERR_INVALID, "pysp_develop: chroma pitch %lld is shorter than W/2 = %d",
                             (long long)a->out_chroma_pitch_bytes, W / 2);
        if (a->out_row0 & 1)
            return plan_fail(err, errn, PYSP_ERR_INVALID, "pysp_develop: out_row0 %d must be even for 4:2:0 output", a->out_row0);
    }
    // logical (RGGB-oriented) rows of the band
    const int lb = flip_y ? H - re : rb, le = flip_y ? H - rb : re;
    auto lo = [&](int v) { return v < 0 ? 0 : v; };
    auto hi = [&](int v) { return v > H ? H : v; };
    const int k1b = lo(lb - 4 * S), k1e = hi(le + 4 * S);
    {   // the input buffer must hold the band + halo
        const int nb = lo(k1b - 6), ne = hi(k1e + 6);
        const int sb = flip_y ? H - ne : nb, se = flip_y ? H - nb : ne;
        if (a->in_row0 > sb || a->in_row0 + a->in_rows < se)
            return plan_fail(err, errn, PYSP_ERR_INVALID,
                             "pysp_develop: input holds rows [%d,%d) but rows [%d,%d) are needed (halo %d)", a->in_row0,
                             a->in_row0 + a->in_rows, sb, se, 6 + 4 * S);
    }
    const int64_t need = develop_scratch_bytes(W, re - rb, S);
    if (S > 0 && (!a->scratch || a->scratch_bytes < need || ((uintptr_t)a->scratch % 4)))
        return plan_fail(err, errn, PYSP_ERR_INVALID, "pysp_develop: 4-byte aligned scratch of %lld bytes needed", (long long)need);

    ColorParams c;
    memset(&c, 0, sizeof(c));
    for (int i = 0; i < 3; ++i) c.wb[i] = a->wb[i];
    for (int i = 0; i < 9; ++i) c.m_metric[i] = c.m_out[i] = a->cam_to_srgb[i];
    c.hdr = a->is_hdr ? 1 : 0;
    c.gamma = a->apply_gamma ? 1 : 0;
    FrameGeom g = {H, W, flip_y, flip_x};

    const int64_t scratch_rows = (re - rb) + 8 * S;
    auto final_store = [&](StoreParams& st) {
        st.mode = OUT_FINAL; st.kind = a->out_kind;
        st.img.base = (char*)a->out + (int64_t)(rb - a->out_row0) * a->out_pitch_bytes;
        st.img.pitch = a->out_pitch_bytes; st.img.rows = re - rb; st.img.cols = out_cols; st.img.elem = (int)osz;
        st.img_row0 = rb;
        if (ycc) {
            const int64_t c0 = (int64_t)(rb - a->out_row0) / 2 * a->out_chroma_pitch_bytes;   // chroma row rb/2 of the views
            st.cb.base = (char*)a->out_cb + c0; st.cr.base = (char*)a->out_cr + c0;
            st.cb.pitch = st.cr.pitch = a->out_chroma_pitch_bytes;
            st.cb.rows = st.cr.rows = (re - rb) / 2; st.cb.cols = st.cr.cols = W / 2; st.cb.elem = st.cr.elem = 1;
        }
        st.tma = osz == 4 && tma_ok(st.img, flip_x != 0, (long long)W * 12);
    };
    auto plane_store = [&](StoreParams& st, int buf, int row0, int rows) {
        st.mode = OUT_PLANES; st.kind = OUT_CAM_F32;
        st.tma = 1;
        for (int k = 0; k < 3; ++k) {
            st.plane[k].base = (float*)a->scratch + ((int64_t)buf * 3 + k) * scratch_rows * W;
            st.plane[k].pitch = (long long)W * 4; st.plane[k].rows = rows; st.plane[k].cols = W; st.plane[k].elem = 4;
            st.tma = st.tma && tma_ok(st.plane[k]);
        }
        st.plane_row0 = row0;
    };

    memset(&plan->select, 0, sizeof(plan->select));
    plan->median.assign((size_t)S, MedianParams());
    for (auto& mp : plan->median) memset(&mp, 0, sizeof(mp));
    SelectParams& sp = plan->select;
    sp.g = g; sp.c = c;
    sp.in_kind = a->in_kind;
    sp.in.base = (void*)a->in; sp.in.pitch = a->in_pitch_bytes; sp.in.rows = a->in_rows; sp.in.cols = W; sp.in.elem = (int)esz;
    sp.in_row0 = a->in_row0;
    sp.tma_in = tma_ok(sp.in, flip_x != 0, (long long)W * esz);
    const int perm[4] = {0, 1, 3, 2};          // [TL,TR,BR,BL] -> index (sy&1)*2+(sx&1)
    for (int i = 0; i < 4; ++i) { sp.black[perm[i]] = a->black[i]; sp.white[perm[i]] = a->white[i]; }
    if (a->in_kind == PYSP_IN_U16) {
        for (int i = 0; i < 4; ++i) sp.rwhite[i] = 1.0f / sp.white[i];
        sp.fast_div = fast_division_is_exact(sp.black, sp.white) ? 1 : 0;
    }
    sp.lut = (const uint4*)a->lab_lut;
    sp.algo = a->quality == PYSP_QUALITY_FAST ? ALGO_EAG : ALGO_AHD;
    if (a->dir_map && sp.algo == ALGO_AHD) {
        if (a->dir_map_pitch_bytes < W)
            return plan_fail(err, errn, PYSP_ERR_INVALID, "pysp_develop: dir_map pitch %lld is shorter than a row", (long long)a->dir_map_pitch_bytes);
        sp.dir_map = a->dir_map; sp.dir_pitch = a->dir_map_pitch_bytes; sp.dir_row0 = a->out_row0; sp.dir_rb = rb; sp.dir_re = re;
    }
    sp.y_begin = k1b; sp.y_end = k1e;
    sp.tiles_x = (W + tw1 - 1) / tw1;
    sp.n_tiles = sp.tiles_x * ((k1e - k1b + th1 - 1) / th1);
    if (S == 0) final_store(sp.st); else plane_store(sp.st, 0, k1b, k1e - k1b);
    plan->n_stages = S;
    for (int s = 1; s <= S; ++s) {
        MedianParams& mp = plan->median[s - 1];
        const StoreParams& prev = s == 1 ? sp.st : plan->median[s - 2].st;
        mp.g = g; mp.c = c;
        for (int k = 0; k < 3; ++k) mp.in[k] = prev.plane[k];
        mp.in_row0 = prev.plane_row0;
        mp.tma_in = prev.tma;
        mp.y_begin = lo(lb - 4 * (S - s)); mp.y_end = hi(le + 4 * (S - s));
        mp.tiles_x = (W + tw2 - 1) / tw2;
        mp.n_tiles = mp.tiles_x * ((mp.y_end - mp.y_begin + th2 - 1) / th2);
        if (s == S) final_store(mp.st); else plane_store(mp.st, s & 1, mp.y_begin, mp.y_end - mp.y_begin);
    }
    return PYSP_OK;
}

}  // namespace pysp
