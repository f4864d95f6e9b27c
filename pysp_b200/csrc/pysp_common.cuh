// pysp_b200 -- shared definitions for the develop-path kernels (sm_100a).
//
// All arithmetic on the path is specified operation by operation (oracle/ahd_spec.py, SURVEY.md
// Appendix B): every float32 op is rounded individually.  The device build therefore uses
// `-fmad=false` (no implicit FMA contraction); `fmaf()` is written explicitly only where the product
// is exact (power-of-two weights), so that it equals mul-then-add bit for bit.
//
// The tile functions in ahd_select.cuh / median_stage.cuh are written as *phases* separated by
// block barriers.  Inside a phase every work item is independent, so the same source also compiles
// for the host (PYSP_HOST_EMU, used only by tests/host_emu to debug tile logic without a GPU) where a
// phase simply runs its work items serially.  The product library never contains that build.
#pragma once
#include <stdint.h>

#ifdef PYSP_HOST_EMU
#include <math.h>
#include <string.h>
#define PYSP_HD inline
#define PYSP_D inline
#define PYSP_NOINLINE inline
#define PYSP_SYNC() ((void)0)
#define PYSP_ITEMS(var, n) for (int var = 0; var < (n); ++var)
#define PYSP_ROW_ITEMS32(row, col, nrows, ncols)            \
    for (int row = 0; row < (nrows); ++row)                 \
        for (int col = 0; col < (ncols); ++col)
static inline float pysp_as_float(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
static inline uint32_t pysp_as_uint(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }
template <typename T> static inline T pysp_ldg(const T* p) { return *p; }
#else
#include <cuda_runtime.h>
#define PYSP_HD __device__ __forceinline__
#define PYSP_D __device__ __forceinline__
// called once per pixel and direction: kept out of line so that the phase bodies fit the instruction cache
#define PYSP_NOINLINE __device__ __noinline__
#define PYSP_SYNC() __syncthreads()
#define PYSP_ITEMS(var, n) for (int var = threadIdx.x; var < (n); var += blockDim.x)
// Work items on an nrows x ncols grid (ncols <= 32), one grid row per warp pass: the lanes of a warp never straddle two
// rows, so unit-stride shared-memory accesses of a row stay free of bank conflicts (a flat item index wraps mid-warp and
// costs a second wavefront on every access).  `continue` in the body skips the item.
#define PYSP_ROW_ITEMS32(row, col, nrows, ncols)                                                    \
    for (int it_ = threadIdx.x; it_ < (nrows) * 32; it_ += blockDim.x)                              \
        for (int row = it_ >> 5, col = it_ & 31, once_ = 1; once_ && col < (ncols); once_ = 0)
__device__ __forceinline__ float pysp_as_float(uint32_t u) { return __uint_as_float(u); }
__device__ __forceinline__ uint32_t pysp_as_uint(float f) { return __float_as_uint(f); }
template <typename T> __device__ __forceinline__ T pysp_ldg(const T* p) { return __ldg(p); }
#endif

// Developer instrumentation (tools/kbench.py --phases, -DPYSP_PHASE_CLOCKS): thread 0 of every CTA accumulates the
// SM clock between phase boundaries into g_phase_clk.  Compiled out of the product build.
#if defined(PYSP_PHASE_CLOCKS) && !defined(PYSP_HOST_EMU)
__device__ unsigned long long g_phase_clk[2][16];
#define PYSP_PHASE_BEGIN() long long ph_t_ = clock64()
#define PYSP_PHASE_MARK(k, i)                                                          \
    if (threadIdx.x == 0) {                                                            \
        long long n_ = clock64();                                                      \
        atomicAdd(&g_phase_clk[k][i], (unsigned long long)(n_ - ph_t_));               \
        ph_t_ = n_;                                                                    \
    }
#else
#define PYSP_PHASE_BEGIN() ((void)0)
#define PYSP_PHASE_MARK(k, i) ((void)0)
#endif

namespace pysp {

// ---- constants of the reference algorithm ---------------------------------------------------------
// debayer/ahd.py:89-94: h = normalise(0.125*h_optimal + 0.875*h_fast) evaluated in float32.
#define PYSP_H0 (-0x1.053316p-2f)
#define PYSP_H1 (0x1p-1f)
#define PYSP_H2 (0x1.053316p-1f)
// cv2.getGaussianKernel(3, 1.0) in float32 (debayer/ahd.py:120-121)
#define PYSP_GK0 (0.27406862f)
#define PYSP_GK1 (0.45186275f)

enum InKind { IN_U16 = 0, IN_F32 = 1 };
enum OutKind { OUT_CAM_F32 = 0, OUT_LIN_F32 = 1, OUT_LIN_F16 = 2, OUT_SRGB_U8 = 3, OUT_SRGB_U16 = 4, OUT_YCC420_U8 = 5 };
#ifdef __CUDACC__
#define PYSP_HOSTDEV __host__ __device__
#else
#define PYSP_HOSTDEV
#endif
// bytes per stored element (for OUT_YCC420_U8: per sample of any of its three planes)
PYSP_HOSTDEV constexpr int out_kind_bytes(int kind) {
    return (kind == OUT_SRGB_U8 || kind == OUT_YCC420_U8) ? 1 : ((kind == OUT_LIN_F16 || kind == OUT_SRGB_U16) ? 2 : 4);
}

struct FrameGeom {
    int H, W;            // frame size (even); flips keep the size
    int flip_y, flip_x;  // image.py:143-152: logical RGGB coord (y,x) <-> stored (fy?H-1-y:y, fx?W-1-x:x)
};

struct ColorParams {
    float wb[3];         // reciprocal neutral multipliers (wb_cct/cam_wb.py:243)
    double m_metric[9];  // camera -> linear sRGB used by the homogeneity metric (debayer/ahd.py:45-48)
    double m_out[9];     // camera -> linear sRGB of to_lin_srgb (base_types/image_base.py:62-64)
    int hdr;             // debayer/ahd.py:52-59
    int gamma;           // apply lin_srgb_to_srgb in the epilogue (colorize/transform.py:89-99)
};

struct View2D {          // plain description of a 2-D tensor (rows x cols elements), see tma.cuh
    void* base;
    long long pitch;     // bytes
    int rows, cols;
    int elem;            // bytes per element
};

// Output of a kernel of the chain: either the final image (interleaved RGB, stored orientation, clipped to the
// rows of the band) or the scratch handed to the next median stage: three float planes r-g, b-g, g in logical
// orientation (debayer/ahd.py:153-154 needs exactly these), so that the next stage loads them by TMA as is.
enum OutMode { OUT_FINAL = 0, OUT_PLANES = 1 };
enum Algo { ALGO_AHD = 0, ALGO_EAG = 1 };

struct StoreParams {
    int mode;            // OutMode
    int kind;            // OutKind (final only)
    View2D img;          // final: [band rows][3*W] of f32/f16; row 0 = first stored row of the band
                         //   (OUT_YCC420_U8: the Y plane, [band rows][W])
    View2D cb, cr;       // OUT_YCC420_U8 only: [band rows / 2][W / 2]; row 0 = stored chroma row img_row0 / 2
    int img_row0;        // stored row number of img row 0
    View2D plane[3];     // planes: [rows][W] f32, row 0 = logical row plane_row0
    int plane_row0;
    int tma;             // 1: the views are also described by the tensor maps passed to the kernel
};

struct SelectParams {    // K1: mosaic -> selected camera RGB
    FrameGeom g;
    ColorParams c;
    int in_kind;
    View2D in;           // stored orientation; row 0 = stored row in_row0
    int in_row0;
    int tma_in;
    float black[4], white[4];   // by stored-mosaic position TL,TR,BL,BR (normalization.py:20-23)
    float rwhite[4];     // float(1/white)
    int fast_div;        // 1: reciprocal + FMA correction verified equal to IEEE division for these levels
    const uint4* lut;    // paired-node Lab table (device), see lab_lookup
    int algo;            // ALGO_AHD (QualityDemosaic.Best) or ALGO_EAG (QualityDemosaic.Fast)
    StoreParams st;
    int y_begin, y_end;  // logical rows to produce (even)
    int tiles_x, n_tiles;
    // optional export of the direction choice (one byte per pixel, stored orientation): rows [dir_rb, dir_re) of the
    // frame as stored are written, map row 0 = stored row dir_row0
    uint8_t* dir_map;
    long long dir_pitch;
    int dir_row0, dir_rb, dir_re;
};

struct MedianParams {    // K2: one postprocess stage (debayer/ahd.py:148-161)
    FrameGeom g;
    ColorParams c;
    View2D in[3];        // r-g, b-g, g planes, logical orientation, row 0 = logical row in_row0
    int in_row0;
    int tma_in;
    StoreParams st;
    int y_begin, y_end;
    int tiles_x, n_tiles;
};

// ---- border index maps -----------------------------------------------------------------------------
PYSP_HD int clampi(int v, int n) { return v < 0 ? 0 : (v >= n ? n - 1 : v); }          // REPLICATE / 1-px BORDER_REFLECT
PYSP_HD int reflect101(int v, int n) { return v < 0 ? -v : (v >= n ? 2 * n - 2 - v : v); }
// quarter-plane edge duplication expressed on full-res mosaic coordinates (debayer/ahd.py:77-80):
// keeps the CFA phase.
PYSP_HD int phase_clamp(int v, int n) { return v < 0 ? (v & 1) : (v >= n ? n - 2 + (v & 1) : v); }

// ---- float64 3x3, result rounded to float32 ---------------------------------------------------------
// Accumulation order of the reference's np.dot (OpenBLAS dgemm, K = 3): acc = m0*c0; acc = fma(m1, c1, acc);
// acc = fma(m2, c2, acc) -- pinned by tests/golden/dot_fma_pins.npz (colorize/transform.py:52-53).
PYSP_HD float dot3_f64(const double* m, float c0, float c1, float c2) {
#ifdef __CUDA_ARCH__
    double a = __dmul_rn(m[0], (double)c0);
    a = __fma_rn(m[1], (double)c1, a);
    return __double2float_rn(__fma_rn(m[2], (double)c2, a));
#else
    volatile double a = m[0] * (double)c0;
    a = fma(m[1], (double)c1, a);
    a = fma(m[2], (double)c2, a);
    return (float)a;
#endif
}

#ifdef __CUDA_ARCH__
__device__ __forceinline__ float exp2f_fast(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
#endif

// np.clip(v, 0, 1) (colorize/transform.py:6-19): NaN stays NaN (max.NaN / min.NaN: one FMNMX each, as fminf/fmaxf)
PYSP_HD float clip01(float v) {
#ifdef __CUDA_ARCH__
    float t, r;
    asm("max.NaN.f32 %0, %1, 0f00000000;" : "=f"(t) : "f"(v));
    asm("min.NaN.f32 %0, %1, 0f3F800000;" : "=f"(r) : "f"(t));
    return r;
#else
    return v != v ? v : fminf(fmaxf(v, 0.0f), 1.0f);
#endif
}
// cv2's clamp in front of the Lab quantisation: NaN -> 0, +inf -> 1, -inf -> 0 (probed on cv2 4.13, both code paths)
PYSP_HD float sat01(float v) { return fminf(fmaxf(v, 0.0f), 1.0f); }

// colorize/transform.py:98-99 in float32.  x^(1/2.4) = exp2(log2(x) / 2.4) with the hardware approximations (MUFU.LG2 /
// MUFU.EX2): relative error of the curve about 1e-6, inside the 1e-4 the parity contract states for the gamma.
PYSP_HD float srgb_gamma(float v) {
    float x = clip01(v);
#ifdef __CUDA_ARCH__
    const float pw = exp2f_fast(__log2f(x) * (float)(1.0 / 2.4));
#else
    const float pw = powf(x, (float)(1.0 / 2.4));
#endif
    return x <= 0.0031308f ? x * 12.92f : (1.055f * pw) - 0.055f;
}

// wire-format quantisation of a gamma-encoded value in [0, 1] (NaN -> 0): round half to even of v * scale
PYSP_HD uint32_t quantise(float v, float scale) {
    float y = fmaf(sat01(v), scale, 8388608.0f);        // v * scale <= 65535 is below 2^23: adding 2^23 rounds to an integer
    return pysp_as_uint(y) & 0x7FFFFFu;
}

// libjpeg's full-range R'G'B' -> YCbCr (jccolor.c rgb_ycc_convert, 16-bit fixed point) and 2x2 chroma average
// (jcsample.c h2v2_downsample) of one 2x2 block of 8-bit pixels.  r[k], g[k], b[k]: pixels TL, TR, BL, BR.  bias: 1 for an
// even stored chroma column, 2 for an odd one.  y01 / y23: the block's top / bottom Y pair, left pixel in the low byte.
// Every intermediate is non-negative (the chroma offset (128 << 16) + 32767 exceeds 0.5 * 255 * 65536), so the shifts
// are the arithmetic shifts of the C source.
struct Ycc2x2 { uint32_t y01, y23, cb, cr; };
PYSP_HD Ycc2x2 ycc_block(const uint32_t r[4], const uint32_t g[4], const uint32_t b[4], uint32_t bias) {
    Ycc2x2 o;
    uint32_t y[4], cb = 0, cr = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        y[k] = (19595u * r[k] + 38470u * g[k] + 7471u * b[k] + 32768u) >> 16;
        cb += (32768u * b[k] + (128u << 16) + 32767u - 11059u * r[k] - 21709u * g[k]) >> 16;
        cr += (32768u * r[k] + (128u << 16) + 32767u - 27439u * g[k] - 5329u * b[k]) >> 16;
    }
    o.y01 = y[0] | (y[1] << 8); o.y23 = y[2] | (y[3] << 8);
    o.cb = (cb + bias) >> 2; o.cr = (cr + bias) >> 2;
    return o;
}

// ---- cv2 RGB->Lab (float32 path) : quantise, trilinear in the 33^3 int16 table -----------------------
// Returns L as the reference float (v*100/16384) and (a,b) as the raw integers v (a = v/64-128 exactly,
// so differences and squared distances of the integers are the reference's scaled by exact powers of
// two; every comparison in the homogeneity count is unchanged).
//
// Device table layout (pysp_lab_lut_pack_host): node (ir, ig, ib), ir, ig in 0..33 (index 33 repeats 32 so the
// upper corner needs no clamp: its weight is zero there), ib in 0..32, is a uint4
//     { L[ib] | L[ib+1] << 16,  a[ib] | a[ib+1] << 16,  b[ib] | b[ib+1] << 16,  0 }
// so one 16-byte load brings both blue corners of all three channels and the blue interpolation is a 2-way
// 16x8-bit dot product (IDP.2A).  The sum of the eight weighted corners is integer arithmetic, hence exact in
// any association: interpolate along blue, then green, then red.
struct LabQ { float L; uint32_t ab; };
#define PYSP_LUT_NR 34
#define PYSP_LUT_NG 34
#define PYSP_LUT_NB 33

#if !defined(PYSP_HOST_EMU) && !defined(__CUDACC__)
struct uint4 { unsigned int x, y, z, w; };
#endif

PYSP_HD uint32_t quant14(float v) {
    // cvRound(clip(v,0,1)*16384): the product is exact, adding 2^23 rounds half-to-even (one FMA: exact product)
#ifdef __CUDA_ARCH__
    float y = fmaf(__saturatef(v), 16384.0f, 8388608.0f);
#else
    float y = fmaf(sat01(v), 16384.0f, 8388608.0f);
#endif
    return pysp_as_uint(y) & 0x7FFFFFu;
}

PYSP_HD uint32_t dot2_u16_u8(uint32_t pair16, uint32_t w8, uint32_t acc) {
#ifdef __CUDA_ARCH__
    return __dp2a_lo(pair16, w8, acc);
#else
    return acc + (pair16 & 0xFFFFu) * (w8 & 0xFFu) + (pair16 >> 16) * ((w8 >> 8) & 0xFFu);
#endif
}

struct LabKey { const uint4* base; uint32_t sr, sg, sb; };        // first of the four table nodes + the three 4-bit fractions

PYSP_HD LabKey lab_key(const uint4* __restrict__ lut, float r, float g, float b) {
    const uint32_t cr = quant14(r), cg = quant14(g), cb = quant14(b);
    const uint32_t tr = cr >> 9, tg = cg >> 9, tb = cb >> 9;
    LabKey k;
    k.sr = (cr >> 5) & 15u; k.sg = (cg >> 5) & 15u; k.sb = (cb >> 5) & 15u;
    k.base = lut + (tr * PYSP_LUT_NG + tg) * PYSP_LUT_NB + tb;
    return k;
}

PYSP_HD LabQ lab_interp(const LabKey& k, const uint4& e00, const uint4& e01, const uint4& e10, const uint4& e11) {
    const uint32_t sr = k.sr, sg = k.sg, sb = k.sb;
    const uint32_t wb = (16u - sb) | (sb << 8), wg0 = 16u - sg, wr0 = 16u - sr;
    // the four (red, green) corner weights are shared by the three channels: 4 + 3 x 4 multiplies instead of 3 x 6.
    // Integer arithmetic: any association of the weighted corner sum is exact (at most 16384 * 4096 < 2^32).
    const uint32_t w00 = wr0 * wg0, w01 = wr0 * sg, w10 = sr * wg0, w11 = sr * sg;
    uint32_t v[3];
#define PYSP_CH(c, f)                                                                              \
    {                                                                                              \
        uint32_t p00 = dot2_u16_u8(e00.f, wb, 0u), p01 = dot2_u16_u8(e01.f, wb, 0u);               \
        uint32_t p10 = dot2_u16_u8(e10.f, wb, 0u), p11 = dot2_u16_u8(e11.f, wb, 0u);               \
        v[c] = (p00 * w00 + p01 * w01 + p10 * w10 + p11 * w11 + 2048u) >> 12;                      \
    }
    PYSP_CH(0, x) PYSP_CH(1, y) PYSP_CH(2, z)
#undef PYSP_CH
    LabQ q;
    q.L = (pysp_as_float(0x4B000000u | v[0]) - 8388608.0f) * (100.0f / 16384.0f);
    q.ab = v[1] | (v[2] << 16);
    return q;
}

PYSP_HD LabQ lab_lookup(const uint4* __restrict__ lut, float r, float g, float b) {
    const LabKey k = lab_key(lut, r, g, b);
    const uint4 e00 = pysp_ldg(k.base);
    const uint4 e01 = pysp_ldg(k.base + PYSP_LUT_NB);
    const uint4 e10 = pysp_ldg(k.base + PYSP_LUT_NG * PYSP_LUT_NB);
    const uint4 e11 = pysp_ldg(k.base + PYSP_LUT_NG * PYSP_LUT_NB + PYSP_LUT_NB);
    return lab_interp(k, e00, e01, e10, e11);
}

// integer-valued float from a 16-bit field, offset by 2^23 (differences of two such values are exact)
#ifdef __CUDA_ARCH__
PYSP_HD float ab_lo(uint32_t ab) { return pysp_as_float(__byte_perm(ab, 0x4B000000u, 0x7610)); }   // one PRMT each
PYSP_HD float ab_hi(uint32_t ab) { return pysp_as_float(__byte_perm(ab, 0x4B000000u, 0x7632)); }
#else
PYSP_HD float ab_lo(uint32_t ab) { return pysp_as_float(0x4B000000u | (ab & 0xFFFFu)); }
PYSP_HD float ab_hi(uint32_t ab) { return pysp_as_float(0x4B000000u | (ab >> 16)); }
#endif

// 8-byte shared-memory pairs (one LDS.64)
struct __attribute__((aligned(8))) F2 { float x, y; };
struct __attribute__((aligned(8))) U2 { uint32_t x, y; };

// homogeneity test of one window cell (ahd_homogeneity_cython.pyx:56-58): all ones when both the lightness and the
// chroma test pass.  pass_ge takes the lightness difference seen from the other end of the pair (-dl <= eps).
// n + 1 if the window cell passes both tests (ahd_homogeneity_cython.pyx:56-58), else n: two compares and one predicated add
PYSP_HD uint32_t count_le(uint32_t n, float dl, float epsl, float d2, float epsc) {
#ifdef __CUDA_ARCH__
    asm("{ .reg .pred p, q; setp.le.f32 p, %1, %2; setp.le.and.f32 q, %3, %4, p; @q add.u32 %0, %0, 1; }" : "+r"(n) : "f"(dl), "f"(epsl), "f"(d2), "f"(epsc));
    return n;
#else
    return n + ((dl <= epsl && d2 <= epsc) ? 1u : 0u);
#endif
}
PYSP_HD uint32_t count_ge(uint32_t n, float dl, float neg_epsl, float d2, float epsc) {
#ifdef __CUDA_ARCH__
    asm("{ .reg .pred p, q; setp.ge.f32 p, %1, %2; setp.le.and.f32 q, %3, %4, p; @q add.u32 %0, %0, 1; }" : "+r"(n) : "f"(dl), "f"(neg_epsl), "f"(d2), "f"(epsc));
    return n;
#else
    return n + ((dl >= neg_epsl && d2 <= epsc) ? 1u : 0u);
#endif
}
PYSP_HD uint32_t pass_le(float dl, float epsl, float d2, float epsc) {
#ifdef __CUDA_ARCH__
    uint32_t m;
    asm("{ .reg .pred p; setp.le.f32 p, %1, %2; set.le.and.u32.f32 %0, %3, %4, p; }" : "=r"(m) : "f"(dl), "f"(epsl), "f"(d2), "f"(epsc));
    return m;
#else
    return (dl <= epsl && d2 <= epsc) ? 0xFFFFFFFFu : 0u;
#endif
}
PYSP_HD uint32_t pass_ge(float dl, float neg_epsl, float d2, float epsc) {
#ifdef __CUDA_ARCH__
    uint32_t m;
    asm("{ .reg .pred p; setp.ge.f32 p, %1, %2; set.le.and.u32.f32 %0, %3, %4, p; }" : "=r"(m) : "f"(dl), "f"(neg_epsl), "f"(d2), "f"(epsc));
    return m;
#else
    return (dl >= neg_epsl && d2 <= epsc) ? 0xFFFFFFFFu : 0u;
#endif
}

// debayer/ahd.py:45-59 : candidate camera RGB -> the RGB that goes into the Lab conversion (and, for HDR frames, the luma
// that replaces L): white balance a second time (ahd.py:46-48), float64 matrix, HDR tone curve x/(1+x) (ahd.py:52-57)
PYSP_HD void metric_rgb(const ColorParams& c, float r, float g, float b, float* o, float* luma) {
    float c0 = r * c.wb[0], c1 = g * c.wb[1], c2 = b * c.wb[2];
    float sr = dot3_f64(c.m_metric + 0, c0, c1, c2);
    float sg = dot3_f64(c.m_metric + 3, c0, c1, c2);
    float sb = dot3_f64(c.m_metric + 6, c0, c1, c2);
    *luma = 0.0f;
    if (c.hdr) {
        *luma = ((0.2126f * sr) + (0.7152f * sg)) + (0.0722f * sb);
        sr = sr / (1.0f + sr); sg = sg / (1.0f + sg); sb = sb / (1.0f + sb);
    }
    o[0] = sr; o[1] = sg; o[2] = sb;
}

// debayer/ahd.py:45-62 : candidate camera RGB -> (L, a, b) of the homogeneity metric
PYSP_HD LabQ metric_lab(const ColorParams& c, const uint4* __restrict__ lut, float r, float g, float b) {
    float m[3], luma;
    metric_rgb(c, r, g, b, m, &luma);
    LabQ q = lab_lookup(lut, m[0], m[1], m[2]);
    if (c.hdr) q.L = luma;
    return q;
}

// ---- output epilogue ------------------------------------------------------------------------------------
// camera RGB -> stored pixel.  OUT_CAM_F32: as is.  OUT_LIN_*: clip to [0,1], float64 3x3
// (colorize/transform.py:37-53), optional gamma.
struct Rgb { float r, g, b; };

PYSP_HD Rgb finish_pixel(const ColorParams& c, int out_kind, Rgb v) {
    if (out_kind == OUT_CAM_F32) return v;
    float c0 = clip01(v.r), c1 = clip01(v.g), c2 = clip01(v.b);
    Rgb o;
    o.r = dot3_f64(c.m_out + 0, c0, c1, c2);
    o.g = dot3_f64(c.m_out + 3, c0, c1, c2);
    o.b = dot3_f64(c.m_out + 6, c0, c1, c2);
    if (c.gamma || out_kind >= OUT_SRGB_U8) { o.r = srgb_gamma(o.r); o.g = srgb_gamma(o.g); o.b = srgb_gamma(o.b); }
    return o;
}

}  // namespace pysp
