/* pysp_b200 -- C ABI of the B200-native develop path (libpysp_b200.so).
 *
 * Drop-in boundary for bullbin/pySP's raw -> linear-sRGB develop path.  The reference has no FFI of its
 * own: the seams are Python callables plus one Cython `cpdef` (SURVEY.md section 8b).  Each entry point
 * below names the reference callable(s) it replaces (file:line in the reference tree); INTEGRATION.md
 * shows the ctypes binding a pySP maintainer would add.
 *
 * Conventions
 *  - plain C types only; every image pointer is a DEVICE pointer owned by the caller (e.g. a torch
 *    tensor's data_ptr()) unless the name ends in `_host`;
 *  - asynchronous on the CUDA stream passed as `stream` (a cudaStream_t cast to void*; NULL = default
 *    stream) on the current device.  The library allocates NO device memory and makes no synchronising
 *    call: scratch and workspaces are caller-provided.  What it does keep, all host-side and mutex-guarded, so
 *    calls are re-entrant across streams, devices and threads:
 *      . per device, the launch set-up of the develop kernels (shared-memory opt-in, persistent grid sizes),
 *        queried on the first pysp_develop on that device; later calls only launch kernels (capturable in a
 *        CUDA graph);
 *      . the verdict of the last normalisation-division check (exhaustive over the 65536 sensor codes of one
 *        level set; re-done when the levels change);
 *      . the event pairs of the bench instrumentation while pysp_timing_enable(1) is in effect;
 *      . the test hook PYSP_DISABLE_TMA, read once per process;
 *  - return value: PYSP_OK or a negative code; pysp_last_error() returns the calling thread's message.
 *    PYSP_ERR_INVALID maps to the reference's ValueError/AssertionError cases, PYSP_ERR_UNSUPPORTED to
 *    NotImplementedError (image.py:152,176), PYSP_ERR_CUDA to a CUDA runtime failure;
 *  - there is no CPU path: without a CUDA device every compute entry point fails with PYSP_ERR_CUDA.
 */
#ifndef PYSP_B200_H
#define PYSP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PYSP_OK 0
#define PYSP_ERR_INVALID (-1)
#define PYSP_ERR_UNSUPPORTED (-2)
#define PYSP_ERR_CUDA (-3)

/* base_types/image_base.py:13-17 (BayerPattern) */
#define PYSP_CFA_RGGB 1
#define PYSP_CFA_BGGR 2
#define PYSP_CFA_GRBG 3
#define PYSP_CFA_GBRG 4

#define PYSP_IN_U16 0      /* sensor counts; normalisation (normalization.py:4-25) is fused into the load */
#define PYSP_IN_F32 1      /* `sensor_scaled` float32 mosaic (RawRggbBayerData, HDR mosaics) */

#define PYSP_OUT_CAM_F32 0 /* RawDemosaicData.image: camera RGB, WB applied once (debayer/ahd.py:167) */
#define PYSP_OUT_LIN_F32 1 /* ... .to_lin_srgb() (base_types/image_base.py:62-64) */
#define PYSP_OUT_LIN_F16 2 /* same, stored as half */
/* Wire-format outputs: lin_srgb_to_srgb (colorize/transform.py:89-99) applied to the linear-sRGB result and rounded to
 * nearest into 8 / 16 bits (x * 255, x * 65535).  The reference stops at float32; these are what a caller that encodes
 * or displays the image needs, at 3 / 6 instead of 12 bytes per pixel over PCIe. */
#define PYSP_OUT_SRGB_U8 3
#define PYSP_OUT_SRGB_U16 4
/* JPEG-ready planes, 1.5 bytes per pixel: the PYSP_OUT_SRGB_U8 result S[y][x][0..2] = R, G, B of the same call, converted
 * exactly as libjpeg converts and subsamples it for a 4:2:0 JPEG (jccolor.c rgb_ycc_convert, full-range JFIF / BT.601;
 * jcsample.c h2v2_downsample), so that a JPEG encoded from the planes is byte-identical to one libjpeg encodes from S.
 * Integer arithmetic, arithmetic shifts, stored orientation:
 *     Y [y][x]   = (19595*R + 38470*G + 7471*B + 32768) >> 16
 *     cb[y][x]   = (-11059*R - 21709*G + 32768*B + (128 << 16) + 32767) >> 16
 *     cr[y][x]   = (32768*R - 27439*G - 5329*B + (128 << 16) + 32767) >> 16
 *     Cb[cy][cx] = (cb[2cy][2cx] + cb[2cy][2cx+1] + cb[2cy+1][2cx] + cb[2cy+1][2cx+1] + 1 + (cx & 1)) >> 2   (Cr alike)
 * cx is the chroma column of the whole stored frame.  `out` holds Y ([rows][width], pitch out_pitch_bytes >= width),
 * `out_cb` / `out_cr` hold Cb / Cr ([rows/2][width/2], pitch out_chroma_pitch_bytes >= width/2).  Y row 0 is stored row
 * out_row0 (which must be even), chroma row 0 is stored chroma row out_row0/2; a band [row_begin, row_end) writes Y rows
 * [row_begin, row_end) and chroma rows [row_begin/2, row_end/2) only. */
#define PYSP_OUT_YCC420_U8 5

/* const.py:3-6 (QualityDemosaic); Draft is not on the B200 path */
#define PYSP_QUALITY_BEST 0
#define PYSP_QUALITY_FAST 1

#define PYSP_MAX_BRACKETS 16

/* One develop call = RawBayerData.demosaic(QualityDemosaic.Best, stages) [+ .to_lin_srgb()
 * [+ lin_srgb_to_srgb]] on one frame or one row band of it.
 * Replaces: image.py:191-197 (to_rggb, demosaic), image.py:156-183 (dispatch, un-flip),
 * debayer/ahd.py:14-170 (debayer_ahd incl. the Cython build_map, ahd_homogeneity_cython.pyx:61),
 * debayer/edge_assisted_gaussian.py:188-201 (debayer_eag) for PYSP_QUALITY_FAST,
 * normalization.py:4-25 when in_kind == PYSP_IN_U16, base_types/image_base.py:62-64 and
 * colorize/transform.py:21-53,76-99 for the PYSP_OUT_LIN_* kinds. */
typedef struct pysp_develop_args {
    int32_t height, width;       /* whole frame, both even and >= 4 */
    int32_t cfa_pattern;         /* PYSP_CFA_*; non-RGGB frames are flipped on load/store (image.py:143-152) */
    int32_t in_kind;             /* PYSP_IN_* */
    const void* in;              /* rows [in_row0, in_row0 + in_rows) of the frame as stored */
    int64_t in_pitch_bytes;
    int32_t in_row0, in_rows;
    float black[4];              /* per CFA site of the STORED mosaic, reference order [TL, TR, BR, BL] */
    float white[4];              /*   (normalization.py:20-23); ignored for PYSP_IN_F32 */
    float wb[3];                 /* cam_wb.get_reciprocal_multipliers() (wb_cct/cam_wb.py:236-243), float32 */
    double cam_to_srgb[9];       /* row-major 3x3 of colorize/transform.py:40-49, built on the host in float64 */
    int32_t stages;              /* postprocess_stages, clamped at 0 (debayer/ahd.py:163) */
    int32_t is_hdr;              /* image.get_hdr() (debayer/ahd.py:52-59) */
    int32_t apply_gamma;         /* fuse lin_srgb_to_srgb (colorize/transform.py:89-99) into the epilogue */
    int32_t out_kind;            /* PYSP_OUT_* */
    void* out;                   /* [rows][width][3], rows [out_row0, ...) of the frame as stored (Y plane
                                    [rows][width] for PYSP_OUT_YCC420_U8) */
    int64_t out_pitch_bytes;
    int32_t out_row0;
    int32_t row_begin, row_end;  /* stored rows to produce, even; whole frame = [0, height) */
    void* scratch;               /* >= pysp_develop_scratch_bytes(...) bytes when stages > 0 */
    int64_t scratch_bytes;
    const void* lab_lut;         /* device copy of the table packed by pysp_lab_lut_pack_host (Best only) */
    int32_t quality;             /* PYSP_QUALITY_BEST: debayer_ahd; PYSP_QUALITY_FAST: debayer_eag
                                    (debayer/edge_assisted_gaussian.py:188-201; stages and is_hdr are ignored) */
    uint8_t* dir_map;            /* optional (NULL = none; Best only): the AHD direction choice `map_h < map_v`
                                    (debayer/ahd.py:136-139), one byte per pixel, 1 = horizontal candidate taken;
                                    [rows][width] for rows [out_row0, ...) of the frame as stored.  The reference never
                                    returns this map; it is exported so that parity of the choice can be checked. */
    int64_t dir_map_pitch_bytes;
    /* PYSP_OUT_YCC420_U8 only (appended: the library reads these three fields for that kind alone, so callers built
       against the struct without them stay valid for every other kind) */
    void* out_cb;                /* [rows/2][width/2] Cb, chroma rows [out_row0/2, ...) of the frame as stored */
    void* out_cr;                /* [rows/2][width/2] Cr, same rows */
    int64_t out_chroma_pitch_bytes;
} pysp_develop_args;

int pysp_develop(const pysp_develop_args* args, void* stream);

/* Bytes of device scratch pysp_develop needs for a band of `rows` output rows (0 when stages <= 0). */
int64_t pysp_develop_scratch_bytes(int32_t width, int32_t rows, int32_t stages);

/* Rows of mosaic needed above/below a band: 6 + 4*stages (SURVEY.md section 8a, stencil reach). */
int32_t pysp_develop_halo_rows(int32_t stages);

/* cv2.cvtColor(COLOR_RGB2LAB) float32 table (debayer/ahd.py:58,62): pack int16 [33][33][33][3] (L,a,b)
 * into the device layout (pysp_lab_lut_bytes() bytes); the caller uploads the result. */
int64_t pysp_lab_lut_bytes(void);
int pysp_lab_lut_pack_host(const int16_t* lut33_host, void* packed_host);

/* bayer_normalize (normalization.py:4-25): u16 [H][W] -> float32 [H][W]; black/white in [TL,TR,BR,BL]. */
int pysp_normalize_u16(const uint16_t* in, int64_t in_pitch_bytes, float* out, int64_t out_pitch_bytes,
                       int32_t height, int32_t width, const float black[4], const float white[4],
                       void* stream);

/* cam_to_rgb_norm / cam_to_lin_srgb (colorize/transform.py:21-53,76-87): n_pixels RGB float32 ->
 * float32 (or half when out_f16); `m` row-major float64; clip = clip_highlights. */
int pysp_cam_to_lin_srgb(const float* in, void* out, int64_t n_pixels, const double m[9], int32_t clip,
                         int32_t apply_gamma, int32_t out_f16, void* stream);

/* RawDemosaicData.wb_apply / wb_undo (base_types/image_base.py:45-60) and clip_rgb (colorize/transform.py:6-19) on
 * n_pixels RGB float32.  mode 0 (PYSP_WB_APPLY): x * wb[c].  mode 1 (PYSP_WB_UNDO): float32(float64(x) / wb[c]), after
 * x * max_wb when `normalized`.  mode 2 (PYSP_CLIP01): clip to [0,1].  `out` may alias `in`.
 * The reference multiplies with whatever dtype its coefficient object has (NumPy promotion): wb_is_f64 = 0 means float32
 * coefficients (products in float32, the EXIF path), 1 means float64 coefficients or a Python list (product / quotient in
 * float64, rounded to float32 once); max_is_f64 = 1 when max(wb) is a NumPy float64 scalar (the image is then promoted
 * to float64 before the division), 0 when it is a float32 or a Python float (product rounded to float32 first). */
#define PYSP_WB_APPLY 0
#define PYSP_WB_UNDO 1
#define PYSP_CLIP01 2
int pysp_wb_scale(const float* in, float* out, int64_t n_pixels, const double wb[3], double max_wb, int32_t mode,
                  int32_t normalized, int32_t wb_is_f64, int32_t max_is_f64, void* stream);

/* cv2.cvtColor(float32 RGB -> Lab) as the homogeneity metric uses it (debayer/ahd.py:58,62), stand-alone for stage tests:
 * n_pixels RGB float32 -> Lab float32.  `lab_lut` is the packed device table (pysp_lab_lut_pack_host). */
int pysp_rgb_to_lab_cv2(const float* in, float* out, int64_t n_pixels, const void* lab_lut, void* stream);

/* lin_srgb_to_srgb (colorize/transform.py:89-99) on n float32 values. */
int pysp_lin_srgb_to_srgb(const float* in, float* out, int64_t n_values, void* stream);

/* fuse_exposures_to_raw (raw_hdr.py:85-158), arithmetic lines 108-148: n float32 RGGB mosaics ->
 * HDR mosaic (+ optional int32 contribution count).  ev_offset[i] = float32(2**(ev_i - target_ev));
 * bias[i*3+c] = 1.6**(-0.1*|ev_offset[i]*wb[c]|) evaluated by the host in float32 (it has three distinct
 * values per bracket, so the device needs no pow).  Brackets are accumulated strictly in list order. */
int pysp_fuse_exposures(const float* const* brackets, int32_t n, int64_t in_pitch_bytes, int32_t height,
                        int32_t width, const float* ev_offset, const float* bias, int32_t brightest,
                        float* out, int64_t out_pitch_bytes, int32_t* count, int64_t count_pitch_bytes,
                        void* stream);

/* ---- steps either side of the develop path (SURVEY.md section 8f) ------------------------------------------------ */

/* Bytes of device workspace pysp_flat_frame_correction / pysp_bayer_plane_means need for an H x W mosaic. */
int64_t pysp_flat_workspace_bytes(int32_t height, int32_t width);

/* np.mean of the four CFA planes R, G1, B, G2 of a float32 mosaic (raw_correction.py:45), bit-identical to NumPy:
 * the float32 pairwise summation tree of NumPy is evaluated in its own order on the device.  means: 4 floats (device). */
int pysp_bayer_plane_means(const float* mosaic, int64_t pitch_bytes, int32_t height, int32_t width, float* means,
                           void* workspace, int64_t workspace_bytes, void* stream);

/* flat_frame_correction (raw_correction.py:25-63): per CFA plane out = (sensor * mean(flat)) / flat; +inf -> largest
 * finite quotient of the plane, negative -> 0, optional clamp at 1; a plane whose quotients are all infinite is
 * copied unchanged.  `out` may alias `sensor`. */
int pysp_flat_frame_correction(const float* sensor, int64_t sensor_pitch_bytes, const float* flat, int64_t flat_pitch_bytes,
                               float* out, int64_t out_pitch_bytes, int32_t height, int32_t width, int32_t clamp_high,
                               void* workspace, int64_t workspace_bytes, void* stream);

/* find_erroneous_pixels_threshold (raw_bad_pixel_corr.py:30-65): masks[4][H/2][W/2] bytes (planes R, G1, B, G2), 1 where
 * (value - min_delta) exceeds more than min_neighbour_count of the eight same-colour neighbours (reflected border). */
int pysp_find_hot_pixels_threshold(const float* sensor, int64_t pitch_bytes, int32_t height, int32_t width, float min_delta,
                                   int32_t min_neighbour_count, uint8_t* masks, void* stream);

/* fuse_exposures_from_debayer (raw_hdr.py:7-83): n demosaiced exposures (float32 [n_pixels][3], white balance applied)
 * -> linear sRGB float32 (+ optional int32 [n_pixels][3] contribution count).  Per exposure, in list order: wb_undo
 * (float64 division, base_types/image_base.py:52-60), saturation weight x bias[i], wb_apply, accumulation x
 * ev_offset[i]; where the weights sum to zero the brightest exposure x offset_max (float64) is used; then the camera
 * -> linear-sRGB matrix without clipping.  ev_offset[i] = float32(2**(ev_i - target)), bias[i] =
 * float32(1.6**(-0.1 * 2**(ev_i - target))), brightest = last i whose offset equals offset_max.  With write_back the
 * exposures are left as the reference leaves them (after its wb_undo/wb_apply round trip). */
int pysp_fuse_exposures_from_debayer(float* const* images, int32_t n, int64_t n_pixels, const float wb[3], float max_wb,
                                     const int32_t* wb_normalized, const float* ev_offset, const float* bias,
                                     int32_t brightest, double offset_max, const double m[9], float* out, int32_t* count,
                                     int32_t write_back, void* stream);

/* ---- post-demosaic lens correction: DNG WarpRectilinear (SURVEY.md section 8f-4) -------------------------------------- */

/* compute_remapping_table (dng_warp_corr/dng_warp_rectilinear_coords.pyx:67-80) and, with `seed`,
 * compute_offset_remapping_table (pyx:82-95): table[H][W][2] float32 = the source position (x', y') of every pixel under
 * the radial (kr0..kr3) + tangential (kt0, kt1) model, k = {kr0, kr1, kr2, kr3, kt0, kt1}; cam_center_norm in [0,1];
 * seed = prior mapping [H][W][2] or NULL for the pixel grid.  Within 2 ulp of the reference (it calls libm's powf). */
int pysp_warp_rectilinear_table(float* table, int64_t table_pitch_bytes, int32_t height, int32_t width, const float k[6],
                                float cam_center_norm_x, float cam_center_norm_y, float scale, const float* seed,
                                int64_t seed_pitch_bytes, void* stream);

/* cv2.remap(plane, clip(map_x, 0, W-1), clip(map_y, 0, H-1), cv2.INTER_LANCZOS4) as apply_opcode_3_warp calls it
 * (dng_warp_corr/chan_distortion_corr.py:94-97) on one plane of an interleaved float32 image: element (y, x) of the plane
 * is src[y * pitch/4 + x * step].  map = [H][W][2] float32 (x', y'), e.g. from pysp_warp_rectilinear_table.
 * lanczos_tab: device copy of OpenCV's float32 [32][8] Lanczos-4 table (pysp_b200/data/lanczos4_tab_f32.npy).
 * dst must not overlap src. */
int pysp_remap_lanczos4(const float* src, int64_t src_pitch_bytes, int32_t src_step, float* dst, int64_t dst_pitch_bytes,
                        int32_t dst_step, int32_t height, int32_t width, const float* map, int64_t map_pitch_bytes,
                        const float* lanczos_tab, void* stream);

/* opcode_warp_rectilinear (dng_warp_corr/chan_distortion_corr.py:53-98) for all planes of a contiguous interleaved image
 * [H][W][planes] in one kernel: coordinates are computed in registers, no table goes through HBM.  coeffs[planes][6];
 * prior = optional [H][W][planes][2] (stack_warp_prior, chan_distortion_corr.py:10-41).  dst must not overlap src (the
 * reference writes each plane back in place after remapping it; the caller copies dst over src for that). */
int pysp_warp_rectilinear_apply(const float* src, float* dst, int32_t height, int32_t width, int32_t planes, const float* coeffs,
                                float cam_center_norm_x, float cam_center_norm_y, float scale, const float* prior,
                                const float* lanczos_tab, void* stream);

/* ---- baseline JPEG of the PYSP_OUT_YCC420_U8 planes --------------------------------------------------------------------
 *
 * pysp_jpeg_encode_ycc420 writes one complete JFIF file byte-identical to libjpeg(-turbo)'s encode of the same planes with
 * its defaults, i.e. Pillow's
 *     Image.merge("YCbCr", [Y, upsample2x2(Cb), upsample2x2(Cr)]).save(f, "JPEG", quality=quality, subsampling=2)
 * When W is a multiple of 16 and the planes are PYSP_OUT_YCC420_U8 of a develop, that is also byte-identical to the JPEG
 * libjpeg writes from the PYSP_OUT_SRGB_U8 image of the same call (for other widths libjpeg pads the chroma's right edge from
 * full-resolution chroma, which the planes do not hold; pysp_jpeg_encode_rgb below encodes the RGB image at any size).  What
 * it does, all in integers (tests/jpeg_ref.py restates it):
 *  - markers SOI, APP0 (JFIF 1.01, density 1:1, no units), DQT luma, DQT chroma (8-bit, zigzag order), SOF0, DHT DC0, AC0,
 *    DC1, AC1 (the standard tables of Annex K.3), SOS, the entropy-coded data, EOI; MCU = Y00 Y01 Y10 Y11 Cb Cr, no restarts;
 *  - quantisation tables: scale = quality < 50 ? 5000/quality : 200 - 2*quality, clamp((std*scale + 50)/100, 1, 255) on
 *    the Annex K.1 tables;
 *  - jfdctint.c ISLOW forward DCT of x - 128; coefficient c is quantised as sign(c) * ((|c| + d/2) / d), d = 8*qtab[k];
 *  - each plane is padded to whole 8x8 blocks by repeating its last column and row; a Y slot of an MCU outside the Y blocks
 *    is a dummy block: AC zero, DC = the DC of the block before it in the MCU;
 *  - DC prediction per component across the scan, ZRL for runs of 16 zeros, EOB for trailing zeros, the last byte padded
 *    with 1-bits, 0x00 after every 0xFF of the entropy-coded data.
 * y: [height][width] (pitch y_pitch >= width), cb / cr: [height/2][width/2] (one pitch chroma_pitch >= width/2); height and
 * width even, 2..65535; quality 1..100.  out: >= pysp_jpeg_max_bytes(height, width) bytes (out_capacity); *out_len (a DEVICE
 * int64) receives the file's length, and no byte of `out` past it is written.  workspace: >= pysp_jpeg_workspace_bytes.
 * Every argument is checked before any CUDA call (PYSP_ERR_INVALID).  The header and the quantisation tables are written by a
 * kernel and the Huffman tables live in constant memory: a call makes no host <-> device copy and can be captured in a CUDA
 * graph. */
/* The worst case of the file.  A block codes its DC difference (category <= 11: a code of at most 11 bits plus 11 magnitude
 * bits) and its 63 AC coefficients; each AC symbol (a code of at most 16 bits plus at most 10 magnitude bits) accounts for at
 * least one coefficient, and so do ZRL (16 coefficients) and EOB (at least one), so a block takes at most
 * 11 + 11 + 63 * (16 + 10) = 1660 bits.  With 6 blocks per MCU the entropy-coded data is at most ceil(6 * MCUs * 1660 / 8)
 * bytes (the padding completes the last byte); stuffing at most doubles it.  Plus the 623-byte header and the 2-byte EOI.
 * 0 for an invalid size. */
int64_t pysp_jpeg_max_bytes(int32_t height, int32_t width);
/* Bytes of device workspace pysp_jpeg_encode_ycc420 needs (0 for an invalid size). */
int64_t pysp_jpeg_workspace_bytes(int32_t height, int32_t width);
int pysp_jpeg_encode_ycc420(const uint8_t* y, int64_t y_pitch, const uint8_t* cb, const uint8_t* cr, int64_t chroma_pitch,
                            int32_t height, int32_t width, int32_t quality, uint8_t* out, int64_t out_capacity,
                            int64_t* out_len, void* workspace, int64_t workspace_bytes, void* stream);

/* ---- baseline JPEG of an 8-bit RGB image at 4:4:4, 4:2:2 or 4:2:0 ------------------------------------------------------
 *
 * pysp_jpeg_encode_rgb writes one complete JFIF file byte-identical to libjpeg(-turbo)'s encode of the image with its
 * defaults, i.e. Pillow's
 *     Image.fromarray(S, "RGB").save(f, "JPEG", quality=quality, subsampling=subsampling)
 * for any height and width.  `subsampling` takes Pillow's integers: */
#define PYSP_JPEG_444 0    /* Y sampled 1x1: an MCU is Y Cb Cr */
#define PYSP_JPEG_422 1    /* Y 2x1: Y0 Y1 Cb Cr */
#define PYSP_JPEG_420 2    /* Y 2x2: Y00 Y01 Y10 Y11 Cb Cr */
/* With (h, v) the Y sampling factors, MCUs mx = ceil(W / 8h) across and my = ceil(H / 8v) down, all in integers
 * (tests/jpeg_rgb_ref.py restates it):
 *  - colour: Y, cb, cr of every pixel as PYSP_OUT_YCC420_U8 states it (jccolor.c rgb_ycc_convert);
 *  - chroma (jcsample.c): cb / cr with the last column repeated out to 8h * mx columns and the last row out to a multiple of v
 *    rows, then downsampled: 4:4:4 a copy, 4:2:2 (a + b + bias) >> 1 with bias 0, 1, 0, 1, ... along the row, 4:2:0 the
 *    2x2 average of PYSP_OUT_YCC420_U8 (bias 1, 2, 1, 2, ...); the last downsampled row is repeated out to 8 * my rows.
 *    Repeating after the downsample instead is not the same: that is why planes developed at 4:2:0 give libjpeg's file of the
 *    RGB image only when W % 16 == 0, and why this entry point takes the RGB image;
 *  - Y: padded to whole blocks by repeating its last column and row; an MCU holds h x v Y slots in raster order, then Cb, Cr;
 *    a Y slot outside the Y blocks is a dummy (AC zero, DC = the DC of the slot before it);
 *  - header: that of pysp_jpeg_encode_ycc420 with the Y sampling byte of SOF0 set to (h << 4) | v; the rest (tables, DCT,
 *    quantisation, Huffman coding, padding, stuffing) is the same.
 * rgb: [height][width][3] R, G, B bytes, row pitch pitch_bytes >= 3 * width, any alignment; height and width 1..65535;
 * quality 1..100.  out: >= pysp_jpeg_rgb_max_bytes(height, width, subsampling) bytes (out_capacity); *out_len (a DEVICE
 * int64) receives the file's length, and no byte of `out` past it is written.  workspace: >=
 * pysp_jpeg_rgb_workspace_bytes(...) bytes (the converted planes live there).  As for pysp_jpeg_encode_ycc420: every argument
 * is checked before any CUDA call, nothing is allocated, no host <-> device copy, no synchronise, capturable in a CUDA graph. */
/* The worst case of the file: pysp_jpeg_max_bytes's derivation with h * v + 2 blocks of at most 1660 bits per MCU:
 * 623 + 2 * ceil((h * v + 2) * mx * my * 1660 / 8) + 2 bytes.  0 for an invalid size or subsampling. */
int64_t pysp_jpeg_rgb_max_bytes(int32_t height, int32_t width, int32_t subsampling);
/* Bytes of device workspace pysp_jpeg_encode_rgb needs (0 for an invalid size or subsampling). */
int64_t pysp_jpeg_rgb_workspace_bytes(int32_t height, int32_t width, int32_t subsampling);
int pysp_jpeg_encode_rgb(const uint8_t* rgb, int64_t pitch_bytes, int32_t height, int32_t width, int32_t quality,
                         int32_t subsampling, uint8_t* out, int64_t out_capacity, int64_t* out_len, void* workspace,
                         int64_t workspace_bytes, void* stream);

/* Bench instrumentation (no reference counterpart): when enabled, pysp_develop brackets each kernel launch
 * with CUDA events on the launching stream; collect() synchronises them and returns, per kernel slot
 * (0 = ahd_select_kernel, 1 = median_stage_kernel; 4 slots), the summed device milliseconds and launch
 * count since the last enable/collect. */
void pysp_timing_enable(int32_t on);
int pysp_timing_collect(double total_ms[4], int64_t launches[4]);

/* Developer hook: SM clocks per kernel phase, summed over CTAs since the last call ([kernel 0..1][phase 0..15]);
 * all zeros unless the library was built with -DPYSP_PHASE_CLOCKS (tools/kbench.py --phases). */
int pysp_debug_phase_clocks(uint64_t out[32]);

const char* pysp_last_error(void);
const char* pysp_version(void);
/* Number of kernels this library has launched in this process (for bench accounting). */
int64_t pysp_kernel_launches(void);

#ifdef __cplusplus
}
#endif
#endif
