// libpysp_b200.so: kernels + C ABI (include/pysp_b200.h).  sm_100a only, no CPU path.
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <map>
#include <mutex>
#include <vector>

#include "../../include/pysp_b200.h"
#include "ahd_select.cuh"
#include "eag.cuh"
#include "median_stage.cuh"
#include "pointwise.cuh"
#include "prepost.cuh"
#include "warp.cuh"
#include "jpeg.cuh"
#include "develop_plan.h"

namespace pysp {

// tile sizes (compile-time; the -D overrides exist for tools/kbench.py A/B builds)
#ifndef PYSP_K1_TW
#define PYSP_K1_TW 60
#endif
#ifndef PYSP_K1_TH
#define PYSP_K1_TH 60
#endif
#ifndef PYSP_K2_TW
#define PYSP_K2_TW 60
#endif
#ifndef PYSP_K2_TH
#define PYSP_K2_TH 60
#endif
#ifndef PYSP_K1_THREADS
#define PYSP_K1_THREADS 512
#endif
constexpr int K1_TW = PYSP_K1_TW, K1_TH = PYSP_K1_TH, K1_THREADS = PYSP_K1_THREADS;
// QualityDemosaic.Fast runs the same pipeline with its own tile: it needs no Lab / candidate planes (98 KB of shared memory on
// 60x44 tiles instead of 208 KB on 60x60), so two 256-thread CTAs fit on an SM.  Measured on a 12 MP frame: 0.1075 ms, against
// 0.126 ms in the AHD configuration (one 512-thread CTA, 60x60) and 0.124 ms on 60x28 tiles with two CTAs (0.1075 with three).
#ifndef PYSP_EAG_TH
#define PYSP_EAG_TH 44
#endif
#ifndef PYSP_EAG_THREADS
#define PYSP_EAG_THREADS 256
#endif
#ifndef PYSP_EAG_CTAS
#define PYSP_EAG_CTAS 2
#endif
constexpr int EAG_TW = PYSP_K1_TW, EAG_TH = PYSP_EAG_TH, EAG_THREADS = PYSP_EAG_THREADS;
#ifndef PYSP_K2_THREADS
#define PYSP_K2_THREADS 512
#endif
#ifndef PYSP_K2_CTAS
#define PYSP_K2_CTAS 1
#endif
constexpr int K2_TW = PYSP_K2_TW, K2_TH = PYSP_K2_TH, K2_THREADS = PYSP_K2_THREADS;
// work item of the median phases: a 2x4 block of outputs (60.75 min/max per median) or a 2x2 block (67.5)
#ifndef PYSP_K2_BLOCK4
#define PYSP_K2_BLOCK4 1
#endif
#if PYSP_K2_BLOCK4
#define PYSP_K2_PHASE_B median_phase_b4
#define PYSP_K2_PHASE_C median_phase_c4
#else
#define PYSP_K2_PHASE_B median_phase_b
#define PYSP_K2_PHASE_C median_phase_c
#endif

struct OutMaps { CUtensorMap m[3]; };     // final image: m[0]; planes: m[0..2]

// stage-out: TMA store of the finished staging tile (one elected thread), or the generic clipped store
template <int TW, int TH>
__device__ __forceinline__ void store_tile(const float* out, const StoreParams& st, const FrameGeom& g, const OutMaps& maps,
                                           int x0, int y0) {
    int bx, by;
    tile_output_box<TW, TH>(st, g, x0, y0, &bx, &by);
    // A TMA store clips a box that overshoots the tensor on the high side, but a negative origin is illegal
    // (measured on B200, tools/probe/tma_store_probe.cu): partial tiles of flipped frames take the generic store.
    if (st.tma && bx >= 0 && by >= 0) {
        if (threadIdx.x == 0) {
            if (st.mode == OUT_FINAL) {
                tma_store_2d(out, &maps.m[0], bx, by);
            } else {
#pragma unroll
                for (int k = 0; k < 3; ++k) tma_store_2d(out + k * OutPlane<TW, TH>::FLOATS, &maps.m[k], bx, by);
            }
            tma_store_commit();
        }
    } else {
        store_tile_generic<TW, TH>(out, st, g, x0, y0);
    }
}

// K1, persistent: grid = resident CTAs (one 512-thread CTA per SM on 60x60 tiles: measured 4.6 % faster than two 256-thread
// CTAs on 60x28 tiles -- the Lab region shrinks from 1.22x to 1.14x the tile, the raw box from 1.9x to 1.6x); each CTA
// walks tiles blockIdx.x, +gridDim.x, ...  The raw box of the next
// tile is in flight (TMA -> staging, mbarrier) while phases 1-4 of the current tile run; the finished tile leaves
// through the staging tile by TMA store, overlapped with the next tile's phases 0-3.
// ALGO_EAG (QualityDemosaic.Fast) runs its own phases 1-2 (eag.cuh) in the same pipeline.
#ifndef PYSP_K1_CTAS
#define PYSP_K1_CTAS 1
#endif
template <int ALGO, int TW, int TH, int THREADS, int CTAS>
__global__ void __launch_bounds__(THREADS, CTAS)
ahd_select_kernel(const __grid_constant__ SelectParams p, const __grid_constant__ CUtensorMap in_map,
                  const __grid_constant__ OutMaps out_maps) {
    typedef SelectTile<TW, TH> L;
    extern __shared__ __align__(128) char smem[];
    uint64_t* bar = (uint64_t*)(smem + L::OFF_BAR);
    void* stage = smem + L::OFF_STAGE;
    const uint32_t box_bytes = L::BOXW * L::BOXH * (p.in_kind == IN_U16 ? 2 : 4);
    int tile = blockIdx.x;
    uint32_t parity = 0;
    if (threadIdx.x == 0) mbar_init(bar, 1);
    __syncthreads();
    auto fetch = [&](int t) {       // start (TMA) or perform (generic) the load of tile t's raw box
        const int ty = t / p.tiles_x, tx = t - ty * p.tiles_x;
        int bx, by;
        select_input_box<TW, TH>(p, tx, ty, &bx, &by);
        if (p.tma_in) {
            if (threadIdx.x == 0) {
                fence_async_smem();
                mbar_expect_tx(bar, box_bytes);
                tma_load_2d(stage, &in_map, bx, by, bar);
            }
        } else {
            box_load_generic(stage, p.in, bx, by, L::BOXW, L::BOXH);
        }
    };
    if (tile < p.n_tiles) fetch(tile);
    if (!p.tma_in) __syncthreads();
    PYSP_PHASE_BEGIN();
    for (; tile < p.n_tiles; tile += gridDim.x) {
        const int tile_y = tile / p.tiles_x, tile_x = tile - tile_y * p.tiles_x;
        const bool edge = select_tile_is_edge<TW, TH>(p, tile_x, tile_y);
        if (p.tma_in) { mbar_wait(bar, parity); parity ^= 1; }
        PYSP_PHASE_MARK(0, 0);                            // wait for the raw box
        if (edge) select_phase0<TW, TH, true>(p, smem, tile_x, tile_y);
        else select_phase0<TW, TH, false>(p, smem, tile_x, tile_y);
        __syncthreads();                                  // staging consumed, quarter planes complete
        PYSP_PHASE_MARK(0, 1);
        const int next = tile + gridDim.x;
        if (p.tma_in && next < p.n_tiles) fetch(next);
        auto before_out = [&]() { if (p.st.tma && threadIdx.x == 0) tma_store_wait_read(); };
        if (ALGO == ALGO_EAG) {
            before_out();
            __syncthreads();
            if (edge) eag_phases<TW, TH, true>(p, smem, tile_x, tile_y);
            else eag_phases<TW, TH, false>(p, smem, tile_x, tile_y);
        } else {
            if (edge) select_phases<TW, TH, true>(p, smem, tile_x, tile_y, before_out);
            else select_phases<TW, TH, false>(p, smem, tile_x, tile_y, before_out);
        }
        if (p.st.tma) fence_async_smem();                 // staging tile written by the generic proxy, read by TMA
        __syncthreads();
        PYSP_PHASE_MARK(0, 6);
        store_tile<TW, TH>((const float*)(smem + L::OFF_OUT), p.st, p.g, out_maps, tile_x * TW,
                                 p.y_begin + tile_y * TH);
        if (!p.tma_in) {                                  // generic load of the next box by the whole CTA: phase 0 reads it
            if (next < p.n_tiles) fetch(next);
            __syncthreads();
        }
        // (with TMA loads no barrier is needed here: phase 0 of the next tile only writes the native planes, which every
        // thread has finished reading before the barrier above, and the staging tile is next written two barriers later)
        PYSP_PHASE_MARK(0, 7);
    }
    if (p.st.tma && threadIdx.x == 0) tma_store_wait_read();
}

// K2, persistent, same pipeline: the three input planes of the next tile are fetched by TMA while phase C runs.
// One 512-thread CTA per SM on 60x60 tiles (measured 6 % faster than two 256-thread CTAs on 60x28 tiles: the tile + 2 px
// region of the first median pair shrinks from 1.22x to 1.14x the tile, and K2 is bound by the min/max pipe, not latency).
__global__ void __launch_bounds__(K2_THREADS, PYSP_K2_CTAS)
median_stage_kernel(const __grid_constant__ MedianParams p, const __grid_constant__ OutMaps in_maps,
                    const __grid_constant__ OutMaps out_maps) {
    typedef MedianTile<K2_TW, K2_TH> L;
    extern __shared__ __align__(128) char smem[];
    uint64_t* bar = (uint64_t*)(smem + L::OFF_BAR);
    int tile = blockIdx.x;
    uint32_t parity = 0;
    if (threadIdx.x == 0) mbar_init(bar, 1);
    __syncthreads();
    auto fetch = [&](int t) {
        const int ty = t / p.tiles_x, tx = t - ty * p.tiles_x;
        const int bx = tx * K2_TW - 4, by = p.y_begin + ty * K2_TH - 4 - p.in_row0;
        if (p.tma_in) {
            if (threadIdx.x == 0) {
                fence_async_smem();
                mbar_expect_tx(bar, 3 * L::AW * L::AH * 4);
#pragma unroll
                for (int k = 0; k < 3; ++k) tma_load_2d(smem + L::OFF_IN + k * L::PLANE_BYTES, &in_maps.m[k], bx, by, bar);
            }
        } else {
            for (int k = 0; k < 3; ++k) box_load_generic(smem + L::OFF_IN + k * L::PLANE_BYTES, p.in[k], bx, by, L::AW, L::AH);
        }
    };
    if (tile < p.n_tiles) fetch(tile);
    if (!p.tma_in) __syncthreads();
    for (; tile < p.n_tiles; tile += gridDim.x) {
        const int tile_y = tile / p.tiles_x, tile_x = tile - tile_y * p.tiles_x;
        const bool edge = median_tile_is_edge<K2_TW, K2_TH>(p, tile_x, tile_y);
        if (p.tma_in) { mbar_wait(bar, parity); parity ^= 1; }
        if (edge) {
            median_fix_border<K2_TW, K2_TH>(p, smem, tile_x, tile_y);
            __syncthreads();
            PYSP_K2_PHASE_B<K2_TW, K2_TH, true>(p, smem, tile_x, tile_y);
        } else {
            PYSP_K2_PHASE_B<K2_TW, K2_TH, false>(p, smem, tile_x, tile_y);
        }
        if (p.st.tma && threadIdx.x == 0) tma_store_wait_read();     // previous tile's store has read the staging tile
        __syncthreads();                                             // input planes consumed
        const int next = tile + gridDim.x;
        if (p.tma_in && next < p.n_tiles) fetch(next);
        if (edge) PYSP_K2_PHASE_C<K2_TW, K2_TH, true>(p, smem, tile_x, tile_y);
        else PYSP_K2_PHASE_C<K2_TW, K2_TH, false>(p, smem, tile_x, tile_y);
        if (p.st.tma) fence_async_smem();
        __syncthreads();
        store_tile<K2_TW, K2_TH>((const float*)(smem + L::OFF_OUT), p.st, p.g, out_maps, tile_x * K2_TW,
                                 p.y_begin + tile_y * K2_TH);
        if (!p.tma_in && next < p.n_tiles) fetch(next);
        __syncthreads();
    }
    if (p.st.tma && threadIdx.x == 0) tma_store_wait_read();
}

}  // namespace pysp

using namespace pysp;

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

static int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

static int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(PYSP_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
    g_launches.fetch_add(1);
    return PYSP_OK;
}

// ---- optional per-kernel timing (bench only): CUDA events recorded on the launching stream ---------------
#define PYSP_TIMING_SLOTS 4
struct TimedEvents { cudaEvent_t a, b; int slot; };
static std::mutex g_tmutex;
static bool g_timing = false;
static std::vector<TimedEvents> g_tev;      // one pair per launch since the last enable/collect; grows as needed
static std::atomic<long long> g_tfail{0};   // launches whose events could not be created (reported by collect)

struct TimedLaunch {     // records an event pair around one launch when timing is enabled
    cudaStream_t s; cudaEvent_t b; bool on;
    TimedLaunch(int slot, cudaStream_t stream) : s(stream), b(nullptr), on(false) {
        if (!g_timing) return;
        TimedEvents e;
        e.slot = slot;
        if (cudaEventCreate(&e.a) != cudaSuccess) { g_tfail.fetch_add(1); return; }
        if (cudaEventCreate(&e.b) != cudaSuccess) { cudaEventDestroy(e.a); g_tfail.fetch_add(1); return; }
        cudaEventRecord(e.a, s);
        b = e.b; on = true;
        std::lock_guard<std::mutex> lk(g_tmutex);
        g_tev.push_back(e);
    }
    ~TimedLaunch() { if (on) cudaEventRecord(b, s); }
};

static int ensure_device() {
    int dev = -1;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return fail(PYSP_ERR_CUDA, "no CUDA device: %s (pysp_b200 has no CPU path)", cudaGetErrorString(e));
    return PYSP_OK;
}

static int grid_for(long long n, int threads) {
    long long b = (n + threads - 1) / threads;
    const long long cap = 148LL * 16;          // a few waves of the 148 SMs; kernels grid-stride
    return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}

extern "C" {

const char* pysp_last_error(void) { return g_err; }
const char* pysp_version(void) { return "pysp_b200 0.1 (sm_100a)"; }
int64_t pysp_kernel_launches(void) { return g_launches.load(); }

void pysp_timing_enable(int32_t on) {
    std::lock_guard<std::mutex> lk(g_tmutex);
    for (auto& e : g_tev) { cudaEventDestroy(e.a); cudaEventDestroy(e.b); }
    g_tev.clear();
    g_tfail.store(0);
    g_timing = on != 0;
}

int pysp_timing_collect(double* total_ms, int64_t* launches) {
    std::lock_guard<std::mutex> lk(g_tmutex);
    for (int k = 0; k < PYSP_TIMING_SLOTS; ++k) { total_ms[k] = 0.0; launches[k] = 0; }
    int rc = PYSP_OK;
    for (auto& ev : g_tev) {
        cudaError_t e = cudaEventSynchronize(ev.b);
        float ms = 0.f;
        if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, ev.a, ev.b);
        if (e != cudaSuccess) rc = fail(PYSP_ERR_CUDA, "pysp_timing_collect: %s", cudaGetErrorString(e));
        else { total_ms[ev.slot] += ms; launches[ev.slot] += 1; }
        cudaEventDestroy(ev.a); cudaEventDestroy(ev.b);
    }
    g_tev.clear();
    const long long lost = g_tfail.exchange(0);
    if (rc == PYSP_OK && lost) rc = fail(PYSP_ERR_CUDA, "pysp_timing_collect: %lld launches were not timed (event creation failed)", lost);
    return rc;
}

// developer hook: per-phase SM clocks summed over CTAs (zeros unless built with -DPYSP_PHASE_CLOCKS); resets them
int pysp_debug_phase_clocks(uint64_t out[32]) {
    memset(out, 0, 32 * sizeof(uint64_t));
#ifdef PYSP_PHASE_CLOCKS
    unsigned long long z[32] = {0};
    if (cudaMemcpyFromSymbol(out, g_phase_clk, sizeof(z)) != cudaSuccess) return fail(PYSP_ERR_CUDA, "phase clocks");
    if (cudaMemcpyToSymbol(g_phase_clk, z, sizeof(z)) != cudaSuccess) return fail(PYSP_ERR_CUDA, "phase clocks");
#endif
    return PYSP_OK;
}

int32_t pysp_develop_halo_rows(int32_t stages) { return 6 + 4 * (stages > 0 ? stages : 0); }

int64_t pysp_develop_scratch_bytes(int32_t width, int32_t rows, int32_t stages) {
    return develop_scratch_bytes(width, rows, stages);
}

int64_t pysp_lab_lut_bytes(void) { return (int64_t)PYSP_LUT_NR * PYSP_LUT_NG * PYSP_LUT_NB * 16; }

int pysp_lab_lut_pack_host(const int16_t* lut, void* packed) {
    if (!lut || !packed) return fail(PYSP_ERR_INVALID, "pysp_lab_lut_pack_host: null pointer");
    uint32_t* o = (uint32_t*)packed;
    auto at = [&](int r, int g, int b, int ch) -> uint32_t {
        r = r > 32 ? 32 : r; g = g > 32 ? 32 : g; b = b > 32 ? 32 : b;
        return (uint16_t)lut[((r * 33 + g) * 33 + b) * 3 + ch];
    };
    for (int r = 0; r < PYSP_LUT_NR; ++r)
        for (int g = 0; g < PYSP_LUT_NG; ++g)
            for (int b = 0; b < PYSP_LUT_NB; ++b) {
                uint32_t* e = o + (((size_t)r * PYSP_LUT_NG + g) * PYSP_LUT_NB + b) * 4;
                for (int ch = 0; ch < 3; ++ch) e[ch] = at(r, g, b, ch) | (at(r, g, b + 1, ch) << 16);
                e[3] = 0;
            }
    return PYSP_OK;
}

// ---- tensor maps (driver entry point fetched through the runtime: no link-time dependency on libcuda) ----------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled_fn() {
    static std::atomic<EncodeTiledFn> cached{nullptr};
    EncodeTiledFn f = cached.load();
    if (f) return f;
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q) != cudaSuccess || !sym) return nullptr;
    cached.store((EncodeTiledFn)sym);
    return (EncodeTiledFn)sym;
}

static int make_map(CUtensorMap* m, const View2D& v, int box_w, int box_h) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) return fail(PYSP_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
    cuuint64_t dims[2] = {(cuuint64_t)v.cols, (cuuint64_t)v.rows};
    cuuint64_t strides[1] = {(cuuint64_t)v.pitch};
    cuuint32_t box[2] = {(cuuint32_t)box_w, (cuuint32_t)box_h};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(m, v.elem == 2 ? CU_TENSOR_MAP_DATA_TYPE_UINT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, v.base, dims, strides,
                     box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(PYSP_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) for a %dx%d view, pitch %lld", (int)r,
                                       v.rows, v.cols, v.pitch);
    return PYSP_OK;
}

static int make_out_maps(OutMaps* om, const StoreParams& st, int tw, int th) {
    memset(om, 0, sizeof(*om));
    if (!st.tma) return PYSP_OK;
    if (st.mode == OUT_FINAL) return make_map(&om->m[0], st.img, 3 * tw, th);
    for (int k = 0; k < 3; ++k) {
        int rc = make_map(&om->m[k], st.plane[k], tw, th);
        if (rc) return rc;
    }
    return PYSP_OK;
}

static int resident_ctas(const void* kernel, int threads, int smem_bytes, int* out) {
    int dev = 0, sms = 0, per_sm = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem_bytes);
    if (e != cudaSuccess) return fail(PYSP_ERR_CUDA, "occupancy query: %s", cudaGetErrorString(e));
    if (per_sm < 1) return fail(PYSP_ERR_CUDA, "kernel does not fit on an SM");
#ifdef PYSP_GRID_PER_SM            // A/B builds (tools/overlap_bench.py): fewer CTAs per SM than would fit, to leave room for another kernel
    if (per_sm > PYSP_GRID_PER_SM) per_sm = PYSP_GRID_PER_SM;
#endif
    *out = sms * per_sm;
    return PYSP_OK;
}

// Per-device launch set-up of the develop chain (shared-memory opt-in, persistent grid sizes), done once per device
struct ChainSetup { int grid_ahd, grid_eag, grid_median; };
#define PYSP_AHD_KERNEL ahd_select_kernel<ALGO_AHD, K1_TW, K1_TH, K1_THREADS, PYSP_K1_CTAS>
#define PYSP_EAG_KERNEL ahd_select_kernel<ALGO_EAG, EAG_TW, EAG_TH, EAG_THREADS, PYSP_EAG_CTAS>
constexpr int SMEM_AHD = SelectTile<K1_TW, K1_TH>::SMEM_BYTES, SMEM_EAG = SelectTile<EAG_TW, EAG_TH>::SMEM_BYTES_EAG;

static int chain_setup(const ChainSetup** out) {
    static std::mutex mu;
    static std::map<int, ChainSetup> cache;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return fail(PYSP_ERR_CUDA, "no current CUDA device");
    std::lock_guard<std::mutex> lk(mu);
    auto it = cache.find(dev);
    if (it == cache.end()) {
        const int smem2 = MedianTile<K2_TW, K2_TH>::SMEM_BYTES;
        cudaError_t e1 = cudaFuncSetAttribute(PYSP_AHD_KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_AHD);
        cudaError_t e2 = cudaFuncSetAttribute(median_stage_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem2);
        cudaError_t e3 = cudaFuncSetAttribute(PYSP_EAG_KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_EAG);
        if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess)
            return fail(PYSP_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e1 != cudaSuccess ? e1 : (e2 != cudaSuccess ? e2 : e3)));
        ChainSetup cs;
        int rc = resident_ctas((const void*)PYSP_AHD_KERNEL, K1_THREADS, SMEM_AHD, &cs.grid_ahd);
        if (!rc) rc = resident_ctas((const void*)PYSP_EAG_KERNEL, EAG_THREADS, SMEM_EAG, &cs.grid_eag);
        if (!rc) rc = resident_ctas((const void*)median_stage_kernel, K2_THREADS, smem2, &cs.grid_median);
        if (rc) return rc;
        it = cache.emplace(dev, cs).first;
    }
    *out = &it->second;
    return PYSP_OK;
}

// Test hook, read ONCE per process: PYSP_DISABLE_TMA bit 0 = loads, bit 1 = stores take the generic (non-TMA) path that
// unaligned tensors take anyway, bit 2 = IEEE division instead of the verified reciprocal form.  tests/test_gpu_parity.py
// sets it in a fresh process to prove those paths give the same bits.
static int debug_path_bits() {
    static const int bits = [] { const char* e = getenv("PYSP_DISABLE_TMA"); return e ? atoi(e) : 0; }();
    return bits;
}

int pysp_develop(const pysp_develop_args* a, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    DevelopPlan plan;
    const bool fast = a && a->quality == PYSP_QUALITY_FAST;           // QualityDemosaic.Fast has its own K1 tile
    int rc = plan_develop(a, fast ? EAG_TW : K1_TW, fast ? EAG_TH : K1_TH, K2_TW, K2_TH, &plan, g_err, sizeof(g_err));
    if (rc) return rc;
    rc = ensure_device();
    if (rc) return rc;
    if (const int bits = debug_path_bits()) {
        if (bits & 1) { plan.select.tma_in = 0; for (auto& mp : plan.median) mp.tma_in = 0; }
        if (bits & 2) { plan.select.st.tma = 0; for (auto& mp : plan.median) mp.st.tma = 0; }
        if (bits & 4) plan.select.fast_div = 0;
    }
    const int smem2 = MedianTile<K2_TW, K2_TH>::SMEM_BYTES;
    const ChainSetup* cs = nullptr;
    rc = chain_setup(&cs);
    if (rc) return rc;
    const bool eag = plan.select.algo == ALGO_EAG;
    const int grid1 = eag ? cs->grid_eag : cs->grid_ahd, grid2 = cs->grid_median;
    {
        CUtensorMap in_map;
        memset(&in_map, 0, sizeof(in_map));
        OutMaps om;
        if (plan.select.tma_in) {
            rc = eag ? make_map(&in_map, plan.select.in, SelectTile<EAG_TW, EAG_TH>::BOXW, SelectTile<EAG_TW, EAG_TH>::BOXH)
                     : make_map(&in_map, plan.select.in, SelectTile<K1_TW, K1_TH>::BOXW, SelectTile<K1_TW, K1_TH>::BOXH);
            if (rc) return rc;
        }
        rc = eag ? make_out_maps(&om, plan.select.st, EAG_TW, EAG_TH) : make_out_maps(&om, plan.select.st, K1_TW, K1_TH);
        if (rc) return rc;
        const int grid = plan.select.n_tiles < grid1 ? plan.select.n_tiles : grid1;
        {
            TimedLaunch t(eag ? 2 : 0, stream);
            if (eag) PYSP_EAG_KERNEL<<<grid, EAG_THREADS, SMEM_EAG, stream>>>(plan.select, in_map, om);
            else PYSP_AHD_KERNEL<<<grid, K1_THREADS, SMEM_AHD, stream>>>(plan.select, in_map, om);
        }
        rc = check_launch("ahd_select_kernel");
        if (rc) return rc;
    }
    for (int s = 0; s < plan.n_stages; ++s) {
        const MedianParams& mp = plan.median[s];
        OutMaps im, om;
        memset(&im, 0, sizeof(im));
        if (mp.tma_in)
            for (int k = 0; k < 3; ++k) {
                rc = make_map(&im.m[k], mp.in[k], MedianTile<K2_TW, K2_TH>::AW, MedianTile<K2_TW, K2_TH>::AH);
                if (rc) return rc;
            }
        rc = make_out_maps(&om, mp.st, K2_TW, K2_TH);
        if (rc) return rc;
        const int grid = mp.n_tiles < grid2 ? mp.n_tiles : grid2;
        {
            TimedLaunch t(1, stream);
            median_stage_kernel<<<grid, K2_THREADS, smem2, stream>>>(mp, im, om);
        }
        rc = check_launch("median_stage_kernel");
        if (rc) return rc;
    }
    return PYSP_OK;
}

int pysp_normalize_u16(const uint16_t* in, int64_t in_pitch, float* out, int64_t out_pitch, int32_t H, int32_t W,
                       const float black[4], const float white[4], void* stream) {
    if (!in || !out || !black || !white) return fail(PYSP_ERR_INVALID, "pysp_normalize_u16: null pointer");
    if (H < 2 || W < 2 || (H & 1) || (W & 1)) return fail(PYSP_ERR_INVALID, "pysp_normalize_u16: dims must be even");
    if (in_pitch < 2LL * W || out_pitch < 4LL * W) return fail(PYSP_ERR_INVALID, "pysp_normalize_u16: bad pitch");
    int rc = ensure_device();
    if (rc) return rc;
    NormalizeParams p;
    p.in = in; p.in_pitch = in_pitch; p.out = out; p.out_pitch = out_pitch; p.H = H; p.W = W;
    const int perm[4] = {0, 1, 3, 2};
    for (int i = 0; i < 4; ++i) { p.black[perm[i]] = black[i]; p.white[perm[i]] = white[i]; }
    normalize_kernel<<<grid_for((long long)H * (W / 2), 256), 256, 0, (cudaStream_t)stream>>>(p);
    return check_launch("normalize_kernel");
}

int pysp_cam_to_lin_srgb(const float* in, void* out, int64_t n, const double m[9], int32_t clip, int32_t gamma,
                         int32_t out_f16, void* stream) {
    if (!in || !out || !m || n < 0) return fail(PYSP_ERR_INVALID, "pysp_cam_to_lin_srgb: bad argument");
    if (n == 0) return PYSP_OK;
    int rc = ensure_device();
    if (rc) return rc;
    MatrixParams p;
    p.in = in; p.out = out; p.n = n; p.clip = clip; p.gamma = gamma; p.out_f16 = out_f16;
    for (int i = 0; i < 9; ++i) p.m[i] = m[i];
    matrix_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(p);
    return check_launch("matrix_kernel");
}

int pysp_wb_scale(const float* in, float* out, int64_t n, const double wb[3], double max_wb, int32_t mode, int32_t normalized,
                  int32_t wb_is_f64, int32_t max_is_f64, void* stream) {
    if (!in || !out || n < 0 || mode < 0 || mode > 2 || (mode != 2 && !wb)) return fail(PYSP_ERR_INVALID, "pysp_wb_scale: bad argument");
    if (n == 0) return PYSP_OK;
    int rc = ensure_device();
    if (rc) return rc;
    WbParams p;
    p.in = in; p.out = out; p.n = n; p.max_wb = max_wb; p.mode = mode; p.normalized = normalized;
    p.wb_f64 = wb_is_f64 ? 1 : 0; p.max_f64 = max_is_f64 ? 1 : 0;
    for (int c = 0; c < 3; ++c) p.wb[c] = wb ? wb[c] : 1.0;
    wb_kernel<<<grid_for(3 * n, 256), 256, 0, (cudaStream_t)stream>>>(p);
    return check_launch("wb_kernel");
}

int pysp_rgb_to_lab_cv2(const float* in, float* out, int64_t n, const void* lab_lut, void* stream) {
    if (!in || !out || !lab_lut || n < 0) return fail(PYSP_ERR_INVALID, "pysp_rgb_to_lab_cv2: bad argument");
    if (n == 0) return PYSP_OK;
    int rc = ensure_device();
    if (rc) return rc;
    LabParams p = {in, out, n, (const uint4*)lab_lut};
    lab_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(p);
    return check_launch("lab_kernel");
}

int pysp_lin_srgb_to_srgb(const float* in, float* out, int64_t n, void* stream) {
    if (!in || !out || n < 0) return fail(PYSP_ERR_INVALID, "pysp_lin_srgb_to_srgb: bad argument");
    if (n == 0) return PYSP_OK;
    int rc = ensure_device();
    if (rc) return rc;
    GammaParams p = {in, out, n};
    gamma_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(p);
    return check_launch("gamma_kernel");
}

int pysp_fuse_exposures(const float* const* brackets, int32_t n, int64_t in_pitch, int32_t H, int32_t W,
                        const float* ev_offset, const float* bias, int32_t brightest, float* out, int64_t out_pitch,
                        int32_t* count, int64_t count_pitch, void* stream) {
    if (!brackets || !ev_offset || !bias || !out) return fail(PYSP_ERR_INVALID, "pysp_fuse_exposures: null pointer");
    if (n < 1 || n > PYSP_MAX_BRACKETS) return fail(PYSP_ERR_INVALID, "pysp_fuse_exposures: 1..%d brackets", PYSP_MAX_BRACKETS);
    if (H < 2 || W < 2 || (H & 1) || (W & 1)) return fail(PYSP_ERR_INVALID, "pysp_fuse_exposures: dims must be even");
    if (brightest < 0 || brightest >= n) return fail(PYSP_ERR_INVALID, "pysp_fuse_exposures: bad brightest index");
    int rc = ensure_device();
    if (rc) return rc;
    FuseParams p;
    memset(&p, 0, sizeof(p));
    for (int i = 0; i < n; ++i) {
        if (!brackets[i]) return fail(PYSP_ERR_INVALID, "pysp_fuse_exposures: null bracket %d", i);
        p.in[i] = brackets[i]; p.ev_off[i] = ev_offset[i];
        for (int c = 0; c < 3; ++c) p.bias[i][c] = bias[3 * i + c];
    }
    p.in_pitch = in_pitch; p.n = n; p.H = H; p.W = W; p.brightest = brightest;
    p.out = out; p.out_pitch = out_pitch; p.count = count; p.count_pitch = count_pitch;
    bool vec = (W % 4 == 0) && (in_pitch % 16 == 0) && (out_pitch % 16 == 0) && ((uintptr_t)out % 16 == 0) &&
               (!count || (count_pitch % 16 == 0 && (uintptr_t)count % 16 == 0));
    for (int i = 0; i < n; ++i) vec = vec && ((uintptr_t)brackets[i] % 16 == 0);
    if (vec) fuse_kernel<true><<<grid_for((long long)H * (W / 4), 256), 256, 0, (cudaStream_t)stream>>>(p);
    else fuse_kernel<false><<<grid_for((long long)H * W, 256), 256, 0, (cudaStream_t)stream>>>(p);
    return check_launch("fuse_kernel");
}

}  // extern "C"

// ---- NumPy-ordered float32 plane sums (prepost.cuh) -----------------------------------------------------------------
namespace {
long long align16(long long v) { return (v + 15) / 16 * 16; }

struct FlatWorkspace { long long off_val, off_mean, off_stat, total; };

// the workspace depends on the plane's element count n alone: the tree's values (heap order, four planes), mean[4], stat[8]
FlatWorkspace flat_workspace_layout(long long n) {
    FlatWorkspace w;
    long long o = 0;
    w.off_val = o; o = align16(o + 4 * 4 * ((2LL << plane_sum_tree(n, nullptr).L) - 1));
    w.off_mean = o; o = align16(o + 16);
    w.off_stat = o; o = align16(o + 32);
    w.total = o;
    return w;
}

// the summation kernels on the caller's stream; mean[4] lands at `mean`.  With `stat`, tree_sum_kernel also resets the
// flat-field statistics words.
int launch_plane_means(const float* mosaic, long long pitch, int H, int W, char* ws, const FlatWorkspace& lay, float* mean,
                       int* stat, cudaStream_t stream) {
    const PlaneSumTree t = plane_sum_tree((long long)(H / 2) * (W / 2), (float*)(ws + lay.off_val));
    leaf_sum_kernel<<<grid_for(32LL << t.L, 256), 256, 0, stream>>>(mosaic, pitch, W, t);   // eight lanes per (plane, node)
    int rc = check_launch("leaf_sum_kernel");
    if (rc) return rc;
    // wide levels of the tree (4096 nodes and more) run on the whole GPU, the narrow top of the tree in one block per plane
    int d = t.L - 1;
    for (; d >= 12; --d) {
        tree_level_kernel<<<dim3((1u << d) / 256, 4), 256, 0, stream>>>(t, d);
        rc = check_launch("tree_level_kernel");
        if (rc) return rc;
    }
    tree_sum_kernel<<<4, 1024, 0, stream>>>(t, d, mean, stat);
    return check_launch("tree_sum_kernel");
}
}  // namespace

extern "C" {

int64_t pysp_flat_workspace_bytes(int32_t H, int32_t W) {
    if (H < 2 || W < 2 || (H & 1) || (W & 1)) return 0;
    return flat_workspace_layout((long long)(H / 2) * (W / 2)).total;
}

int pysp_bayer_plane_means(const float* mosaic, int64_t pitch, int32_t H, int32_t W, float* means, void* workspace,
                           int64_t workspace_bytes, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!mosaic || !means || !workspace) return fail(PYSP_ERR_INVALID, "pysp_bayer_plane_means: null pointer");
    if (H < 2 || W < 2 || (H & 1) || (W & 1)) return fail(PYSP_ERR_INVALID, "pysp_bayer_plane_means: dims must be even");
    if (pitch < 4LL * W) return fail(PYSP_ERR_INVALID, "pysp_bayer_plane_means: bad pitch");
    int rc = ensure_device();
    if (rc) return rc;
    const FlatWorkspace lay = flat_workspace_layout((long long)(H / 2) * (W / 2));
    if (workspace_bytes < lay.total) return fail(PYSP_ERR_INVALID, "pysp_bayer_plane_means: workspace too small (%lld < %lld)", (long long)workspace_bytes, lay.total);
    return launch_plane_means(mosaic, pitch, H, W, (char*)workspace, lay, means, nullptr, stream);
}

int pysp_flat_frame_correction(const float* sensor, int64_t sensor_pitch, const float* flat, int64_t flat_pitch, float* out,
                               int64_t out_pitch, int32_t H, int32_t W, int32_t clamp_high, void* workspace,
                               int64_t workspace_bytes, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!sensor || !flat || !out || !workspace) return fail(PYSP_ERR_INVALID, "pysp_flat_frame_correction: null pointer");
    if (H < 2 || W < 2 || (H & 1) || (W & 1)) return fail(PYSP_ERR_INVALID, "pysp_flat_frame_correction: dims must be even");
    if (sensor_pitch < 4LL * W || flat_pitch < 4LL * W || out_pitch < 4LL * W) return fail(PYSP_ERR_INVALID, "pysp_flat_frame_correction: bad pitch");
    int rc = ensure_device();
    if (rc) return rc;
    const FlatWorkspace lay = flat_workspace_layout((long long)(H / 2) * (W / 2));
    if (workspace_bytes < lay.total) return fail(PYSP_ERR_INVALID, "pysp_flat_frame_correction: workspace too small (%lld < %lld)", (long long)workspace_bytes, lay.total);
    char* ws = (char*)workspace;
    FlatParams p;
    p.sensor = sensor; p.sensor_pitch = sensor_pitch; p.flat = flat; p.flat_pitch = flat_pitch; p.out = out; p.out_pitch = out_pitch;
    p.H = H; p.W = W; p.clamp_high = clamp_high;
    p.mean = (float*)(ws + lay.off_mean); p.stat = (int*)(ws + lay.off_stat);
    rc = launch_plane_means(flat, flat_pitch, H, W, ws, lay, p.mean, p.stat, stream);
    if (rc) return rc;
    flat_stats_kernel<<<grid_for((long long)H * W, 256), 256, 0, stream>>>(p);
    rc = check_launch("flat_stats_kernel");
    if (rc) return rc;
    flat_apply_kernel<<<grid_for((long long)H * W, 256), 256, 0, stream>>>(p);
    return check_launch("flat_apply_kernel");
}

int pysp_find_hot_pixels_threshold(const float* sensor, int64_t pitch, int32_t H, int32_t W, float min_delta,
                                   int32_t min_neighbour_count, uint8_t* masks, void* stream) {
    if (!sensor || !masks) return fail(PYSP_ERR_INVALID, "pysp_find_hot_pixels_threshold: null pointer");
    if (H < 4 || W < 4 || (H & 1) || (W & 1)) return fail(PYSP_ERR_INVALID, "pysp_find_hot_pixels_threshold: dims must be even and >= 4");
    if (pitch < 4LL * W) return fail(PYSP_ERR_INVALID, "pysp_find_hot_pixels_threshold: bad pitch");
    int rc = ensure_device();
    if (rc) return rc;
    HotParams p;
    p.sensor = sensor; p.pitch = pitch; p.H = H; p.W = W; p.min_delta = min_delta; p.min_count = min_neighbour_count; p.masks = masks;
    hot_pixel_kernel<<<grid_for((long long)H * W, 256), 256, 0, (cudaStream_t)stream>>>(p);
    return check_launch("hot_pixel_kernel");
}

int pysp_fuse_exposures_from_debayer(float* const* images, int32_t n, int64_t n_pixels, const float wb[3], float max_wb,
                                     const int32_t* wb_normalized, const float* ev_offset, const float* bias, int32_t brightest,
                                     double offset_max, const double m[9], float* out, int32_t* count, int32_t write_back,
                                     void* stream) {
    if (!images || !wb || !ev_offset || !bias || !m || !out) return fail(PYSP_ERR_INVALID, "pysp_fuse_exposures_from_debayer: null pointer");
    if (n < 1 || n > PYSP_MAX_EXPOSURES) return fail(PYSP_ERR_INVALID, "pysp_fuse_exposures_from_debayer: 1..%d exposures", PYSP_MAX_EXPOSURES);
    if (brightest < 0 || brightest >= n || n_pixels < 0) return fail(PYSP_ERR_INVALID, "pysp_fuse_exposures_from_debayer: bad argument");
    if (n_pixels == 0) return PYSP_OK;
    int rc = ensure_device();
    if (rc) return rc;
    FuseCamParams p;
    memset(&p, 0, sizeof(p));
    for (int i = 0; i < n; ++i) {
        if (!images[i]) return fail(PYSP_ERR_INVALID, "pysp_fuse_exposures_from_debayer: null exposure %d", i);
        p.img[i] = images[i]; p.ev_off[i] = ev_offset[i]; p.bias[i] = bias[i];
        p.normalized[i] = wb_normalized ? wb_normalized[i] : 0;
    }
    p.n = n; p.n_px = n_pixels; p.brightest = brightest; p.off_max = offset_max; p.out = out; p.count = count; p.write_back = write_back;
    p.max_wb = max_wb;
    for (int c = 0; c < 3; ++c) p.wb[c] = wb[c];
    for (int i = 0; i < 9; ++i) p.m[i] = m[i];
    fuse_cam_kernel<<<grid_for(n_pixels, 256), 256, 0, (cudaStream_t)stream>>>(p);
    return check_launch("fuse_cam_kernel");
}

}  // extern "C"

// ---- DNG WarpRectilinear (warp.cuh) ---------------------------------------------------------------------------------
namespace {
// host scalars of the entry points (dng_warp_rectilinear_coords.pyx:73-77), with the reference's C types: unsigned * float,
// libm powf, np.sqrt of the float sum as a Python float rounded into `cdef float m`
WarpGeom warp_geom(int H, int W, float cnx, float cny, float scale) {
    WarpGeom g;
    g.H = H; g.W = W; g.scale = scale;
    const unsigned width = (unsigned)W, height = (unsigned)H;
    g.cx = (width - 1) * cnx;
    g.cy = (height - 1) * cny;
    float a = fabsf((width - 1) - g.cx), b = fabsf(-g.cx);
    const float mdx = a > b ? a : b;
    a = fabsf((height - 1) - g.cy); b = fabsf(-g.cy);
    const float mdy = a > b ? a : b;
    volatile float s = powf(mdx, 2.0f) + powf(mdy, 2.0f);
    g.m = (float)sqrt((double)s);
    return g;
}
}  // namespace

extern "C" {

int pysp_warp_rectilinear_table(float* table, int64_t table_pitch, int32_t H, int32_t W, const float k[6], float cnx, float cny,
                                float scale, const float* seed, int64_t seed_pitch, void* stream) {
    if (!table || !k) return fail(PYSP_ERR_INVALID, "pysp_warp_rectilinear_table: null pointer");
    if (H < 1 || W < 1) return fail(PYSP_ERR_INVALID, "pysp_warp_rectilinear_table: empty image");
    if (table_pitch < 8LL * W || (table_pitch % 8) || ((uintptr_t)table % 8) || (seed && (seed_pitch < 8LL * W || (seed_pitch % 8) || ((uintptr_t)seed % 8))))
        return fail(PYSP_ERR_INVALID, "pysp_warp_rectilinear_table: tables are [H][W][2] float32, 8-byte aligned rows");
    int rc = ensure_device();
    if (rc) return rc;
    WarpTableParams p;
    p.g = warp_geom(H, W, cnx, cny, scale);
    if (!(p.g.m > 0.0f)) return fail(PYSP_ERR_INVALID, "float division");      // the reference raises ZeroDivisionError (1x1 image)
    for (int i = 0; i < 6; ++i) p.k[i] = k[i];
    p.seed = seed; p.seed_pitch = seed_pitch; p.table = table; p.table_pitch = table_pitch;
    warp_table_kernel<<<grid_for((long long)H * W, 256), 256, 0, (cudaStream_t)stream>>>(p);
    return check_launch("warp_table_kernel");
}

int pysp_remap_lanczos4(const float* src, int64_t src_pitch, int32_t src_step, float* dst, int64_t dst_pitch, int32_t dst_step,
                        int32_t H, int32_t W, const float* map, int64_t map_pitch, const float* lanczos_tab, void* stream) {
    if (!src || !dst || !map || !lanczos_tab) return fail(PYSP_ERR_INVALID, "pysp_remap_lanczos4: null pointer");
    if (H < 1 || W < 1 || src_step < 1 || dst_step < 1) return fail(PYSP_ERR_INVALID, "pysp_remap_lanczos4: bad geometry");
    if (src == dst) return fail(PYSP_ERR_INVALID, "pysp_remap_lanczos4: in-place remapping is not possible (gather)");
    if ((src_pitch % 4) || (dst_pitch % 4) || map_pitch < 8LL * W || (map_pitch % 8) || ((uintptr_t)map % 8))
        return fail(PYSP_ERR_INVALID, "pysp_remap_lanczos4: bad pitch / alignment");
    int rc = ensure_device();
    if (rc) return rc;
    RemapParams p;
    p.H = H; p.W = W; p.src = src; p.src_pitch = src_pitch; p.src_step = src_step; p.dst = dst; p.dst_pitch = dst_pitch;
    p.dst_step = dst_step; p.map = map; p.map_pitch = map_pitch; p.tab = lanczos_tab;
    remap_lanczos4_kernel<<<grid_for((long long)H * W, 256), 256, 0, (cudaStream_t)stream>>>(p);
    return check_launch("remap_lanczos4_kernel");
}

int pysp_warp_rectilinear_apply(const float* src, float* dst, int32_t H, int32_t W, int32_t planes, const float* coeffs, float cnx,
                                float cny, float scale, const float* prior, const float* lanczos_tab, void* stream) {
    if (!src || !dst || !coeffs || !lanczos_tab) return fail(PYSP_ERR_INVALID, "pysp_warp_rectilinear_apply: null pointer");
    if (src == dst) return fail(PYSP_ERR_INVALID, "pysp_warp_rectilinear_apply: source and destination must differ (gather)");
    if (H < 1 || W < 1 || planes < 1 || planes > PYSP_WARP_MAX_PLANES)
        return fail(PYSP_ERR_INVALID, "pysp_warp_rectilinear_apply: 1..%d planes", PYSP_WARP_MAX_PLANES);
    if (prior && ((uintptr_t)prior % 8)) return fail(PYSP_ERR_INVALID, "pysp_warp_rectilinear_apply: prior must be 8-byte aligned");
    int rc = ensure_device();
    if (rc) return rc;
    WarpApplyParams p;
    p.g = warp_geom(H, W, cnx, cny, scale);
    if (!(p.g.m > 0.0f)) return fail(PYSP_ERR_INVALID, "float division");
    p.planes = planes;
    for (int c = 0; c < planes; ++c)
        for (int i = 0; i < 6; ++i) p.k[c][i] = coeffs[c * 6 + i];
    p.prior = prior; p.src = src; p.dst = dst; p.tab = lanczos_tab;
    const long long tiles = (long long)((W + 31) / 32) * ((H + 7) / 8);
    const long long cap = 148LL * 32;
    warp_apply_kernel<<<(int)(tiles < cap ? tiles : cap), 256, 0, (cudaStream_t)stream>>>(p);
    return check_launch("warp_apply_kernel");
}

}  // extern "C"

// ---- baseline JPEG of YCbCr 4:2:0 planes or of RGB images (jpeg.cuh) ---------------------------------------------------
// the phases of one encode, in order; the convert phase only for RGB input
static int jpeg_launch(const JpegParams& p, cudaStream_t stream) {
    int rc;
    const long long cap = 148LL * 8;                     // fixed grids of the kernels whose item count is on the device
    const int block_grid = (int)((p.n_blocks + JPEG_THREADS - 1) / JPEG_THREADS);
    const long long bchunks = (p.n_blocks + JPEG_SCAN_CHUNK - 1) / JPEG_SCAN_CHUNK;
    const long long fchunks = (p.max_items + JPEG_SCAN_CHUNK - 1) / JPEG_SCAN_CHUNK;
    const JpegScan bscan = {p.bits, p.boff, p.bchunk, p.totals, p.n_blocks, nullptr};
    const JpegScan fscan = {p.ffcnt, p.foff, p.fchunk, p.totals + 1, 0, p.totals};
    jpeg_header_kernel<<<1, JPEG_THREADS, 0, stream>>>(p);
    if ((rc = check_launch("jpeg_header_kernel"))) return rc;
    if (p.rgb) {
        jpeg_convert_kernel<<<dim3((p.cw + JPEG_THREADS - 1) / JPEG_THREADS, p.ch), JPEG_THREADS, 0, stream>>>(p);
        if ((rc = check_launch("jpeg_convert_kernel"))) return rc;
    }
    jpeg_block_kernel<<<block_grid, JPEG_THREADS, 0, stream>>>(p);
    if ((rc = check_launch("jpeg_block_kernel"))) return rc;
    jpeg_scan_reduce_kernel<<<(int)std::min(bchunks, cap), JPEG_THREADS, 0, stream>>>(bscan);
    if ((rc = check_launch("jpeg_scan_reduce_kernel"))) return rc;
    jpeg_scan_top_kernel<<<1, JPEG_THREADS, 0, stream>>>(bscan);
    if ((rc = check_launch("jpeg_scan_top_kernel"))) return rc;
    jpeg_scan_down_kernel<<<(int)std::min(bchunks, cap), JPEG_THREADS, 0, stream>>>(bscan);
    if ((rc = check_launch("jpeg_scan_down_kernel"))) return rc;
    jpeg_zero_kernel<<<(int)cap, JPEG_THREADS, 0, stream>>>(p);
    if ((rc = check_launch("jpeg_zero_kernel"))) return rc;
    jpeg_pack_kernel<<<block_grid, JPEG_THREADS, 0, stream>>>(p);
    if ((rc = check_launch("jpeg_pack_kernel"))) return rc;
    jpeg_count_kernel<<<(int)cap, JPEG_THREADS, 0, stream>>>(p);
    if ((rc = check_launch("jpeg_count_kernel"))) return rc;
    jpeg_scan_reduce_kernel<<<(int)std::min(fchunks, cap), JPEG_THREADS, 0, stream>>>(fscan);
    if ((rc = check_launch("jpeg_scan_reduce_kernel"))) return rc;
    jpeg_scan_top_kernel<<<1, JPEG_THREADS, 0, stream>>>(fscan);
    if ((rc = check_launch("jpeg_scan_top_kernel"))) return rc;
    jpeg_scan_down_kernel<<<(int)std::min(fchunks, cap), JPEG_THREADS, 0, stream>>>(fscan);
    if ((rc = check_launch("jpeg_scan_down_kernel"))) return rc;
    jpeg_emit_kernel<<<(int)cap, JPEG_THREADS, 0, stream>>>(p);
    return check_launch("jpeg_emit_kernel");
}

extern "C" {

int64_t pysp_jpeg_max_bytes(int32_t H, int32_t W) { return jpeg_size_ok(H, W) ? jpeg_max_bytes(H, W, 2, 2) : 0; }

int64_t pysp_jpeg_workspace_bytes(int32_t H, int32_t W) { return jpeg_size_ok(H, W) ? jpeg_layout(H, W, nullptr, nullptr) : 0; }

int pysp_jpeg_encode_ycc420(const uint8_t* y, int64_t y_pitch, const uint8_t* cb, const uint8_t* cr, int64_t chroma_pitch, int32_t H,
                            int32_t W, int32_t quality, uint8_t* out, int64_t out_capacity, int64_t* out_len, void* workspace,
                            int64_t workspace_bytes, void* stream) {
    JpegParams p;
    if (plan_jpeg(y, y_pitch, cb, cr, chroma_pitch, H, W, quality, out, out_capacity, out_len, workspace, workspace_bytes, &p, g_err,
                  sizeof(g_err)))
        return PYSP_ERR_INVALID;
    int rc = ensure_device();
    if (rc) return rc;
    return jpeg_launch(p, (cudaStream_t)stream);
}

int64_t pysp_jpeg_rgb_max_bytes(int32_t H, int32_t W, int32_t subsampling) {
    return jpeg_rgb_size_ok(H, W, subsampling) ? jpeg_max_bytes(H, W, jpeg_h(subsampling), jpeg_v(subsampling)) : 0;
}

int64_t pysp_jpeg_rgb_workspace_bytes(int32_t H, int32_t W, int32_t subsampling) {
    return jpeg_rgb_size_ok(H, W, subsampling) ? jpeg_layout(H, W, jpeg_h(subsampling), jpeg_v(subsampling), true, nullptr, nullptr)
                                               : 0;
}

int pysp_jpeg_encode_rgb(const uint8_t* rgb, int64_t pitch_bytes, int32_t H, int32_t W, int32_t quality, int32_t subsampling,
                         uint8_t* out, int64_t out_capacity, int64_t* out_len, void* workspace, int64_t workspace_bytes, void* stream) {
    JpegParams p;
    if (plan_jpeg_rgb(rgb, pitch_bytes, H, W, quality, subsampling, out, out_capacity, out_len, workspace, workspace_bytes, &p, g_err,
                      sizeof(g_err)))
        return PYSP_ERR_INVALID;
    int rc = ensure_device();
    if (rc) return rc;
    return jpeg_launch(p, (cudaStream_t)stream);
}

}  // extern "C"
