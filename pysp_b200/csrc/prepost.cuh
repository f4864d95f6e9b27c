// Steps either side of the develop path (SURVEY.md section 8f): flat-field correction and hot-pixel detection on the
// mosaic before it, camera-space HDR fusion of demosaiced exposures after it.  All HBM-bound point/stencil work.
//
// flat_frame_correction (raw_correction.py:25-63) needs np.mean of each CFA plane of the flat field in float32, and
// NumPy's float32 sum is a *pairwise* sum with a fixed shape (loops_utils.h.src, @TYPE@_pairwise_sum): blocks of at
// most 128 elements are summed with eight strided accumulators, blocks are combined by recursive halving (left half
// rounded down to a multiple of 8).  The tree only depends on the element count, and a node's elements follow from its
// position: node (d, i), the i-th node from the left at depth d, is reached from the root by applying NumPy's split once
// per bit of i (sum_node).  So the device evaluates the tree in exactly NumPy's order without a table: leaf_sum_kernel,
// then tree_level_kernel / tree_sum_kernel level by level.  np.mean then divides the float32 sum by the integer count in
// float64 and rounds the quotient to float32 once (numpy/_core/_methods.py, _mean); tree_sum_kernel does the same.  (A
// float32 divisor agrees only up to 2^24 sites: above that float32(n) may differ from n.)  The result is bit-identical
// to np.mean.
#pragma once
#include "pysp_common.cuh"

namespace pysp {

// NumPy's pairwise-sum tree of one plane of n elements.  With n = 8K + t, every left part is a whole number of 8-element
// units (floor(k/2) of a node's k), so the sizes of the nodes at one depth differ by at most one unit plus the t-element
// tail, which stays on the right spine, the largest node of every depth.  Every leaf therefore sits on depth D, where the
// right spine first holds at most 128 elements, or on D - 1, and every node on level L = max(D - 1, 0) is a leaf or the
// parent of two leaves.  leaf_sum_kernel writes level L, the levels above it are sums of two children.  Values are kept
// in heap order: node (d, i) in slot s = 2^d - 1 + i, its children in slots 2s + 1 and 2s + 2, 2^(L+1) - 1 slots per plane.
struct PlaneSumTree {
    long long n;
    int L;
    float* val;                 // [4][2^(L+1) - 1] in the caller's workspace
};

// NumPy's split of a run of more than 128 elements: the left part is half of it, rounded down to a multiple of 8
template <typename T> PYSP_HOSTDEV inline T pairwise_left(T n) { return n / 2 - (n / 2) % 8; }

PYSP_HOSTDEV inline PlaneSumTree plane_sum_tree(long long n, float* val) {
    int D = 0;
    for (long long r = n; r > 128; r -= pairwise_left(r)) ++D;          // down the right spine
    return {n, D > 0 ? D - 1 : 0, val};
}

struct SumNode { int first, count; };   // plane elements [first, first + count); a leaf iff count <= 128

// node (d, i): NumPy's split applied along the path from the root, bit b of i choosing the right part at depth d - b
PYSP_HD SumNode sum_node(const PlaneSumTree& s, int d, int i) {
    SumNode e = {0, (int)s.n};
    for (int b = d - 1; b >= 0; --b) {
        const int l = pairwise_left(e.count);
        if ((i >> b) & 1) { e.first += l; e.count -= l; } else e.count = l;
    }
    return e;
}

// node e on level L is summed as two runs [first, first + l) and [first + l, first + count): a leaf as itself and an empty
// run, an internal node as its two leaf children
PYSP_HD int leaf_part(const SumNode& e) { return e.count > 128 ? pairwise_left(e.count) : e.count; }

struct FlatParams {             // raw_correction.py:25-63
    const float* sensor; long long sensor_pitch;
    const float* flat; long long flat_pitch;
    float* out; long long out_pitch;
    int H, W;
    int clamp_high;
    float* mean;                // [4] device
    int* stat;                  // [4][2]: ordered-int maximum of the finite quotients, number of quotients that are not +-inf
};

struct HotParams {              // raw_bad_pixel_corr.py:30-65
    const float* sensor; long long pitch;
    int H, W;
    float min_delta;
    int min_count;
    uint8_t* masks;             // [4][h][w], planes in the reference's order R, G1, B, G2
};

#define PYSP_MAX_EXPOSURES 16
struct FuseCamParams {          // raw_hdr.py:7-83
    float* img[PYSP_MAX_EXPOSURES];     // [n_px][3] camera RGB, white balance applied; rewritten when write_back
    int n;
    long long n_px;
    float wb[3], max_wb;
    int normalized[PYSP_MAX_EXPOSURES];
    float ev_off[PYSP_MAX_EXPOSURES];   // float32(2**(ev_i - target))
    float bias[PYSP_MAX_EXPOSURES];     // float32(1.6**(-0.1*ev_off_i))
    int brightest;                      // last exposure whose offset equals the maximum
    double off_max;                     // the maximum offset as float64 (np.max returns a strong float64 scalar)
    double m[9];
    float* out; int32_t* count;
    int write_back;
};

// order-preserving float <-> int map (for atomicMax on floats of either sign)
PYSP_HD int float_key(float f) { int b = (int)pysp_as_uint(f); return b >= 0 ? b : b ^ 0x7FFFFFFF; }
PYSP_HD float key_float(int k) { return pysp_as_float((uint32_t)(k >= 0 ? k : k ^ 0x7FFFFFFF)); }
#define PYSP_KEY_NONE ((int)0x80000000)     // below every finite float's key: "no finite value seen"

#ifndef PYSP_HOST_EMU
// plane p in the reference's order R(TL), G1(TR), B(BR), G2(BL): row / column parity of its sites
__device__ __forceinline__ int plane_py(int p) { return p >> 1; }
__device__ __forceinline__ int plane_px(int p) { return (p == 1 || p == 2) ? 1 : 0; }

__device__ __forceinline__ float plane_elem(const float* base, long long pitch, int w, int py, int px, int e) {
    int i = e / w, j = e - i * w;
    return *((const float*)((const char*)base + (long long)(2 * i + py) * pitch) + 2 * j + px);
}

// eight lanes sum the leaf [off, off + n) of one plane (n <= 128, 0 for nothing) exactly as NumPy's unrolled block sum:
// lane j owns the strided partial sum r[j]; the fixed combine ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)) is an xor-butterfly
// (float addition commutes), the tail elements are added by lane 0 in order.  Eight consecutive plane elements are 64
// contiguous bytes of the mosaic.  Every lane of the warp calls it; the sum is lane 0's result.
__device__ __forceinline__ float leaf_sum(const float* mosaic, long long pitch, int w, int py, int px, int off, int n, int lane8) {
    float res = 0.0f;
    if (n < 8) {
        if (lane8 == 0) for (int i = 0; i < n; ++i) res = res + plane_elem(mosaic, pitch, w, py, px, off + i);
    } else {
        // walk (row, column) of the plane incrementally: one division per leaf instead of one per element
        int e = off + lane8, i = e / w, j = e - i * w;
        float r = *((const float*)((const char*)mosaic + (long long)(2 * i + py) * pitch) + 2 * j + px);
        for (int k = 8; k < n - (n % 8); k += 8) {
            j += 8;
            while (j >= w) { j -= w; ++i; }
            r = r + *((const float*)((const char*)mosaic + (long long)(2 * i + py) * pitch) + 2 * j + px);
        }
        res = r;
    }
    // groups with n < 8 carry zeros that only lane 0's own sum replaces
    float s = res;
    s = s + __shfl_xor_sync(0xFFFFFFFFu, s, 1);
    s = s + __shfl_xor_sync(0xFFFFFFFFu, s, 2);
    s = s + __shfl_xor_sync(0xFFFFFFFFu, s, 4);
    if (lane8 == 0 && n >= 8) {
        res = s;
        for (int i = n - (n % 8); i < n; ++i) res = res + plane_elem(mosaic, pitch, w, py, px, off + i);
    }
    return res;
}

// one work item = eight lanes = node (L, i) of one plane: a leaf, or two leaves summed one after the other and added
// left + right, as NumPy's recursion adds them
__global__ void __launch_bounds__(256) leaf_sum_kernel(const float* mosaic, long long pitch, int W, PlaneSumTree t) {
    const int w = W >> 1;
    const int total = 4 << t.L;                                 // a multiple of 4: whole warps stay together for the shuffles
    const int lane8 = threadIdx.x & 7;
    const int groups = (gridDim.x * blockDim.x) >> 3;
    for (int id = (blockIdx.x * blockDim.x + threadIdx.x) >> 3; id < total; id += groups) {
        const int p = id >> t.L, i = id & ((1 << t.L) - 1);
        const int py = plane_py(p), px = plane_px(p);
        const SumNode e = sum_node(t, t.L, i);
        const int l = leaf_part(e);
        const float a = leaf_sum(mosaic, pitch, w, py, px, e.first, l, lane8);
        const float b = leaf_sum(mosaic, pitch, w, py, px, e.first + l, e.count - l, lane8);
        if (lane8 == 0) t.val[(long long)p * ((2 << t.L) - 1) + (1 << t.L) - 1 + i] = l < e.count ? a + b : a;
    }
}

// one wide level d of the tree (its 2^d nodes are independent), all four planes: blockIdx.y = plane.  Node = left child
// + right child, as NumPy's recursion adds them.
__global__ void __launch_bounds__(256) tree_level_kernel(PlaneSumTree t, int d) {
    float* val = t.val + (long long)blockIdx.y * ((2 << t.L) - 1);
    for (int s = (1 << d) - 1 + blockIdx.x * blockDim.x + threadIdx.x; s < (2 << d) - 1; s += gridDim.x * blockDim.x)
        val[s] = val[2 * s + 1] + val[2 * s + 2];
}

// one block = one plane: combine levels d0 .. 0 (the narrow top of the tree), then mean = float32(float64(sum) /
// float64(n)), the division np.mean does.  With `stat` (flat-field correction) it also resets the plane's statistics words
// that flat_stats_kernel, launched next on the same stream, accumulates into.
__global__ void __launch_bounds__(1024) tree_sum_kernel(PlaneSumTree t, int d0, float* mean, int* stat) {
    float* val = t.val + (long long)blockIdx.x * ((2 << t.L) - 1);
    for (int d = d0; d >= 0; --d) {
        for (int s = (1 << d) - 1 + threadIdx.x; s < (2 << d) - 1; s += blockDim.x) val[s] = val[2 * s + 1] + val[2 * s + 2];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        mean[blockIdx.x] = __double2float_rn(__ddiv_rn((double)val[0], (double)t.n));
        if (stat) { stat[2 * blockIdx.x] = PYSP_KEY_NONE; stat[2 * blockIdx.x + 1] = 0; }
    }
}

// work item of the two flat-field passes: four photosites of a row (two CFA sites, alternating)
struct FlatItem { float c[4], q[4]; int plane0, plane1, n; };

__device__ __forceinline__ FlatItem flat_item(const FlatParams& p, const float* mean, long long y, int x0, bool vec) {
    FlatItem it;
    const int row = (int)y & 1;
    it.plane0 = row ? 3 : 0; it.plane1 = row ? 2 : 1;              // even columns: R / G2, odd columns: G1 / B
    const float* s = (const float*)((const char*)p.sensor + y * p.sensor_pitch) + x0;
    const float* f = (const float*)((const char*)p.flat + y * p.flat_pitch) + x0;
    float fv[4] = {1, 1, 1, 1};
    it.n = vec ? 4 : min(4, p.W - x0);
    if (vec) {
        const float4 a = *(const float4*)s, b = *(const float4*)f;
        it.c[0] = a.x; it.c[1] = a.y; it.c[2] = a.z; it.c[3] = a.w;
        fv[0] = b.x; fv[1] = b.y; fv[2] = b.z; fv[3] = b.w;
    } else {
        for (int j = 0; j < 4; ++j) { it.c[j] = j < it.n ? s[j] : 0.0f; fv[j] = j < it.n ? f[j] : 1.0f; }
    }
    const float m0 = mean[it.plane0], m1 = mean[it.plane1];
#pragma unroll
    for (int j = 0; j < 4; ++j) it.q[j] = (it.c[j] * ((j & 1) ? m1 : m0)) / fv[j];      // raw_correction.py:46
    return it;
}

__device__ __forceinline__ bool flat_vec_ok(const FlatParams& p) {
    return (p.W % 4 == 0) && (p.sensor_pitch % 16 == 0) && (p.flat_pitch % 16 == 0) && (p.out_pitch % 16 == 0) &&
           (((size_t)p.sensor | (size_t)p.flat | (size_t)p.out) % 16 == 0);
}

__global__ void __launch_bounds__(256) flat_stats_kernel(FlatParams p) {
    __shared__ int s_max[4], s_cnt[4];
    __shared__ float s_mean[4];
    if (threadIdx.x < 4) { s_max[threadIdx.x] = PYSP_KEY_NONE; s_cnt[threadIdx.x] = 0; s_mean[threadIdx.x] = p.mean[threadIdx.x]; }
    __syncthreads();
    int lmax[4] = {PYSP_KEY_NONE, PYSP_KEY_NONE, PYSP_KEY_NONE, PYSP_KEY_NONE}, lcnt[4] = {0, 0, 0, 0};
    const RowItems ri(p.H, p.W, 4);
    const bool vec = flat_vec_ok(p);
    PYSP_ROW_ITEMS(ri, y, c) {
        const FlatItem it = flat_item(p, s_mean, y, (int)c * 4, vec);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (j >= it.n) continue;
            const float q = it.q[j];
            const bool inf = isinf(q), fin = !inf && !isnan(q);
            const int pl = (j & 1) ? it.plane1 : it.plane0;
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (pl == k) {
                    if (fin) lmax[k] = max(lmax[k], float_key(q));
                    lcnt[k] += inf ? 0 : 1;
                }
        }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (lmax[k] != PYSP_KEY_NONE) atomicMax(&s_max[k], lmax[k]);
        if (lcnt[k]) atomicAdd(&s_cnt[k], lcnt[k]);
    }
    __syncthreads();
    if (threadIdx.x < 4) {
        if (s_max[threadIdx.x] != PYSP_KEY_NONE) atomicMax(&p.stat[2 * threadIdx.x], s_max[threadIdx.x]);
        if (s_cnt[threadIdx.x]) atomicAdd(&p.stat[2 * threadIdx.x + 1], s_cnt[threadIdx.x]);
    }
}

__global__ void __launch_bounds__(256) flat_apply_kernel(FlatParams p) {
    __shared__ float s_mean[4], s_vmax[4];
    __shared__ int s_allinf[4];
    if (threadIdx.x < 4) {
        s_mean[threadIdx.x] = p.mean[threadIdx.x];
        const int key = p.stat[2 * threadIdx.x];
        s_vmax[threadIdx.x] = key == PYSP_KEY_NONE ? pysp_as_float(0x7FC00000u) : key_float(key);
        s_allinf[threadIdx.x] = p.stat[2 * threadIdx.x + 1] == 0;   // np.isinf(output).all(): leave the plane alone
    }
    __syncthreads();
    const RowItems ri(p.H, p.W, 4);
    const bool vec = flat_vec_ok(p);
    PYSP_ROW_ITEMS(ri, y, c) {
        const int x0 = (int)c * 4;
        const FlatItem it = flat_item(p, s_mean, y, x0, vec);
        float o[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int pl = (j & 1) ? it.plane1 : it.plane0;
            float q = it.q[j];
            if (s_allinf[pl]) {
                q = it.c[j];
            } else {
                if (q == pysp_as_float(0x7F800000u)) q = s_vmax[pl];   // +inf -> largest finite value of the plane
                if (q < 0.0f) q = 0.0f;
                if (p.clamp_high && q > 1.0f) q = 1.0f;
            }
            o[j] = q;
        }
        float* dst = (float*)((char*)p.out + y * p.out_pitch) + x0;
        if (vec) *(float4*)dst = make_float4(o[0], o[1], o[2], o[3]);
        else for (int j = 0; j < it.n; ++j) dst[j] = o[j];
    }
}

// One work item = four horizontally adjacent 2x2 quads: the four planes' sites at quarter coordinates (qy, qx0..qx0+3).
// It reads mosaic rows 2qy-2..2qy+3, columns 2qx0-2..2qx0+9 (np.pad mode="reflect" on the plane = REFLECT_101 on the
// quarter grid) and writes four bytes per plane.
__global__ void __launch_bounds__(256) hot_pixel_kernel(HotParams p) {
    const int h = p.H >> 1, w = p.W >> 1;
    const RowItems ri(h, w, 4);
    const bool vec_st = (w % 4 == 0) && ((size_t)p.masks % 4 == 0);
    PYSP_ROW_ITEMS(ri, qy, c) {
        const int qx0 = (int)c * 4;
        const bool interior = qy >= 1 && qy + 1 < h && qx0 >= 1 && qx0 + 4 < w;
        float v[6][12];                                     // [row][col] of the 6 x 12 mosaic window
        if (interior) {
            // columns 2*qx0-2 .. 2*qx0+9: qx0 is a multiple of 4, so the run starts on an 8-byte boundary when the rows do
            const bool al = (p.pitch % 8 == 0) && ((size_t)p.sensor % 8 == 0);
#pragma unroll
            for (int r = 0; r < 6; ++r) {
                const float* row = (const float*)((const char*)p.sensor + (long long)(2 * ((int)qy - 1) + r) * p.pitch) + 2 * qx0 - 2;
                if (al) {
#pragma unroll
                    for (int k = 0; k < 6; ++k) { const float2 t = ((const float2*)row)[k]; v[r][2 * k] = t.x; v[r][2 * k + 1] = t.y; }
                } else {
#pragma unroll
                    for (int k = 0; k < 12; ++k) v[r][k] = row[k];
                }
            }
        } else {
#pragma unroll
            for (int r = 0; r < 6; ++r) {
                const int ny = reflect101((int)qy - 1 + (r >> 1), h);
                const float* row = (const float*)((const char*)p.sensor + (long long)(2 * ny + (r & 1)) * p.pitch);
#pragma unroll
                for (int k = 0; k < 12; ++k) {
                    const int nx = reflect101(min(qx0 - 1 + (k >> 1), w), w);
                    v[r][k] = row[2 * nx + (k & 1)];
                }
            }
        }
        uint32_t bits[4] = {0, 0, 0, 0};                    // byte j of plane k
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int sy = 0; sy < 2; ++sy)
#pragma unroll
                for (int sx = 0; sx < 2; ++sx) {
                    const int r0 = 2 + sy, k0 = 2 + 2 * j + sx;         // the site itself in the window
                    const float ref = v[r0][k0] - p.min_delta;
                    int cnt = 0;
#pragma unroll
                    for (int dy = -2; dy <= 2; dy += 2)
#pragma unroll
                        for (int dx = -2; dx <= 2; dx += 2) {
                            if (dy == 0 && dx == 0) continue;
                            cnt += ref > v[r0 + dy][k0 + dx] ? 1 : 0;
                        }
                    const int plane = sy == 0 ? sx : (sx ? 2 : 3);
                    if (cnt > p.min_count) bits[plane] |= 1u << (8 * j);
                }
        const int nq = min(4, w - qx0);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            uint8_t* dst = p.masks + (long long)k * h * w + (long long)qy * w + qx0;
            if (vec_st) *(uint32_t*)dst = bits[k];
            else for (int j = 0; j < nq; ++j) dst[j] = (uint8_t)(bits[k] >> (8 * j));
        }
    }
}

// one work item = four pixels = twelve consecutive floats (three 16-byte vectors per exposure), exposures strictly in
// list order
__global__ void __launch_bounds__(256) fuse_cam_kernel(FuseCamParams p) {
    bool vec = ((size_t)p.out % 16 == 0) && (!p.count || (size_t)p.count % 16 == 0);
    for (int k = 0; k < p.n; ++k) vec = vec && ((size_t)p.img[k] % 16 == 0);
    const long long items = (p.n_px + 3) / 4;
    for (long long it = blockIdx.x * (long long)blockDim.x + threadIdx.x; it < items; it += (long long)gridDim.x * blockDim.x) {
        const long long e0 = it * 12;                                   // first float of the item
        const int nv = (int)min(12LL, 3 * p.n_px - e0);
        const bool full = vec && nv == 12;
        float sum_w[12], sum_p[12], bright[12];
        int cnt[12];
#pragma unroll
        for (int j = 0; j < 12; ++j) { sum_w[j] = 0.0f; sum_p[j] = 0.0f; bright[j] = 0.0f; cnt[j] = 0; }
        for (int k = 0; k < p.n; ++k) {
            float v[12];
            float* src = p.img[k] + e0;
            if (full) {
#pragma unroll
                for (int q = 0; q < 3; ++q) { const float4 t = ((const float4*)src)[q]; v[4 * q] = t.x; v[4 * q + 1] = t.y; v[4 * q + 2] = t.z; v[4 * q + 3] = t.w; }
            } else {
#pragma unroll
                for (int j = 0; j < 12; ++j) v[j] = j < nv ? src[j] : 0.0f;
            }
            const float bias = p.bias[k], ev = p.ev_off[k];
            const bool norm = p.normalized[k] != 0;
#pragma unroll
            for (int j = 0; j < 12; ++j) {
                const float wbc = p.wb[j % 3];
                float x = v[j];
                if (norm) x = x * p.max_wb;                                               // image_base.py:56-57
                const float u = __double2float_rn(__ddiv_rn((double)x, (double)wbc));     // wb_undo (float64 division)
                const float wgt = (0.5f - fabsf(u - 0.5f)) * bias;                        // raw_hdr.py:59-62
                sum_w[j] = sum_w[j] + wgt;
                const float a = u * wbc;                                                  // wb_apply
                v[j] = a;
                if (k == p.brightest) bright[j] = a;
                sum_p[j] = sum_p[j] + ((a * wgt) * ev);                                   // raw_hdr.py:71
                cnt[j] += wgt > 0.0f ? 1 : 0;
            }
            if (p.write_back) {
                if (full) {
#pragma unroll
                    for (int q = 0; q < 3; ++q) ((float4*)src)[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
                } else {
#pragma unroll
                    for (int j = 0; j < 12; ++j) if (j < nv) src[j] = v[j];
                }
            }
        }
        float fused[12], o[12];
#pragma unroll
        for (int j = 0; j < 12; ++j) {
            const float q = sum_p[j] / sum_w[j];
            fused[j] = sum_w[j] == 0.0f ? __double2float_rn(__dmul_rn((double)bright[j], p.off_max)) : q;   // raw_hdr.py:75-80
        }
#pragma unroll
        for (int px = 0; px < 4; ++px)                                                    // clip_highlights=False (raw_hdr.py:81)
#pragma unroll
            for (int r = 0; r < 3; ++r) o[3 * px + r] = dot3_f64(p.m + 3 * r, fused[3 * px], fused[3 * px + 1], fused[3 * px + 2]);
        float* dst = p.out + e0;
        int32_t* dc = p.count ? p.count + e0 : nullptr;
        if (full) {
#pragma unroll
            for (int q = 0; q < 3; ++q) {
                ((float4*)dst)[q] = make_float4(o[4 * q], o[4 * q + 1], o[4 * q + 2], o[4 * q + 3]);
                if (dc) ((int4*)dc)[q] = make_int4(cnt[4 * q], cnt[4 * q + 1], cnt[4 * q + 2], cnt[4 * q + 3]);
            }
        } else {
#pragma unroll
            for (int j = 0; j < 12; ++j) if (j < nv) { dst[j] = o[j]; if (dc) dc[j] = cnt[j]; }
        }
    }
}
#endif

}  // namespace pysp
