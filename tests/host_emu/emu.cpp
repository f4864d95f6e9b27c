// TEST INFRASTRUCTURE ONLY -- host emulation of the tile functions in pysp_b200/csrc/*.cuh.
//
// The CUDA tile functions are written as barrier-separated phases whose work items are independent, so
// the very same source compiles for the host (PYSP_HOST_EMU): a phase runs its items serially, a barrier
// is a no-op.  The TMA box transfers are replaced by `box_load_generic` / `store_tile_generic`, which the
// device build also uses when a tensor cannot be described by a tensor map and which have the TMA's
// semantics (zero fill on load, clipping on store).  This lets tests/test_tile_logic.py diff the exact kernel
// logic (tiling, halos, the six border rules, band seams, flips) against the oracle in a container without a
// GPU.  It is NOT a CPU fallback: it is never built into libpysp_b200.so, never imported by the pysp_b200
// package, and its entry point takes HOST pointers.  Build: tests/host_emu/build.sh (g++ -ffp-contract=off).
#define PYSP_HOST_EMU 1
#include <stdlib.h>
#include <vector>

struct uint4 { unsigned int x, y, z, w; };

#include "../../pysp_b200/csrc/ahd_select.cuh"
#include "../../pysp_b200/csrc/eag.cuh"
#include "../../pysp_b200/csrc/median_stage.cuh"
#include "../../pysp_b200/csrc/develop_plan.h"
#include "../../pysp_b200/csrc/prepost.cuh"

using namespace pysp;

static char g_err[512];

extern "C" const char* emu_last_error(void) { return g_err; }

template <int TW, int TH, int TW2 = TW, int TH2 = TH>
static void run_chain(const DevelopPlan& plan) {
    typedef SelectTile<TW, TH> LS;
    typedef MedianTile<TW2, TH2> LM;
    std::vector<float> buf((LS::SMEM_BYTES > LM::SMEM_BYTES ? LS::SMEM_BYTES : LM::SMEM_BYTES) / 4 + 64);
    char* smem = (char*)buf.data();
    auto poison = [&]() { for (size_t i = 0; i < buf.size(); ++i) buf[i] = __builtin_nanf(""); };
    {
        const SelectParams& p = plan.select;
        for (int t = 0; t < p.n_tiles; ++t) {
            int ty = t / p.tiles_x, tx = t - ty * p.tiles_x;
            poison();
            int bx, by;
            select_input_box<TW, TH>(p, tx, ty, &bx, &by);
            box_load_generic(smem + LS::OFF_STAGE, p.in, bx, by, LS::BOXW, LS::BOXH);
            const bool eag = p.algo == ALGO_EAG;
            if (select_tile_is_edge<TW, TH>(p, tx, ty)) {
                select_phase0<TW, TH, true>(p, smem, tx, ty);
                if (eag) eag_phases<TW, TH, true>(p, smem, tx, ty); else select_phases<TW, TH, true>(p, smem, tx, ty, []() {});
            } else {
                select_phase0<TW, TH, false>(p, smem, tx, ty);
                if (eag) eag_phases<TW, TH, false>(p, smem, tx, ty); else select_phases<TW, TH, false>(p, smem, tx, ty, []() {});
            }
            store_tile_generic<TW, TH>((const float*)(smem + LS::OFF_OUT), p.st, p.g, tx * TW, p.y_begin + ty * TH);
        }
    }
    for (int s = 0; s < plan.n_stages; ++s) {
        const MedianParams& p = plan.median[s];
        for (int t = 0; t < p.n_tiles; ++t) {
            int ty = t / p.tiles_x, tx = t - ty * p.tiles_x;
            poison();
            const int bx = tx * TW2 - 4, by = p.y_begin + ty * TH2 - 4 - p.in_row0;
            for (int k = 0; k < 3; ++k) box_load_generic(smem + LM::OFF_IN + k * LM::PLANE_BYTES, p.in[k], bx, by, LM::AW, LM::AH);
            // the product runs the 2x4-block phases; odd stages of the emulation run the 2x2-block ones so that both stay covered
            const bool block4 = (s & 1) == 0;
            if (median_tile_is_edge<TW2, TH2>(p, tx, ty)) {
                median_fix_border<TW2, TH2>(p, smem, tx, ty);
                if (block4) { median_phase_b4<TW2, TH2, true>(p, smem, tx, ty); median_phase_c4<TW2, TH2, true>(p, smem, tx, ty); }
                else { median_phase_b<TW2, TH2, true>(p, smem, tx, ty); median_phase_c<TW2, TH2, true>(p, smem, tx, ty); }
            } else {
                if (block4) { median_phase_b4<TW2, TH2, false>(p, smem, tx, ty); median_phase_c4<TW2, TH2, false>(p, smem, tx, ty); }
                else { median_phase_b<TW2, TH2, false>(p, smem, tx, ty); median_phase_c<TW2, TH2, false>(p, smem, tx, ty); }
            }
            store_tile_generic<TW2, TH2>((const float*)(smem + LM::OFF_OUT), p.st, p.g, tx * TW2, p.y_begin + ty * TH2);
        }
    }
}

// NumPy's pairwise-sum tree of an n-element plane as leaf_sum_kernel walks it (prepost.cuh): one row (depth, index, first
// element, count) per leaf, from left to right, and the level L of the kernel's work items in *L.  Returns the number of
// leaves, or -1 when there are more than `cap`.
extern "C" int emu_plane_sum_leaves(long long n, int* L, int64_t* rows, int cap) {
    const PlaneSumTree t = plane_sum_tree(n, nullptr);
    *L = t.L;
    int k = 0;
    auto leaf = [&](int d, int i, int first, int count) {
        if (k == cap) return false;
        int64_t* r = rows + 4 * (long long)k++;
        r[0] = d; r[1] = i; r[2] = first; r[3] = count;
        return true;
    };
    for (int i = 0; i < (1 << t.L); ++i) {
        const SumNode e = sum_node(t, t.L, i);
        const int l = leaf_part(e);
        const bool ok = l == e.count ? leaf(t.L, i, e.first, l)
                                     : leaf(t.L + 1, 2 * i, e.first, l) && leaf(t.L + 1, 2 * i + 1, e.first + l, e.count - l);
        if (!ok) return -1;
    }
    return k;
}

extern "C" int emu_develop(const pysp_develop_args* a, int tw, int th) {
    // tile sizes are compile-time in the kernels; the emulation instantiates the product's tiles (K1 60x60, K2 60x60), the
    // 60x28 K1 tile of earlier builds and small ones (16x8, 20x8) that put many tile seams and partial tiles into small frames
    DevelopPlan plan;
    const bool old = tw == 60 && th == 28;
    int rc = plan_develop(a, tw, th, tw, old ? 60 : th, &plan, g_err, sizeof(g_err));
    if (rc) return rc;
    if (old) run_chain<60, 28, 60, 60>(plan);
    else if (tw == 60 && th == 60) run_chain<60, 60>(plan);   // the product's tiles
    else if (tw == 60 && th == 44) run_chain<60, 44>(plan);   // the K1 tile of QualityDemosaic.Fast
    else if (tw == 56 && th == 30) run_chain<56, 30>(plan);   // a box with the fixed 8-px margin (tile width 0 mod 8)
    else if (tw == 16 && th == 8) run_chain<16, 8>(plan);
    else if (tw == 20 && th == 8) run_chain<20, 8>(plan);     // tile width 4 mod 8: box margin alternates 8 / 12 px
    else {
        snprintf(g_err, sizeof(g_err), "emu_develop: tile %dx%d not instantiated", tw, th);
        return PYSP_ERR_INVALID;
    }
    return PYSP_OK;
}
