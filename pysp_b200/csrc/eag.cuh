// QualityDemosaic.Fast: edge-assisted Gaussian demosaic (debayer/edge_assisted_gaussian.py:188-201) in the same
// tile pipeline as K1.  Phase 0 (ahd_select.cuh) leaves the greens un-balanced here, because the reference
// interpolates the raw greens and multiplies by wb[1] afterwards (edge_assisted_gaussian.py:193).
//   phase 1  green at R/B sites by the delta-mix bilinear kernel (l.10-49, 92-124), white balance, colour differences;
//   phase 2  per 2x2 quad: green high-pass (l.157), 4-phase Gaussian upsample of (c-g) and g (l.126-143) -> staging tile,
//            by K1's quad_resample.
#pragma once
#include "ahd_select.cuh"

namespace pysp {

// edge_assisted_gaussian.py:33-49, float32, evaluated operation by operation
PYSP_HD float delta_mix(float top, float bottom, float left, float right) {
    float dy = fabsf(top - bottom), dx = fabsf(left - right);
    float total = dy + dx;
    float avg_x = (left + right) / 2.0f, avg_y = (top + bottom) / 2.0f;
    float sy = total != 0.0f ? dy / total : 0.5f;
    float sx = 1.0f - sy;
    return (avg_y * sx) + (avg_x * sy);
}

template <int TW, int TH, bool EDGE>
PYSP_D void eag_phases(const SelectParams& p, char* __restrict__ smem, int tile_x, int tile_y) {
    typedef SelectTile<TW, TH> L;
    constexpr int QW = L::QW, QN = L::QN;
    const int H = p.g.H, W = p.g.W;
    const int hq = H >> 1, wq = W >> 1;
    const int x0 = tile_x * TW, y0 = p.y_begin + tile_y * TH;
    constexpr int JX = L::JX, IY = L::IY;
    const int qx0 = (x0 >> 1) - JX, qy0 = (y0 >> 1) - IY;
    float* Q = (float*)(smem + L::OFF_Q);
    float* out = (float*)(smem + L::OFF_OUT);
    // plane roles in this mode: P_R = R*wb0, P_B = B*wb2, P_G1/P_G2 = raw greens;
    // P_GHR / P_GHB = balanced green at R / B sites, P_GVR / P_GVB = balanced G1 / G2, P_DHR / P_DHB = c - g
    {
        constexpr int GW = TW / 2 + 2, GH = TH / 2 + 2;      // tile quads with a 1-quad halo
        const float wbg = p.c.wb[1];
        PYSP_ITEMS(it, GW * GH) {
            int gy = it / GW, gx = it - gy * GW;
            int i = gy + IY - 1, j = gx + JX - 1;
            if (EDGE) {
                int fi = qy0 + i, fj = qx0 + j;
                if (fi < 0 || fi >= hq || fj < 0 || fj >= wq || 2 * fi >= p.y_end + 2) continue;
            }
            int c = i * QW + j;
            const float* G1 = Q + L::P_G1 * QN; const float* G2 = Q + L::P_G2 * QN;
            float g1 = G1[c], g2 = G2[c];
            float gr = delta_mix(G2[c - QW], g2, G1[c - 1], g1) * wbg;        // l.101-104
            float gb = delta_mix(g1, G1[c + QW], g2, G2[c + 1]) * wbg;        // l.95-98
            Q[L::P_GHR * QN + c] = gr; Q[L::P_GHB * QN + c] = gb;
            Q[L::P_GVR * QN + c] = g1 * wbg; Q[L::P_GVB * QN + c] = g2 * wbg;
            Q[L::P_DHR * QN + c] = Q[L::P_R * QN + c] - gr;
            Q[L::P_DHB * QN + c] = Q[L::P_B * QN + c] - gb;
        }
    }
    PYSP_SYNC();
    {
        constexpr int OW = TW / 2, OH = TH / 2;
        PYSP_ITEMS(it, OW * OH) {
            int oy = it / OW, ox = it - oy * OW;
            int i = oy + IY, j = ox + JX;
            int fi = qy0 + i, fj = qx0 + j;
            if (EDGE) { if (fi >= hq || fj >= wq || 2 * fi >= p.y_end) continue; }
            Rgb v[4];
            quad_resample<TW, TH, EDGE>(Q + L::P_GHR * QN, Q + L::P_GHB * QN, Q + L::P_DHR * QN, Q + L::P_DHB * QN,
                                        Q + L::P_GVR * QN, Q + L::P_GVB * QN, i, j, qy0, qx0, H, W, v);
#pragma unroll
            for (int k = 0; k < 4; ++k) stage_pixel<TW, TH>(out, p.st, p.g, p.c, 2 * oy + (k >> 1), 2 * ox + (k & 1), v[k]);
        }
    }
}

}  // namespace pysp
