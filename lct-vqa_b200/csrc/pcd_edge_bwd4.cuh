// pcd_edge_bwd4.cuh — stage-A backward DATA kernels of the MixedOp edges for the production geometries, v4.
//
// Where the generic kernel (pcd_edge.cuh) runs six or seven blocks per (edge, image, tile), one per candidate op, each
// storing its own partial d xs plane that source_grad masks and sums, v4 runs TWO blocks per (edge, image, tile):
//   conv block : A5, D5, A3, D3 (+ FactorizedReduce at stride 2) one after the other, the partial input gradients summed in
//                REGISTERS across the units, the ReLU mask applied at the end (x re-read from L2), ONE plain store;
//   pool block : max-pool (argmax recomputed from the raw tile) + avg-pool (+ identity skip at stride 1), ONE plain store.
// No atomics, no memset of the slots, a fifth of the d xs traffic, and the depthwise-transpose phase uses the tap tables /
// narrow segment loads of pcd_edge_v4.cuh.  At stride 2 the transposed depthwise convs are evaluated per input parity
// plane (input pixel (2i+a, 2j+b) only sees the taps of parity (a, b)): unit-stride everywhere, a thread produces the
// interleaved even/odd columns of its rows and stores whole float4s.
// The two slots are the first two planes of the edge's partial-gradient region (EdgeG::pd): slot 0 = masked conv/FR
// partial, slot 1 = pool partial (SrcEdge::merged set).
#pragma once
#include "pcd_edge_bwd2.cuh"
#include "pcd_edge_v4.cuh"

namespace pcd {

// acc[oy][j] += sum over the taps (ky, kx) of parity (A, B) of w[ky][kx] * dt[oy - pos(ky)][j - pos(kx)]
// (transpose of dw_plane: `base` = dt plane element of (patch row 0, patch column 0), 16-byte aligned, pitch P)
template <int KS, int DIL, int S, int PR, int A, int B, int P>
PCD_HD void dw_plane_bwd(const float* PCD_RESTRICT base, const float (&w)[KS * KS], float (&acc)[PR][4]) {
    using G = TapGeo<KS, DIL, S>;
    if constexpr (G::any(A) && G::any(B)) {
        constexpr int RMIN = -G::pmax(A), RMAX = -G::pmin(A) + PR - 1;
        constexpr int LO = seg_lo(-G::pmax(B)), HI = seg_hi(3 - G::pmin(B));
#pragma unroll
        for (int rr = RMIN; rr <= RMAX; ++rr) {
            float v[HI - LO + 1];
            load_seg<LO, HI>(base + rr * P, v);
#pragma unroll
            for (int oy = 0; oy < PR; ++oy) {
                const int ky = G::find(A, oy - rr);
                if (ky < 0) continue;
#pragma unroll
                for (int kx = 0; kx < KS; ++kx) {
                    if (G::par(kx) != B) continue;
                    const int g = -G::pos(kx) - LO;
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[oy][j] = fmaf(w[ky * KS + kx], v[j + g], acc[oy][j]);
                }
            }
        }
    }
}

template <int C, int S, int W>
struct V4GeoBwd {
    static constexpr int TH = (S == 1) ? 16 : 8;             // output rows per tile (= rows of each input parity plane)
    static constexpr int HYMAX = (S == 1) ? 4 : 2;
    static constexpr int RHMAX = TH + 2 * HYMAX;
    static constexpr int P = W + 8 + (W == 16 ? 4 : 0);
    static constexpr int WS4 = W / 4, NRB = TH / 4;
    static constexpr int DZ_FLOATS = C * RHMAX * W, DT_FLOATS = C * RHMAX * P;
    static constexpr int NCOEF = 5 * 4 * C;                  // A3 A5 D3 D5 FR
    static constexpr int NW = 68 * C + 4 * C * C;            // depthwise taps (A5 D5 A3 D3) + the four transposed pointwise matrices
    static constexpr size_t CONV_SMEM_FLOATS = (size_t)DZ_FLOATS + DT_FLOATS + NCOEF + NW + 16;
    // pool block (V4GeoPool below): raw input tile + three planes over the row-haloed output tile, C/2 channels per pass
    static constexpr size_t POOL_SMEM_FLOATS = (size_t)(C / 2) * ((S * TH + 8) * (S * W + 8) + 3 * (TH + 2) * P) + 2 * 4 * C + 16;
    static constexpr size_t SMEM_FLOATS = CONV_SMEM_FLOATS > POOL_SMEM_FLOATS ? CONV_SMEM_FLOATS : POOL_SMEM_FLOATS;
    static_assert((S == 1 ? 1 : 2) * C * NRB * WS4 == kThreads, "one input-gradient patch per thread");
};

// ---- conv block --------------------------------------------------------------------------------------------------
// one unit: dz on the row-haloed tile -> dt = Wpw^T dz -> this thread's patch of the transposed depthwise conv, added to acc
template <int C, int S, int W, int KS, int DIL, int U, class AccT>
PCD_HD void bwdA4_unit(const EdgeBwdArgs& a, const EdgeG& e, int n, int oy0, float* DZ, float* DT, const float* COEF, const float* WT,
                       const float* WDW, AccT& PCD_TPASS(accs)) {
    using G = V4GeoBwd<C, S, W>;
    constexpr int PAD = DIL * (KS - 1) / 2;
    constexpr int HY = (S == 1) ? PAD : (PAD + 1) / 2;
    constexpr int RH = G::TH + 2 * HY, P = G::P;
    const long long HW = (long long)a.Ho * W, nslot = (long long)a.B * C * HW;
    constexpr bool isA = (U == 0 || U == 2);
    constexpr int which = (U == 2) ? 1 : 0;
    const float* dy_img = isA ? e.ga + which * nslot + (long long)n * C * HW : e.dn + (long long)n * e.dn_ns;
    dz_stage<C, RH, W>(DZ, DT, dy_img, HW, isA ? 1 : 4, e.saved + slot_z(U) * nslot + (long long)n * C * HW, HW, oy0 - HY, a.Ho);
    cp16_wait();
    PCD_SYNC();
    dz_finish<C, RH, W>(DZ, DT, COEF, oy0 - HY, a.Ho);
    PCD_SYNC();                                     // raw z consumed: DT can be rewritten
    zero_col_halo<C * RH, W, P>(DT);
    dt_rows<C, RH, W, P, 4>(DT, DZ, WT, oy0 - HY, a.Ho);
    PCD_SYNC();
    PCD_EACH(t) {
        auto& acc = PCD_TREF(accs, t);
        const int strip = t % G::WS4, rb = (t / G::WS4) % G::NRB, ch = (t / (G::WS4 * G::NRB)) % C;
        const int py = rb * 4, px = strip * 4;
        float w[KS * KS];
#pragma unroll
        for (int i = 0; i < KS * KS; ++i) w[i] = WDW[ch * KS * KS + i];
        const float* base = DT + (ch * RH + py + HY) * P + 4 + px;
        if (S == 1) {
            dw_plane_bwd<KS, DIL, 1, 4, 0, 0, P>(base, w, acc[0]);
        } else if (t < kThreads / 2) {               // even input rows (warp-uniform: the row parity is the outermost task index)
            dw_plane_bwd<KS, DIL, 2, 4, 0, 0, P>(base, w, acc[0]);
            dw_plane_bwd<KS, DIL, 2, 4, 0, 1, P>(base, w, acc[1]);
        } else {
            dw_plane_bwd<KS, DIL, 2, 4, 1, 0, P>(base, w, acc[0]);
            dw_plane_bwd<KS, DIL, 2, 4, 1, 1, P>(base, w, acc[1]);
        }
    }
    PCD_SYNC();                                     // DZ / DT are rewritten by the next unit
}

template <int C, int S, int W>
PCD_HD void bwdA4_conv_block(const EdgeBwdArgs& a, const EdgeG& e, int tile, int n, float* smem) {
    using G = V4GeoBwd<C, S, W>;
    constexpr int TH = G::TH, NB = (S == 1) ? 1 : 2;
    float* DZ = smem;
    float* DT = DZ + G::DZ_FLOATS;
    float* COEF = DT + G::DT_FLOATS;               // [A3 | A5 | D3 | D5 | FR][4C]
    float* WDW = COEF + G::NCOEF;                  // [A5 25C | D5 25C | A3 9C | D3 9C]
    float* WT = WDW + 68 * C;                      // [A5 | D5 | A3 | D3][ci][co]
    const int oy0 = tile * TH;
    const long long HW = (long long)a.Ho * W, nslot = (long long)a.B * C * HW;
    const double cnt = (double)a.B * a.Ho * W;
    const float beta = e.beta ? e.beta[0] : 1.f;
    {   // the edge's weights, once per block: depthwise taps as they are, pointwise matrices transposed
        const int us[4] = {2, 5, 0, 4}, ks2[4] = {25, 25, 9, 9}, wo[4] = {0, 25 * C, 50 * C, 59 * C};
        for (int q = 0; q < 4; ++q) {
            const float* wd = e.par + edge_dw_off(C, S, us[q]);
            const float* wp = e.par + edge_pw_off(C, S, us[q]);
            PCD_FOR(i, ks2[q] * C) WDW[wo[q] + i] = wd[i];
            PCD_FOR(i, C * C) WT[q * C * C + (i % C) * C + i / C] = wp[i];
        }
    }
    PCD_FOR(i, 5 * C) {
        const int k = i / C, j = i - k * C;
        if (k < 2) {                                // A3 / A5: dy = GA (kappa already inside)
            const int u = k == 0 ? 0 : 2, bn = bn_unit(S, u);
            edge_coef(COEF + k * 4 * C, j, dz_consts(e.stats, C, bn, j, cnt, a.eps, e.bstats[bs_ga(k) * C + j],
                                                     e.bstats[(bs_ga(k) + 1) * C + j], 1.f));
        } else if (k < 4) {                         // D3 / D5: dy = kappa * h
            const int u = k == 2 ? 4 : 5, bn = bn_unit(S, u);
            edge_coef(COEF + k * 4 * C, j, dz_consts(e.stats, C, bn, j, cnt, a.eps, e.bstats[bs_s0() * C + j],
                                                     e.bstats[bs_sz(bn) * C + j], beta * e.alpha[k == 2 ? 6 : 7]));
        } else if (S == 2) {
            edge_coef(COEF + 4 * 4 * C, j, dz_consts(e.stats, C, bn_f(), j, cnt, a.eps, e.bstats[bs_s0() * C + j],
                                                     e.bstats[bs_sz(bn_f()) * C + j], beta * e.alpha[3]));
        }
    }
    PCD_TSTATE(float, acc, [NB][4][4]);
    PCD_EACH(t) {
        auto& ac = PCD_TREF(acc, t);
#pragma unroll
        for (int b = 0; b < NB; ++b)
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) ac[b][i][j] = 0.f;
    }
    PCD_SYNC();
    bwdA4_unit<C, S, W, 5, 1, 2>(a, e, n, oy0, DZ, DT, COEF + 1 * 4 * C, WT + 0 * C * C, WDW, PCD_TPASS(acc));
    bwdA4_unit<C, S, W, 5, 2, 5>(a, e, n, oy0, DZ, DT, COEF + 3 * 4 * C, WT + 1 * C * C, WDW + 25 * C, PCD_TPASS(acc));
    bwdA4_unit<C, S, W, 3, 1, 0>(a, e, n, oy0, DZ, DT, COEF + 0 * 4 * C, WT + 2 * C * C, WDW + 50 * C, PCD_TPASS(acc));
    bwdA4_unit<C, S, W, 3, 2, 4>(a, e, n, oy0, DZ, DT, COEF + 2 * 4 * C, WT + 3 * C * C, WDW + 59 * C, PCD_TPASS(acc));
    if (S == 2) {
        // FactorizedReduce (operations.py:90-104): conv_1 reads relu(x)[2i][2j], conv_2 relu(x)[2i+1][2j+1]
        dz_rows<C, TH, W>(DZ, e.dn + (long long)n * e.dn_ns, HW, 4, e.saved + slot_f() * nslot + (long long)n * C * HW, HW,
                          COEF + 4 * 4 * C, oy0, a.Ho);
        PCD_FOR(i, C * C) WT[i] = e.par[i];        // [co][ci], conv_1 rows then conv_2 rows
        PCD_SYNC();
        PCD_EACH(t) {
            auto& ac = PCD_TREF(acc, t);
            const int strip = t % G::WS4, rb = (t / G::WS4) % G::NRB, ch = (t / (G::WS4 * G::NRB)) % C;
            const int py = rb * 4, px = strip * 4, par = t < kThreads / 2 ? 0 : 1;
#pragma unroll 4
            for (int k = 0; k < C / 2; ++k) {
                const int co = par * (C / 2) + k;
                const float wv = WT[co * C + ch];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const F4 d = ld4(DZ + (co * TH + py + i) * W + px);
                    if (par == 0) {                  // warp-uniform; static accumulator indices keep acc in registers
                        float (&row)[4] = ac[0][i];
                        row[0] = fmaf(wv, d.x, row[0]); row[1] = fmaf(wv, d.y, row[1]);
                        row[2] = fmaf(wv, d.z, row[2]); row[3] = fmaf(wv, d.w, row[3]);
                    } else {
                        float (&row)[4] = ac[NB - 1][i];
                        row[0] = fmaf(wv, d.x, row[0]); row[1] = fmaf(wv, d.y, row[1]);
                        row[2] = fmaf(wv, d.z, row[2]); row[3] = fmaf(wv, d.w, row[3]);
                    }
                }
            }
        }
    }
    // ---- ReLU mask (every conv candidate and FactorizedReduce starts with ReLU(x)), one plain store ---------------------
    const float* x_img = e.x + (long long)n * e.x_ns;
    float* pd_img = e.pd + (long long)n * C * a.Hs * a.Ws;                  // slot 0
    PCD_EACH(t) {
        auto& ac = PCD_TREF(acc, t);
        const int strip = t % G::WS4, rb = (t / G::WS4) % G::NRB, ch = (t / (G::WS4 * G::NRB)) % C;
        const int py = rb * 4, px = strip * 4;
        if (S == 1) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const long long o = ((long long)ch * a.Hs + oy0 + py + i) * W + px;
                const F4 x = ld4(x_img + o);
                st4(pd_img + o, x.x > 0.f ? ac[0][i][0] : 0.f, x.y > 0.f ? ac[0][i][1] : 0.f, x.z > 0.f ? ac[0][i][2] : 0.f,
                    x.w > 0.f ? ac[0][i][3] : 0.f);
            }
        } else {
            const int par = t < kThreads / 2 ? 0 : 1;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const long long o = ((long long)ch * a.Hs + 2 * (oy0 + py + i) + par) * (2 * W) + 2 * px;
                const F4 x0 = ld4(x_img + o), x1 = ld4(x_img + o + 4);
                const float (&e0)[4] = ac[0][i];
                const float (&o1)[4] = ac[NB - 1][i];
                st4(pd_img + o, x0.x > 0.f ? e0[0] : 0.f, x0.y > 0.f ? o1[0] : 0.f, x0.z > 0.f ? e0[1] : 0.f, x0.w > 0.f ? o1[1] : 0.f);
                st4(pd_img + o + 4, x1.x > 0.f ? e0[2] : 0.f, x1.y > 0.f ? o1[2] : 0.f, x1.z > 0.f ? e0[3] : 0.f, x1.w > 0.f ? o1[3] : 0.f);
            }
        }
    }
}

// ---- pool block: max-pool (argmax recomputed from the raw tile) + avg-pool (+ identity skip at stride 1) ---------------
// acc[oy][j] += sum over the 3x3 windows o that contain input pixel (oy, j) of parity plane (A, B):
//               dta[o]  +  (code[o] == tap of this pixel inside o ? dtm[o] : 0)
// dta = avg-pool dz / window count, dtm = max-pool dz, code = argmax tap (ky*3 + kx, as a float) of window o; all three are
// [rows][P] planes over the row-haloed output tile (same tap enumeration as dw_plane_bwd).
template <int S, int PR, int A, int B, int P>
PCD_HD void pool_plane_bwd(const float* PCD_RESTRICT dta, const float* PCD_RESTRICT dtm, const float* PCD_RESTRICT cod, float (&acc)[PR][4]) {
    using G = TapGeo<3, 1, S>;
    if constexpr (G::any(A) && G::any(B)) {
        constexpr int RMIN = -G::pmax(A), RMAX = -G::pmin(A) + PR - 1;
        constexpr int LO = seg_lo(-G::pmax(B)), HI = seg_hi(3 - G::pmin(B));
#pragma unroll
        for (int rr = RMIN; rr <= RMAX; ++rr) {
            float va[HI - LO + 1], vm[HI - LO + 1], vc[HI - LO + 1];
            load_seg<LO, HI>(dta + rr * P, va);
            load_seg<LO, HI>(dtm + rr * P, vm);
            load_seg<LO, HI>(cod + rr * P, vc);
#pragma unroll
            for (int oy = 0; oy < PR; ++oy) {
                const int ky = G::find(A, oy - rr);
                if (ky < 0) continue;
#pragma unroll
                for (int kx = 0; kx < 3; ++kx) {
                    if (G::par(kx) != B) continue;
                    const int g = -G::pos(kx) - LO;
                    const float tap = (float)(ky * 3 + kx);
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[oy][j] += va[j + g] + (vc[j + g] == tap ? vm[j + g] : 0.f);
                }
            }
        }
    }
}

template <int C, int S, int W>
struct V4GeoPool {
    using GB = V4GeoBwd<C, S, W>;
    static constexpr int TH = GB::TH, P = GB::P, WS4 = W / 4, NRB = TH / 4;
    static constexpr int CP = C / 2;                          // channels per pass: keeps the pool block below the conv block's smem
    static constexpr int IH = S * TH + 8, XW = S * W + 8;     // raw input tile: rows S*oy0-4 .., columns -4 ..
    static constexpr int RH = TH + 2;                         // output rows oy0-1 .. oy0+TH
    static constexpr int X_FLOATS = CP * IH * XW, PL_FLOATS = CP * RH * P;
    static constexpr size_t SMEM_FLOATS = (size_t)X_FLOATS + 3 * PL_FLOATS + 2 * 4 * C + 16;
};

template <int C, int S, int W>
PCD_HD void bwdA4_pool_block(const EdgeBwdArgs& a, const EdgeG& e, int tile, int n, float* smem) {
    using G = V4GeoPool<C, S, W>;
    constexpr int TH = G::TH, RH = G::RH, P = G::P, IH = G::IH, XW = G::XW, CP = G::CP, WS4 = G::WS4, NRB = G::NRB;
    float* XIN = smem;                              // [CP][IH][XW] raw input
    float* DTA = XIN + G::X_FLOATS;                 // [CP][RH][P] avg-pool dz / window count, data columns at [4, 4+W)
    float* DTM = DTA + G::PL_FLOATS;                // max-pool dz
    float* COD = DTM + G::PL_FLOATS;                // argmax tap of every window, as a float
    float* COEF = COD + G::PL_FLOATS;               // [max | avg][4C]
    const int oy0 = tile * TH;
    const long long HW = (long long)a.Ho * W, nslot = (long long)a.B * C * HW;
    const double cnt = (double)a.B * a.Ho * W;
    const float beta = e.beta ? e.beta[0] : 1.f;
    const long long xcs = (long long)a.Hs * a.Ws;
    PCD_FOR(i, 2 * C) {
        const int k = i / C, j = i - k * C, bn = k ? bn_p2() : bn_p1();
        edge_coef(COEF + k * 4 * C, j, dz_consts(e.stats, C, bn, j, cnt, a.eps, e.bstats[bs_s0() * C + j], e.bstats[bs_sz(bn) * C + j],
                                                 beta * e.alpha[k ? 2 : 1]));
    }
    const float idc = beta * e.alpha[3];
    for (int c0 = 0; c0 < C; c0 += CP) {
        const float* xi = e.x + (long long)n * e.x_ns + c0 * xcs;
        PCD_SYNC();                                 // the previous pass's readers are done (first pass: COEF is complete)
        for_tasks<CP * IH * (XW / 4)>([&](int i) {
            const int c4 = i % (XW / 4), r = (i / (XW / 4)) % IH, ch = i / ((XW / 4) * IH);
            const int gy = S * oy0 - 4 + r, gx = 4 * c4 - 4;
            const bool ok = gy >= 0 && gy < a.Hs && gx >= 0 && gx < a.Ws;
            cp16(XIN + (size_t)i * 4, ok ? xi + ch * xcs + (long long)gy * a.Ws + gx : xi, ok);
        });
        for_tasks<CP * RH * 2>([&](int i) {         // column halos of the three planes
            const int side = i & 1, row = i >> 1;
            const int o = row * P + (side ? 4 + W : 0);
            st4(DTA + o, 0.f, 0.f, 0.f, 0.f);
            st4(DTM + o, 0.f, 0.f, 0.f, 0.f);
            st4(COD + o, -1.f, -1.f, -1.f, -1.f);
        });
        cp16_wait();
        PCD_SYNC();
        const float* dn_img = e.dn + (long long)n * e.dn_ns + (long long)(4 * c0) * HW;
        const float* Z1 = e.saved + slot_p1() * nslot + ((long long)n * C + c0) * HW;
        const float* Z2 = e.saved + slot_p2() * nslot + ((long long)n * C + c0) * HW;
        // ---- dz of both pools and the max-pool argmax tap of every window whose rows touch the tile ---------------------
        for_tasks<CP * RH * WS4>([&](int i) {
            const int strip = i % WS4, r = (i / WS4) % RH, ch = i / (WS4 * RH);
            const int oy = oy0 + r - 1, ox = strip * 4;
            float dm[4] = {0.f, 0.f, 0.f, 0.f}, da[4] = {0.f, 0.f, 0.f, 0.f}, cd[4] = {-1.f, -1.f, -1.f, -1.f};
            if (oy >= 0 && oy < a.Ho) {
                const long long o = (long long)oy * W + ox;
                const F4 h4 = ld4(dn_img + (long long)(4 * ch) * HW + o);
                const F4 z1 = ld4(Z1 + (long long)ch * HW + o), z2 = ld4(Z2 + (long long)ch * HW + o);
                const float h[4] = {h4.x, h4.y, h4.z, h4.w}, zm[4] = {z1.x, z1.y, z1.z, z1.w}, za[4] = {z2.x, z2.y, z2.z, z2.w};
                const float* cm = COEF + 4 * (c0 + ch);
                const float* ca = COEF + 4 * C + 4 * (c0 + ch);
                const bool rok[3] = {oy > 0, true, (S == 2) || (oy < a.Ho - 1)};
                const int nrow = (int)rok[0] + 1 + (int)rok[2];
                // the three input rows of the windows: columns S*ox - 1 .. S*(ox + 3) + 1
                constexpr int NV = 3 * S + 3;
                float xv[3][NV];
#pragma unroll
                for (int dy = 0; dy < 3; ++dy) {
                    const float* rowp = XIN + (ch * IH + S * (r - 1) + dy - 1 + 4) * XW + 4 + S * ox;
                    if constexpr (S == 1) load_seg<-1, 4>(rowp, xv[dy]);
                    else {
                        float t[12];
                        load_seg<-4, 7>(rowp, t);         // 2*ox - 4 .. 2*ox + 7
#pragma unroll
                        for (int k = 0; k < NV; ++k) xv[dy][k] = t[k + 3];
                    }
                }
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    const bool left = (ox + t == 0), right = (S == 1) && (ox + t == W - 1);
                    const int ncol = 3 - (left ? 1 : 0) - (right ? 1 : 0);
                    dm[t] = cm[0] * (h[t] - cm[1] - (zm[t] - cm[2]) * cm[3]);
                    da[t] = ca[0] * (h[t] - ca[1] - (za[t] - ca[2]) * ca[3]) / (float)(nrow * ncol);
                    float m = -INFINITY, best = -1.f;      // first maximum in scan order (ATen's max_pool2d rule)
#pragma unroll
                    for (int dy = 0; dy < 3; ++dy)
#pragma unroll
                        for (int dx = 0; dx < 3; ++dx) {
                            bool ok = rok[dy];
                            if (dx == 0) ok = ok && !left;
                            if (dx == 2) ok = ok && !right;
                            const float v = xv[dy][S * t + dx];
                            const bool take = ok && (v > m || best < 0.f);
                            m = take ? v : m;
                            best = take ? (float)(dy * 3 + dx) : best;
                        }
                    cd[t] = best;
                }
            }
            const int o = (ch * RH + r) * P + 4 + ox;
            st4(DTM + o, dm[0], dm[1], dm[2], dm[3]);
            st4(DTA + o, da[0], da[1], da[2], da[3]);
            st4(COD + o, cd[0], cd[1], cd[2], cd[3]);
        });
        PCD_SYNC();
        // ---- gather over the windows that contain each input pixel: one 4x4 patch (stride 2: of both column parities) ---
        float* pd_img = e.pd + (long long)a.B * C * a.Hs * a.Ws + ((long long)n * C + c0) * a.Hs * a.Ws;      // slot 1
        constexpr int NPAR = (S == 1) ? 1 : 2;
        for_tasks<NPAR * CP * NRB * WS4>([&](int t) {
            const int strip = t % WS4, rb = (t / WS4) % NRB, ch = (t / (WS4 * NRB)) % CP, par = t / (WS4 * NRB * CP);
            const int py = rb * 4, px = strip * 4;
            const int o = (ch * RH + py + 1) * P + 4 + px;
            float acc0[4][4], acc1[4][4];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) { acc0[i][j] = 0.f; acc1[i][j] = 0.f; }
            if (S == 1) {
                pool_plane_bwd<1, 4, 0, 0, P>(DTA + o, DTM + o, COD + o, acc0);
#pragma unroll
                for (int i = 0; i < 4; ++i) {       // identity skip: d xs += beta * w3 * dN[:, 0::4]
                    const long long g = ((long long)ch * a.Hs + oy0 + py + i) * W + px;
                    const F4 h = ld4(dn_img + (long long)(4 * ch) * HW + (long long)(oy0 + py + i) * W + px);
                    st4(pd_img + g, fmaf(idc, h.x, acc0[i][0]), fmaf(idc, h.y, acc0[i][1]), fmaf(idc, h.z, acc0[i][2]), fmaf(idc, h.w, acc0[i][3]));
                }
            } else {
                if (par == 0) {
                    pool_plane_bwd<2, 4, 0, 0, P>(DTA + o, DTM + o, COD + o, acc0);
                    pool_plane_bwd<2, 4, 0, 1, P>(DTA + o, DTM + o, COD + o, acc1);
                } else {
                    pool_plane_bwd<2, 4, 1, 0, P>(DTA + o, DTM + o, COD + o, acc0);
                    pool_plane_bwd<2, 4, 1, 1, P>(DTA + o, DTM + o, COD + o, acc1);
                }
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const long long g = ((long long)ch * a.Hs + 2 * (oy0 + py + i) + par) * (2 * W) + 2 * px;
                    st4(pd_img + g, acc0[i][0], acc1[i][0], acc0[i][1], acc1[i][1]);
                    st4(pd_img + g + 4, acc0[i][2], acc1[i][2], acc0[i][3], acc1[i][3]);
                }
            }
        });
    }
}

template <int C, int S, int W>
PCD_HD void bwdA4_body(const EdgeBwdArgs& a, int tile, int n, int z, float* smem) {
    const EdgeG& e = a.e[z >> 1];
    if ((z & 1) == 0) bwdA4_conv_block<C, S, W>(a, e, tile, n, smem);
    else bwdA4_pool_block<C, S, W>(a, e, tile, n, smem);
}

}  // namespace pcd
