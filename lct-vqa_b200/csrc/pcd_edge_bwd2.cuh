// pcd_edge_bwd2.cuh — backward kernels of the MixedOp edges (model_search.py:44-58) for the production geometries:
// the stage-B data kernel and the weight-gradient kernel (the stage-A data kernel is pcd_edge_bwd4.cuh).  Compile-time
// tile <TH, TW> with TW == the full output width (so the column halo of every tile is zero padding) and full tiles.
// Other shapes run the generic kernels of pcd_edge.cuh.
//
// Every depthwise->pointwise unit's backward is split into two independent jobs:
//   data  job : dz on the row-haloed tile -> dt = Wpw^T dz -> flipped depthwise correlation -> grad of the unit input
//   wgrad job : dz, dt on the tile centre only + the unit's input tile and its saved depthwise output
//               -> dW(pointwise), dW(depthwise)       (deferred: one launch per cell covers every edge)
// Jobs per block (blockIdx.z):  stage B data: B3 | B5          wgrad: A3 | B3 | A5 | B5 | D3 | D5 | [FR]
// The building blocks below (dz_rows, dz_stage / dz_finish, dt_rows, zero_col_halo, edge_coef) serve pcd_edge_bwd4.cuh too.
#pragma once
#include "pcd_edge.cuh"

namespace pcd {

// ---- shared building blocks -----------------------------------------------------------------------------
// DZ[co][r][x] = BN-backward(dy, z) for image rows oyf + r (zero outside the image); full-width rows.
template <int C, int RH, int TW>
PCD_HD void dz_rows(float* DZ, const float* PCD_RESTRICT dy_img, long long dy_cs, int dy_chm,
                    const float* PCD_RESTRICT z_img, long long HW, const float* COEF, int oyf, int Ho) {
    constexpr int W4 = TW / 4;
    for_tasks<C * RH * W4>([&](int i) {
        const int x4 = i % W4, r = (i / W4) % RH, co = i / (W4 * RH);
        const int oy = oyf + r;
        float o[4] = {0.f, 0.f, 0.f, 0.f};
        if (oy >= 0 && oy < Ho) {
            const F4 dy = ld4(dy_img + (long long)(co * dy_chm) * dy_cs + (long long)oy * TW + 4 * x4);
            const F4 zz = ld4(z_img + (long long)co * HW + (long long)oy * TW + 4 * x4);
            const float c0 = COEF[4 * co], ca = COEF[4 * co + 1], cm = COEF[4 * co + 2], c1 = COEF[4 * co + 3];
            o[0] = c0 * (dy.x - ca - (zz.x - cm) * c1);
            o[1] = c0 * (dy.y - ca - (zz.y - cm) * c1);
            o[2] = c0 * (dy.z - ca - (zz.z - cm) * c1);
            o[3] = c0 * (dy.w - ca - (zz.w - cm) * c1);
        }
        st4(DZ + (co * RH + r) * TW + 4 * x4, o[0], o[1], o[2], o[3]);
    });
}

// the same in two steps: raw dy -> DZ and raw z -> ZR with cp.async (dz_stage: no registers, needs no coefficient, so it
// can be issued before the BN constants are even computed), then DZ = BN-backward(DZ, ZR) in place (dz_finish)
template <int C, int RH, int TW>
PCD_HD void dz_stage(float* DZ, float* ZR, const float* PCD_RESTRICT dy_img, long long dy_cs, int dy_chm,
                     const float* PCD_RESTRICT z_img, long long HW, int oyf, int Ho) {
    constexpr int W4 = TW / 4;
    for_tasks<C * RH * W4>([&](int i) {
        const int x4 = i % W4, r = (i / W4) % RH, co = i / (W4 * RH);
        const int oy = oyf + r;
        const bool ok = oy >= 0 && oy < Ho;
        const long long off = ok ? (long long)oy * TW + 4 * x4 : 0;
        cp16(DZ + (size_t)i * 4, dy_img + (long long)(co * dy_chm) * dy_cs + off, ok);
        cp16(ZR + (size_t)i * 4, z_img + (long long)co * HW + off, ok);
    });
}
template <int C, int RH, int TW>
PCD_HD void dz_finish(float* DZ, const float* ZR, const float* COEF, int oyf, int Ho) {
    constexpr int W4 = TW / 4;
    for_tasks<C * RH * W4>([&](int i) {
        const int r = (i / W4) % RH, co = i / (W4 * RH);
        const int oy = oyf + r;
        if (oy >= 0 && oy < Ho) {           // rows outside the image stay the zeros the copy wrote
            const F4 dy = ld4(DZ + (size_t)i * 4), zz = ld4(ZR + (size_t)i * 4);
            const float c0 = COEF[4 * co], ca = COEF[4 * co + 1], cm = COEF[4 * co + 2], c1 = COEF[4 * co + 3];
            st4(DZ + (size_t)i * 4, c0 * (dy.x - ca - (zz.x - cm) * c1), c0 * (dy.y - ca - (zz.y - cm) * c1),
                c0 * (dy.z - ca - (zz.z - cm) * c1), c0 * (dy.w - ca - (zz.w - cm) * c1));
        }
    });
}

// DT[ci][r][OFF + x] = sum_co WT[ci][co] * DZ[co][r][x]   (pitch P; rows outside the image are written as zeros)
template <int C, int RH, int TW, int P, int OFF>
PCD_HD void dt_rows(float* DT, const float* DZ, const float* WT, int oyf, int Ho) {
    constexpr int W4 = TW / 4, NT = (C / 4) * RH * W4;
    for_tasks_rolled<NT>([&](int i) {
        const int x4 = i % W4, r = (i / W4) % RH, cig = i / (W4 * RH);
        const int oy = oyf + r;
        float s[4][4];
#pragma unroll
        for (int q = 0; q < 4; ++q)
#pragma unroll
            for (int t = 0; t < 4; ++t) s[q][t] = 0.f;
        if (oy >= 0 && oy < Ho) {
#pragma unroll
            for (int c4 = 0; c4 < C / 4; ++c4) {
                F4 d[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) d[k] = ld4(DZ + ((c4 * 4 + k) * RH + r) * TW + 4 * x4);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const F4 w = ld4(WT + (cig * 4 + q) * C + c4 * 4);
                    const float wk[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        s[q][0] = fmaf(wk[k], d[k].x, s[q][0]);
                        s[q][1] = fmaf(wk[k], d[k].y, s[q][1]);
                        s[q][2] = fmaf(wk[k], d[k].z, s[q][2]);
                        s[q][3] = fmaf(wk[k], d[k].w, s[q][3]);
                    }
                }
            }
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) st4(DT + ((cig * 4 + q) * RH + r) * P + OFF + 4 * x4, s[q][0], s[q][1], s[q][2], s[q][3]);
    });
}

// zero the 4-float column halos of a [NPL][P] array of rows whose data sits at [4, 4 + TW)
template <int NROWS, int TW, int P>
PCD_HD void zero_col_halo(float* T) {
    for_tasks<NROWS * 2>([&](int i) {
        const int row = i >> 1, side = i & 1;
        st4(T + row * P + (side ? 4 + TW : 0), 0.f, 0.f, 0.f, 0.f);
    });
}

PCD_HD void edge_coef(float* COEF, int j, const DzC& d) {
    COEF[4 * j] = d.c0; COEF[4 * j + 1] = d.a; COEF[4 * j + 2] = d.m; COEF[4 * j + 3] = d.c1;
}

// ======================================================================================================
// stage B, data job: grad of relu(bn(zA)) (masked) = GA, and its two sums
// ======================================================================================================
template <int C, int TH, int TW>
PCD_HOSTDEV size_t bwdB2_smem_floats() {
    return (size_t)C * (TH + 4) * TW + (size_t)C * (TH + 4) * (TW + 8) + 6 * C + C * C + 2 * C * 8 + 64;
}

template <int C, int KS, int TH, int TW>
PCD_HD void bwdB2_data_job(const EdgeBwdArgs& a, const EdgeG& e, const Geo& g, int half, float* smem) {
    constexpr int PAD = (KS - 1) / 2, RH = TH + 2 * PAD, IW = TW + 8, PW4 = TW / 4, NPATCH = (TH / 4) * PW4;
    const int S = a.S;
    float* DZ = smem;                               // [C][TH+4][TW]   (RH rows used)
    float* DT = DZ + C * (TH + 4) * TW;             // [C][TH+4][IW]
    float* COEF = DT + C * (TH + 4) * IW;           // 4C
    float* BNA = COEF + 4 * C;                      // 2C
    float* WT = BNA + 2 * C;                        // C*C
    float* P2 = WT + C * C;                         // 2*C*8
    float* Pga = DZ;                                // [2][C*NPATCH] (DZ is dead after dt_rows)
    const int uA = half ? 2 : 0, uB = uA + 1;
    const long long nslot = (long long)a.B * C * a.Ho * a.Wo, HW = (long long)a.Ho * a.Wo;
    const double cnt = (double)a.B * a.Ho * a.Wo;
    const float beta = e.beta ? e.beta[0] : 1.f;
    const float kappa = beta * e.alpha[half ? 5 : 4];
    const float* w_dw = e.par + edge_dw_off(C, S, uB);
    const float* w_pw = e.par + edge_pw_off(C, S, uB);
    // the raw dN / zB rows start their way into shared memory (DZ / the DT area) before the BN constants are derived
    const float* zA = e.saved + slot_z(uA) * nslot + (long long)g.n * C * HW;
    const float* zB = e.saved + slot_z(uB) * nslot + (long long)g.n * C * HW;
    dz_stage<C, RH, TW>(DZ, DT, e.dn + (long long)g.n * e.dn_ns, HW, 4, zB, HW, g.oy0 - PAD, a.Ho);
    PCD_FOR(j, C) {
        const int bnB = bn_unit(S, uB);
        edge_coef(COEF, j, dz_consts(e.stats, C, bnB, j, cnt, a.eps, e.bstats[bs_s0() * C + j], e.bstats[bs_sz(bnB) * C + j], kappa));
        BnC b = bn_consts(e.stats, C, bn_unit(S, uA), j, cnt, a.eps);
        BNA[2 * j] = b.mean; BNA[2 * j + 1] = b.rstd;
    }
    PCD_FOR(i, C * C) WT[(i % C) * C + i / C] = w_pw[i];
    cp16_wait();
    PCD_SYNC();
    dz_finish<C, RH, TW>(DZ, DT, COEF, g.oy0 - PAD, a.Ho);
    PCD_SYNC();                                     // raw zB consumed: DT can be rewritten
    zero_col_halo<C * RH, TW, IW>(DT);
    dt_rows<C, RH, TW, IW, 4>(DT, DZ, WT, g.oy0 - PAD, a.Ho);
    PCD_SYNC();
    float* ga = e.ga + half * nslot;
    for_tasks_rolled<C * NPATCH>([&](int task) {
        const int ch = task / NPATCH, patch = task - ch * NPATCH;
        const int py = (patch / PW4) * 4, px = (patch % PW4) * 4;
        F4 za[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) za[i] = ld4(zA + (long long)ch * HW + (long long)(g.oy0 + py + i) * TW + px);
        float acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
        dw_patch<KS, 1, 1, true, false>(DT + ch * RH * IW, IW, py, px, w_dw + ch * KS * KS, acc);
        const float m = BNA[2 * ch], r = BNA[2 * ch + 1];
        float s = 0.f, sz = 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float zv[4] = {za[i].x, za[i].y, za[i].z, za[i].w};
            float o[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                o[j] = ((zv[j] - m) * r > 0.f) ? acc[i][j] : 0.f;
                s += o[j];
                sz = fmaf(o[j], zv[j], sz);
            }
            st4(ga + ((long long)(g.n * C + ch) * a.Ho + g.oy0 + py + i) * TW + px, o[0], o[1], o[2], o[3]);
        }
        Pga[task] = s;
        Pga[C * NPATCH + task] = sz;
    });
    reduce_columns<8>(Pga, P2, 2, C, NPATCH, C * NPATCH, [&](int ch, int k, float v) {
        pcd_atomic_add(e.bstats + (bs_ga(half) + k) * C + ch, (double)v);
    });
}

template <int C, int TH, int TW>
PCD_HD void bwdB2_body(const EdgeBwdArgs& a, int bx, int n, int z, float* smem) {
    Geo g;
    g.n = n; g.TH = TH; g.TW = TW; g.Ho = a.Ho; g.Wo = a.Wo;
    g.oy0 = bx * TH; g.ox0 = 0;
    if ((z & 1) == 0) bwdB2_data_job<C, 3, TH, TW>(a, a.e[z >> 1], g, 0, smem);
    else bwdB2_data_job<C, 5, TH, TW>(a, a.e[z >> 1], g, 1, smem);
}

// ======================================================================================================
// weight-gradient jobs (all six depthwise->pointwise units of an edge, + FactorizedReduce)
// ======================================================================================================
template <int C, int S, int TH, int TW>
PCD_HOSTDEV size_t wgrad2_smem_floats() {
    constexpr size_t npix = (size_t)TH * TW;
    constexpr size_t in = (size_t)C * (S * TH + 8) * (S * TW + 4) + 4;
    return 3 * C * npix + in + 16 * 256 + (size_t)25 * C * 4 + 16 * 16 * 4 + 6 * C + C * C + 64;
}

// unit with input stride SI (1 for the second halves), kernel KS, dilation DIL; BNIN: the unit input is relu(bn(zA)).
// The input tile keeps only the LEFT 4-float column halo: rows are full image width, so the right halo of row r is
// the (zero) left halo of row r + 1 (pitch = width + 4; 4 zero floats follow the last row).
// One block walks every tile of images [n0, n1): the weight-grad partial sums stay in registers across tiles and are
// reduced over the block (and added atomically) once.
template <int C, int SI, int KS, int DIL, int TH, int TW, bool BNIN>
PCD_HD void wgrad2_unit_job(const EdgeBwdArgs& a, const EdgeG& e, int n0, int n1, int u, float* smem) {
    constexpr int PAD = DIL * (KS - 1) / 2, NPIX = TH * TW, PW4 = TW / 4, NPATCH = (TH / 4) * PW4;
    constexpr int IH = SI * TH + 8, XW = SI * TW + 4;
    constexpr int NOG = (C / 4) * (C / 4), NTP = 256, NSL = NTP / NOG;     // pointwise: 4x4 outputs x pixel slices
    static_assert((NPIX / 4) % NSL == 0, "pointwise slices");
    static_assert(C * NPATCH <= kThreads && NTP <= kThreads, "one task per thread");
    const int S = a.S;
    float* DZ = smem;                       // [C][NPIX]
    float* T = DZ + C * NPIX;               // [C][NPIX]   saved depthwise output
    float* DT = T + C * NPIX;               // [C][NPIX]
    float* IN = DT + C * NPIX;              // [C][IH][XW] (+4) unit input: row halo 4, left column halo 4
    float* Ppw = IN + (size_t)C * (S * TH + 8) * (S * TW + 4) + 4;  // [16][256]  (IN sized for the stride-S units)
    float* P2 = Ppw + 16 * 256;             // 25*C*4 + 16*NOG*4
    float* COEF = P2 + 25 * C * 4 + 16 * 16 * 4;
    float* BNA = COEF + 4 * C;
    float* WT = BNA + 2 * C;
    float* Pdw = DZ;                        // [KS*KS][C*NPATCH] (after the tile loop)
    const long long nslot = (long long)a.B * C * a.Ho * a.Wo, HW = (long long)a.Ho * a.Wo;
    const double cnt = (double)a.B * a.Ho * a.Wo;
    const float beta = e.beta ? e.beta[0] : 1.f;
    const float* w_pw = e.par + edge_pw_off(C, S, u);
    const bool isA = (u == 0 || u == 2);
    const int which = (u == 2) ? 1 : 0;
    PCD_FOR(j, C) {
        const int bn = bn_unit(S, u);
        if (isA)
            edge_coef(COEF, j, dz_consts(e.stats, C, bn, j, cnt, a.eps, e.bstats[bs_ga(which) * C + j],
                                         e.bstats[(bs_ga(which) + 1) * C + j], 1.f));
        else
            edge_coef(COEF, j, dz_consts(e.stats, C, bn, j, cnt, a.eps, e.bstats[bs_s0() * C + j], e.bstats[bs_sz(bn) * C + j],
                                         beta * e.alpha[u == 1 ? 4 : u == 3 ? 5 : u == 4 ? 6 : 7]));
        if (BNIN) {
            BnC b = bn_consts(e.stats, C, bn_unit(S, u - 1), j, cnt, a.eps);
            BNA[2 * j] = b.mean; BNA[2 * j + 1] = b.rstd;
        }
    }
    PCD_FOR(i, C * C) WT[(i % C) * C + i / C] = w_pw[i];
    PCD_FOR(i, 4) IN[(size_t)C * IH * XW + i] = 0.f;
    PCD_TSTATE(float, accp, [4][4]);
    PCD_TSTATE(float, accd, [KS * KS]);
    PCD_EACH(task) {
        auto& ap = PCD_TREF(accp, task);
        auto& ad = PCD_TREF(accd, task);
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int k = 0; k < 4; ++k) ap[i][k] = 0.f;
#pragma unroll
        for (int k = 0; k < KS * KS; ++k) ad[k] = 0.f;
    }
    const int H = BNIN ? a.Ho : a.Hs, W = BNIN ? a.Wo : a.Ws;
    const long long scs = (long long)H * W;
    const int tiles = a.Ho / TH;
    for (int n = n0; n < n1; ++n)
    for (int tile = 0; tile < tiles; ++tile) {
        const int oy0 = tile * TH;
        PCD_SYNC();                               // constants ready / previous tile's readers are done
        // ---- tiles: unit input (haloed), saved depthwise output, dz ----------------------------------------
        // the input tile and the saved depthwise output go global -> shared without passing through registers (cp.async),
        // like the raw dy / z rows (staged in DZ / DT): every load of the tile is in flight at once; the input's ReLU / BN+ReLU
        // and the BN-backward that turns (dy, z) into dz are applied in place afterwards
        const float* src = BNIN ? e.saved + slot_z(u - 1) * nslot + (long long)n * C * HW : e.x + (long long)n * e.x_ns;
        for_tasks<C * IH * (XW / 4)>([&](int i) {
            const int c4 = i % (XW / 4), r = (i / (XW / 4)) % IH, ch = i / ((XW / 4) * IH);
            const int gy = SI * oy0 - 4 + r, gx = 4 * c4 - 4;
            const bool ok = gy >= 0 && gy < H && gx >= 0 && gx < W;
            cp16(IN + (size_t)i * 4, ok ? src + ch * scs + (long long)gy * W + gx : src, ok);
        });
        const float* tsl = e.saved + slot_t(u) * nslot + (long long)n * C * HW + (long long)oy0 * TW;
        for_tasks<C * NPIX / 4>([&](int i) {
            const int p4 = i % (NPIX / 4), ch = i / (NPIX / 4);
            cp16(T + (size_t)i * 4, tsl + (long long)ch * HW + 4 * p4, true);
        });
        const float* dy_img = isA ? e.ga + which * nslot + (long long)n * C * HW : e.dn + (long long)n * e.dn_ns;
        dz_stage<C, TH, TW>(DZ, DT, dy_img, HW, isA ? 1 : 4, e.saved + slot_z(u) * nslot + (long long)n * C * HW, HW, oy0, a.Ho);
        cp16_wait();
        PCD_SYNC();
        dz_finish<C, TH, TW>(DZ, DT, COEF, oy0, a.Ho);
        for_tasks<C * IH * (XW / 4)>([&](int i) {
            const int c4 = i % (XW / 4), r = (i / (XW / 4)) % IH, ch = i / ((XW / 4) * IH);
            const int gy = SI * oy0 - 4 + r, gx = 4 * c4 - 4;
            if (gy >= 0 && gy < H && gx >= 0 && gx < W) {
                F4 v = ld4(IN + (size_t)i * 4);
                if (BNIN) {
                    const float m = BNA[2 * ch], r_ = BNA[2 * ch + 1];
                    v.x = relu((v.x - m) * r_); v.y = relu((v.y - m) * r_); v.z = relu((v.z - m) * r_); v.w = relu((v.w - m) * r_);
                } else {
                    v.x = relu(v.x); v.y = relu(v.y); v.z = relu(v.z); v.w = relu(v.w);
                }
                *reinterpret_cast<F4*>(IN + (size_t)i * 4) = v;
            }
        });
        PCD_SYNC();                               // dz complete, the raw z in DT consumed
        // ---- dt on the centre; pointwise weight-grad partials ---------------------------------------------------
        dt_rows<C, TH, TW, TW, 0>(DT, DZ, WT, oy0, a.Ho);
        PCD_EACH(task) {
            auto& acc = PCD_TREF(accp, task);
            const int og = task / NSL, sl = task - og * NSL;
            const int co0 = (og / (C / 4)) * 4, ci0 = (og % (C / 4)) * 4;
#pragma unroll 2
            for (int st = sl; st < NPIX / 4; st += NSL) {
                F4 tv[4], dz[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    tv[k] = ld4(T + (ci0 + k) * NPIX + st * 4);
                    dz[k] = ld4(DZ + (co0 + k) * NPIX + st * 4);
                }
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        acc[i][k] = fmaf(dz[i].x, tv[k].x, fmaf(dz[i].y, tv[k].y, fmaf(dz[i].z, tv[k].z, fmaf(dz[i].w, tv[k].w, acc[i][k]))));
            }
        }
        PCD_SYNC();
        // ---- depthwise weight-grad partials ---------------------------------------------------------------------------
        PCD_EACH(task) {
            if (task < C * NPATCH) {
                auto& acc = PCD_TREF(accd, task);
                const int ch = task / NPATCH, patch = task - ch * NPATCH;
                const int py = (patch / PW4) * 4, px = (patch % PW4) * 4;
                float dt[4][4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const F4 v = ld4(DT + (ch * TH + py + i) * TW + px);
                    dt[i][0] = v.x; dt[i][1] = v.y; dt[i][2] = v.z; dt[i][3] = v.w;
                }
                dw_wgrad_patch<KS, DIL, SI, false>(IN + ch * IH * XW, XW, SI * py - PAD + 4, SI * px, dt, acc);
            }
        }
    }
    PCD_SYNC();
    // ---- block reductions (P aliases DZ | T), 4 partials per output, then atomics ---------------------------------------
    PCD_EACH(task) {
        auto& ap = PCD_TREF(accp, task);
        auto& ad = PCD_TREF(accd, task);
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int k = 0; k < 4; ++k) Ppw[(i * 4 + k) * NTP + task] = ap[i][k];
        if (task < C * NPATCH) {
#pragma unroll
            for (int k = 0; k < KS * KS; ++k) Pdw[k * (C * NPATCH) + task] = ad[k];
        }
    }
    PCD_SYNC();
    constexpr int NP = 4, NDW = KS * KS * C, NPW = 16 * NOG;
    float* P2dw = P2;
    float* P2pw = P2 + 25 * C * 4;
    for_tasks_rolled<(NDW + NPW) * NP>([&](int q) {
        if (q < NDW * NP) {
            const int part = q % NP, kg = q / NP, k = kg / C, ch = kg - k * C;
            float s = 0.f;
            for (int t = part; t < NPATCH; t += NP) s += Pdw[k * (C * NPATCH) + ch * NPATCH + t];
            P2dw[q] = s;
        } else {
            const int q2 = q - NDW * NP;
            const int part = q2 % NP, kg = q2 / NP, k = kg / NOG, og = kg - k * NOG;
            float s = 0.f;
            for (int t = part; t < NSL; t += NP) s += Ppw[k * NTP + og * NSL + t];
            P2pw[q2] = s;
        }
    });
    PCD_SYNC();
    float* gdw = e.gpar + edge_dw_off(C, S, u);
    float* gpw = e.gpar + edge_pw_off(C, S, u);
    for_tasks_rolled<NDW + NPW>([&](int kg) {
        if (kg < NDW) {
            const int k = kg / C, ch = kg - k * C;
            pcd_atomic_add(gdw + ch * KS * KS + k, (P2dw[kg * NP] + P2dw[kg * NP + 1]) + (P2dw[kg * NP + 2] + P2dw[kg * NP + 3]));
        } else {
            const int kg2 = kg - NDW, k = kg2 / NOG, og = kg2 - k * NOG;
            const int co = (og / (C / 4)) * 4 + (k >> 2), ci = (og % (C / 4)) * 4 + (k & 3);
            pcd_atomic_add(gpw + co * C + ci, (P2pw[kg2 * NP] + P2pw[kg2 * NP + 1]) + (P2pw[kg2 * NP + 2] + P2pw[kg2 * NP + 3]));
        }
    });
}

// FactorizedReduce weight grads: dW_fr[co][ci] += sum_p dz[co][p] * relu(x[ci][2p + off(co)])
template <int C, int TH, int TW>
PCD_HD void wgrad2_fr_job(const EdgeBwdArgs& a, const EdgeG& e, const Geo& g, float* smem) {
    constexpr int NPIX = TH * TW, NOG = (C / 4) * (C / 4), NSL = 256 / NOG;
    static_assert((NPIX / 4) % NSL == 0, "FR slices");
    float* DZ = smem;                       // [C][NPIX]
    float* R = DZ + C * NPIX;               // [C][NPIX]  relu(x) at the sampling grid of each input channel's ... (2 grids)
    float* R1 = R + C * NPIX;               // second grid
    float* P = R1 + C * NPIX;               // [16][256]  (fits: IN region of the unit jobs is larger)
    float* P2 = P + 16 * 256;
    float* COEF = P2 + 16 * 16 * 4;
    const long long nslot = (long long)a.B * C * a.Ho * a.Wo, HW = (long long)a.Ho * a.Wo;
    const double cnt = (double)a.B * a.Ho * a.Wo;
    const float beta = e.beta ? e.beta[0] : 1.f;
    PCD_FOR(j, C) {
        edge_coef(COEF, j, dz_consts(e.stats, C, bn_f(), j, cnt, a.eps, e.bstats[bs_s0() * C + j], e.bstats[bs_sz(bn_f()) * C + j],
                                     beta * e.alpha[3]));
    }
    PCD_SYNC();
    dz_rows<C, TH, TW>(DZ, e.dn + (long long)g.n * e.dn_ns, HW, 4, e.saved + slot_f() * nslot + (long long)g.n * C * HW, HW, COEF,
                       g.oy0, a.Ho);
    const float* xi = e.x + (long long)g.n * e.x_ns;
    const long long xcs = (long long)a.Hs * a.Ws;
    for_tasks<C * NPIX / 4>([&](int i) {
        const int x4 = i % (TW / 4), r = (i / (TW / 4)) % TH, ch = i / ((TW / 4) * TH);
        const float* p0 = xi + ch * xcs + (long long)(2 * (g.oy0 + r)) * a.Ws + 8 * x4;
        const F4 a0 = ld4(p0), b0 = ld4(p0 + 4), a1 = ld4(p0 + a.Ws), b1 = ld4(p0 + a.Ws + 4);
        st4(R + (size_t)i * 4, relu(a0.x), relu(a0.z), relu(b0.x), relu(b0.z));
        st4(R1 + (size_t)i * 4, relu(a1.y), relu(a1.w), relu(b1.y), relu(b1.w));
    });
    PCD_SYNC();
    for_tasks_rolled<256>([&](int task) {
        const int og = task / NSL, sl = task - og * NSL;
        const int co0 = (og / (C / 4)) * 4, ci0 = (og % (C / 4)) * 4;
        const float* Rr = (co0 >= C / 2) ? R1 : R;
        float acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int k = 0; k < 4; ++k) acc[i][k] = 0.f;
#pragma unroll 2
        for (int st = sl; st < NPIX / 4; st += NSL) {
            F4 rv[4], dz[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                rv[k] = ld4(Rr + (ci0 + k) * NPIX + st * 4);
                dz[k] = ld4(DZ + (co0 + k) * NPIX + st * 4);
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    acc[i][k] = fmaf(dz[i].x, rv[k].x, fmaf(dz[i].y, rv[k].y, fmaf(dz[i].z, rv[k].z, fmaf(dz[i].w, rv[k].w, acc[i][k]))));
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int k = 0; k < 4; ++k) P[(i * 4 + k) * 256 + task] = acc[i][k];
    });
    reduce_columns<4>(P, P2, 16, NOG, NSL, 256, [&](int og, int k, float v) {
        const int co = (og / (C / 4)) * 4 + (k >> 2), ci = (og % (C / 4)) * 4 + (k & 3);
        pcd_atomic_add(e.gpar + co * C + ci, v);
    });
}

constexpr int kWgradImages = 4;      // images per weight-grad block

template <int C, int S, int TH, int TW>
PCD_HD void wgrad2_body(const EdgeBwdArgs& a, int bx, int by, int z, float* smem) {
    constexpr int NJ = 6 + (S == 2);
    const int ez = z / NJ, job = z - ez * NJ;
    const EdgeG& e = a.e[ez];
    const int n0 = by * kWgradImages, n1 = (n0 + kWgradImages < a.B) ? n0 + kWgradImages : a.B;
    (void)bx;
    if (job == 0) wgrad2_unit_job<C, S, 3, 1, TH, TW, false>(a, e, n0, n1, 0, smem);
    else if (job == 1) wgrad2_unit_job<C, 1, 3, 1, TH, TW, true>(a, e, n0, n1, 1, smem);
    else if (job == 2) wgrad2_unit_job<C, S, 5, 1, TH, TW, false>(a, e, n0, n1, 2, smem);
    else if (job == 3) wgrad2_unit_job<C, 1, 5, 1, TH, TW, true>(a, e, n0, n1, 3, smem);
    else if (job == 4) wgrad2_unit_job<C, S, 3, 2, TH, TW, false>(a, e, n0, n1, 4, smem);
    else if (job == 5) wgrad2_unit_job<C, S, 5, 2, TH, TW, false>(a, e, n0, n1, 5, smem);
    else if (S == 2) {
        for (int n = n0; n < n1; ++n)
            for (int tile = 0; tile < a.Ho / TH; ++tile) {
                Geo g;
                g.n = n; g.TH = TH; g.TW = TW; g.Ho = a.Ho; g.Wo = a.Wo;
                g.oy0 = tile * TH; g.ox0 = 0;
                PCD_SYNC();
                wgrad2_fr_job<C, TH, TW>(a, e, g, smem);
            }
    }
}

}  // namespace pcd
