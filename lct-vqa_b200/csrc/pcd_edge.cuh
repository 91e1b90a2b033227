// pcd_edge.cuh — forward and backward kernels of the MixedOp edges (model_search.py:44-58), v2.
//
// One thread block = one JOB on one output tile of one image of one edge:
//   forward  stage A jobs: A3 | A5 | D3 | D5 (depthwise->pointwise on relu(xs))  | pools (+FactorizedReduce)
//            stage B jobs: B3 | B5 (second half of the separable convs, BN+ReLU applied on load)
//   backward stage B jobs: B3 | B5  -> grad of the mid tensors (GA) + its sums + weight grads
//            stage A jobs: A3 | A5 | D3 | D5 | max-pool | avg-pool(+identity) | FactorizedReduce
//                          each writes its own partial d xs (summed, with the ReLU mask, by source_grad)
// Splitting by job instead of looping over the candidate ops inside a block multiplies the number of
// resident blocks (B=64 gives only 64..256 tiles per edge) and keeps shared memory per block small.
//
// These are the generic kernels (run-time tile, masked edges): they run every edge geometry except the five
// production edge shapes, which take the v4 forward (pcd_edge_v4.cuh), the stage-B backward and weight-gradient
// kernels of pcd_edge_bwd2.cuh and the v4 stage-A backward (pcd_edge_bwd4.cuh).  This file also holds the argument
// structs and the small building blocks those kernels share.
#pragma once
#include "pcd_common.cuh"

namespace pcd {

struct EdgeF {
    const float* x;        // source state (B, C, Hs, Ws)
    long long x_ns;        // its batch stride (floats)
    const float* par;      // edge parameter block
    float* saved;          // edge saved-activation slots
    double* stats;         // edge forward sums
};

struct PassArgs {
    int B, Hs, Ws, Ho, Wo, S;
    int TH, TW, tiles_x;
    float eps;
    int nedges;
    EdgeF e[kMaxEdgesPerLaunch];
};

struct Geo {
    int n, oy0, ox0, TH, TW, Ho, Wo;
};

PCD_HD long long out_index(const Geo& g, int C, int ch, int oy, int ox) {
    return (((long long)g.n * C + ch) * g.Ho + oy) * g.Wo + ox;
}

// store 4 consecutive pixels of row oy starting at ox (the part inside the image)
PCD_HD void store4(float* base, const Geo& g, int C, int ch, int oy, int ox, const float (&v)[4]) {
    float* p = base + out_index(g, C, ch, oy, ox);
    if (oy >= g.Ho) return;
    if (ox + 3 < g.Wo && (((uintptr_t)p) & 15) == 0) {
        F4 t = {v[0], v[1], v[2], v[3]};
        *reinterpret_cast<F4*>(p) = t;
    } else {
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (ox + j < g.Wo) p[j] = v[j];
    }
}

// 4 consecutive pixels of an image row; zero outside [0,W)
PCD_HD void load4(const float* row, int x, int W, float (&v)[4]) {
    if (x >= 0 && x + 3 < W && (((uintptr_t)(row + x)) & 15) == 0) {
        const F4 t = *reinterpret_cast<const F4*>(row + x);
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = (x + j >= 0 && x + j < W) ? row[x + j] : 0.f;
    }
}

// dst[C][rows][pitch] <- f(ch, src[ch*cs + gy*W + gx]) inside the image, 0 outside.  gx0 is a multiple of 4.
template <class F>
PCD_HD void load_tile(float* dst, const float* src, long long cs, int C, int rows, int pitch, int gy0, int gx0, int H,
                      int W, F f) {
    const int p4 = pitch >> 2;
    PCD_FOR(i, C * rows * p4) {
        const int c4 = i % p4, rr = i / p4, r = rr % rows, ch = rr / rows;
        const int gy = gy0 + r, gx = gx0 + 4 * c4;
        float v[4] = {0.f, 0.f, 0.f, 0.f};
        if (gy >= 0 && gy < H && gx + 3 >= 0 && gx < W) {
            load4(src + ch * cs + (long long)gy * W, gx, W, v);
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (gx + j >= 0 && gx + j < W) v[j] = f(ch, v[j]);
        }
        F4 t = {v[0], v[1], v[2], v[3]};
        *reinterpret_cast<F4*>(dst + (size_t)i * 4) = t;
    }
}

// f(i) for i in [0, N): strided over the block's threads, fully unrolled (N is a compile-time constant)
template <int N, class F>
PCD_HD void for_tasks(F f) {
#if PCD_CUDA
    constexpr int IT = (N + kThreads - 1) / kThreads;
#pragma unroll
    for (int it = 0; it < IT; ++it) {
        const int i = (int)threadIdx.x + it * kThreads;
        if (N % kThreads == 0 || i < N) f(i);
    }
#else
    for (int i = 0; i < N; ++i) f(i);
#endif
}
// same, rolled (heavy bodies)
template <int N, class F>
PCD_HD void for_tasks_rolled(F f) {
#if PCD_CUDA
#pragma unroll 1
    for (int i = (int)threadIdx.x; i < N; i += kThreads) f(i);
#else
    for (int i = 0; i < N; ++i) f(i);
#endif
}

PCD_HD F4 ld4(const float* p) { return *reinterpret_cast<const F4*>(p); }
PCD_HD void st4(float* p, float a, float b, float c, float d) {
    F4 t = {a, b, c, d};
    *reinterpret_cast<F4*>(p) = t;
}

// 16-byte global -> shared copy that does not occupy a register (cp.async; zero fill when !valid); cp16_wait() makes this
// thread's copies visible to it (a barrier then publishes them to the block)
PCD_HD void cp16(float* dst, const float* src, bool valid) {
#if PCD_CUDA
    const unsigned d = (unsigned)__cvta_generic_to_shared(dst);
    const int nbytes = valid ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(src), "r"(nbytes) : "memory");
#else
    if (valid) { dst[0] = src[0]; dst[1] = src[1]; dst[2] = src[2]; dst[3] = src[3]; }
    else { dst[0] = dst[1] = dst[2] = dst[3] = 0.f; }
#endif
}
PCD_HD void cp16_wait() {
#if PCD_CUDA
    asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory");
#endif
}

// ======================================================================================================
// forward
// ======================================================================================================
// One depthwise->pointwise unit on a shared-memory input tile [C][rows][pitch] (col halo 4, row halo halo_y).
template <int C, int KS, int DIL, int S, bool RELU>
PCD_HD void unit_forward(const float* tile, int rows, int pitch, int halo_y, const float* w_dw, const float* w_pw,
                         float* T, float* P, float* P2, float* WS, float* t_out, float* z_out, double* st, const Geo& g) {
    constexpr int PAD = DIL * (KS - 1) / 2;
    const int TH = g.TH, TW = g.TW, NPIX = TH * TW, NSTRIP = NPIX / 4, PW4 = TW / 4;
    const int NPATCH = (TH / 4) * PW4;
    PCD_FOR(i, C * C) WS[i] = w_pw[i];
    PCD_FOR(task, C * NPATCH) {
        const int ch = task / NPATCH, patch = task - ch * NPATCH;
        const int py = (patch / PW4) * 4, px = (patch % PW4) * 4;
        float acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
        dw_patch<KS, DIL, S, false, RELU>(tile + ch * rows * pitch, pitch, S * py - PAD + halo_y, S * px,
                                          w_dw + ch * KS * KS, acc);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            F4 v = {acc[i][0], acc[i][1], acc[i][2], acc[i][3]};
            *reinterpret_cast<F4*>(T + ch * NPIX + (py + i) * TW + px) = v;
            store4(t_out, g, C, ch, g.oy0 + py + i, g.ox0 + px, acc[i]);
        }
    }
    PCD_SYNC();
    constexpr int NCG = C / 4;
    PCD_FOR(task, NCG * NSTRIP) {
        const int cg = task / NSTRIP, strip = task - cg * NSTRIP;
        const int oyl = strip / PW4, oxl = (strip - oyl * PW4) * 4;
        float z[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) z[i][j] = 0.f;
#pragma unroll
        for (int c4 = 0; c4 < C / 4; ++c4) {
            F4 t[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) t[k] = *reinterpret_cast<const F4*>(T + (c4 * 4 + k) * NPIX + strip * 4);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const F4 w = *reinterpret_cast<const F4*>(WS + (cg * 4 + i) * C + c4 * 4);
                const float wk[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    z[i][0] = fmaf(wk[k], t[k].x, z[i][0]);
                    z[i][1] = fmaf(wk[k], t[k].y, z[i][1]);
                    z[i][2] = fmaf(wk[k], t[k].z, z[i][2]);
                    z[i][3] = fmaf(wk[k], t[k].w, z[i][3]);
                }
            }
        }
        const int oy = g.oy0 + oyl, ox = g.ox0 + oxl;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            store4(z_out, g, C, cg * 4 + i, oy, ox, z[i]);
            float s = 0.f, q = 0.f;
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (oy < g.Ho && ox + j < g.Wo) {
                    s += z[i][j];
                    q = fmaf(z[i][j], z[i][j], q);
                }
            P[(2 * i) * (NCG * NSTRIP) + task] = s;
            P[(2 * i + 1) * (NCG * NSTRIP) + task] = q;
        }
    }
    reduce_columns<(C == 16 ? 16 : 32)>(P, P2, 8, NCG, NSTRIP, NCG * NSTRIP, [&](int grp, int k, float v) {
        pcd_atomic_add(st + (k & 1) * C + grp * 4 + (k >> 1), (double)v);
    });
}

constexpr int kFwdAJobs = 5;

// partial sums per column in the block reductions of the forward kernels: 16 for C = 16 keeps the 16x16 stride-1 job at
// 75 KB (3 blocks/SM)
PCD_HOSTDEV int fwd_np(int C) { return C == 16 ? 16 : 32; }

PCD_HOSTDEV size_t fwdA_smem_floats(int C, int S, int TH, int TW) {
    const int IH = S * TH + 8, IW = S * TW + 8;
    return (size_t)C * IH * IW + (size_t)C * TH * TW * 2 + 4 * C * fwd_np(C) + C * C + 64;
}

template <int C, int S>
PCD_HD void fwdA_body(const PassArgs& a, int bx, int n, int z, float* smem) {
    const int TH = a.TH, TW = a.TW;
    const int ez = z / kFwdAJobs, job = z - ez * kFwdAJobs;
    const EdgeF& e = a.e[ez];
    Geo g;
    g.n = n; g.TH = TH; g.TW = TW; g.Ho = a.Ho; g.Wo = a.Wo;
    g.oy0 = (bx / a.tiles_x) * TH;
    g.ox0 = (bx % a.tiles_x) * TW;
    const int NPIX = TH * TW, NSTRIP = NPIX / 4, PW4 = TW / 4;
    const int IH = S * TH + 8, IW = S * TW + 8;
    float* XIN = smem;
    float* T = XIN + C * IH * IW;
    float* P = T + C * NPIX;
    float* P2 = P + C * NPIX;
    float* WS = P2 + 4 * C * fwd_np(C);
    const long long nslot = (long long)a.B * C * a.Ho * a.Wo;
    load_tile(XIN, e.x + (long long)n * e.x_ns, (long long)a.Hs * a.Ws, C, IH, IW, S * g.oy0 - 4, S * g.ox0 - 4, a.Hs, a.Ws,
              [](int, float v) { return v; });
    PCD_SYNC();

#define PCD_UNIT_A(U, KS, DIL)                                                                                     \
    unit_forward<C, KS, DIL, S, true>(XIN, IH, IW, 4, e.par + edge_dw_off(C, S, U), e.par + edge_pw_off(C, S, U),  \
                                      T, P, P2, WS, e.saved + slot_t(U) * nslot, e.saved + slot_z(U) * nslot,       \
                                      e.stats + bn_unit(S, U) * 2 * C, g)
    if (job == 0) { PCD_UNIT_A(0, 3, 1); return; }
    if (job == 1) { PCD_UNIT_A(2, 5, 1); return; }
    if (job == 2) { PCD_UNIT_A(4, 3, 2); return; }
    if (job == 3) { PCD_UNIT_A(5, 5, 2); return; }
#undef PCD_UNIT_A

    // ---- job 4: 3x3 max / avg pool (operations.py:6-7), stride S, pad 1, count_include_pad=False ---------
    PCD_FOR(task, C * NSTRIP) {
        const int ch = task / NSTRIP, strip = task - ch * NSTRIP;
        const int oyl = strip / PW4, oxl = (strip - oyl * PW4) * 4;
        const float* pl = XIN + ch * IH * IW;
        const int oy = g.oy0 + oyl;
        float mx[4], sm[4];
        int nrow = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) { mx[j] = -INFINITY; sm[j] = 0.f; }
#pragma unroll
        for (int dy = 0; dy < 3; ++dy) {
            const int gy = S * oy + dy - 1;
            if (gy < 0 || gy >= a.Hs) continue;
            ++nrow;
            const F4* rp = reinterpret_cast<const F4*>(pl + (S * oyl + dy + 3) * IW + S * oxl);
            float v[12];
#pragma unroll
            for (int q = 0; q < 3; ++q) { const F4 t = rp[q]; v[4 * q] = t.x; v[4 * q + 1] = t.y; v[4 * q + 2] = t.z; v[4 * q + 3] = t.w; }
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int dx = 0; dx < 3; ++dx) {
                    const int gx = S * (g.ox0 + oxl + j) + dx - 1;
                    const float val = v[S * j + dx + 3];
                    if (gx >= 0 && gx < a.Ws) {
                        mx[j] = val > mx[j] ? val : mx[j];
                        sm[j] += val;
                    }
                }
        }
        float av[4], s1 = 0.f, q1 = 0.f, s2 = 0.f, q2 = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int ox = g.ox0 + oxl + j;
            int ncol = 0;
#pragma unroll
            for (int dx = 0; dx < 3; ++dx) {
                const int gx = S * ox + dx - 1;
                ncol += (gx >= 0 && gx < a.Ws) ? 1 : 0;
            }
            const int cnt = nrow * ncol;
            mx[j] = cnt ? mx[j] : 0.f;
            av[j] = cnt ? sm[j] / (float)cnt : 0.f;
            if (oy < a.Ho && ox < a.Wo) {
                s1 += mx[j]; q1 = fmaf(mx[j], mx[j], q1);
                s2 += av[j]; q2 = fmaf(av[j], av[j], q2);
            }
        }
        store4(e.saved + slot_p1() * nslot, g, C, ch, oy, g.ox0 + oxl, mx);
        store4(e.saved + slot_p2() * nslot, g, C, ch, oy, g.ox0 + oxl, av);
        const int NT = C * NSTRIP;
        P[0 * NT + task] = s1; P[1 * NT + task] = q1; P[2 * NT + task] = s2; P[3 * NT + task] = q2;
    }
    reduce_columns<(C == 16 ? 16 : 32)>(P, P2, 4, C, NSTRIP, C * NSTRIP, [&](int ch, int k, float v) {
        const int bn = (k < 2) ? bn_p1() : bn_p2();
        pcd_atomic_add(e.stats + (bn * 2 + (k & 1)) * C + ch, (double)v);
    });

    // ---- skip_connect at stride 2 = FactorizedReduce (operations.py:90-104) ------------------------------
    if (S == 2) {
        PCD_FOR(task, C * NSTRIP) {
            const int co = task / NSTRIP, strip = task - co * NSTRIP;
            const int oyl = strip / PW4, oxl = (strip - oyl * PW4) * 4;
            const int off = (co >= C / 2) ? 1 : 0;
            const float* w = e.par + co * C;
            float f[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int ci = 0; ci < C; ++ci) {
                const float* pl = XIN + ci * IH * IW + (2 * oyl + off + 4) * IW + 2 * oxl + off + 4;
                const float wv = w[ci];
#pragma unroll
                for (int j = 0; j < 4; ++j) f[j] = fmaf(wv, relu(pl[2 * j]), f[j]);
            }
            const int oy = g.oy0 + oyl, ox = g.ox0 + oxl;
            store4(e.saved + slot_f() * nslot, g, C, co, oy, ox, f);
            float s = 0.f, q = 0.f;
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (oy < a.Ho && ox + j < a.Wo) { s += f[j]; q = fmaf(f[j], f[j], q); }
            const int NT = C * NSTRIP;
            P[task] = s; P[NT + task] = q;
        }
        reduce_columns(P, P2, 2, C, NSTRIP, C * NSTRIP, [&](int ch, int k, float v) {
            pcd_atomic_add(e.stats + (bn_f() * 2 + k) * C + ch, (double)v);
        });
    }
}

PCD_HOSTDEV size_t fwdB_smem_floats(int C, int TH, int TW) {
    return (size_t)C * (TH + 4) * (TW + 8) + (size_t)C * TH * TW * 2 + 4 * C * 32 + C * C + 2 * C + 64;
}

// second half of SepConv: BN -> ReLU -> dw (stride 1) -> pw   (operations.py:58-62); job = half (k=3 | k=5)
template <int C>
PCD_HD void fwdB_body(const PassArgs& a, int bx, int n, int z, float* smem) {
    const int TH = a.TH, TW = a.TW;
    const int ez = z >> 1, half = z & 1;
    const EdgeF& e = a.e[ez];
    Geo g;
    g.n = n; g.TH = TH; g.TW = TW; g.Ho = a.Ho; g.Wo = a.Wo;
    g.oy0 = (bx / a.tiles_x) * TH;
    g.ox0 = (bx % a.tiles_x) * TW;
    const int NPIX = TH * TW, IW = TW + 8;
    const int HY = half ? 2 : 1, IH = TH + 2 * HY;
    float* Q = smem;
    float* T = Q + C * (TH + 4) * IW;
    float* P = T + C * NPIX;
    float* P2 = P + C * NPIX;
    float* WS = P2 + 4 * C * 32;
    float* BNC = WS + C * C;
    const long long nslot = (long long)a.B * C * a.Ho * a.Wo;
    const double cnt = (double)a.B * a.Ho * a.Wo;
    const int S = a.S, uA = half ? 2 : 0, uB = uA + 1;
    const float* src = e.saved + slot_z(uA) * nslot + (long long)n * C * a.Ho * a.Wo;
    PCD_FOR(j, C) {
        BnC b = bn_consts(e.stats, C, bn_unit(S, uA), j, cnt, a.eps);
        BNC[2 * j] = b.mean;
        BNC[2 * j + 1] = b.rstd;
    }
    PCD_SYNC();
    load_tile(Q, src, (long long)a.Ho * a.Wo, C, IH, IW, g.oy0 - HY, g.ox0 - 4, a.Ho, a.Wo,
              [&](int ch, float v) { return relu((v - BNC[2 * ch]) * BNC[2 * ch + 1]); });
    PCD_SYNC();
    if (half == 0)
        unit_forward<C, 3, 1, 1, false>(Q, IH, IW, 1, e.par + edge_dw_off(C, S, uB), e.par + edge_pw_off(C, S, uB), T,
                                        P, P2, WS, e.saved + slot_t(uB) * nslot, e.saved + slot_z(uB) * nslot,
                                        e.stats + bn_unit(S, uB) * 2 * C, g);
    else
        unit_forward<C, 5, 1, 1, false>(Q, IH, IW, 2, e.par + edge_dw_off(C, S, uB), e.par + edge_pw_off(C, S, uB), T,
                                        P, P2, WS, e.saved + slot_t(uB) * nslot, e.saved + slot_z(uB) * nslot,
                                        e.stats + bn_unit(S, uB) * 2 * C, g);
}

// ======================================================================================================
// backward
// ======================================================================================================
// dz = c0 * (dy - a - (z - m) * c1)        (BatchNorm backward, affine=False, batch statistics)
struct DzC { float c0, a, m, c1; };

PCD_HD DzC dz_consts(const double* st, int c, int bn, int j, double n, float eps, double sum_dy, double sum_dyz,
                     float kappa) {
    BnC b = bn_consts(st, c, bn, j, n, eps);
    DzC r;
    r.c0 = b.rstd * kappa;
    r.a = (float)(sum_dy / n);
    r.m = b.mean;
    r.c1 = (float)((double)b.rstd * (double)b.rstd * (sum_dyz - (double)b.mean * sum_dy) / n);
    return r;
}

struct EdgeG {
    const float* x;        // source state
    long long x_ns;
    const float* dn;       // grad of the node this edge feeds (B, 4c, Ho, Wo) view
    long long dn_ns;
    const float* saved;
    const double* stats;
    double* bstats;
    const float* par;
    float* gpar;           // null when need_wgrad == 0
    const float* alpha;
    const float* beta;     // null => 1
    float* ga;             // 2 slots: grad wrt BN(A3) / BN(A5) outputs (post ReLU mask)
    float* pd;             // partial d xs slots, each (B, c, Hs, Ws): A3 A5 D3 D5 (pre ReLU mask) | max | avg(+id) | FR
};

PCD_HOSTDEV int edge_npd(int s) { return 6 + (s == 2); }

struct EdgeBwdArgs {
    int B, Hs, Ws, Ho, Wo, S;
    int TH, TW, tiles_x;
    float eps;
    int nedges, need_wgrad;
    EdgeG e[kMaxEdgesPerLaunch];
};

// dz on the haloed output tile -> dt = Wpw^T dz into DT[C][RH][IW] (row halo halo_y, col halo 4);
// centre dz into DZ[C][NPIX] when DZ != null.  WT holds Wpw transposed: WT[ci][co].
template <int C>
PCD_HD void dz_dt_tile(float* DT, float* DZ, int RH, int IW, int halo_y, const float* dy_img, long long dy_cs, int dy_chm,
                       const float* z_img, const float* WT, const float* COEF, const Geo& g) {
    const int NPIX = g.TH * g.TW, p4 = IW >> 2;
    const long long HW = (long long)g.Ho * g.Wo;
    PCD_FOR(i, RH * p4) {
        const int r = i / p4, c4 = i - r * p4;
        const int oyl = r - halo_y, oxl = 4 * c4 - 4;
        const int oy = g.oy0 + oyl, ox = g.ox0 + oxl;
        const bool in = (oy >= 0 && oy < g.Ho && ox + 3 >= 0 && ox < g.Wo);
        float dz[C][4];
#pragma unroll
        for (int j = 0; j < C; ++j) {
            float dy[4] = {0.f, 0.f, 0.f, 0.f}, zz[4] = {0.f, 0.f, 0.f, 0.f};
            if (in) {
                load4(dy_img + (long long)(j * dy_chm) * dy_cs + (long long)oy * g.Wo, ox, g.Wo, dy);
                load4(z_img + (long long)j * HW + (long long)oy * g.Wo, ox, g.Wo, zz);
            }
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const bool ok = in && ox + t >= 0 && ox + t < g.Wo;
                dz[j][t] = ok ? COEF[4 * j] * (dy[t] - COEF[4 * j + 1] - (zz[t] - COEF[4 * j + 2]) * COEF[4 * j + 3]) : 0.f;
            }
        }
#pragma unroll
        for (int ci = 0; ci < C; ++ci) {
            float s[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int c4o = 0; c4o < C / 4; ++c4o) {
                const F4 w = *reinterpret_cast<const F4*>(WT + ci * C + c4o * 4);
                const float wk[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
                for (int k = 0; k < 4; ++k)
#pragma unroll
                    for (int t = 0; t < 4; ++t) s[t] = fmaf(wk[k], dz[c4o * 4 + k][t], s[t]);
            }
            F4 o = {s[0], s[1], s[2], s[3]};
            *reinterpret_cast<F4*>(DT + (ci * RH + r) * IW + 4 * c4) = o;
        }
        if (DZ && oyl >= 0 && oyl < g.TH && oxl >= 0 && oxl < g.TW) {
#pragma unroll
            for (int j = 0; j < C; ++j) {
                F4 o = {dz[j][0], dz[j][1], dz[j][2], dz[j][3]};
                *reinterpret_cast<F4*>(DZ + j * NPIX + oyl * g.TW + oxl) = o;
            }
        }
    }
}

// dWpw[co][ci] += sum_p DZ[co][p] * t[ci][p] over the tile.  (C/4)^2 output groups x NSL pixel slices.
template <int C>
struct WgradPw {
    static constexpr int NOG = (C / 4) * (C / 4);
    static constexpr int NT = (C == 16) ? 128 : 256;      // tasks (C == 16: fewer, to keep P small)
    static constexpr int NSL = NT / NOG;
    static constexpr int PFLOATS = 16 * NT;
};

template <int C>
PCD_HD void wgrad_pw(const float* DZ, const float* t_slot, float* gw, float* P, float* P2, const Geo& g) {
    constexpr int NOG = WgradPw<C>::NOG, NSL = WgradPw<C>::NSL, NT = WgradPw<C>::NT;
    const int NPIX = g.TH * g.TW, SPS = (NPIX / 4 + NSL - 1) / NSL, PW4 = g.TW / 4;   // strips per slice
    PCD_FOR(task, NT) {
        const int og = task / NSL, sl = task - og * NSL;
        const int co0 = (og / (C / 4)) * 4, ci0 = (og % (C / 4)) * 4;
        float acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int k = 0; k < 4; ++k) acc[i][k] = 0.f;
        for (int st = sl * SPS; st < (sl + 1) * SPS && st < NPIX / 4; ++st) {
            const int oyl = st / PW4, oxl = (st - oyl * PW4) * 4;
            const int oy = g.oy0 + oyl, ox = g.ox0 + oxl;
            if (oy >= g.Ho) continue;
            float tv[4][4], dz[4][4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                load4(t_slot + out_index(g, C, ci0 + k, oy, 0), ox, g.Wo, tv[k]);
                const F4 d = *reinterpret_cast<const F4*>(DZ + (co0 + k) * NPIX + st * 4);
                dz[k][0] = d.x; dz[k][1] = d.y; dz[k][2] = d.z; dz[k][3] = d.w;
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int k = 0; k < 4; ++k)
#pragma unroll
                    for (int t = 0; t < 4; ++t) acc[i][k] = fmaf(dz[i][t], tv[k][t], acc[i][k]);
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int k = 0; k < 4; ++k) P[(i * 4 + k) * NT + task] = acc[i][k];
    }
    reduce_columns<4>(P, P2, 16, NOG, NSL, NT, [&](int og, int k, float v) {
        const int co = (og / (C / 4)) * 4 + (k >> 2), ci = (og % (C / 4)) * 4 + (k & 3);
        pcd_atomic_add(gw + co * C + ci, v);
    });
}

// dWdw[ch][tap] += sum over tile patches of dt(centre of DT) * in(tile)
template <int C, int KS, int DIL, int S, bool RELU>
PCD_HD void wgrad_dw(const float* DT, int RH, int IW, int halo_y, const float* IN, int in_rows, int in_pitch,
                     int in_halo_y, float* gw, float* P, float* P2, const Geo& g) {
    constexpr int PAD = DIL * (KS - 1) / 2;
    const int PW4 = g.TW / 4, NPATCH = (g.TH / 4) * PW4, NT = C * NPATCH;
    PCD_FOR(task, NT) {
        const int ch = task / NPATCH, patch = task - ch * NPATCH;
        const int py = (patch / PW4) * 4, px = (patch % PW4) * 4;
        float dt[4][4], acc[KS * KS];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const F4 v = *reinterpret_cast<const F4*>(DT + (ch * RH + py + i + halo_y) * IW + px + 4);
            dt[i][0] = v.x; dt[i][1] = v.y; dt[i][2] = v.z; dt[i][3] = v.w;
        }
#pragma unroll
        for (int k = 0; k < KS * KS; ++k) acc[k] = 0.f;
        dw_wgrad_patch<KS, DIL, S, RELU>(IN + ch * in_rows * in_pitch, in_pitch, S * py - PAD + in_halo_y, S * px, dt, acc);
#pragma unroll
        for (int k = 0; k < KS * KS; ++k) P[k * NT + task] = acc[k];
    }
    reduce_columns<4>(P, P2, KS * KS, C, NPATCH, NT, [&](int ch, int k, float v) {
        pcd_atomic_add(gw + ch * KS * KS + k, v);
    });
}

constexpr int kWgradNP = 4;     // partials per (value, group) in the weight-grad column reductions

PCD_HOSTDEV size_t wgrad_p2_floats(int C) { return (size_t)25 * C * kWgradNP + 64; }

PCD_HOSTDEV size_t wgrad_scratch_floats(int C, int TH, int TW) {
    // DZ [C][NPIX] + P for wgrad_pw (16 * tasks); wgrad_dw's P (25*C*NPATCH) aliases the same region; then P2
    size_t a = (size_t)C * TH * TW + 16 * (C == 16 ? 128 : 256), b = (size_t)25 * C * (TH / 4) * (TW / 4);
    return (a > b ? a : b) + wgrad_p2_floats(C);
}

// ---- stage B ------------------------------------------------------------------------------------------------
PCD_HOSTDEV size_t bwdB_smem_floats(int C, int TH, int TW, int need_wgrad) {
    const size_t tile = (size_t)C * (TH + 4) * (TW + 8);
    const int NPATCH = (TH / 4) * (TW / 4);
    size_t scratch = need_wgrad ? wgrad_scratch_floats(C, TH, TW) : (size_t)2 * C * NPATCH + 2 * C * 8 + 64;
    return 2 * tile + scratch + 6 * C + C * C + 64;
}

template <int C, int KS>
PCD_HD void bwdB_job(const EdgeBwdArgs& a, const EdgeG& e, const Geo& g, int half, float* smem) {
    constexpr int PAD = (KS - 1) / 2;
    const int S = a.S, TH = g.TH, TW = g.TW, NPIX = TH * TW, RH = TH + 2 * PAD, IW = TW + 8;
    const int PW4 = TW / 4, NPATCH = (TH / 4) * PW4;
    const size_t tile = (size_t)C * (TH + 4) * IW;
    float* DT = smem;
    float* Q = DT + tile;
    float* COEF = Q + tile;
    float* BNA = COEF + 4 * C;
    float* WT = BNA + 2 * C;
    float* SCR = WT + C * C;
    // scratch: [DZ | P(pw)] then reused as P(dw); P2 at the end
    float* DZ = a.need_wgrad ? SCR : nullptr;
    float* Ppw = SCR + C * NPIX;
    float* Pdw = SCR;
    float* P2 = a.need_wgrad ? SCR + (wgrad_scratch_floats(C, TH, TW) - wgrad_p2_floats(C)) : SCR + 2 * C * NPATCH;
    const int uA = half ? 2 : 0, uB = uA + 1;
    const long long nslot = (long long)a.B * C * a.Ho * a.Wo, HW = (long long)a.Ho * a.Wo;
    const double cnt = (double)a.B * a.Ho * a.Wo;
    const float beta = e.beta ? e.beta[0] : 1.f;
    const float kappa = beta * e.alpha[half ? 5 : 4];
    const float* w_dw = e.par + edge_dw_off(C, S, uB);
    const float* w_pw = e.par + edge_pw_off(C, S, uB);
    PCD_FOR(j, C) {
        const int bnB = bn_unit(S, uB);
        DzC d = dz_consts(e.stats, C, bnB, j, cnt, a.eps, e.bstats[bs_s0() * C + j], e.bstats[bs_sz(bnB) * C + j], kappa);
        COEF[4 * j] = d.c0; COEF[4 * j + 1] = d.a; COEF[4 * j + 2] = d.m; COEF[4 * j + 3] = d.c1;
        BnC b = bn_consts(e.stats, C, bn_unit(S, uA), j, cnt, a.eps);
        BNA[2 * j] = b.mean; BNA[2 * j + 1] = b.rstd;
    }
    PCD_FOR(i, C * C) WT[(i % C) * C + i / C] = w_pw[i];
    PCD_SYNC();
    const float* zA = e.saved + slot_z(uA) * nslot + (long long)g.n * C * HW;
    const float* zB = e.saved + slot_z(uB) * nslot + (long long)g.n * C * HW;
    dz_dt_tile<C>(DT, DZ, RH, IW, PAD, e.dn + (long long)g.n * e.dn_ns, HW, 4, zB, WT, COEF, g);
    load_tile(Q, zA, HW, C, RH, IW, g.oy0 - PAD, g.ox0 - 4, a.Ho, a.Wo,
              [&](int ch, float v) { return relu((v - BNA[2 * ch]) * BNA[2 * ch + 1]); });
    PCD_SYNC();
    // grad wrt relu(bn(zA)) = flipped depthwise correlation of dt; mask by the ReLU; sums for BN-A backward
    float* ga = e.ga + half * nslot;
    float* Pga = a.need_wgrad ? Ppw : SCR;      // [2][C*NPATCH]
    PCD_FOR(task, C * NPATCH) {
        const int ch = task / NPATCH, patch = task - ch * NPATCH;
        const int py = (patch / PW4) * 4, px = (patch % PW4) * 4;
        float acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
        dw_patch<KS, 1, 1, true, false>(DT + ch * RH * IW, IW, py, px, w_dw + ch * KS * KS, acc);
        float s = 0.f, sz = 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int oy = g.oy0 + py + i;
            const F4 q4 = *reinterpret_cast<const F4*>(Q + (ch * RH + py + i + PAD) * IW + px + 4);
            const float q[4] = {q4.x, q4.y, q4.z, q4.w};
            float o[4], za[4] = {0.f, 0.f, 0.f, 0.f};
            if (oy < a.Ho) load4(zA + (long long)ch * HW + (long long)oy * a.Wo, g.ox0 + px, a.Wo, za);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                o[j] = q[j] > 0.f ? acc[i][j] : 0.f;
                if (oy < a.Ho && g.ox0 + px + j < a.Wo) {
                    s += o[j];
                    sz = fmaf(o[j], za[j], sz);
                }
            }
            store4(ga, g, C, ch, oy, g.ox0 + px, o);
        }
        Pga[task] = s;
        Pga[C * NPATCH + task] = sz;
    }
    reduce_columns<8>(Pga, P2, 2, C, NPATCH, C * NPATCH, [&](int ch, int k, float v) {
        pcd_atomic_add(e.bstats + (bs_ga(half) + k) * C + ch, (double)v);
    });
    if (a.need_wgrad) {
        wgrad_pw<C>(DZ, e.saved + slot_t(uB) * nslot, e.gpar + edge_pw_off(C, S, uB), Ppw, P2, g);
        wgrad_dw<C, KS, 1, 1, false>(DT, RH, IW, PAD, Q, RH, IW, PAD, e.gpar + edge_dw_off(C, S, uB), Pdw, P2, g);
    }
}

template <int C>
PCD_HD void bwdB_body(const EdgeBwdArgs& a, int bx, int n, int z, float* smem) {
    Geo g;
    g.n = n; g.TH = a.TH; g.TW = a.TW; g.Ho = a.Ho; g.Wo = a.Wo;
    g.oy0 = (bx / a.tiles_x) * a.TH;
    g.ox0 = (bx % a.tiles_x) * a.TW;
    if ((z & 1) == 0) bwdB_job<C, 3>(a, a.e[z >> 1], g, 0, smem);
    else bwdB_job<C, 5>(a, a.e[z >> 1], g, 1, smem);
}

// ---- stage A ------------------------------------------------------------------------------------------------
PCD_HOSTDEV int bwdA_njobs(int S) { return 6 + (S == 2); }

PCD_HOSTDEV size_t bwdA_smem_floats(int C, int S, int TH, int TW, int need_wgrad) {
    const size_t xin = (size_t)C * (S * TH + 8) * (S * TW + 8);
    const size_t tile = (size_t)C * (TH + 8) * (TW + 8);
    // conv job: DT + [XIN + scratch if wgrad]; max-pool job: XIN + 2 tiles; FR job: XIN + DZ + P
    size_t conv = tile + (need_wgrad ? xin + wgrad_scratch_floats(C, TH, TW) : 0);
    size_t pool = xin + 2 * tile;
    size_t fr = S == 2 ? xin + (size_t)C * TH * TW + 16 * 256 + 16 * 16 * 8 : 0;
    size_t m = conv > pool ? conv : pool;
    if (fr > m) m = fr;
    return m + 4 * C + C * C + 64;
}

// gather d relu(x) for one stride-2 depthwise conv: in pixel q gets sum_tap w[tap] * dt[(q + PAD - tap*DIL)/2]
template <int KS, int DIL>
PCD_HD void dw_bwd_data_s2(const float* dtp /* plane [RH][IW], row halo HY, col halo 4 */, int IW, int HY, int qy0, int qx0,
                           const float* w, float (&acc)[4][4]) {
    constexpr int PAD = DIL * (KS - 1) / 2;
#pragma unroll
    for (int iy = 0; iy < 4; ++iy)
#pragma unroll
        for (int ky = 0; ky < KS; ++ky) {
            const int ty = iy + PAD - ky * DIL;               // qy0 is a multiple of 4 (even)
            if ((ty & 1) != 0) continue;
            const int prow = (qy0 + ty) / 2 + HY;
#pragma unroll
            for (int ix = 0; ix < 4; ++ix)
#pragma unroll
                for (int kx = 0; kx < KS; ++kx) {
                    const int tx = ix + PAD - kx * DIL;
                    if ((tx & 1) != 0) continue;
                    const int pcol = (qx0 + tx) / 2 + 4;
                    acc[iy][ix] = fmaf(w[ky * KS + kx], dtp[prow * IW + pcol], acc[iy][ix]);
                }
        }
}

PCD_HD void store_in4(float* pd_img, int ch, int gy, int gx, int Hs, int Ws, const float (&v)[4]) {
    float* p = pd_img + ((long long)ch * Hs + gy) * Ws + gx;
    if (gy >= Hs) return;
#pragma unroll
    for (int j = 0; j < 4; ++j)
        if (gx + j < Ws) p[j] = v[j];
}

// conv job: unit u (A3/A5: dy = GA, D3/D5: dy = dN[:, 0::4]) -> partial d relu(xs) (pre mask), weight grads
template <int C, int S, int KS, int DIL>
PCD_HD void bwdA_conv_job(const EdgeBwdArgs& a, const EdgeG& e, const Geo& g, int u, int slot, float* smem) {
    constexpr int PAD = DIL * (KS - 1) / 2;
    constexpr int HY = (S == 1) ? PAD : (PAD + 1) / 2;
    const int TH = g.TH, TW = g.TW, NPIX = TH * TW, RH = TH + 2 * HY, IW = TW + 8, IH = S * TH + 8, XW = S * TW + 8;
    float* COEF = smem;
    float* WT = COEF + 4 * C;
    float* DT = WT + C * C;
    float* XIN = DT + (size_t)C * (TH + 8) * IW;
    float* SCR = XIN + (size_t)C * IH * XW;
    float* DZ = a.need_wgrad ? SCR : nullptr;
    float* Ppw = SCR + C * NPIX;
    float* Pdw = SCR;
    float* P2 = SCR + (wgrad_scratch_floats(C, TH, TW) - wgrad_p2_floats(C));
    const long long nslot = (long long)a.B * C * a.Ho * a.Wo, HW = (long long)a.Ho * a.Wo;
    const double cnt = (double)a.B * a.Ho * a.Wo;
    const float beta = e.beta ? e.beta[0] : 1.f;
    const float* w_dw = e.par + edge_dw_off(C, S, u);
    const float* w_pw = e.par + edge_pw_off(C, S, u);
    const bool isA = (u == 0 || u == 2);
    const int which = (u == 2) ? 1 : 0;
    PCD_FOR(j, C) {
        DzC d;
        const int bn = bn_unit(S, u);
        if (isA)
            d = dz_consts(e.stats, C, bn, j, cnt, a.eps, e.bstats[bs_ga(which) * C + j], e.bstats[(bs_ga(which) + 1) * C + j], 1.f);
        else
            d = dz_consts(e.stats, C, bn, j, cnt, a.eps, e.bstats[bs_s0() * C + j], e.bstats[bs_sz(bn) * C + j],
                          beta * e.alpha[u == 4 ? 6 : 7]);
        COEF[4 * j] = d.c0; COEF[4 * j + 1] = d.a; COEF[4 * j + 2] = d.m; COEF[4 * j + 3] = d.c1;
    }
    PCD_FOR(i, C * C) WT[(i % C) * C + i / C] = w_pw[i];
    if (a.need_wgrad)
        load_tile(XIN, e.x + (long long)g.n * e.x_ns, (long long)a.Hs * a.Ws, C, IH, XW, S * g.oy0 - 4, S * g.ox0 - 4,
                  a.Hs, a.Ws, [](int, float v) { return v; });
    PCD_SYNC();
    const float* dy_img = isA ? e.ga + which * nslot + (long long)g.n * C * HW : e.dn + (long long)g.n * e.dn_ns;
    dz_dt_tile<C>(DT, DZ, RH, IW, HY, dy_img, HW, isA ? 1 : 4, e.saved + slot_z(u) * nslot + (long long)g.n * C * HW,
                  WT, COEF, g);
    PCD_SYNC();
    float* pd_img = e.pd + (long long)slot * a.B * C * a.Hs * a.Ws + (long long)g.n * C * a.Hs * a.Ws;
    const int AH = S * TH, AW = S * TW, APW4 = AW / 4, ANP = (AH / 4) * APW4;
    PCD_FOR(task, C * ANP) {
        const int ch = task / ANP, patch = task - ch * ANP;
        const int qy = (patch / APW4) * 4, qx = (patch % APW4) * 4;
        float acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
        if (S == 1)
            dw_patch<KS, DIL, 1, true, false>(DT + ch * RH * IW, IW, qy, qx, w_dw + ch * KS * KS, acc);
        else
            dw_bwd_data_s2<KS, DIL>(DT + ch * RH * IW, IW, HY, qy, qx, w_dw + ch * KS * KS, acc);
#pragma unroll
        for (int i = 0; i < 4; ++i) store_in4(pd_img, ch, S * g.oy0 + qy + i, S * g.ox0 + qx, a.Hs, a.Ws, acc[i]);
    }
    if (a.need_wgrad) {
        wgrad_pw<C>(DZ, e.saved + slot_t(u) * nslot, e.gpar + edge_pw_off(C, S, u), Ppw, P2, g);
        wgrad_dw<C, KS, DIL, S, true>(DT, RH, IW, HY, XIN, IH, XW, 4, e.gpar + edge_dw_off(C, S, u), Pdw, P2, g);
    }
}

// pool jobs: which = 0 max-pool (argmax recomputed from the raw tile), 1 avg-pool (+ identity skip at stride 1)
template <int C, int S>
PCD_HD void bwdA_pool_job(const EdgeBwdArgs& a, const EdgeG& e, const Geo& g, int which, float* smem) {
    const int TH = g.TH, TW = g.TW, RH = TH + 2, IW = TW + 8, IH = S * TH + 8, XW = S * TW + 8, p4 = IW >> 2;
    float* COEF = smem;
    float* DT = COEF + 4 * C + C * C;
    float* AM = DT + (size_t)C * (TH + 8) * IW;
    float* XIN = AM + (size_t)C * (TH + 8) * IW;
    const long long nslot = (long long)a.B * C * a.Ho * a.Wo, HW = (long long)a.Ho * a.Wo;
    const double cnt = (double)a.B * a.Ho * a.Wo;
    const float beta = e.beta ? e.beta[0] : 1.f;
    const int bn = which ? bn_p2() : bn_p1();
    PCD_FOR(j, C) {
        DzC d = dz_consts(e.stats, C, bn, j, cnt, a.eps, e.bstats[bs_s0() * C + j], e.bstats[bs_sz(bn) * C + j],
                          beta * e.alpha[which ? 2 : 1]);
        COEF[4 * j] = d.c0; COEF[4 * j + 1] = d.a; COEF[4 * j + 2] = d.m; COEF[4 * j + 3] = d.c1;
    }
    if (!which)
        load_tile(XIN, e.x + (long long)g.n * e.x_ns, (long long)a.Hs * a.Ws, C, IH, XW, S * g.oy0 - 4, S * g.ox0 - 4,
                  a.Hs, a.Ws, [](int, float v) { return v; });
    PCD_SYNC();
    const float* dn_img = e.dn + (long long)g.n * e.dn_ns;
    const float* Z = e.saved + (which ? slot_p2() : slot_p1()) * nslot + (long long)g.n * C * HW;
    // dz (and, for max-pool, the argmax code) of every output pixel within one pixel of the tile
    PCD_FOR(i, C * RH * p4) {
        const int c4 = i % p4, rr = i / p4, r = rr % RH, ch = rr / RH;
        const int oyl = r - 1, oxl = 4 * c4 - 4;
        const int oy = g.oy0 + oyl, ox = g.ox0 + oxl;
        float dz[4] = {0.f, 0.f, 0.f, 0.f}, code[4] = {-1.f, -1.f, -1.f, -1.f};
        if (oy >= 0 && oy < a.Ho && ox + 3 >= 0 && ox < a.Wo) {
            float h[4], zz[4];
            load4(dn_img + (long long)(4 * ch) * HW + (long long)oy * a.Wo, ox, a.Wo, h);
            load4(Z + (long long)ch * HW + (long long)oy * a.Wo, ox, a.Wo, zz);
            int nrow = 0;
#pragma unroll
            for (int dy = 0; dy < 3; ++dy) {
                const int gy = S * oy + dy - 1;
                nrow += (gy >= 0 && gy < a.Hs) ? 1 : 0;
            }
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                if (ox + t < 0 || ox + t >= a.Wo) continue;
                float v = COEF[4 * ch] * (h[t] - COEF[4 * ch + 1] - (zz[t] - COEF[4 * ch + 2]) * COEF[4 * ch + 3]);
                if (which) {
                    int ncol = 0;
#pragma unroll
                    for (int dx = 0; dx < 3; ++dx) {
                        const int gx = S * (ox + t) + dx - 1;
                        ncol += (gx >= 0 && gx < a.Ws) ? 1 : 0;
                    }
                    v = v / (float)(nrow * ncol);
                } else if (oyl >= -1 && oyl <= TH && oxl + t >= -1 && oxl + t <= TW) {
                    float m = -INFINITY;
                    int best = -1;
#pragma unroll
                    for (int dy = 0; dy < 3; ++dy)
#pragma unroll
                        for (int dx = 0; dx < 3; ++dx) {
                            const int gy = S * oy + dy - 1, gx = S * (ox + t) + dx - 1;
                            if (gy >= 0 && gy < a.Hs && gx >= 0 && gx < a.Ws) {
                                const float xv = XIN[(ch * IH + S * oyl + dy + 3) * XW + S * (oxl + t) + dx + 3];
                                if (xv > m || best < 0) { m = xv; best = dy * 3 + dx; }
                            }
                        }
                    code[t] = (float)best;
                }
                dz[t] = v;
            }
        }
        F4 o = {dz[0], dz[1], dz[2], dz[3]};
        *reinterpret_cast<F4*>(DT + (ch * RH + r) * IW + 4 * c4) = o;
        if (!which) {
            F4 c = {code[0], code[1], code[2], code[3]};
            *reinterpret_cast<F4*>(AM + (ch * RH + r) * IW + 4 * c4) = c;
        }
    }
    PCD_SYNC();
    // gather over the windows that contain each input pixel
    const int AH = S * TH, AW = S * TW, AW4 = AW / 4;
    float* pd_img = e.pd + (long long)(4 + which) * a.B * C * a.Hs * a.Ws + (long long)g.n * C * a.Hs * a.Ws;
    const float idc = beta * e.alpha[3];
    PCD_FOR(task, C * AH * AW4) {
        const int q4 = task % AW4, rr = task / AW4, qy = rr % AH, ch = rr / AH;
        const int qx0 = q4 * 4;
        float s[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int dy = 0; dy < 3; ++dy) {
            const int ty = qy + 1 - dy;
            if (ty % S != 0) continue;
            const int pr = ty / S + 1;             // ty >= -1 (only when S == 1)
#pragma unroll
            for (int t = 0; t < 4; ++t)
#pragma unroll
                for (int dx = 0; dx < 3; ++dx) {
                    const int tx = qx0 + t + 1 - dx;
                    if (tx % S != 0) continue;
                    const int idx = (ch * RH + pr) * IW + tx / S + 4;
                    if (which) s[t] += DT[idx];
                    else if (AM[idx] == (float)(dy * 3 + dx)) s[t] += DT[idx];
                }
        }
        const int gy = S * g.oy0 + qy, gx = S * g.ox0 + qx0;
        if (which && S == 1 && gy < a.Ho) {       // identity skip: d xs += beta * w3 * dN[:, 0::4]
            float h[4];
            load4(dn_img + (long long)(4 * ch) * HW + (long long)gy * a.Wo, gx, a.Wo, h);
#pragma unroll
            for (int t = 0; t < 4; ++t) s[t] = fmaf(idc, h[t], s[t]);
        }
        store_in4(pd_img, ch, gy, gx, a.Hs, a.Ws, s);
    }
}

// FactorizedReduce backward (stride-2 skip): partial d relu(xs) (pre mask) + the two 1x1 weight grads
template <int C>
PCD_HD void bwdA_fr_job(const EdgeBwdArgs& a, const EdgeG& e, const Geo& g, float* smem) {
    const int TH = g.TH, TW = g.TW, NPIX = TH * TW, IH = 2 * TH + 8, XW = 2 * TW + 8, PW4 = TW / 4;
    float* COEF = smem;
    float* XIN = COEF + 4 * C + C * C;
    float* DZ = XIN + (size_t)C * IH * XW;
    float* P = DZ + C * NPIX;
    float* P2 = P + 16 * 256;
    const long long nslot = (long long)a.B * C * a.Ho * a.Wo, HW = (long long)a.Ho * a.Wo;
    const double cnt = (double)a.B * a.Ho * a.Wo;
    const float beta = e.beta ? e.beta[0] : 1.f;
    PCD_FOR(j, C) {
        DzC d = dz_consts(e.stats, C, bn_f(), j, cnt, a.eps, e.bstats[bs_s0() * C + j], e.bstats[bs_sz(bn_f()) * C + j],
                          beta * e.alpha[3]);
        COEF[4 * j] = d.c0; COEF[4 * j + 1] = d.a; COEF[4 * j + 2] = d.m; COEF[4 * j + 3] = d.c1;
    }
    if (a.need_wgrad)
        load_tile(XIN, e.x + (long long)g.n * e.x_ns, (long long)a.Hs * a.Ws, C, IH, XW, 2 * g.oy0 - 4, 2 * g.ox0 - 4,
                  a.Hs, a.Ws, [](int, float v) { return v; });
    PCD_SYNC();
    const float* dn_img = e.dn + (long long)g.n * e.dn_ns;
    const float* F = e.saved + slot_f() * nslot + (long long)g.n * C * HW;
    float* pd_img = e.pd + 6LL * a.B * C * a.Hs * a.Ws + (long long)g.n * C * a.Hs * a.Ws;
    PCD_FOR(st, NPIX / 4) {
        const int oyl = st / PW4, oxl = (st - oyl * PW4) * 4;
        const int oy = g.oy0 + oyl, ox = g.ox0 + oxl;
        float dz[C][4];
#pragma unroll
        for (int j = 0; j < C; ++j) {
            float h[4] = {0.f, 0.f, 0.f, 0.f}, f[4] = {0.f, 0.f, 0.f, 0.f};
            const bool in = oy < a.Ho;
            if (in) {
                load4(dn_img + (long long)(4 * j) * HW + (long long)oy * a.Wo, ox, a.Wo, h);
                load4(F + (long long)j * HW + (long long)oy * a.Wo, ox, a.Wo, f);
            }
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const bool ok = in && ox + t < a.Wo;
                dz[j][t] = ok ? COEF[4 * j] * (h[t] - COEF[4 * j + 1] - (f[t] - COEF[4 * j + 2]) * COEF[4 * j + 3]) : 0.f;
            }
            if (a.need_wgrad) {
                F4 o = {dz[j][0], dz[j][1], dz[j][2], dz[j][3]};
                *reinterpret_cast<F4*>(DZ + j * NPIX + st * 4) = o;
            }
        }
#pragma unroll
        for (int ci = 0; ci < C; ++ci) {
            float r0[8], r1[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) { r0[k] = 0.f; r1[k] = 0.f; }
#pragma unroll
            for (int co = 0; co < C / 2; ++co) {
                const float w0 = e.par[co * C + ci], w1 = e.par[(co + C / 2) * C + ci];
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    r0[2 * t] = fmaf(w0, dz[co][t], r0[2 * t]);
                    r1[2 * t + 1] = fmaf(w1, dz[co + C / 2][t], r1[2 * t + 1]);
                }
            }
            const float a0[4] = {r0[0], r0[1], r0[2], r0[3]}, a1[4] = {r0[4], r0[5], r0[6], r0[7]};
            const float b0[4] = {r1[0], r1[1], r1[2], r1[3]}, b1[4] = {r1[4], r1[5], r1[6], r1[7]};
            store_in4(pd_img, ci, 2 * oy, 2 * ox, a.Hs, a.Ws, a0);
            store_in4(pd_img, ci, 2 * oy, 2 * ox + 4, a.Hs, a.Ws, a1);
            store_in4(pd_img, ci, 2 * oy + 1, 2 * ox, a.Hs, a.Ws, b0);
            store_in4(pd_img, ci, 2 * oy + 1, 2 * ox + 4, a.Hs, a.Ws, b1);
        }
    }
    if (a.need_wgrad) {
        PCD_SYNC();
        // dW_fr[co][ci] += sum_p dz[co][p] * relu(x[ci][2p + off(co)])
        constexpr int NOG = (C / 4) * (C / 4), NSL = 256 / NOG;
        const int PPS = (NPIX + NSL - 1) / NSL;
        PCD_FOR(task, 256) {
            const int og = task / NSL, sl = task - og * NSL;
            const int co0 = (og / (C / 4)) * 4, ci0 = (og % (C / 4)) * 4;
            float acc[4][4];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int k = 0; k < 4; ++k) acc[i][k] = 0.f;
            for (int pp = sl * PPS; pp < (sl + 1) * PPS && pp < NPIX; ++pp) {
                const int oyl = pp / TW, oxl = pp - oyl * TW;
                float rv[2][4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    rv[0][k] = relu(XIN[((ci0 + k) * IH + 2 * oyl + 4) * XW + 2 * oxl + 4]);
                    rv[1][k] = relu(XIN[((ci0 + k) * IH + 2 * oyl + 5) * XW + 2 * oxl + 5]);
                }
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float d = DZ[(co0 + i) * NPIX + pp];
                    const int off = (co0 + i) >= C / 2 ? 1 : 0;
#pragma unroll
                    for (int k = 0; k < 4; ++k) acc[i][k] = fmaf(d, rv[off][k], acc[i][k]);
                }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int k = 0; k < 4; ++k) P[(i * 4 + k) * 256 + task] = acc[i][k];
        }
        reduce_columns<4>(P, P2, 16, NOG, NSL, 256, [&](int og, int k, float v) {
            const int co = (og / (C / 4)) * 4 + (k >> 2), ci = (og % (C / 4)) * 4 + (k & 3);
            pcd_atomic_add(e.gpar + co * C + ci, v);
        });
    }
}

template <int C, int S>
PCD_HD void bwdA_body(const EdgeBwdArgs& a, int bx, int n, int z, float* smem) {
    const int NJ = 6 + (S == 2);
    const int ez = z / NJ, job = z - ez * NJ;
    const EdgeG& e = a.e[ez];
    Geo g;
    g.n = n; g.TH = a.TH; g.TW = a.TW; g.Ho = a.Ho; g.Wo = a.Wo;
    g.oy0 = (bx / a.tiles_x) * a.TH;
    g.ox0 = (bx % a.tiles_x) * a.TW;
    if (job == 0) bwdA_conv_job<C, S, 3, 1>(a, e, g, 0, 0, smem);
    else if (job == 1) bwdA_conv_job<C, S, 5, 1>(a, e, g, 2, 1, smem);
    else if (job == 2) bwdA_conv_job<C, S, 3, 2>(a, e, g, 4, 2, smem);
    else if (job == 3) bwdA_conv_job<C, S, 5, 2>(a, e, g, 5, 3, smem);
    else if (job == 4) bwdA_pool_job<C, S>(a, e, g, 0, smem);
    else if (job == 5) bwdA_pool_job<C, S>(a, e, g, 1, smem);
    else if (S == 2) bwdA_fr_job<C>(a, e, g, smem);
}

}  // namespace pcd
