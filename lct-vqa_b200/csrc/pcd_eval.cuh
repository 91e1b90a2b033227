// pcd_eval.cuh — eval-mode forward kernels: BatchNorm from running statistics (ATen's inference form
// y = scale * z + shift, scale = gamma / sqrt(running_var + eps), shift = beta - running_mean * scale).
//
// With fixed per-channel affine maps there are no batch-statistic barriers, so one block computes a whole
// node of a cell for its (image, output-row tile): for every incoming edge it stages the partial-channel
// input tile x[:, :c] once (halo 4, or 6 on the input grid of a stride-2 edge: enough for the two 5x5 stages
// of sep_conv_5x5 and for dil_conv_5x5), runs all 8 candidate ops from shared memory (the first separable
// stage recomputed over the halo the second needs), accumulates sum_e beta_e * sum_k alpha_ek * op_k and
// writes the node's slice of the cell output once, channel-shuffled, bypass channels included.  Nothing
// else reaches HBM: no statistics, no running-stat updates, no saved activations.
//
// Written in the phase style of pcd_common.cuh so the -DPCD_EMU build runs the same bodies on the CPU.
#pragma once
#include "pcd_common.cuh"

namespace pcd {

// ---- one node (or a stand-alone MixedOp: one edge, beta = 1) ------------------------------------------------
constexpr int kEvalMaxIn = 5;
constexpr int kEvalTH = 4;          // output rows per block

struct EvalEdge {
    const float* x;                 // source state, image 0
    long long x_ns;                 // floats between images
    int stride, Hs, Ws;
    const float* par;               // edge parameter block (layout of edge_param_floats)
    const float* running;           // per BN of the edge: running_mean[c], running_var[c]
    const float* alpha;             // 8 softmaxed op weights
    const float* beta;              // edge weight; null => 1
};

struct EvalNodeArgs {
    int B, Ho, Wo, TH, nin, maxS;
    float eps;
    float* out;                     // node slice (channels 4c) of the output, image 0
    long long out_ns;
    EvalEdge e[kEvalMaxIn];
};

PCD_HOSTDEV int eval_halo(int S) { return S == 1 ? 4 : 6; }
PCD_HOSTDEV int eval_xs_rows(int S, int TH) { return S * TH + 2 * eval_halo(S); }
PCD_HOSTDEV int eval_xs_cols(int S, int Wo) { return S * Wo + 2 * eval_halo(S); }

// shared-memory carve-up (floats): input tile | edge parameters | BN scale, shift | two mid buffers | edge sum | node sum
struct EvalSmem { int par, bn, t, m, ea, acc, total; };
PCD_HOSTDEV EvalSmem eval_smem(int c, int TH, int Wo, int maxS) {
    EvalSmem s;
    const int xs = c * eval_xs_rows(maxS, TH) * eval_xs_cols(maxS, Wo);
    const int mid = c * (TH + 4) * (Wo + 4), tile = c * TH * Wo;
    s.par = round_up(xs, 4);
    s.bn = s.par + round_up(edge_param_floats(c, 2), 4);
    s.t = s.bn + 2 * 9 * c;
    s.m = s.t + mid;
    s.ea = s.m + mid;
    s.acc = s.ea + tile;
    s.total = s.acc + tile;
    return s;
}

// depthwise KSxKS stencil (dilation DIL) whose first tap is plane[r][q]
template <int KS, int DIL, bool RELU>
PCD_HD float dw_at(const float* PCD_RESTRICT plane, int pitch, int r, int q, const float* PCD_RESTRICT w) {
    float s = 0.f;
#pragma unroll
    for (int ky = 0; ky < KS; ++ky)
#pragma unroll
        for (int kx = 0; kx < KS; ++kx) {
            const float v = plane[(r + DIL * ky) * pitch + q + DIL * kx];
            s = fmaf(w[ky * KS + kx], RELU ? relu(v) : v, s);
        }
    return s;
}

// 1x1 conv of channel `co` at position p of a [C][n] buffer, then the BN affine
template <int C>
PCD_HD float pw_bn(const float* PCD_RESTRICT t, int n, int p, const float* PCD_RESTRICT w, int co, const float* bns) {
    float s = 0.f;
#pragma unroll
    for (int ci = 0; ci < C; ++ci) s = fmaf(w[co * C + ci], t[ci * n + p], s);
    return fmaf(s, bns[co], bns[C + co]);
}

// one separable conv (units u, u+1: KS x KS, first stage with the edge's stride) from the staged tile into T (tile
// layout).  Stage 1 runs over the tile plus the (KS/2)-pixel halo stage 2 needs, masked to zero outside the image.
template <int C, int KS>
PCD_HD void eval_sep(const EvalNodeArgs& a, int S, int r0, const float* XS, int XR, int XP, const float* PAR,
                     const float* BNS, float* T, float* M, int u) {
    constexpr int P = KS / 2;
    const int TH = a.TH, Wo = a.Wo, HI = eval_halo(S), MR = TH + 2 * P, MP = Wo + 2 * P, NM = MR * MP;
    const float* w1 = PAR + edge_dw_off(C, S, u);
    const float* p1 = PAR + edge_pw_off(C, S, u);
    const float* w2 = PAR + edge_dw_off(C, S, u + 1);
    (void)XR;
    PCD_FOR(i, C * NM) {
        const int ch = i / NM, m = i - ch * NM, mi = m / MP, mj = m - mi * MP;
        T[i] = dw_at<KS, 1, true>(XS + ch * XR * XP, XP, S * (mi - P) - P + HI, S * (mj - P) - P + HI, w1 + ch * KS * KS);
    }
    PCD_SYNC();
    const float* bn1 = BNS + 2 * C * bn_unit(S, u);
    PCD_FOR(i, C * NM) {
        const int co = i / NM, m = i - co * NM, mi = m / MP, mj = m - mi * MP;
        const int oy = r0 - P + mi, ox = mj - P;
        M[i] = (oy >= 0 && oy < a.Ho && ox >= 0 && ox < Wo) ? relu(pw_bn<C>(T, NM, m, p1, co, bn1)) : 0.f;
    }
    PCD_SYNC();
    PCD_FOR(i, C * TH * Wo) {
        const int ch = i / (TH * Wo), p = i - ch * TH * Wo, oi = p / Wo, oj = p - oi * Wo;
        T[i] = dw_at<KS, 1, false>(M + ch * NM, MP, oi, oj, w2 + ch * KS * KS);
    }
    PCD_SYNC();
}

template <int C>
PCD_HD void eval_node_body(const EvalNodeArgs& a, int tile, int n, float* smem) {
    const int TH = a.TH, Wo = a.Wo, r0 = tile * TH, NP = TH * Wo, NT = C * NP;
    const EvalSmem L = eval_smem(C, TH, Wo, a.maxS);
    float* XS = smem;
    float* PAR = smem + L.par;
    float* BNS = smem + L.bn;           // per BN: scale[C], shift[C]
    float* T = smem + L.t;
    float* M = smem + L.m;
    float* EA = smem + L.ea;
    float* ACC = smem + L.acc;
    for (int ei = 0; ei < a.nin; ++ei) {
        const EvalEdge& e = a.e[ei];
        const int S = e.stride, HI = eval_halo(S), XR = eval_xs_rows(S, TH), XP = eval_xs_cols(S, Wo);
        const int gy0 = S * r0 - HI;
        const long long plane = (long long)e.Hs * e.Ws;
        const float* xb = e.x + (long long)n * e.x_ns;
        // 1. stage the partial-channel tile (zero outside the image), the edge's weights and BN affine maps
        PCD_FOR(i, C * XR * XP) {
            const int ch = i / (XR * XP), r = (i / XP) % XR, q = i % XP;
            const int gy = gy0 + r, gx = q - HI;
            XS[i] = (gy >= 0 && gy < e.Hs && gx >= 0 && gx < e.Ws) ? xb[ch * plane + (long long)gy * e.Ws + gx] : 0.f;
        }
        PCD_FOR(i, edge_param_floats(C, S)) PAR[i] = e.par[i];
        PCD_FOR(i, edge_nbn(S) * C) {
            const int bn = i / C, j = i - bn * C;
            const float sc = 1.f / sqrtf(e.running[bn * 2 * C + C + j] + a.eps);
            BNS[bn * 2 * C + j] = sc;
            BNS[bn * 2 * C + C + j] = -e.running[bn * 2 * C + j] * sc;
        }
        PCD_SYNC();
        // 2. depthwise halves of the two dilated convs
        {
            const float* w3 = PAR + edge_dw_off(C, S, 4);
            const float* w5 = PAR + edge_dw_off(C, S, 5);
            PCD_FOR(i, NT) {
                const int ch = i / NP, p = i - ch * NP, oi = p / Wo, oj = p - oi * Wo;
                const float* pl = XS + ch * XR * XP;
                T[i] = dw_at<3, 2, true>(pl, XP, S * oi - 2 + HI, S * oj - 2 + HI, w3 + ch * 9);
                M[i] = dw_at<5, 2, true>(pl, XP, S * oi - 4 + HI, S * oj - 4 + HI, w5 + ch * 25);
            }
        }
        PCD_SYNC();
        // 3. pools, skip / FactorizedReduce, dilated convs' pointwise halves
        {
            const float* al = e.alpha;
            const float a1 = al[1], a2 = al[2], a3 = al[3], a6 = al[6], a7 = al[7];
            const float* pd3 = PAR + edge_pw_off(C, S, 4);
            const float* pd5 = PAR + edge_pw_off(C, S, 5);
            PCD_FOR(i, NT) {
                const int co = i / NP, p = i - co * NP, oi = p / Wo, oj = p - oi * Wo;
                const float* pl = XS + co * XR * XP;
                float mx = -INFINITY, sm = 0.f;
                int cnt = 0;
#pragma unroll
                for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx) {
                        const int r = S * oi - 1 + ky + HI, q = S * oj - 1 + kx + HI;
                        const int gy = gy0 + r, gx = q - HI;
                        if (gy >= 0 && gy < e.Hs && gx >= 0 && gx < e.Ws) {
                            const float v = pl[r * XP + q];
                            mx = v > mx ? v : mx;
                            sm += v;
                            ++cnt;
                        }
                    }
                const float* b1 = BNS + 2 * C * bn_p1();
                const float* b2 = BNS + 2 * C * bn_p2();
                float acc = a1 * fmaf(mx, b1[co], b1[C + co]);
                acc = fmaf(a2, fmaf(sm / (float)cnt, b2[co], b2[C + co]), acc);
                float sk;
                if (S == 1) {
                    sk = pl[(oi + HI) * XP + oj + HI];
                } else {          // FactorizedReduce: conv_1 on the even grid, conv_2 on the (1,1)-shifted one
                    const int sh = co < C / 2 ? 0 : 1;
                    const int r = 2 * oi + sh + HI, q = 2 * oj + sh + HI;
                    float s = 0.f;
#pragma unroll
                    for (int ci = 0; ci < C; ++ci) s = fmaf(PAR[co * C + ci], relu(XS[(ci * XR + r) * XP + q]), s);
                    const float* bf = BNS + 2 * C * bn_f();
                    sk = fmaf(s, bf[co], bf[C + co]);
                }
                acc = fmaf(a3, sk, acc);
                acc = fmaf(a6, pw_bn<C>(T, NP, p, pd3, co, BNS + 2 * C * bn_unit(S, 4)), acc);
                acc = fmaf(a7, pw_bn<C>(M, NP, p, pd5, co, BNS + 2 * C * bn_unit(S, 5)), acc);
                EA[i] = acc;
            }
        }
        PCD_SYNC();
        // 4. the two separable convs; the edge sum joins the node sum with beta
        eval_sep<C, 3>(a, S, r0, XS, XR, XP, PAR, BNS, T, M, 0);
        {
            const float a4 = e.alpha[4];
            const float* p3 = PAR + edge_pw_off(C, S, 1);
            const float* bn3 = BNS + 2 * C * bn_unit(S, 1);
            PCD_FOR(i, NT) {
                const int co = i / NP, p = i - co * NP;
                EA[i] = fmaf(a4, pw_bn<C>(T, NP, p, p3, co, bn3), EA[i]);
            }
        }
        PCD_SYNC();
        eval_sep<C, 5>(a, S, r0, XS, XR, XP, PAR, BNS, T, M, 2);
        {
            const float a5 = e.alpha[5];
            const float beta = e.beta ? e.beta[0] : 1.f;
            const float* p5 = PAR + edge_pw_off(C, S, 3);
            const float* bn5 = BNS + 2 * C * bn_unit(S, 3);
            PCD_FOR(i, NT) {
                const int co = i / NP, p = i - co * NP;
                const float es = fmaf(a5, pw_bn<C>(T, NP, p, p5, co, bn5), EA[i]);
                ACC[i] = ei == 0 ? beta * es : fmaf(beta, es, ACC[i]);
            }
        }
        PCD_SYNC();
    }
    // 5. out[:, 4j] = node sum of channel j; out[:, 4j+q] = sum_e beta_e * bypass_e[q*C + j] (2x2 max-pool at stride 2)
    const long long HWo = (long long)a.Ho * Wo;
    PCD_FOR(i, NT) {
        const int j = i / NP, p = i - j * NP, oi = p / Wo, oj = p - oi * Wo, oy = r0 + oi;
        if (oy < a.Ho) {
            float by[3] = {0.f, 0.f, 0.f};
            for (int ei = 0; ei < a.nin; ++ei) {
                const EvalEdge& e = a.e[ei];
                const float beta = e.beta ? e.beta[0] : 1.f;
                const float* xb = e.x + (long long)n * e.x_ns;
                const long long plane = (long long)e.Hs * e.Ws;
#pragma unroll
                for (int q = 1; q < 4; ++q) {
                    const float* pl = xb + (q * C + j) * plane;
                    float v;
                    if (e.stride == 1) {
                        v = pl[(long long)oy * e.Ws + oj];
                    } else {
                        const float* w = pl + (long long)(2 * oy) * e.Ws + 2 * oj;
                        v = w[0];
                        v = w[1] > v ? w[1] : v;
                        v = w[e.Ws] > v ? w[e.Ws] : v;
                        v = w[e.Ws + 1] > v ? w[e.Ws + 1] : v;
                    }
                    by[q - 1] = fmaf(beta, v, by[q - 1]);
                }
            }
            float* ob = a.out + (long long)n * a.out_ns + (long long)oy * Wo + oj;
            ob[(4 * j) * HWo] = ACC[i];
#pragma unroll
            for (int q = 1; q < 4; ++q) ob[(4 * j + q) * HWo] = by[q - 1];
        }
    }
}

// ---- preprocess: ReLU -> 1x1 conv (or FactorizedReduce) -> BN affine from running statistics ----------------
// Block = 128 output pixels x 16 output channels of one image; thread = 4 pixels x 2 channels; input channels
// streamed through shared memory in chunks of 32.  FP32 FMA like the training forward (pcd_pre.cuh).
struct EvalPreArgs {
    int B, Cin, Cout, Hin, Win, Ho, Wo, fr;
    float eps;
    const float* x;                 // (B, Cin, Hin, Win)
    const float* w;                 // [Cout][Cin] (FactorizedReduce: conv_1 rows then conv_2 rows)
    const float* running;           // running_mean[Cout], running_var[Cout]
    const float* gamma;             // null => 1
    const float* beta;              // null => 0
    float* y;                       // (B, Cout, Ho, Wo)
};

constexpr int kEvalPrePx = 128, kEvalPreKC = 32, kEvalPreCO = 16;
PCD_HOSTDEV size_t eval_pre_smem_floats() { return (size_t)kEvalPreKC * kEvalPrePx + kEvalPreCO * kEvalPreKC + 2 * kEvalPreCO; }

PCD_HD void eval_pre_body(const EvalPreArgs& a, int bx, int n, int z, float* smem) {
    float* XS = smem;                                   // [KC][128]
    float* WS = XS + kEvalPreKC * kEvalPrePx;           // [16][KC]
    float* SC = WS + kEvalPreCO * kEvalPreKC;           // [16] scale, [16] shift
    const int HW = a.Ho * a.Wo, p0 = bx * kEvalPrePx, co_base = z * kEvalPreCO;
    const int shift = (a.fr && co_base >= a.Cout / 2) ? 1 : 0;
    const long long cs = (long long)a.Hin * a.Win;
    const float* xb = a.x + (long long)n * a.Cin * cs;
    PCD_TSTATE(float, acc, [2][4]);
    PCD_EACH(t) {
        auto& ac = PCD_TREF(acc, t);
        for (int r = 0; r < 2; ++r)
            for (int q = 0; q < 4; ++q) ac[r][q] = 0.f;
    }
    PCD_FOR(i, kEvalPreCO) {
        const int co = co_base + i;
        const float sc = (1.f / sqrtf(a.running[a.Cout + co] + a.eps)) * (a.gamma ? a.gamma[co] : 1.f);
        SC[i] = sc;
        SC[kEvalPreCO + i] = (a.beta ? a.beta[co] : 0.f) - a.running[co] * sc;
    }
    for (int kc = 0; kc < a.Cin; kc += kEvalPreKC) {
        PCD_FOR(i, kEvalPreKC * kEvalPrePx) {
            const int k = i / kEvalPrePx, p = p0 + (i - k * kEvalPrePx), ci = kc + k;
            float v = 0.f;
            if (ci < a.Cin && p < HW) {
                const float* pl = xb + ci * cs;
                if (a.fr) {
                    const int oy = p / a.Wo, ox = p - oy * a.Wo;
                    v = pl[(long long)(2 * oy + shift) * a.Win + 2 * ox + shift];
                } else {
                    v = pl[p];
                }
            }
            XS[i] = relu(v);
        }
        PCD_FOR(i, kEvalPreCO * kEvalPreKC) {
            const int col = i / kEvalPreKC, k = i - col * kEvalPreKC;
            WS[i] = kc + k < a.Cin ? a.w[(long long)(co_base + col) * a.Cin + kc + k] : 0.f;
        }
        PCD_SYNC();
        PCD_EACH(t) {
            auto& ac = PCD_TREF(acc, t);
            const int quad = t & 31, g = t >> 5;
            const float* ws0 = WS + (2 * g) * kEvalPreKC;
            const float* ws1 = ws0 + kEvalPreKC;
#pragma unroll 8
            for (int k = 0; k < kEvalPreKC; ++k) {
                const F4 x4 = *reinterpret_cast<const F4*>(XS + k * kEvalPrePx + 4 * quad);
                const float w0 = ws0[k], w1 = ws1[k];
                ac[0][0] = fmaf(w0, x4.x, ac[0][0]); ac[0][1] = fmaf(w0, x4.y, ac[0][1]);
                ac[0][2] = fmaf(w0, x4.z, ac[0][2]); ac[0][3] = fmaf(w0, x4.w, ac[0][3]);
                ac[1][0] = fmaf(w1, x4.x, ac[1][0]); ac[1][1] = fmaf(w1, x4.y, ac[1][1]);
                ac[1][2] = fmaf(w1, x4.z, ac[1][2]); ac[1][3] = fmaf(w1, x4.w, ac[1][3]);
            }
        }
        PCD_SYNC();
    }
    PCD_EACH(t) {
        auto& ac = PCD_TREF(acc, t);
        const int quad = t & 31, g = t >> 5;
        for (int r = 0; r < 2; ++r) {
            const int cl = 2 * g + r;
            float* yb = a.y + ((long long)n * a.Cout + co_base + cl) * HW;
            for (int q = 0; q < 4; ++q) {
                const int p = p0 + 4 * quad + q;
                if (p < HW) yb[p] = fmaf(ac[r][q], SC[cl], SC[kEvalPreCO + cl]);
            }
        }
    }
}

// ---- stem: Conv2d(3, Cout, 3, padding=1) + affine BN from running statistics, one launch ---------------------
struct EvalStemArgs {
    int B, Cout, H, W, rows;        // rows: image rows per block
    float eps;
    const float* x;                 // (B, 3, H, W)
    const float* par;               // conv weight (Cout,3,3,3), bn weight (Cout), bn bias (Cout)
    const float* running;           // running_mean[Cout], running_var[Cout]
    float* out;                     // (B, Cout, H, W)
};

PCD_HOSTDEV size_t eval_stem_smem_floats(int Cout, int rows, int W) { return (size_t)Cout * 29 + (size_t)3 * (rows + 2) * (W + 2); }

PCD_HD void eval_stem_body(const EvalStemArgs& a, int bx, int n, float* smem) {
    const int Cout = a.Cout, rows = a.rows, PW = a.W + 2, y0 = bx * rows;
    const long long HW = (long long)a.H * a.W;
    float* Wt = smem;                    // [Cout][27]
    float* SC = Wt + Cout * 27;          // scale[Cout], shift[Cout]
    float* XS = SC + 2 * Cout;           // [3][rows + 2][W + 2]
    const float* xb = a.x + (long long)n * 3 * HW;
    PCD_FOR(i, Cout * 27) Wt[i] = a.par[i];
    PCD_FOR(co, Cout) {
        const float sc = (1.f / sqrtf(a.running[Cout + co] + a.eps)) * a.par[Cout * 27 + co];
        SC[co] = sc;
        SC[Cout + co] = a.par[Cout * 28 + co] - a.running[co] * sc;
    }
    PCD_FOR(i, 3 * (rows + 2) * PW) {
        const int ci = i / ((rows + 2) * PW), r = (i / PW) % (rows + 2), q = i % PW;
        const int gy = y0 + r - 1, gx = q - 1;
        XS[i] = (gy >= 0 && gy < a.H && gx >= 0 && gx < a.W) ? xb[ci * HW + (long long)gy * a.W + gx] : 0.f;
    }
    PCD_SYNC();
    const int npx = rows * a.W;
    PCD_FOR(i, Cout * npx) {
        const int co = i / npx, p = i - co * npx, r = p / a.W, q = p - r * a.W;
        if (y0 + r < a.H) {
            const float* w = Wt + co * 27;
            float s = 0.f;
#pragma unroll
            for (int ci = 0; ci < 3; ++ci)
#pragma unroll
                for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx)
                        s = fmaf(w[ci * 9 + ky * 3 + kx], XS[(ci * (rows + 2) + r + ky) * PW + q + kx], s);
            a.out[((long long)n * Cout + co) * HW + (long long)(y0 + r) * a.W + q] = fmaf(s, SC[co], SC[Cout + co]);
        }
    }
}

// host launchers (pcd_k_eval.cu)
int launch_eval_node(const EvalNodeArgs& a, int c, void* stream);
int launch_eval_pre(const EvalPreArgs& a, void* stream);
int launch_eval_stem(const EvalStemArgs& a, void* stream);

}  // namespace pcd
