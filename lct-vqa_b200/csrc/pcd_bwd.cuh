// pcd_bwd.cuh — backward kernel bodies.
//
// Backward of a node sum + its incoming MixedOp edges, split at the BatchNorm-backward reductions:
//   node_stats  : per node   sum h, sum h*z_k, sum h*xs, bypass dot  (h = dN[:, 0::4])
//   edge_bwdB   : second halves of the separable convs -> grad of the mid tensor (GA) + its sums,
//                 weight grads of the second dw/pw pair
//   edge_bwdA   : everything that reads the edge input xs: first sep halves, dilated convs, pools,
//                 skip / FactorizedReduce -> d xs, weight grads
//   source_grad : per source state: d state = [sum_e d xs_e | sum_e beta_e * unshuffled dN] (+ cell-output grad)
//   arch_grads  : d softmax(alpha) rows and d beta from the reduction scratch
#pragma once
#include "pcd_fwd.cuh"

namespace pcd {

// ---- node_stats -------------------------------------------------------------------------------------
struct EdgeS {
    const float* x;
    long long x_ns;
    int stride, Hs, Ws;
    const float* saved;
    double* bstats;
};

struct NodeStatsArgs {
    int B, Ho, Wo, px_per_block;
    const float* dn;       // node grad (B, C, Ho, Wo) view
    long long dn_ns;
    int nin;
    EdgeS e[kMaxNodeIn];
};

constexpr int kStatK = 9;

PCD_HOSTDEV size_t node_stats_smem_floats(int C) { return (size_t)kStatK * 1024 + (size_t)kStatK * C * 32 + 16; }

template <int C>
PCD_HD void node_stats_body(const NodeStatsArgs& a, int bx, int n, int ez, float* smem) {
    const EdgeS& e = a.e[ez];
    const int HW = a.Ho * a.Wo, PXB = a.px_per_block, NSTRIP = PXB / 4, NT = C * NSTRIP;
    float* P = smem;
    float* P2 = P + kStatK * 1024;
    const int p0 = bx * PXB;
    const long long nslot = (long long)a.B * C * HW;
    const float* dnb = a.dn + (long long)n * a.dn_ns;
    const float* xb = e.x + (long long)n * e.x_ns;
    const int s = e.stride;
    const bool vec = (HW % 4 == 0) && (PXB % 4 == 0) && ((((uintptr_t)a.dn) | ((uintptr_t)e.x) | ((uintptr_t)e.saved)) & 15) == 0 &&
                     a.dn_ns % 4 == 0 && e.x_ns % 4 == 0 && (s == 1 || (a.Wo % 4 == 0 && e.Ws % 4 == 0));
    if (vec) {
        PCD_FOR(task, NT) {
            const int j = task / NSTRIP, strip = task - j * NSTRIP;
            float acc[kStatK];
#pragma unroll
            for (int k = 0; k < kStatK; ++k) acc[k] = 0.f;
            const int p = p0 + strip * 4;
            if (p < HW) {
                const int slots[6] = {slot_p1(), slot_p2(), slot_z(1), slot_z(3), slot_z(4), slot_z(5)};
                const F4 h4 = *reinterpret_cast<const F4*>(dnb + (long long)(4 * j) * HW + p);
                const float h[4] = {h4.x, h4.y, h4.z, h4.w};
                const float* sv = e.saved + ((long long)n * C + j) * HW + p;
                acc[0] = (h[0] + h[1]) + (h[2] + h[3]);
#pragma unroll
                for (int k = 0; k < 6; ++k) {
                    const F4 v = *reinterpret_cast<const F4*>(sv + slots[k] * nslot);
                    acc[1 + k] = fmaf(h[0], v.x, fmaf(h[1], v.y, fmaf(h[2], v.z, h[3] * v.w)));
                }
                if (s == 1) {
                    const F4 v = *reinterpret_cast<const F4*>(xb + (long long)j * HW + p);
                    acc[7] = fmaf(h[0], v.x, fmaf(h[1], v.y, fmaf(h[2], v.z, h[3] * v.w)));
#pragma unroll
                    for (int q = 1; q < 4; ++q) {
                        const F4 d = *reinterpret_cast<const F4*>(dnb + (long long)(4 * j + q) * HW + p);
                        const F4 b = *reinterpret_cast<const F4*>(xb + (long long)(q * C + j) * HW + p);
                        acc[8] += fmaf(d.x, b.x, fmaf(d.y, b.y, fmaf(d.z, b.z, d.w * b.w)));
                    }
                } else {
                    const F4 v = *reinterpret_cast<const F4*>(sv + slot_f() * nslot);
                    acc[7] = fmaf(h[0], v.x, fmaf(h[1], v.y, fmaf(h[2], v.z, h[3] * v.w)));
                    const int oy = p / a.Wo, ox = p - oy * a.Wo;
#pragma unroll
                    for (int q = 1; q < 4; ++q) {
                        const F4 d = *reinterpret_cast<const F4*>(dnb + (long long)(4 * j + q) * HW + p);
                        const float* pl = xb + (long long)(q * C + j) * e.Hs * e.Ws + (long long)(2 * oy) * e.Ws + 2 * ox;
                        const F4 r0a = *reinterpret_cast<const F4*>(pl), r0b = *reinterpret_cast<const F4*>(pl + 4);
                        const F4 r1a = *reinterpret_cast<const F4*>(pl + e.Ws), r1b = *reinterpret_cast<const F4*>(pl + e.Ws + 4);
                        const float w0 = fmaxf(fmaxf(r0a.x, r0a.y), fmaxf(r1a.x, r1a.y));
                        const float w1 = fmaxf(fmaxf(r0a.z, r0a.w), fmaxf(r1a.z, r1a.w));
                        const float w2 = fmaxf(fmaxf(r0b.x, r0b.y), fmaxf(r1b.x, r1b.y));
                        const float w3 = fmaxf(fmaxf(r0b.z, r0b.w), fmaxf(r1b.z, r1b.w));
                        acc[8] += fmaf(d.x, w0, fmaf(d.y, w1, fmaf(d.z, w2, d.w * w3)));
                    }
                }
            }
#pragma unroll
            for (int k = 0; k < kStatK; ++k) P[k * NT + task] = acc[k];
        }
    } else
    PCD_FOR(task, NT) {
        const int j = task / NSTRIP, strip = task - j * NSTRIP;
        float acc[kStatK];
#pragma unroll
        for (int k = 0; k < kStatK; ++k) acc[k] = 0.f;
        const int slots[6] = {slot_p1(), slot_p2(), slot_z(1), slot_z(3), slot_z(4), slot_z(5)};
        for (int t = 0; t < 4; ++t) {
            const int p = p0 + strip * 4 + t;
            if (p >= HW) break;
            const float h = dnb[(long long)(4 * j) * HW + p];
            const long long so = ((long long)n * C + j) * HW + p;
            acc[0] += h;
#pragma unroll
            for (int k = 0; k < 6; ++k) acc[1 + k] = fmaf(h, e.saved[slots[k] * nslot + so], acc[1 + k]);
            if (s == 1) {
                acc[7] = fmaf(h, xb[(long long)j * HW + p], acc[7]);
#pragma unroll
                for (int q = 1; q < 4; ++q)
                    acc[8] = fmaf(dnb[(long long)(4 * j + q) * HW + p], xb[(long long)(q * C + j) * HW + p], acc[8]);
            } else {
                acc[7] = fmaf(h, e.saved[slot_f() * nslot + so], acc[7]);
                const int oy = p / a.Wo, ox = p - oy * a.Wo;
#pragma unroll
                for (int q = 1; q < 4; ++q) {
                    const float* pl = xb + (long long)(q * C + j) * e.Hs * e.Ws + (2 * oy) * e.Ws + 2 * ox;
                    float v = pl[0];
                    v = pl[1] > v ? pl[1] : v;
                    v = pl[e.Ws] > v ? pl[e.Ws] : v;
                    v = pl[e.Ws + 1] > v ? pl[e.Ws + 1] : v;
                    acc[8] = fmaf(dnb[(long long)(4 * j + q) * HW + p], v, acc[8]);
                }
            }
        }
#pragma unroll
        for (int k = 0; k < kStatK; ++k) P[k * NT + task] = acc[k];
    }
    reduce_columns(P, P2, kStatK, C, NSTRIP, NT, [&](int j, int k, float v) {
        int row;
        if (k == 0) row = bs_s0();
        else if (k == 1) row = bs_sz(bn_p1());
        else if (k == 2) row = bs_sz(bn_p2());
        else if (k == 3) row = bs_sz(bn_unit(s, 1));
        else if (k == 4) row = bs_sz(bn_unit(s, 3));
        else if (k == 5) row = bs_sz(bn_unit(s, 4));
        else if (k == 6) row = bs_sz(bn_unit(s, 5));
        else if (k == 7) row = (s == 2) ? bs_sz(bn_f()) : bs_sx();
        else { pcd_atomic_add(e.bstats + 15 * C, (double)v); return; }
        pcd_atomic_add(e.bstats + row * C + j, (double)v);
    });
}

// ---- source_grad ----------------------------------------------------------------------------------------
struct SrcEdge {
    const float* pd;       // partial d xs slots of this edge (see EdgeG::pd), each (B, c, Hs, Ws)
    const float* dn;       // node grad of the consumer (B, C, Ho, Wo) view
    long long dn_ns;
    const float* beta;     // null => 1
    int stride;
    int merged;            // set: the two slots of the production backward (bwdA4): slot 0 = the ReLU-masked sum of the conv / FR
                           // partials, slot 1 = max-pool + avg-pool(+identity).  Clear: the generic kernels' per-job slots
};

constexpr int kMaxSrcEdges = 4;

struct SourceGradArgs {
    int B, C, Hs, Ws;
    const float* x;        // the source state itself (ReLU mask; 2x2 max-pool argmax at stride 2)
    long long x_ns;
    const float* g0;       // optional initial grad (cell-output slice), same view geometry as `out`
    long long g0_ns;
    float* out;            // d source (B, C, Hs, Ws) view
    long long out_ns;
    int nedges;
    int nimg;              // images per block (blockIdx.z covers ceil(B / nimg)); >1 when planes are small
    double* bn_sums;       // optional [2][C]: += sum out, sum out * x per channel — the BatchNorm-backward reductions of the
                           // preprocess op that produced x (x is its normalised output), fused here instead of a separate pass
    SrcEdge e[kMaxSrcEdges];
};

// block total of two per-thread partial sums -> two fp64 atomics per warp (emulation: the block's tasks ran in one loop)
PCD_HD void src_bn_flush(double* dst, int C, int ch, float s, float q) {
#if PCD_CUDA
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        q += __shfl_xor_sync(0xffffffffu, q, o);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(dst + ch, (double)s);
        atomicAdd(dst + C + ch, (double)q);
    }
#else
    dst[ch] += (double)s;
    dst[C + ch] += (double)q;
#endif
}

// d x[:, ch<c]  = g0 + sum_e [ relu'(x) * (A3 + A5 + D3 + D5 (+ FR)) + max-pool + avg-pool(+identity) partials ]
// d x[:, q*c+j] = g0 + sum_e beta_e * (dN_e[:, 4j+q]  |  routed through the 2x2 max-pool argmax at stride 2)
// block (bx, ch, nz): pixel chunk bx of channel ch for images nz*nimg .. (several images per block when planes are small)
PCD_HD void source_grad_body(const SourceGradArgs& a, int bx, int ch, int nz) {
    const int HW = a.Hs * a.Ws, c = a.C / 4;
    const int p0 = bx * 4096;
    const int npx = (HW - p0) < 4096 ? (HW - p0) : 4096;
    const int nimg = a.nimg > 0 ? a.nimg : 1, n0 = nz * nimg;
    const long long pslot = (long long)a.B * c * HW;
    const bool vec = (HW % 4 == 0) && (p0 % 4 == 0) && ((((uintptr_t)a.out) | ((uintptr_t)a.x)) & 15) == 0 &&
                     a.out_ns % 4 == 0 && a.x_ns % 4 == 0 && (!a.g0 || (((((uintptr_t)a.g0) & 15) == 0) && a.g0_ns % 4 == 0));
    const int tpp = npx / 4;          // float4 tasks per plane chunk
    bool all_merged = true, all_s1 = true;
    for (int k = 0; k < a.nedges; ++k) {
        all_merged = all_merged && a.e[k].merged;
        all_s1 = all_s1 && a.e[k].stride == 1;
    }
    float bs = 0.f, bq = 0.f;          // BatchNorm-backward partial sums (bn_sums): per thread; the emulation loops once per block
    if (ch < c && vec && all_merged) {
        // production path: every load of a task (2 per edge + x + initial grad) is issued before the first use
        PCD_FOR(tt, nimg * tpp) {
            const int n = n0 + tt / tpp, i4 = tt % tpp;
            if (n >= a.B) continue;
            const int p = p0 + i4 * 4;
            const long long off = ((long long)n * c + ch) * HW + p;
            F4 m[kMaxSrcEdges], q4[kMaxSrcEdges];
#pragma unroll
            for (int k = 0; k < kMaxSrcEdges; ++k)
                if (k < a.nedges) {
                    m[k] = *reinterpret_cast<const F4*>(a.e[k].pd + off);
                    q4[k] = *reinterpret_cast<const F4*>(a.e[k].pd + off + pslot);
                }
            const F4 xv = *reinterpret_cast<const F4*>(a.x + (long long)n * a.x_ns + (long long)ch * HW + p);
            F4 v = {0.f, 0.f, 0.f, 0.f};
            if (a.g0) v = *reinterpret_cast<const F4*>(a.g0 + (long long)n * a.g0_ns + (long long)ch * HW + p);
#pragma unroll
            for (int k = 0; k < kMaxSrcEdges; ++k)
                if (k < a.nedges) {
                    v.x += m[k].x + q4[k].x;
                    v.y += m[k].y + q4[k].y;
                    v.z += m[k].z + q4[k].z;
                    v.w += m[k].w + q4[k].w;
                }
            *reinterpret_cast<F4*>(a.out + (long long)n * a.out_ns + (long long)ch * HW + p) = v;
            bs += (v.x + v.y) + (v.z + v.w);
            bq = fmaf(v.x, xv.x, fmaf(v.y, xv.y, fmaf(v.z, xv.z, fmaf(v.w, xv.w, bq))));
        }
        if (a.bn_sums) src_bn_flush(a.bn_sums, a.C, ch, bs, bq);
        return;
    }
    if (ch < c && vec) {
        PCD_FOR(tt, nimg * tpp) {
            const int n = n0 + tt / tpp, i4 = tt % tpp;
            if (n >= a.B) continue;
            float* ob = a.out + (long long)n * a.out_ns + (long long)ch * HW;
            const float* xb = a.x + (long long)n * a.x_ns + (long long)ch * HW;
            const int p = p0 + i4 * 4;
            F4 v = {0.f, 0.f, 0.f, 0.f};
            if (a.g0) v = *reinterpret_cast<const F4*>(a.g0 + (long long)n * a.g0_ns + (long long)ch * HW + p);
            const F4 xv = *reinterpret_cast<const F4*>(xb + p);
            for (int k = 0; k < a.nedges; ++k) {
                const SrcEdge& e = a.e[k];
                const float* pd = e.pd + ((long long)n * c + ch) * HW + p;
                if (e.merged) {
                    const F4 m = *reinterpret_cast<const F4*>(pd), q4 = *reinterpret_cast<const F4*>(pd + pslot);
                    v.x += m.x + q4.x;
                    v.y += m.y + q4.y;
                    v.z += m.z + q4.z;
                    v.w += m.w + q4.w;
                    continue;
                }
                F4 m = {0.f, 0.f, 0.f, 0.f};
                for (int s = 0; s < 4; ++s) {
                    const F4 t = *reinterpret_cast<const F4*>(pd + s * pslot);
                    m.x += t.x; m.y += t.y; m.z += t.z; m.w += t.w;
                }
                if (e.stride == 2) {
                    const F4 t = *reinterpret_cast<const F4*>(pd + 6 * pslot);
                    m.x += t.x; m.y += t.y; m.z += t.z; m.w += t.w;
                }
                const F4 p4 = *reinterpret_cast<const F4*>(pd + 4 * pslot);
                const F4 p5 = *reinterpret_cast<const F4*>(pd + 5 * pslot);
                v.x += (xv.x > 0.f ? m.x : 0.f) + p4.x + p5.x;
                v.y += (xv.y > 0.f ? m.y : 0.f) + p4.y + p5.y;
                v.z += (xv.z > 0.f ? m.z : 0.f) + p4.z + p5.z;
                v.w += (xv.w > 0.f ? m.w : 0.f) + p4.w + p5.w;
            }
            *reinterpret_cast<F4*>(ob + p) = v;
            bs += (v.x + v.y) + (v.z + v.w);
            bq = fmaf(v.x, xv.x, fmaf(v.y, xv.y, fmaf(v.z, xv.z, fmaf(v.w, xv.w, bq))));
        }
        if (a.bn_sums) src_bn_flush(a.bn_sums, a.C, ch, bs, bq);
        return;
    }
    bool vecb = vec && ch >= c && a.Ws % 4 == 0;
    for (int k = 0; k < a.nedges; ++k)
        vecb = vecb && ((((uintptr_t)a.e[k].dn) & 15) == 0) && a.e[k].dn_ns % 4 == 0 && (a.e[k].stride == 1 || a.Ws % 8 == 0);
    if (vecb && all_s1) {
        // bypass channels, every consumer at stride 1: one load per edge, all in flight together
        const int q = ch / c, j = ch - q * c;
        PCD_FOR(tt, nimg * tpp) {
            const int n = n0 + tt / tpp, i4 = tt % tpp;
            if (n >= a.B) continue;
            const int p = p0 + i4 * 4;
            F4 d[kMaxSrcEdges];
#pragma unroll
            for (int k = 0; k < kMaxSrcEdges; ++k)
                if (k < a.nedges) d[k] = *reinterpret_cast<const F4*>(a.e[k].dn + (long long)n * a.e[k].dn_ns + (long long)(4 * j + q) * HW + p);
            F4 v = {0.f, 0.f, 0.f, 0.f};
            if (a.g0) v = *reinterpret_cast<const F4*>(a.g0 + (long long)n * a.g0_ns + (long long)ch * HW + p);
#pragma unroll
            for (int k = 0; k < kMaxSrcEdges; ++k)
                if (k < a.nedges) {
                    const float beta = a.e[k].beta ? a.e[k].beta[0] : 1.f;
                    v.x = fmaf(beta, d[k].x, v.x); v.y = fmaf(beta, d[k].y, v.y); v.z = fmaf(beta, d[k].z, v.z); v.w = fmaf(beta, d[k].w, v.w);
                }
            *reinterpret_cast<F4*>(a.out + (long long)n * a.out_ns + (long long)ch * HW + p) = v;
            if (a.bn_sums) {
                const F4 xv = *reinterpret_cast<const F4*>(a.x + (long long)n * a.x_ns + (long long)ch * HW + p);
                bs += (v.x + v.y) + (v.z + v.w);
                bq = fmaf(v.x, xv.x, fmaf(v.y, xv.y, fmaf(v.z, xv.z, fmaf(v.w, xv.w, bq))));
            }
        }
        if (a.bn_sums) src_bn_flush(a.bn_sums, a.C, ch, bs, bq);
        return;
    }
    if (vecb) {
        const int q = ch / c, j = ch - q * c;
        PCD_FOR(tt, nimg * tpp) {
            const int n = n0 + tt / tpp, i4 = tt % tpp;
            if (n >= a.B) continue;
            float* ob = a.out + (long long)n * a.out_ns + (long long)ch * HW;
            const float* xb = a.x + (long long)n * a.x_ns + (long long)ch * HW;
            const int p = p0 + i4 * 4;
            F4 v = {0.f, 0.f, 0.f, 0.f};
            if (a.g0) v = *reinterpret_cast<const F4*>(a.g0 + (long long)n * a.g0_ns + (long long)ch * HW + p);
            for (int k = 0; k < a.nedges; ++k) {
                const SrcEdge& e = a.e[k];
                const float beta = e.beta ? e.beta[0] : 1.f;
                if (e.stride == 1) {
                    const F4 d = *reinterpret_cast<const F4*>(e.dn + (long long)n * e.dn_ns + (long long)(4 * j + q) * HW + p);
                    v.x = fmaf(beta, d.x, v.x); v.y = fmaf(beta, d.y, v.y); v.z = fmaf(beta, d.z, v.z); v.w = fmaf(beta, d.w, v.w);
                } else {
                    const int y = p / a.Ws, x = p - y * a.Ws;           // x is a multiple of 4: two 2x2 windows
                    const int oy = y >> 1, ox = x >> 1, Ho = a.Hs >> 1, Wo = a.Ws >> 1;
                    const float* pl = xb + (long long)(2 * oy) * a.Ws + x;
                    const F4 r0 = *reinterpret_cast<const F4*>(pl), r1 = *reinterpret_cast<const F4*>(pl + a.Ws);
                    const float* dp = e.dn + (long long)n * e.dn_ns + ((long long)(4 * j + q) * Ho + oy) * Wo + ox;
                    const float d0 = dp[0], d1 = dp[1];
                    const float w0[4] = {r0.x, r0.y, r1.x, r1.y}, w1[4] = {r0.z, r0.w, r1.z, r1.w};
                    int b0 = 0, b1 = 0;
                    float m0 = w0[0], m1 = w1[0];
#pragma unroll
                    for (int t = 1; t < 4; ++t) {
                        if (w0[t] > m0) { m0 = w0[t]; b0 = t; }
                        if (w1[t] > m1) { m1 = w1[t]; b1 = t; }
                    }
                    const int row = (y & 1) * 2;
                    if (b0 == row) v.x = fmaf(beta, d0, v.x);
                    if (b0 == row + 1) v.y = fmaf(beta, d0, v.y);
                    if (b1 == row) v.z = fmaf(beta, d1, v.z);
                    if (b1 == row + 1) v.w = fmaf(beta, d1, v.w);
                }
            }
            *reinterpret_cast<F4*>(ob + p) = v;
            if (a.bn_sums) {
                const F4 xv = *reinterpret_cast<const F4*>(xb + p);
                bs += (v.x + v.y) + (v.z + v.w);
                bq = fmaf(v.x, xv.x, fmaf(v.y, xv.y, fmaf(v.z, xv.z, fmaf(v.w, xv.w, bq))));
            }
        }
        if (a.bn_sums) src_bn_flush(a.bn_sums, a.C, ch, bs, bq);
        return;
    }
    PCD_FOR(tt, nimg * npx) {
        const int n = n0 + tt / npx, i = tt % npx;
        if (n >= a.B) continue;
        float* ob = a.out + (long long)n * a.out_ns + (long long)ch * HW;
        const float* xb = a.x + (long long)n * a.x_ns + (long long)ch * HW;
        const int p = p0 + i;
        float v = a.g0 ? a.g0[(long long)n * a.g0_ns + (long long)ch * HW + p] : 0.f;
        for (int k = 0; k < a.nedges; ++k) {
            const SrcEdge& e = a.e[k];
            if (ch < c) {
                const float* pd = e.pd + ((long long)n * c + ch) * HW + p;
                if (e.merged) {
                    v += pd[0] + pd[pslot];
                    continue;
                }
                float m = pd[0] + pd[pslot] + pd[2 * pslot] + pd[3 * pslot];
                if (e.stride == 2) m += pd[6 * pslot];
                v += (xb[p] > 0.f ? m : 0.f) + pd[4 * pslot] + pd[5 * pslot];
            } else {
                const int q = ch / c, j = ch - q * c;     // x channel q*c + j  <->  node channel 4j + q
                const float beta = e.beta ? e.beta[0] : 1.f;
                if (e.stride == 1) {
                    v = fmaf(beta, e.dn[(long long)n * e.dn_ns + (long long)(4 * j + q) * HW + p], v);
                } else {
                    const int y = p / a.Ws, x = p - y * a.Ws;
                    const int oy = y >> 1, ox = x >> 1, Ho = a.Hs >> 1, Wo = a.Ws >> 1;
                    const float* pl = a.x + (long long)n * a.x_ns + (long long)ch * HW + (2 * oy) * a.Ws + 2 * ox;
                    int best = 0;
                    float m = pl[0];
                    if (pl[1] > m) { m = pl[1]; best = 1; }
                    if (pl[a.Ws] > m) { m = pl[a.Ws]; best = 2; }
                    if (pl[a.Ws + 1] > m) { m = pl[a.Ws + 1]; best = 3; }
                    if (best == (y & 1) * 2 + (x & 1))
                        v = fmaf(beta, e.dn[(long long)n * e.dn_ns + ((long long)(4 * j + q) * Ho + oy) * Wo + ox], v);
                }
            }
        }
        ob[p] = v;
        bs += v;
        bq = fmaf(v, xb[p], bq);
    }
    if (a.bn_sums) src_bn_flush(a.bn_sums, a.C, ch, bs, bq);
}

// ---- arch_grads -----------------------------------------------------------------------------------------
struct ArchEdge {
    const double* stats;
    const double* bstats;
    const float* alpha;
    const float* beta;
    int stride;
    double count;
    float* gw;     // 8 floats
    float* gw2;    // 1 float or null
};

struct ArchGradArgs {
    int c, nedges;
    float eps;
    ArchEdge e[PCD_MAX_EDGES_CONST];
};

PCD_HOSTDEV size_t arch_grads_smem_floats() { return 2 * PCD_MAX_EDGES_CONST * 8 + 16; }

PCD_HD void arch_grads_body(const ArchGradArgs& a, float* smem) {
    double* D = reinterpret_cast<double*>(smem);          // [edge][8]
    PCD_FOR(t, a.nedges * 8) {
        const int ei = t >> 3, k = t & 7;
        const ArchEdge& e = a.e[ei];
        const int c = a.c, s = e.stride;
        // primitive k -> BN id (or -1): none | max | avg | skip | sep3 | sep5 | dil3 | dil5
        int bn = -1;
        if (k == 1) bn = bn_p1();
        else if (k == 2) bn = bn_p2();
        else if (k == 3) bn = (s == 2) ? bn_f() : -1;
        else if (k >= 4) bn = bn_unit(s, k == 4 ? 1 : k == 5 ? 3 : k == 6 ? 4 : 5);
        double acc = 0.0;
        if (bn >= 0) {
            for (int j = 0; j < c; ++j) {
                BnC b = bn_consts(e.stats, c, bn, j, e.count, a.eps);
                acc += (double)b.rstd * (e.bstats[bs_sz(bn) * c + j] - (double)b.mean * e.bstats[bs_s0() * c + j]);
            }
        } else if (k == 3) {
            for (int j = 0; j < c; ++j) acc += e.bstats[bs_sx() * c + j];
        }
        D[t] = acc;
        const float beta = e.beta ? e.beta[0] : 1.f;
        e.gw[k] = (float)(beta * acc);
    }
    PCD_SYNC();
    PCD_FOR(ei, a.nedges) {
        const ArchEdge& e = a.e[ei];
        if (e.gw2) {
            double db = e.bstats[15 * a.c];
            for (int k = 0; k < 8; ++k) db += (double)e.alpha[k] * D[ei * 8 + k];
            e.gw2[0] = (float)db;
        }
    }
}

// ---- preprocess backward ---------------------------------------------------------------------------------
struct BnBwdStatArgs {
    int B, C, HW;
    const float* dy;       // (B, C, HW)
    const float* y;        // normalised output (affine=False) or pre-BN z when `stats` is given
    const double* stats;   // null => y is already normalised
    float eps;
    double* bstats;        // sum dy [C], sum dy*yhat [C]
};

PCD_HOSTDEV size_t bn_bwd_stats_smem_floats() { return 2 * 1024 + 2 * 32 + 16; }

// block (bx, ch): 4096 elements of channel ch, flattened over (image, pixel)
PCD_HD void bn_bwd_stats_body(const BnBwdStatArgs& a, int bx, int ch, int, float* smem) {
    float* P = smem;
    float* P2 = P + 2 * 1024;
    float mean = 0.f, rstd = 1.f;
    if (a.stats) {
        BnC b = bn_consts(a.stats, a.C, 0, ch, (double)a.B * a.HW, a.eps);
        mean = b.mean; rstd = b.rstd;
    }
    const bool vec = (a.HW % 4 == 0) && ((((uintptr_t)a.dy) | ((uintptr_t)a.y)) & 15) == 0;
    const long long total = (long long)a.B * a.HW;
    PCD_FOR(task, 1024) {
        float s = 0.f, q = 0.f;
        const long long t0 = (long long)bx * 4096 + 4 * task;
        if (vec) {
            if (t0 < total) {
                const long long n = t0 / a.HW, p = t0 - n * a.HW;
                const long long o = (n * a.C + ch) * a.HW + p;
                const F4 d = *reinterpret_cast<const F4*>(a.dy + o), y = *reinterpret_cast<const F4*>(a.y + o);
                s = (d.x + d.y) + (d.z + d.w);
                q = fmaf(d.x, (y.x - mean) * rstd, fmaf(d.y, (y.y - mean) * rstd, fmaf(d.z, (y.z - mean) * rstd, d.w * ((y.w - mean) * rstd))));
            }
        } else {
            for (int t = 0; t < 4; ++t) {
                const long long tt = t0 + t;
                if (tt < total) {
                    const long long n = tt / a.HW, p = tt - n * a.HW;
                    const long long o = (n * a.C + ch) * a.HW + p;
                    const float d = a.dy[o];
                    s += d;
                    q = fmaf(d, (a.y[o] - mean) * rstd, q);
                }
            }
        }
        P[task] = s;
        P[1024 + task] = q;
    }
    reduce_columns(P, P2, 2, 1, 1024, 1024, [&](int, int k, float v) {
        pcd_atomic_add(a.bstats + k * a.C + ch, (double)v);
    });
}

// ---- stem backward ---------------------------------------------------------------------------------------
struct StemBwdArgs {
    int B, Cout, H, W, PXB, nblocks_px, nblocks_launch;
    const float* x;
    const float* z;        // pre-BN conv output
    const float* dy;
    const float* gamma;
    const double* stats;
    const double* bstats;  // sum dy, sum dy*yhat
    float eps;
    float* gw;             // conv weight grad [Cout][27]
    float* ggamma;
    float* gbias;
};

PCD_HOSTDEV size_t stem_bwd_smem_floats(int Cout, int PXB) { return (size_t)Cout * 27 + (size_t)Cout * PXB + 5 * Cout + 16; }

PCD_HD void stem_bwd_body(const StemBwdArgs& a, int bx, int nblk, float* smem) {
    const int Cout = a.Cout, PXB = a.PXB, HW = a.H * a.W;
    float* WACC = smem;
    float* DZ = WACC + Cout * 27;
    float* COEF = DZ + Cout * PXB;
    const double cnt = (double)a.B * HW;
    PCD_FOR(i, Cout * 27) WACC[i] = 0.f;
    PCD_FOR(co, Cout) {
        BnC b = bn_consts(a.stats, Cout, 0, co, cnt, a.eps);
        COEF[5 * co] = b.rstd * a.gamma[co];
        COEF[5 * co + 1] = (float)(a.bstats[co] / cnt);
        COEF[5 * co + 2] = (float)(a.bstats[Cout + co] / cnt);
        COEF[5 * co + 3] = b.mean;
        COEF[5 * co + 4] = b.rstd;
        if (bx == 0) {
            a.gbias[co] = (float)a.bstats[co];
            a.ggamma[co] = (float)a.bstats[Cout + co];
        }
    }
    PCD_SYNC();
    const int per_img = (HW + PXB - 1) / PXB;
    for (int blk = bx; blk < a.nblocks_px; blk += nblk) {
        const int n = blk / per_img, p0 = (blk - n * per_img) * PXB;
        PCD_FOR(i, Cout * PXB) {
            const int co = i / PXB, t = i - co * PXB, p = p0 + t;
            float v = 0.f;
            if (p < HW) {
                const long long o = ((long long)n * Cout + co) * HW + p;
                const float yh = (a.z[o] - COEF[5 * co + 3]) * COEF[5 * co + 4];
                v = COEF[5 * co] * (a.dy[o] - COEF[5 * co + 1] - yh * COEF[5 * co + 2]);
            }
            DZ[i] = v;
        }
        PCD_SYNC();
        const float* xb = a.x + (long long)n * 3 * HW;
        PCD_FOR(task, (Cout / 4) * 27) {
            const int co0 = (task / 27) * 4, tap = task % 27;
            const int ci = tap / 9, ky = (tap / 3) % 3, kx = tap % 3;
            float acc[4] = {0.f, 0.f, 0.f, 0.f};
            for (int t = 0; t < PXB; ++t) {
                const int p = p0 + t;
                if (p >= HW) break;
                const int oy = p / a.W, ox = p - oy * a.W;
                const int gy = oy + ky - 1, gx = ox + kx - 1;
                if (gy < 0 || gy >= a.H || gx < 0 || gx >= a.W) continue;
                const float xv = xb[(long long)ci * HW + gy * a.W + gx];
#pragma unroll
                for (int i = 0; i < 4; ++i) acc[i] = fmaf(DZ[(co0 + i) * PXB + t], xv, acc[i]);
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) WACC[(co0 + i) * 27 + tap] += acc[i];
        }
        PCD_SYNC();
    }
    PCD_FOR(i, Cout * 27) pcd_atomic_add(a.gw + i, WACC[i]);
}

// ---- stem backward, v2: 4-row x full-width tiles, register accumulators across tiles -------------------------------
// dW[co][ci][ky][kx] = sum_{n,p} dz[co][p] * x[ci][p + (ky-1, kx-1)].  Task = (4 output channels, ci, ky) x pixel part;
// per float4 strip of pixels: 4 + 3 LDS.128, 48 FMA into 12 accumulators that live in registers over all the block's tiles.
constexpr int kStemTR = 4;
PCD_HOSTDEV bool stem_bwd2_ok(int Cout, int H, int W) { return Cout % 4 == 0 && (Cout / 4) * 9 <= kThreads && W % 4 == 0 && W <= 64 && H % kStemTR == 0; }
PCD_HOSTDEV size_t stem_bwd2_smem_floats(int Cout, int W) {
    return (size_t)Cout * kStemTR * W + (size_t)3 * (kStemTR + 2) * (W + 8) + 5 * Cout + 16;
}

PCD_HD void stem_bwd2_body(const StemBwdArgs& a, int bx, int nblk, float* smem) {
    const int Cout = a.Cout, W = a.W, H = a.H, HW = H * W, NPX = kStemTR * W, W4 = W / 4, XP = W + 8, XR = kStemTR + 2;
    float* DZ = smem;                         // [Cout][NPX]
    float* XT = DZ + Cout * NPX;              // [3][XR][XP]   (row halo 1, column halo 4)
    float* COEF = XT + 3 * XR * XP;
    float* P = DZ;                            // [12][kThreads] after the tile loop
    const int ncombo = (Cout / 4) * 9, nparts = kThreads / ncombo;
    const double cnt = (double)a.B * HW;
    PCD_FOR(co, Cout) {
        BnC b = bn_consts(a.stats, Cout, 0, co, cnt, a.eps);
        COEF[5 * co] = b.rstd * a.gamma[co];
        COEF[5 * co + 1] = (float)(a.bstats[co] / cnt);
        COEF[5 * co + 2] = (float)(a.bstats[Cout + co] / cnt);
        COEF[5 * co + 3] = b.mean;
        COEF[5 * co + 4] = b.rstd;
        if (bx == 0) {
            a.gbias[co] = (float)a.bstats[co];
            a.ggamma[co] = (float)a.bstats[Cout + co];
        }
    }
    PCD_TSTATE(float, acc, [4][3]);
    PCD_EACH(task) {
        auto& ac = PCD_TREF(acc, task);
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int k = 0; k < 3; ++k) ac[i][k] = 0.f;
    }
    const int tiles_per_img = H / kStemTR, ntiles = a.B * tiles_per_img;
    for (int tile = bx; tile < ntiles; tile += nblk) {
        const int n = tile / tiles_per_img, y0 = (tile - n * tiles_per_img) * kStemTR;
        PCD_SYNC();                           // COEF ready / previous tile's readers done
        PCD_FOR(i, Cout * NPX / 4) {
            const int co = i / (NPX / 4), s4 = i - co * (NPX / 4);
            const long long o = ((long long)n * Cout + co) * HW + (long long)y0 * W + 4 * s4;
            const F4 z4 = *reinterpret_cast<const F4*>(a.z + o), d4 = *reinterpret_cast<const F4*>(a.dy + o);
            const float c0 = COEF[5 * co], c1 = COEF[5 * co + 1], c2 = COEF[5 * co + 2], m = COEF[5 * co + 3], r = COEF[5 * co + 4];
            F4 v = {c0 * (d4.x - c1 - (z4.x - m) * r * c2), c0 * (d4.y - c1 - (z4.y - m) * r * c2),
                    c0 * (d4.z - c1 - (z4.z - m) * r * c2), c0 * (d4.w - c1 - (z4.w - m) * r * c2)};
            *reinterpret_cast<F4*>(DZ + co * NPX + 4 * s4) = v;
        }
        PCD_FOR(i, 3 * XR * (XP / 4)) {
            const int c4 = i % (XP / 4), rr = i / (XP / 4), r = rr % XR, ci = rr / XR;
            const int gy = y0 - 1 + r, gx = 4 * c4 - 4;
            F4 v = {0.f, 0.f, 0.f, 0.f};
            if (gy >= 0 && gy < H && gx >= 0 && gx < W) v = *reinterpret_cast<const F4*>(a.x + ((long long)n * 3 + ci) * HW + (long long)gy * W + gx);
            *reinterpret_cast<F4*>(XT + (ci * XR + r) * XP + 4 * c4) = v;
        }
        PCD_SYNC();
        PCD_EACH(task) {
            const int combo = task / nparts, part = task - combo * nparts;
            if (combo < ncombo) {
                auto& ac = PCD_TREF(acc, task);
                const int co0 = (combo / 9) * 4, cik = combo % 9, ci = cik / 3, ky = cik - ci * 3;
                for (int st = part; st < NPX / 4; st += nparts) {
                    const int r = st / W4, x4 = st - r * W4;
                    const float* xr = XT + (ci * XR + r + ky) * XP + 4 * x4;
                    const F4 a0 = *reinterpret_cast<const F4*>(xr), a1 = *reinterpret_cast<const F4*>(xr + 4), a2 = *reinterpret_cast<const F4*>(xr + 8);
                    const float v[6] = {a0.w, a1.x, a1.y, a1.z, a1.w, a2.x};        // image columns 4*x4 - 1 .. 4*x4 + 4
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const F4 d = *reinterpret_cast<const F4*>(DZ + (co0 + i) * NPX + 4 * st);
#pragma unroll
                        for (int kx = 0; kx < 3; ++kx)
                            ac[i][kx] = fmaf(d.x, v[kx], fmaf(d.y, v[kx + 1], fmaf(d.z, v[kx + 2], fmaf(d.w, v[kx + 3], ac[i][kx]))));
                    }
                }
            }
        }
    }
    PCD_SYNC();
    PCD_EACH(task) {
        auto& ac = PCD_TREF(acc, task);
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int k = 0; k < 3; ++k) P[(i * 3 + k) * kThreads + task] = ac[i][k];
    }
    PCD_SYNC();
    PCD_FOR(q, ncombo * 12) {
        const int combo = q / 12, ik = q - combo * 12, i = ik / 3, kx = ik - i * 3;
        float s = 0.f;
        for (int part = 0; part < nparts; ++part) s += P[ik * kThreads + combo * nparts + part];
        const int co = (combo / 9) * 4 + i, cik = combo % 9;
        pcd_atomic_add(a.gw + co * 27 + cik * 3 + kx, s);
    }
}

}  // namespace pcd
