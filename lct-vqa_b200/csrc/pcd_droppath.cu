// pcd_droppath.cu — one node of a derived cell with drop-path (pcdarts/model.py Cell.forward):
//     node[b] = d1(b) * h1[b] + d2(b) * h2[b],   d_i(b) x = (x / keep) * m_i(b)  when input i is dropped, else x
// which is DARTS's `x.div_(keep_prob).mul_(mask)` on every non-Identity op output followed by the node's add, in one pass:
// 2 tensors read, 1 written (the stock composite makes up to 11 tensor passes).  The masks are the Philox function of
// pcd_philox.cuh, recomputed in the backward from the seed; the seed and keep are read from device memory, so a CUDA graph
// draws new masks on every replay and follows a changed keep without being captured again.
#include "../../include/pcdarts_sm100.h"
#include "pcd_launch.cuh"
#include "pcd_philox.cuh"

namespace pcd {
namespace droppath {

constexpr int kVecPerThread = 4;
constexpr int kVecPerBlock = kThreads * kVecPerThread;      // float4s of one sample per block

struct Args {
    long long n;                            // elements per sample (C*H*W)
    int drop1, drop2, cell, node, offset, vec;
    const unsigned long long* seed;
    const float* keep;
    const float* a;                         // forward: h1          backward: grad_node
    const float* b;                         // forward: h2          backward: -
    float* y1;                              // forward: node        backward: grad_h1 (may be null)
    float* y2;                              // forward: -           backward: grad_h2 (may be null)
};

// d * x in DARTS's order of operations: IEEE division by keep, then the mask (not a multiplication by 1 / keep)
PCD_HD float scaled(float x, bool drop, float keep, float m) {
#if PCD_CUDA
    return drop ? __fdiv_rn(x, keep) * m : x;
#else
    return drop ? (x / keep) * m : x;
#endif
}

template <bool kBwd>
struct KDropPath {
    static constexpr int kMinBlocks = 4;
    static const char* name() { return kBwd ? "droppath_sum_backward" : "droppath_sum_forward"; }

    static PCD_D void elem(const Args& a, long long i, bool d1, bool d2, float keep, float m1, float m2) {
        if (kBwd) {
            const float g = a.a[i];
            if (a.y1) a.y1[i] = scaled(g, d1, keep, m1);
            if (a.y2) a.y2[i] = scaled(g, d2, keep, m2);
        } else {
            a.y1[i] = scaled(a.a[i], d1, keep, m1) + scaled(a.b[i], d2, keep, m2);
        }
    }

    static PCD_D void run(const Args& a, int x, int s, int, float*) {
        const bool d1 = a.drop1 != 0, d2 = a.drop2 != 0;
        const float keep = (d1 || d2) ? a.keep[0] : 1.f;
        const unsigned long long seed = (d1 || d2) ? a.seed[0] : 0ull;
        const float m1 = d1 ? droppath_mask(seed, a.offset + s, a.cell, 2 * a.node, keep) : 1.f;
        const float m2 = d2 ? droppath_mask(seed, a.offset + s, a.cell, 2 * a.node + 1, keep) : 1.f;
        const long long n = a.n, base = (long long)s * n;
        // scalar head up to the sample's first 16-byte boundary, float4 body, scalar tail (all scalar when a pointer is
        // not 16-byte aligned)
        long long head = a.vec ? ((4 - (base & 3)) & 3) : n;
        if (head > n) head = n;
        const long long nvec = (n - head) >> 2, tail0 = head + 4 * nvec;
        PCD_FOR(t, kThreads) {
            F4 va[kVecPerThread], vb[kVecPerThread];
#pragma unroll
            for (int k = 0; k < kVecPerThread; ++k) {
                const long long q = (long long)x * kVecPerBlock + k * kThreads + t;
                if (q < nvec) {
                    va[k] = *reinterpret_cast<const F4*>(a.a + base + head + 4 * q);
                    if (!kBwd) vb[k] = *reinterpret_cast<const F4*>(a.b + base + head + 4 * q);
                }
            }
#pragma unroll
            for (int k = 0; k < kVecPerThread; ++k) {
                const long long q = (long long)x * kVecPerBlock + k * kThreads + t;
                if (q >= nvec) continue;
                const long long i = base + head + 4 * q;
                if (kBwd) {
                    const F4 g = va[k];
                    if (a.y1) {
                        F4 o;
                        o.x = scaled(g.x, d1, keep, m1); o.y = scaled(g.y, d1, keep, m1);
                        o.z = scaled(g.z, d1, keep, m1); o.w = scaled(g.w, d1, keep, m1);
                        *reinterpret_cast<F4*>(a.y1 + i) = o;
                    }
                    if (a.y2) {
                        F4 o;
                        o.x = scaled(g.x, d2, keep, m2); o.y = scaled(g.y, d2, keep, m2);
                        o.z = scaled(g.z, d2, keep, m2); o.w = scaled(g.w, d2, keep, m2);
                        *reinterpret_cast<F4*>(a.y2 + i) = o;
                    }
                } else {
                    const F4 p = va[k], r = vb[k];
                    F4 o;
                    o.x = scaled(p.x, d1, keep, m1) + scaled(r.x, d2, keep, m2);
                    o.y = scaled(p.y, d1, keep, m1) + scaled(r.y, d2, keep, m2);
                    o.z = scaled(p.z, d1, keep, m1) + scaled(r.z, d2, keep, m2);
                    o.w = scaled(p.w, d1, keep, m1) + scaled(r.w, d2, keep, m2);
                    *reinterpret_cast<F4*>(a.y1 + i) = o;
                }
            }
            if (x == 0) {
                for (long long j = t; j < head; j += kThreads) elem(a, base + j, d1, d2, keep, m1, m2);
                for (long long j = tail0 + t; j < n; j += kThreads) elem(a, base + j, d1, d2, keep, m1, m2);
            }
        }
    }
};

static bool aligned16(const void* p) { return p == nullptr || ((uintptr_t)p & 15) == 0; }

static int validate(const pcd_droppath_args* p) {
    if (!p || p->batch < 0 || p->sample_numel < 0 || p->sample_offset < 0) return PCD_ERR_ARG;
    if ((long long)p->sample_offset + p->batch > 0x7fffffffLL) return PCD_ERR_ARG;     // the sample is one 32-bit counter word
    if ((p->drop1 || p->drop2) && (!p->seed || !p->keep)) return PCD_ERR_ARG;
    return PCD_OK;
}

static Args args_of(const pcd_droppath_args* p) {
    Args a;
    a.n = p->sample_numel;
    a.drop1 = p->drop1 != 0; a.drop2 = p->drop2 != 0;
    a.cell = p->cell; a.node = p->node; a.offset = p->sample_offset;
    a.seed = p->seed; a.keep = p->keep;
    a.a = a.b = nullptr; a.y1 = a.y2 = nullptr; a.vec = 0;
    return a;
}

static int grid_x(long long n) { return (int)((n / 4 + kVecPerBlock - 1) / kVecPerBlock) + (n < 4); }

}  // namespace droppath
}  // namespace pcd

using namespace pcd;
using namespace pcd::droppath;

extern "C" {

int pcd_droppath_sum_forward(const pcd_droppath_args* p, void* stream) {
    PCD_TRY(validate(p));
    if (p->batch == 0 || p->sample_numel == 0) return PCD_OK;
    if (!p->h1 || !p->h2 || !p->out) return PCD_ERR_ARG;
    Args a = args_of(p);
    a.a = p->h1; a.b = p->h2; a.y1 = p->out;
    a.vec = aligned16(a.a) && aligned16(a.b) && aligned16(a.y1);
    return launch<KDropPath<false>, Args>(a, grid_x(a.n), p->batch, 1, 0, stream);
}

int pcd_droppath_sum_backward(const pcd_droppath_args* p, void* stream) {
    PCD_TRY(validate(p));
    if (p->batch == 0 || p->sample_numel == 0) return PCD_OK;
    if (!p->grad_out) return PCD_ERR_ARG;
    if (!p->grad_h1 && !p->grad_h2) return PCD_OK;
    Args a = args_of(p);
    a.a = p->grad_out; a.y1 = p->grad_h1; a.y2 = p->grad_h2;
    a.vec = aligned16(a.a) && aligned16(a.y1) && aligned16(a.y2);
    return launch<KDropPath<true>, Args>(a, grid_x(a.n), p->batch, 1, 0, stream);
}

}  // extern "C"
