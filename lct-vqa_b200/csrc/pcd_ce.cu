// pcd_ce.cu — cross-entropy over the vocabulary logits, fused around the tcgen05 projection (pcd_gemm_sm100.cu):
//   vqa_model.py:192-194  qst_out = fc1(tanh(lstm_out))            -> pcd_gemm_tn_3xtf32 into a padded-pitch buffer
//   vqa_model.py:356-358  CE(qst_out[:, :-1], qst[:, 1:])          -> pcd_ce_forward / pcd_ce_backward on that buffer
// The logits never get sliced / re-laid-out: rows whose target is negative (the last time step) or >= V are ignored, the
// gradient is written straight into the padded-pitch layout the backward GEMMs read through TMA, and
// pcd_transpose_pad produces the K-major operands (dlogits^T, W^T, h^T) of those GEMMs.
#include "../../include/pcdarts_sm100.h"
#include "pcd_launch.cuh"

#if PCD_CUDA

namespace pcd {
namespace ce {

constexpr int kCeThreads = 256;

__device__ __forceinline__ void online(float& m, float& s, float v) {
    if (v > m) { s = s * __expf(m - v) + 1.f; m = v; }
    else s += __expf(v - m);
}

// one block per row: online softmax statistics, lse and the row loss
__global__ void __launch_bounds__(kCeThreads) ce_fwd_kernel(const float* __restrict__ logits, long long ld, int V,
                                                            const long long* __restrict__ targets, float* __restrict__ lse,
                                                            float* __restrict__ loss_rows) {
    const int r = blockIdx.x;
    const float* row = logits + (long long)r * ld;
    float m = -INFINITY, s = 0.f;
    const int V4 = V / 4;
    for (int i = threadIdx.x; i < V4; i += kCeThreads) {
        const float4 v = *reinterpret_cast<const float4*>(row + 4 * i);
        online(m, s, v.x); online(m, s, v.y); online(m, s, v.z); online(m, s, v.w);
    }
    for (int c = 4 * V4 + threadIdx.x; c < V; c += kCeThreads) online(m, s, row[c]);
    __shared__ float sm[kCeThreads / 32], ss[kCeThreads / 32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float m2 = __shfl_xor_sync(0xffffffffu, m, o), s2 = __shfl_xor_sync(0xffffffffu, s, o);
        const float M = fmaxf(m, m2);
        s = (m == -INFINITY ? 0.f : s * __expf(m - M)) + (m2 == -INFINITY ? 0.f : s2 * __expf(m2 - M));
        m = M;
    }
    if ((threadIdx.x & 31) == 0) { sm[threadIdx.x >> 5] = m; ss[threadIdx.x >> 5] = s; }
    __syncthreads();
    if (threadIdx.x == 0) {
        float M = sm[0], S = ss[0];
        for (int w = 1; w < kCeThreads / 32; ++w) {
            const float M2 = fmaxf(M, sm[w]);
            S = (M == -INFINITY ? 0.f : S * __expf(M - M2)) + (sm[w] == -INFINITY ? 0.f : ss[w] * __expf(sm[w] - M2));
            M = M2;
        }
        const float l = M + logf(S);
        lse[r] = l;
        const long long t = targets[r];
        loss_rows[r] = (t >= 0 && t < V) ? l - row[t] : 0.f;
    }
}

// dlogits[r][c] = scale * (exp(x - lse_r) - [c == target_r]) for valid rows, 0 for ignored rows and pad columns
__global__ void __launch_bounds__(kCeThreads) ce_bwd_kernel(const float* __restrict__ logits, long long ld, int V,
                                                            const long long* __restrict__ targets, const float* __restrict__ lse,
                                                            const float* __restrict__ scale, float* __restrict__ dl) {
    const int r = blockIdx.y;
    const int c = (blockIdx.x * kCeThreads + threadIdx.x) * 4;
    if (c >= ld) return;
    const long long t = targets[r];
    const float sc = *scale, l = lse[r];
    const float4 x = *reinterpret_cast<const float4*>(logits + (long long)r * ld + c);
    float o[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int cc = c + j;
        // a row is ignored when its target is negative OR out of range, exactly as ce_fwd scores it (torch raises on >= V)
        o[j] = (t >= 0 && t < V && cc < V) ? sc * (__expf(o[j] - l) - (cc == t ? 1.f : 0.f)) : 0.f;
    }
    *reinterpret_cast<float4*>(dl + (long long)r * ld + c) = make_float4(o[0], o[1], o[2], o[3]);
}

// dst[c][r] = src[r][c] for r < R, c < C; dst columns [R, ld_d) are zero-filled
__global__ void __launch_bounds__(256) transpose_pad_kernel(const float* __restrict__ src, long long ld_s, int R, int C,
                                                            float* __restrict__ dst, long long ld_d) {
    __shared__ float tile[32][33];
    const int r0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;      // 32 x 8
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int r = r0 + ty + 8 * k, c = c0 + tx;
        tile[ty + 8 * k][tx] = (r < R && c < C) ? src[(long long)r * ld_s + c] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int c = c0 + ty + 8 * k, r = r0 + tx;
        if (c < C && r < ld_d) dst[(long long)c * ld_d + r] = tile[tx][ty + 8 * k];
    }
}

static int after_launch(const char* what) {
    LaunchState& L = launch_state();
    count_launch(L);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        snprintf(L.last_err, sizeof L.last_err, "launch %s: %s", what, cudaGetErrorString(e));
        return PCD_ERR_CUDA;
    }
    return PCD_OK;
}

}  // namespace ce
}  // namespace pcd

extern "C" {

int pcd_ce_forward(const float* logits, long long ld, int M, int V, const long long* targets, float* lse, float* loss_rows,
                   void* stream) {
    using namespace pcd;
    if (!logits || !targets || !lse || !loss_rows || M <= 0 || V <= 0 || ld < V) return PCD_ERR_ARG;
    if ((((uintptr_t)logits) & 15) || ld % 4) return PCD_ERR_ALIGN;
    ce::ce_fwd_kernel<<<M, ce::kCeThreads, 0, (cudaStream_t)stream>>>(logits, ld, V, targets, lse, loss_rows);
    return ce::after_launch("ce_fwd");
}

int pcd_ce_backward(const float* logits, long long ld, int M, int V, const long long* targets, const float* lse,
                    const float* scale, float* dlogits, void* stream) {
    using namespace pcd;
    if (!logits || !targets || !lse || !scale || !dlogits || M <= 0 || V <= 0 || ld < V) return PCD_ERR_ARG;
    if (((((uintptr_t)logits) | ((uintptr_t)dlogits)) & 15) || ld % 4) return PCD_ERR_ALIGN;
    dim3 grid((unsigned)((ld / 4 + ce::kCeThreads - 1) / ce::kCeThreads), (unsigned)M);
    ce::ce_bwd_kernel<<<grid, ce::kCeThreads, 0, (cudaStream_t)stream>>>(logits, ld, V, targets, lse, scale, dlogits);
    return ce::after_launch("ce_bwd");
}

int pcd_transpose_pad(const float* src, long long ld_s, int R, int C, float* dst, long long ld_d, void* stream) {
    using namespace pcd;
    if (!src || !dst || R <= 0 || C <= 0 || ld_s < C || ld_d < R) return PCD_ERR_ARG;
    dim3 grid((unsigned)((ld_d + 31) / 32), (unsigned)((C + 31) / 32));
    if (grid.y > 65535) return PCD_ERR_UNSUPPORTED;
    ce::transpose_pad_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(src, ld_s, R, C, dst, ld_d);
    return ce::after_launch("transpose_pad");
}

}  // extern "C"

#else   // ---- CPU emulation build (tests only) ----------------------------------------------------------------------

#include <math.h>

extern "C" {

int pcd_ce_forward(const float* logits, long long ld, int M, int V, const long long* targets, float* lse, float* loss_rows, void*) {
    if (!logits || !targets || !lse || !loss_rows) return PCD_ERR_ARG;
    for (int r = 0; r < M; ++r) {
        const float* row = logits + (long long)r * ld;
        float m = -INFINITY;
        for (int c = 0; c < V; ++c) m = row[c] > m ? row[c] : m;
        double s = 0.0;
        for (int c = 0; c < V; ++c) s += exp((double)row[c] - m);
        lse[r] = (float)(m + log(s));
        const long long t = targets[r];
        loss_rows[r] = (t >= 0 && t < V) ? lse[r] - row[t] : 0.f;
    }
    return PCD_OK;
}

int pcd_ce_backward(const float* logits, long long ld, int M, int V, const long long* targets, const float* lse,
                    const float* scale, float* dl, void*) {
    if (!logits || !targets || !lse || !scale || !dl) return PCD_ERR_ARG;
    for (int r = 0; r < M; ++r)
        for (long long c = 0; c < ld; ++c) {
            const long long t = targets[r];
            dl[r * ld + c] = (t >= 0 && t < V && c < V) ?*scale * (expf(logits[r * ld + c] - lse[r]) - (c == t ? 1.f : 0.f)) : 0.f;
        }
    return PCD_OK;
}

int pcd_transpose_pad(const float* src, long long ld_s, int R, int C, float* dst, long long ld_d, void*) {
    if (!src || !dst) return PCD_ERR_ARG;
    for (int c = 0; c < C; ++c)
        for (long long r = 0; r < ld_d; ++r) dst[c * ld_d + r] = r < R ? src[r * ld_s + c] : 0.f;
    return PCD_OK;
}

}  // extern "C"
#endif
