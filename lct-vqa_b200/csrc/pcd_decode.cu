// pcd_decode.cu — greedy question decode (vqa_model.py:103-136, models_lct.py:124-157) as ONE persistent cooperative
// kernel.  The reference runs, 30 times in a row, embedding -> one LSTM step -> tanh -> Linear(H, V) -> argmax: ~10 small
// launches per word whose next input depends on the previous argmax.  On the LCT path that loop runs three times per
// alpha-step (architect_lct.py:54,69).  Here the time loop lives inside the kernel; per word
//   phase A  (blocks 0 .. H/4-1, as in pcd_lstm.cu: block g owns 4 hidden units, its 16 rows of W_hh AND W_ih stay in
//             shared memory for all steps, the cell state in a register)
//             x = emb[word] (tanh only for <start>, vqa_model.py:119 vs :133);  gates = x W_ih^T + h W_hh^T + b;  h_t -> L2
//   -- grid barrier --
//   phase B  (every block: one 64 x 128 tile of the vocabulary)  logits = tanh(h_t) W_out^T + b_out: K chunks of 32 of
//             (tanh(h_t) rows | W_out tile rows; W_out is L2-resident, 36.6 MB at V = 17858) stream through a 4-stage
//             cp.async ring; 4 x 8 register tiles; row-wise argmax of the tile -> one packed (value, index) candidate per
//             row and tile
//   -- grid barrier --
//   the next phase A starts by reducing the candidates (lowest index wins ties, like torch.argmax) to the new words;
//   the input projection is split four ways along the embedding row (all ~19 float4 loads of a thread independent).
// The logits are never written anywhere.  Sampled decoding (deterministic=False: torch.multinomial over softmax(logits / T))
// is the same kernel with kSample = true: the phase-B epilogue ranks score = logit / T + G(seed, t, row, v) instead of the
// logit (Gumbel-max; G from pcd_philox.cuh, the seed read from device memory, so the kernel stays graph-capturable), and
// everything else — candidates, pick_words, barriers, phase A — is shared.
// Beam search (kMode = kBeam) decodes B items x K beams as B*K rows of the same kernel.  Phase B emits, per (row, tile),
// the tile's top-K (logit, index) pairs and its (max, sum exp(logit - max)); one more grid barrier follows, behind which
// block i merges item i: log-sum-exp per row, then the top K of the K^2 * ntiles candidates s_k + logit - lse_k.  The merge
// writes (word, parent row) packed into tokens[row][t]; the next phase A reads a row's word, stages h_{t-1} and reads c_{t-1}
// of its parent row (c_t goes to a double-buffered [2][rows][H] buffer), and after the last step block 0 backtracks the
// parent pointers in place.  An item's top K lies in the union of its rows' per-tile top K, so the reduction is exact.
// End-of-sequence decoding (kStop = true, one more instantiation per mode): a greedy / sampled row that has emitted
// end_token is fed pad_token and its later words are replaced by it (a per-row flag in shared memory); a finished beam
// contributes the single candidate (k, pad_token) with its score unchanged, the merge ranks by score / L^length_penalty and
// carries the raw score beside that key, and each row's frozen length persists in the workspace.  Every block sees every
// row's state (greedy / sampled: pick_words runs everywhere; beam: the lengths are read behind the merge barrier), so all
// blocks leave the time loop at the same step once every row has finished, without another barrier.
// Truncated sampling (kTrunc, sampled mode only: top-k and nucleus): the phase-B epilogue stores the logits into a
// [rows][V] workspace stash instead of ranking them; behind one more grid barrier each block takes whole rows, finds the
// kept set by radix select (select_words) and draws the Gumbel argmax over it into a word buffer, which the next step
// reads in place of pick_words.
#include "../../include/pcdarts_sm100.h"
#include "pcd_launch.cuh"
#include "pcd_philox.cuh"

#include <limits.h>

namespace pcd {
namespace decode {
enum { kGreedy = PCD_DECODE_GREEDY, kSampled = PCD_DECODE_SAMPLED, kBeam = PCD_DECODE_BEAM };
constexpr int kT = 256, kUnits = 4, kMaxB = 64, kMaxK = 8, kTileN = 128, kKC = 32, kWP = kKC + 4, kStages = 4, kPickJ = 5;
constexpr int kStageFloats = (kMaxB + kTileN) * kWP;
PCD_HOSTDEV int u_floats(int H) { return kMaxB * (H + 4) > kStages * kStageFloats ? kMaxB * (H + 4) : kStages * kStageFloats; }
static inline int tiles_of(int V) { return (V + kTileN - 1) / kTileN; }
static inline bool shape_ok(int T, int B, int H, int E, int V) {
    return T > 0 && B > 0 && B <= kMaxB && H >= 32 && H <= 512 && H % 32 == 0 && E > 0 && E % 4 == 0 && V > 0;
}
static inline bool beam_ok(int B, int K, int V) { return K >= 1 && K <= kMaxK && K <= V && B >= 1 && B <= kMaxB / K; }

// the status of a call before anything device-specific: every PCD_ERR_ARG comes before any shape check, so a beam shape
// outside the envelope is PCD_ERR_UNSUPPORTED only when every pointer is set
static int validate(const pcd_decode_args* a) {
    if (!a || a->mode < kGreedy || a->mode > kBeam || (a->mode != kBeam && a->K != 1)) return PCD_ERR_ARG;
    if (a->mode == kSampled && !(a->seed && a->row_offset >= 0 && isfinite(a->temperature) && a->temperature > 0.f))
        return PCD_ERR_ARG;
    if (a->stop && !(a->end_token >= 0 && a->end_token < a->V && a->pad_token >= 0 && a->pad_token < a->V &&
                     isfinite(a->length_penalty)))
        return PCD_ERR_ARG;
    if (a->truncate && !(a->mode == kSampled && a->top_k >= 0 && isfinite(a->top_p) && a->top_p > 0.f && a->top_p <= 1.f))
        return PCD_ERR_ARG;
    if (!a->emb || !a->w_ih || !a->w_hh || !a->b_ih || !a->b_hh || !a->h0 || !a->c0 || !a->w_out || !a->b_out || !a->tokens ||
        !a->work || (a->mode == kBeam && !a->scores))
        return PCD_ERR_ARG;
    if (a->mode == kBeam && !beam_ok(a->B, a->K, a->V)) return PCD_ERR_UNSUPPORTED;
    if (!shape_ok(a->T, a->B * a->K, a->H, a->E, a->V) || a->start_token < 0 || a->start_token >= a->V) return PCD_ERR_UNSUPPORTED;
    return PCD_OK;
}

// workspace offsets in floats, rows = B x K:  hbuf [2][rows][H] | tbuf [rows][H] | then greedy / sampled: candidates
// [rows][ntiles] float2 | truncated sampling only: logits [rows][V] | words [rows] int;  beam: cbuf [2][rows][H] | top-K
// candidates [rows][ntiles][K] float2 | tile (max, sum exp) [rows][ntiles] float2 | beam scores [rows] | finished lengths
// [rows] int (end-of-sequence decode)
struct Work {
    size_t tbuf, cand, cbuf, bcand, bstat, bscore, blen, stash, words, floats;
};
static Work work_of(int mode, int B, int K, int H, int V, bool truncate) {
    const size_t rows = (size_t)B * K, nt = tiles_of(V), rh = rows * H;
    Work w = {};
    w.tbuf = 2 * rh;
    if (mode == kBeam) {
        w.cbuf = 3 * rh;
        w.bcand = 5 * rh;
        w.bstat = w.bcand + 2 * rows * nt * K;
        w.bscore = w.bstat + 2 * rows * nt;
        w.blen = w.bscore + rows;
        w.floats = w.blen + rows;
    } else {
        w.cand = 3 * rh;
        w.floats = w.cand + 2 * rows * nt;
        if (truncate) {
            w.stash = w.floats;
            w.words = w.stash + rows * (size_t)V;
            w.floats = w.words + rows;
        }
    }
    return w;
}

// truncated sampling (pcdarts_sm100.h): the order-preserving image of (logit, word), larger logit first and ties to the
// lower word (-0 counts as +0), and a word's mass q = expf((l - lmax) / T) in fp32 as an integer multiple of 2^-s,
// s = 63 - bit length of V, so that the masses of a row sum exactly (in any order) below 2^63
PCD_HOSTDEV unsigned long long order_key(float l, int v) {
    const float z = l == 0.f ? 0.f : l;
    uint32_t b;
    memcpy(&b, &z, sizeof b);
    b ^= (b & 0x80000000u) ? 0xffffffffu : 0x80000000u;
    return ((unsigned long long)b << 32) | (0xffffffffu - (uint32_t)v);
}
PCD_HOSTDEV int mass_shift(int V) {
    int bits = 0;
    while (bits < 31 && (V >> bits)) ++bits;
    return 63 - bits;
}
PCD_HOSTDEV unsigned long long mass_of(float l, float lmax, float T, float scale) {
    return (unsigned long long)rintf(expf((l - lmax) / T) * scale);      // scale = 2^s: exact
}
// the nucleus target: Z rounded to fp64, times top_p, rounded up; never above Z
PCD_HOSTDEV unsigned long long nucleus_target(unsigned long long Z, float top_p) {
    const unsigned long long t = (unsigned long long)ceil((double)Z * (double)top_p);
    return t > Z ? Z : t;
}
}  // namespace decode
}  // namespace pcd

extern "C" size_t pcd_decode_work_floats(const pcd_decode_args* a) {
    return a ? pcd::decode::work_of(a->mode, a->B, a->K, a->H, a->V, a->mode == pcd::decode::kSampled && a->truncate).floats : 0;
}

#if PCD_CUDA
#include <cooperative_groups.h>
namespace cg = cooperative_groups;

namespace pcd {
namespace decode {

struct Args {
    int T, B, H, E, V, start, ntiles;
    const float *emb, *w_ih, *w_hh, *b_ih, *b_hh, *h0, *c0, *w_out, *b_out;
    long long* tokens;    // [B][T]
    float* hbuf;          // [2][B][H]  h_t, double-buffered by step parity
    float* tbuf;          // [B][H]     tanh(h_t): the input of the vocabulary projection
    float2* cand;         // [B][ntiles]  (logit or sampled score, index bits): one 8-byte word per row and vocabulary tile
    const unsigned long long* seed;   // sampled decode only: Philox key (device memory)
    float temperature;
    int row_offset;                   // global batch row of row 0 (batches above 64 are decoded in slices)
    // beam decode only (B above counts rows = items x K); tokens[row][t] holds (word | parent row << 32) until the backtrack
    int K;
    float* cbuf;          // [2][B][H]  c_t, double-buffered by step parity: a beam continues its parent's cell state
    float2* bcand;        // [B][ntiles][K]  a tile's top K (logit, index bits) of a row, best first
    float2* bstat;        // [B][ntiles]     (max, sum exp(logit - max)) of a row's tile
    float* bscore;        // [B]  cumulative log-probability of each beam
    float* scores;        // [B]  output
    // end-of-sequence decode only (kStop)
    int end_token, pad_token;
    float length_penalty; // beam: candidates ranked by score / L^length_penalty (0: by score)
    int* blen;            // [B]  beam: length of a finished beam counting end_token, 0 while it is live
    // truncated sampling only (kTrunc)
    int top_k;            // 0: no top-k limit
    float top_p;          // 1: no nucleus
    float* stash;         // [B][V]  the step's fp32 logits
    int* words;           // [B]     the step's words
};

__device__ __forceinline__ float sigm(float x) { return 1.f / (1.f + expf(-x)); }
__device__ __forceinline__ float dot4(float4 a, float4 b, float acc) {
    return fmaf(a.x, b.x, fmaf(a.y, b.y, fmaf(a.z, b.z, fmaf(a.w, b.w, acc))));
}
__device__ __forceinline__ bool better(float v, int i, float best, int bi) { return v > best || (v == best && i < bi); }

// [B][H] (L2: written by other SMs) -> shared memory rows of pitch H + 4, 16-byte cp.async, no commit; kMap: row bb
// takes source row PAR[bb] (a beam continues its parent's state)
template <bool kMap = false>
__device__ __forceinline__ void stage_rows(float* Hs, const float* src, int B, int H, const int* PAR = nullptr) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, HP = H + 4;
    for (int bb = warp; bb < B; bb += kT / 32) {
        const unsigned dst = (unsigned)__cvta_generic_to_shared(Hs + bb * HP);
        const float* s = src + (long long)(kMap ? PAR[bb] : bb) * H;
        for (int k = 4 * lane; k < H; k += 128)
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + 4u * k), "l"(s + k) : "memory");
    }
}

// candidates of the previous step -> TOK[row].  Warp w takes rows 8w .. 8w+7, lane l the tiles l, l+32, ...: the first
// kPickJ x 8 loads of a lane are independent (one L2 round trip for up to 32 kPickJ tiles), then 8 warp reductions.
__device__ __forceinline__ void pick_words(const Args& a, int* TOK) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float2 cv[8][kPickJ];
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        const int row = warp * 8 + r;
        const float2* cr = a.cand + (long long)(row < a.B ? row : 0) * a.ntiles;
#pragma unroll
        for (int j = 0; j < kPickJ; ++j) {
            const int k = lane + 32 * j;
            cv[r][j] = (row < a.B && k < a.ntiles) ? __ldcg(cr + k) : make_float2(-INFINITY, __int_as_float(INT_MAX));
        }
    }
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        const int row = warp * 8 + r;
        float best = -INFINITY;
        int bi = INT_MAX;
#pragma unroll
        for (int j = 0; j < kPickJ; ++j) {
            const int i = __float_as_int(cv[r][j].y);
            if (better(cv[r][j].x, i, best, bi)) { best = cv[r][j].x; bi = i; }
        }
        if (row < a.B)
            for (int k = lane + 32 * kPickJ; k < a.ntiles; k += 32) {          // only for V > 4096 kPickJ
                const float2 c = __ldcg(a.cand + (long long)row * a.ntiles + k);
                if (better(c.x, __float_as_int(c.y), best, bi)) { best = c.x; bi = __float_as_int(c.y); }
            }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (better(ov, oi, best, bi)) { best = ov; bi = oi; }
        }
        if (lane == 0 && row < a.B) TOK[row] = (bi >= 0 && bi < a.V) ? bi : 0;
    }
}

// candidate (score, key) into a list of kMaxK kept in `better` order; key = k * V + v (ties: lower beam, then lower word)
__device__ __forceinline__ void list_insert(float (&ls)[kMaxK], int (&lk)[kMaxK], float sc, int key) {
#pragma unroll
    for (int q = 0; q < kMaxK; ++q)
        if (better(sc, key, ls[q], lk[q])) {
            const float ts = ls[q]; const int tk = lk[q];
            ls[q] = sc; lk[q] = key; sc = ts; key = tk;
        }
}

// best (score, key) of a warp's list heads, in every lane; the lane that holds it drops its head
__device__ __forceinline__ void warp_pop(float (&ls)[kMaxK], int (&lk)[kMaxK], float& best, int& bk) {
    best = ls[0]; bk = lk[0];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, best, o);
        const int ok = __shfl_xor_sync(0xffffffffu, bk, o);
        if (better(ov, ok, best, bk)) { best = ov; bk = ok; }
    }
    if (bk != INT_MAX && lk[0] == bk) {
#pragma unroll
        for (int q = 0; q < kMaxK - 1; ++q) { ls[q] = ls[q + 1]; lk[q] = lk[q + 1]; }
        ls[kMaxK - 1] = -INFINITY; lk[kMaxK - 1] = INT_MAX;
    }
}

// the same two with a third value carried beside each entry (the end-of-sequence merge ranks by key, returns raw scores)
__device__ __forceinline__ void list_insert(float (&ls)[kMaxK], int (&lk)[kMaxK], float (&lr)[kMaxK], float sc, int key, float raw) {
#pragma unroll
    for (int q = 0; q < kMaxK; ++q)
        if (better(sc, key, ls[q], lk[q])) {
            const float ts = ls[q], tr = lr[q]; const int tk = lk[q];
            ls[q] = sc; lk[q] = key; lr[q] = raw; sc = ts; key = tk; raw = tr;
        }
}

__device__ __forceinline__ void warp_pop(float (&ls)[kMaxK], int (&lk)[kMaxK], float (&lr)[kMaxK], float& best, int& bk,
                                         float& braw) {
    best = ls[0]; bk = lk[0]; braw = lr[0];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, best, o);
        const int ok = __shfl_xor_sync(0xffffffffu, bk, o);
        const float orw = __shfl_xor_sync(0xffffffffu, braw, o);
        if (better(ov, ok, best, bk)) { best = ov; bk = ok; braw = orw; }
    }
    if (bk != INT_MAX && lk[0] == bk) {
#pragma unroll
        for (int q = 0; q < kMaxK - 1; ++q) { ls[q] = ls[q + 1]; lk[q] = lk[q + 1]; lr[q] = lr[q + 1]; }
        ls[kMaxK - 1] = -INFINITY; lk[kMaxK - 1] = INT_MAX; lr[kMaxK - 1] = -INFINITY;
    }
}

// ranking key of a hypothesis of length L with raw score s: s / L^alpha (s itself for alpha = 0)
__device__ __forceinline__ float rank_key(float s, int L, float alpha) { return alpha != 0.f ? s / powf((float)L, alpha) : s; }

// step t of the beam decode, behind a grid barrier: block i merges items i, i + gridDim.x, ...  S is free shared memory.
// Every reduction runs in a fixed order, so the result does not change from run to run.
// kStop: a finished beam k (FL[k] = its frozen length) skips its tile candidates and its log-sum-exp and contributes the one
// candidate (k, pad_token) with its score unchanged; candidates are ranked by rank_key, the raw score travels beside the key.
template <bool kStop>
__device__ __forceinline__ void merge_beams(const Args& a, int t, float* S) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, K = a.K, nt = a.ntiles, per_row = nt * K;
    float* LSE = S;                                      // [kMaxK]
    float* SC = S + kMaxK;                               // [kMaxK] scores of the beams at step t - 1
    float* WS = S + 2 * kMaxK;                           // [8 warps][kMaxK] each warp's top K
    int* WK = reinterpret_cast<int*>(WS + 8 * kMaxK);
    float* WR = reinterpret_cast<float*>(WK + 8 * kMaxK);   // kStop: [8 warps][kMaxK] raw scores beside the keys WS
    int* FL = reinterpret_cast<int*>(WR + 8 * kMaxK);       // kStop: [kMaxK] frozen length of a finished beam, 0 while live
    for (int item = blockIdx.x; item < a.B / K; item += gridDim.x) {
        const int r0 = item * K;
        if (warp < K) {                                  // warp k: log-sum-exp of row r0 + k over its tiles
            int fl = 0;
            if constexpr (kStop) fl = t ? __ldcg(a.blen + r0 + warp) : 0;
            const float2* st = a.bstat + (long long)(r0 + warp) * nt;
            float m = -INFINITY;
            float s = 0.f;
            if (!fl) {
                for (int l = lane; l < nt; l += 32) m = fmaxf(m, __ldcg(st + l).x);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
                for (int l = lane; l < nt; l += 32) { const float2 p = __ldcg(st + l); s += p.y * expf(p.x - m); }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
                s = __shfl_sync(0xffffffffu, s, 0);
            }
            if (lane == 0) {
                LSE[warp] = m + logf(s);
                SC[warp] = t ? __ldcg(a.bscore + r0 + warp) : (warp ? -INFINITY : 0.f);   // t = 0: only beam 0 is live
                if constexpr (kStop) FL[warp] = fl;
            }
        }
        __syncthreads();
        // the item's K rows x ntiles x K candidates are contiguous; each thread keeps its best kMaxK
        float ls[kMaxK], lr[kMaxK];
        int lk[kMaxK];
#pragma unroll
        for (int q = 0; q < kMaxK; ++q) { ls[q] = -INFINITY; lk[q] = INT_MAX; lr[q] = -INFINITY; }
        const float2* cb = a.bcand + (long long)r0 * per_row;
        if constexpr (kStop) {
            const float alpha = a.length_penalty;
            for (int i = threadIdx.x; i < K * per_row; i += kT) {
                const int k = i / per_row;
                if (FL[k]) continue;
                const float2 c = __ldcg(cb + i);
                const int v = __float_as_int(c.y);
                if (v < a.V) {
                    const float raw = SC[k] + (c.x - LSE[k]);
                    list_insert(ls, lk, lr, rank_key(raw, t + 1, alpha), k * a.V + v, raw);
                }
            }
            const int k = threadIdx.x;
            if (k < K && FL[k]) list_insert(ls, lk, lr, rank_key(SC[k], FL[k], alpha), k * a.V + a.pad_token, SC[k]);
        } else {
            for (int i = threadIdx.x; i < K * per_row; i += kT) {
                const float2 c = __ldcg(cb + i);
                const int v = __float_as_int(c.y), k = i / per_row;
                if (v < a.V) list_insert(ls, lk, SC[k] + (c.x - LSE[k]), k * a.V + v);
            }
        }
        for (int j = 0; j < K; ++j) {
            float best; int bk;
            if constexpr (kStop) {
                float braw;
                warp_pop(ls, lk, lr, best, bk, braw);
                if (lane == 0) WR[warp * kMaxK + j] = braw;
            } else warp_pop(ls, lk, best, bk);
            if (lane == 0) { WS[warp * kMaxK + j] = best; WK[warp * kMaxK + j] = bk; }
        }
        __syncthreads();
        if (warp == 0) {                                 // the 8 warps' lists -> the item's top K, best first
#pragma unroll
            for (int q = 0; q < kMaxK; ++q) { ls[q] = -INFINITY; lk[q] = INT_MAX; lr[q] = -INFINITY; }
            for (int e = lane; e < 8 * kMaxK; e += 32)
                if (e % kMaxK < K) {
                    if constexpr (kStop) list_insert(ls, lk, lr, WS[e], WK[e], WR[e]);
                    else list_insert(ls, lk, WS[e], WK[e]);
                }
            for (int j = 0; j < K; ++j) {
                float best, braw; int bk;
                if constexpr (kStop) warp_pop(ls, lk, lr, best, bk, braw);
                else warp_pop(ls, lk, best, bk);
                if (lane == 0) {
                    const int k = bk / a.V, v = bk - k * a.V;
                    a.tokens[(long long)(r0 + j) * a.T + t] = (long long)v | ((long long)(r0 + k) << 32);
                    if constexpr (kStop) {
                        a.bscore[r0 + j] = braw;
                        a.blen[r0 + j] = FL[k] ? FL[k] : (v == a.end_token ? t + 1 : 0);
                    } else a.bscore[r0 + j] = best;
                }
            }
        }
        __syncthreads();                                 // LSE / SC / WS / FL reused by the next item
    }
}

// ---- truncated sampling: the select phase ------------------------------------------------------------------------------
constexpr int kSelFloats = 1536;          // tail of the U region: histograms and reduction scratch of the select phase
PCD_HOSTDEV int stage_cap(int H) { return u_floats(H) - kSelFloats; }

// the boundary of a row's kept set by radix select on the 64-bit order keys, 8 bits per pass from the top: the returned
// key C has { v : key_v >= C } = the first `need` words in order (kMass = false), or the shortest prefix whose mass
// reaches `need` (kMass = true), among the words with key >= lo.  A pass stops early once the bucket that holds the
// boundary is taken whole (its remaining bits are then 0, so C is the larger of that prefix and lo).  Counts and masses
// are integers: every pass gives the same histogram whatever the order of its atomics.  The 64-bit shared atomic is a
// compare-and-swap loop, and most words of a row share a few high buckets, so the lanes of a warp that hit one bucket
// add their masses once, through the warp's scratch xs[32].
template <bool kMass, class Load>
__device__ unsigned long long radix_select(Load load, int V, float lmax, float T, float scale, unsigned long long lo,
                                           unsigned long long need, unsigned* cnt, unsigned long long* mass,
                                           unsigned long long* bc, unsigned long long* xs) {
    const int tid = threadIdx.x, lane = tid & 31;
    unsigned long long P = 0, M = 0;
    for (int shift = 56; shift >= 0; shift -= 8) {
        cnt[tid] = 0u;
        if constexpr (kMass) mass[tid] = 0ull;
        __syncthreads();
        for (int base = 0; base < V; base += kT) {          // uniform trip count: the whole warp reaches the match
            const int v = base + tid;
            int d = 256;
            unsigned long long m = 0;
            if (v < V) {
                const float l = load(v);
                const unsigned long long k = order_key(l, v);
                if (k >= lo && (k & M) == P) {
                    d = (int)(k >> shift) & 255;
                    atomicAdd(cnt + d, 1u);
                    if constexpr (kMass) m = mass_of(l, lmax, T, scale);
                }
            }
            if constexpr (kMass) {
                const unsigned peers = __match_any_sync(0xffffffffu, d);
                xs[lane] = m;
                __syncwarp();
                if (d < 256 && lane == __ffs(peers) - 1) {
                    unsigned long long sum = 0;
                    for (unsigned r = peers; r; r &= r - 1) sum += xs[__ffs(r) - 1];
                    atomicAdd(mass + d, sum);
                }
                __syncwarp();
            }
        }
        __syncthreads();
        if (tid < 32) {
            // lane l holds the buckets 255 - 8l .. 248 - 8l (descending); a warp scan finds the bucket where `need` is met
            unsigned long long own = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) own += kMass ? mass[255 - 8 * lane - j] : cnt[255 - 8 * lane - j];
            unsigned long long inc = own;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned long long x = __shfl_up_sync(0xffffffffu, inc, o);
                if (lane >= o) inc += x;
            }
            const int first = __ffs(__ballot_sync(0xffffffffu, inc >= need)) - 1;
            if (lane == first) {
                unsigned long long acc = inc - own;
                for (int j = 0; j < 8; ++j) {
                    const int d = 255 - 8 * lane - j;
                    const unsigned long long x = kMass ? mass[d] : cnt[d];
                    if (acc + x >= need) {
                        const unsigned long long left = need - acc;
                        bc[0] = P | ((unsigned long long)d << shift);
                        bc[1] = left;
                        bc[2] = cnt[d] == 1u || (!kMass && cnt[d] == left) || shift == 0;
                        break;
                    }
                    acc += x;
                }
            }
        }
        __syncthreads();
        P = bc[0];
        need = bc[1];
        const bool done = bc[2] != 0;
        M |= 255ull << shift;
        __syncthreads();                  // bc and the histograms are rewritten by the next pass
        if (done) break;
    }
    return P > lo ? P : lo;
}

// one row: S = the kept set of pcdarts_sm100.h, then the Gumbel argmax over S -> a.words[row]
template <class Load>
__device__ void select_row(const Args& a, int t, int row, Load load, float lmax, unsigned* cnt, unsigned long long* mass,
                           unsigned long long* bc, float* red, unsigned long long* xs) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, V = a.V;
    const float T = a.temperature;
    const int s = mass_shift(V);
    const float scale = __int_as_float((127 + s) << 23);
    unsigned long long C = 0;             // every key is >= 0: no truncation
    if (a.top_k > 0 && a.top_k < V)
        C = radix_select<false>(load, V, lmax, T, scale, 0ull, (unsigned long long)a.top_k, cnt, mass, bc, xs);
    if (a.top_p < 1.f) {
        unsigned long long z = 0;
        for (int v = tid; v < V; v += kT) {
            const float l = load(v);
            if (order_key(l, v) >= C) z += mass_of(l, lmax, T, scale);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) z += __shfl_xor_sync(0xffffffffu, z, o);
        if (lane == 0) mass[warp] = z;
        __syncthreads();
        if (tid == 0) {
            unsigned long long Z = 0;
            for (int w = 0; w < kT / 32; ++w) Z += mass[w];
            bc[3] = nucleus_target(Z, a.top_p);
        }
        __syncthreads();
        const unsigned long long tgt = bc[3];
        __syncthreads();
        C = radix_select<true>(load, V, lmax, T, scale, C, tgt, cnt, mass, bc, xs);
    }
    // Gumbel argmax over S: the score of untruncated sampling, one Philox block per 4 words with a kept word
    const unsigned long long seed = __ldg(a.seed);
    const uint32_t grow = (uint32_t)(a.row_offset + row);
    float best = -INFINITY;
    int bi = INT_MAX;
    for (int j = tid; 4 * j < V; j += kT) {
        float l[4];
        unsigned in = 0u;
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            const int v = 4 * j + w;
            l[w] = v < V ? load(v) : 0.f;
            if (v < V && order_key(l[w], v) >= C) in |= 1u << w;
        }
        if (in) {
            const Philox4 blk = philox4x32_10((uint32_t)j, (uint32_t)t, grow, 0u, (uint32_t)seed, (uint32_t)(seed >> 32));
#pragma unroll
            for (int w = 0; w < 4; ++w)
                if ((in >> w) & 1u) {
                    const float sc = l[w] / T + gumbel_of_bits(blk.w[w]);
                    if (better(sc, 4 * j + w, best, bi)) { best = sc; bi = 4 * j + w; }
                }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (better(ov, oi, best, bi)) { best = ov; bi = oi; }
    }
    if (lane == 0) { red[warp] = best; red[8 + warp] = __int_as_float(bi); }
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < kT / 32; ++w)
            if (better(red[w], __float_as_int(red[8 + w]), best, bi)) { best = red[w]; bi = __float_as_int(red[8 + w]); }
        __stcg(a.words + row, (bi >= 0 && bi < V) ? bi : 0);
    }
    __syncthreads();                      // red reused by the next row
}

// step t of the truncated sampled decode, behind the grid barrier after phase B: block r takes rows r, r + gridDim.x, ...
// A row's logits are staged in the U region when V fits (it does at V = 17858 for every H), else every pass reads L2.
__device__ void select_words(const Args& a, int t, float* U) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, V = a.V;
    float* tail = U + stage_cap(a.H);
    unsigned long long* mass = reinterpret_cast<unsigned long long*>(tail);          // [256]
    unsigned* cnt = reinterpret_cast<unsigned*>(tail + 512);                          // [256]
    unsigned long long* bc = reinterpret_cast<unsigned long long*>(tail + 768);       // [4] pass result
    float* red = tail + 776;                                                          // [16] reductions
    unsigned long long* xs = reinterpret_cast<unsigned long long*>(tail + 800) + 32 * warp;   // [8 warps][32]
    const bool staged = V <= stage_cap(a.H);
    for (int row = blockIdx.x; row < a.B; row += gridDim.x) {
        const float* src = a.stash + (long long)row * V;
        float m = -INFINITY;
        for (int v = tid; v < V; v += kT) {
            const float l = __ldcg(src + v);
            if (staged) U[v] = l;
            m = fmaxf(m, l);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        if (lane == 0) red[warp] = m;
        __syncthreads();
        float lmax = red[0];
        for (int w = 1; w < kT / 32; ++w) lmax = fmaxf(lmax, red[w]);
        __syncthreads();
        if (staged) select_row(a, t, row, [U](int v) { return U[v]; }, lmax, cnt, mass, bc, red, xs);
        else select_row(a, t, row, [src](int v) { return __ldcg(src + v); }, lmax, cnt, mass, bc, red, xs);
    }
}

template <int kMode, bool kStop, bool kTrunc = false>
__global__ void __launch_bounds__(kT, 1) decode_kernel(Args a) {
    constexpr bool kSample = kMode == kSampled, kBeamMode = kMode == kBeam;
    cg::grid_group grid = cg::this_grid();
    extern __shared__ __align__(16) float sm[];
    const int H = a.H, E = a.E, B = a.B, HP = H + 4, EP = E + 4, H4 = H / 4, E4 = E / 4;
    float* Ws = sm;                       // [16][HP]  row q*4+u <- W_hh row q*H + u0 + u
    float* Wi = Ws + 16 * HP;             // [16][EP]  same rows of W_ih
    float* U = Wi + 16 * EP;              // phase A: Hs [B][HP] = h_{t-1};  phase B: kStages x ([64][kWP] | [128][kWP]) chunk ring
    float* Hs = U;
    int* TOK = reinterpret_cast<int*>(U + u_floats(H));            // [64]
    float* XP = reinterpret_cast<float*>(TOK + kMaxB);             // [4 quarters][16 gate rows][64] input-projection partials
    int* PAR = reinterpret_cast<int*>(XP + 64 * kMaxB);            // [64]  beam: the row whose state a row continues
    int* FIN = PAR;                                                // [64]  greedy / sampled kStop: the row emitted end_token
    const int tid = threadIdx.x;
    const bool gate_block = (int)blockIdx.x < H / kUnits;
    const int u0 = blockIdx.x * kUnits;
    const int b = tid & 63, u = tid >> 6, unit = u0 + u;
    const int ty = tid >> 4, tx = tid & 15;
    float bsum[4] = {0.f, 0.f, 0.f, 0.f}, c = 0.f;
    if (gate_block) {
        for (int i = tid; i < 16 * H4; i += kT) {
            const int rr = i / H4, k4 = i - rr * H4;
            *reinterpret_cast<float4*>(Ws + rr * HP + 4 * k4) =
                *reinterpret_cast<const float4*>(a.w_hh + (long long)((rr >> 2) * H + u0 + (rr & 3)) * H + 4 * k4);
        }
        for (int i = tid; i < 16 * E4; i += kT) {
            const int rr = i / E4, k4 = i - rr * E4;
            *reinterpret_cast<float4*>(Wi + rr * EP + 4 * k4) =
                *reinterpret_cast<const float4*>(a.w_ih + (long long)((rr >> 2) * H + u0 + (rr & 3)) * E + 4 * k4);
        }
        if (b < B) {
#pragma unroll
            for (int q = 0; q < 4; ++q) bsum[q] = a.b_ih[q * H + unit] + a.b_hh[q * H + unit];
            if constexpr (!kBeamMode) c = a.c0[(long long)b * H + unit];
        }
    }
    const int nk = H / kKC;
    int t_run = a.T;                      // kStop: steps run before every row had finished
    for (int t = 0; t < a.T; ++t) {
        // ---- the word chosen at the previous step ------------------------------------------------------------------------
        if (t == 0) {
            if (tid < kMaxB) {
                TOK[tid] = a.start;
                if constexpr (kBeamMode) PAR[tid] = tid / a.K;             // every beam of item b starts from h0[b], c0[b]
                else if constexpr (kStop) FIN[tid] = 0;
            }
        } else if constexpr (kBeamMode) {
            if (tid < B) {
                const long long p = __ldcg(a.tokens + (long long)tid * a.T + t - 1);
                TOK[tid] = (int)(p & 0xffffffffll);
                PAR[tid] = (int)(p >> 32);
            }
        } else if constexpr (kTrunc) {
            if (tid < B) TOK[tid] = __ldcg(a.words + tid);
        } else pick_words(a, TOK);
        if constexpr (kStop && kBeamMode) {
            // every block reads every row's finished length behind the merge barrier, so all of them leave at the same step
            if (!__syncthreads_count(t == 0 || (tid < B && __ldcg(a.blen + tid) == 0))) { t_run = t; break; }
        } else __syncthreads();
        if constexpr (kStop && !kBeamMode)
            if (t > 0) {
                // word t - 1 of a finished row is pad_token, and so is its next input; every block picked the same words, so
                // all of them see the last row finish at the same step
                int live = 0;
                if (tid < B) {
                    if (FIN[tid]) TOK[tid] = a.pad_token;
                    else live = !(FIN[tid] = TOK[tid] == a.end_token);
                }
                if (!__syncthreads_count(live)) t_run = t;
            }
        if constexpr (!kBeamMode)
            if (t > 0 && blockIdx.x == 0 && tid < B) a.tokens[(long long)tid * a.T + t - 1] = TOK[tid];
        if constexpr (kStop && !kBeamMode)
            if (t_run == t) break;
        // ---- phase A: one LSTM step for this block's 4 hidden units ----------------------------------------------------------
        if (gate_block) {
            const float* hprev = t ? a.hbuf + (long long)((t - 1) & 1) * B * H : a.h0;
            if constexpr (kBeamMode) stage_rows<true>(Hs, hprev, B, H, PAR);
            else stage_rows(Hs, hprev, B, H);
            asm volatile("cp.async.commit_group;" ::: "memory");
            // input projection while h_{t-1} is in flight: thread (b, u) takes quarter u of x_b against all 16 gate rows of
            // the block (its ~19 float4 of the embedding row are independent loads), partial sums meet in shared memory
            if (b < B) {
                const float4* xr = reinterpret_cast<const float4*>(a.emb + (long long)TOK[b] * E);
                const int kq0 = (E4 * u) >> 2, kq1 = (E4 * (u + 1)) >> 2;
                float p[16];
#pragma unroll
                for (int r = 0; r < 16; ++r) p[r] = 0.f;
                if (t == 0) {                             // <start>: tanh(emb[2]) (vqa_model.py:119)
                    for (int k4 = kq0; k4 < kq1; ++k4) {
                        float4 x = __ldg(xr + k4);
                        x.x = tanhf(x.x); x.y = tanhf(x.y); x.z = tanhf(x.z); x.w = tanhf(x.w);
#pragma unroll
                        for (int r = 0; r < 16; ++r) p[r] = dot4(x, *reinterpret_cast<const float4*>(Wi + r * EP + 4 * k4), p[r]);
                    }
                } else {
#pragma unroll 10
                    for (int k4 = kq0; k4 < kq1; ++k4) {
                        const float4 x = __ldg(xr + k4);
#pragma unroll
                        for (int r = 0; r < 16; ++r) p[r] = dot4(x, *reinterpret_cast<const float4*>(Wi + r * EP + 4 * k4), p[r]);
                    }
                }
#pragma unroll
                for (int r = 0; r < 16; ++r) XP[(u * 16 + r) * kMaxB + b] = p[r];
            }
            asm volatile("cp.async.wait_group 0;" ::: "memory");
            __syncthreads();
            if (b < B) {
                if constexpr (kBeamMode)
                    c = t ? __ldcg(a.cbuf + (long long)((t - 1) & 1) * B * H + (long long)PAR[b] * H + unit)
                          : a.c0[(long long)PAR[b] * H + unit];
                float acc[4];
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    acc[q] = bsum[q] + ((XP[(0 * 16 + q * 4 + u) * kMaxB + b] + XP[(1 * 16 + q * 4 + u) * kMaxB + b]) +
                                        (XP[(2 * 16 + q * 4 + u) * kMaxB + b] + XP[(3 * 16 + q * 4 + u) * kMaxB + b]));
                const float* hr = Hs + b * HP;
#pragma unroll 4
                for (int k4 = 0; k4 < H4; ++k4) {
                    const float4 h4 = *reinterpret_cast<const float4*>(hr + 4 * k4);
#pragma unroll
                    for (int q = 0; q < 4; ++q) acc[q] = dot4(h4, *reinterpret_cast<const float4*>(Ws + (q * 4 + u) * HP + 4 * k4), acc[q]);
                }
                const float gi = sigm(acc[0]), gf = sigm(acc[1]), gg = tanhf(acc[2]), go = sigm(acc[3]);
                c = fmaf(gf, c, gi * gg);
                const float h = go * tanhf(c);
                if constexpr (kBeamMode) __stcg(a.cbuf + (long long)(t & 1) * B * H + (long long)b * H + unit, c);
                __stcg(a.hbuf + (long long)(t & 1) * B * H + (long long)b * H + unit, h);
                __stcg(a.tbuf + (long long)b * H + unit, tanhf(h));
            }
        }
        grid.sync();
        // ---- phase B: vocabulary logits of this block's tiles, row-wise argmax candidates ----------------------------------------
        // K chunks of 32: (tanh(h_t) rows | W_out tile rows) pairs through a kStages-deep cp.async ring in the U region
        for (int tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x) {
            {
                const int col0 = tile * kTileN;
                auto issue = [&](int kc) {
                    float* sbuf = U + (kc % kStages) * kStageFloats;
                    float* wbuf = sbuf + kMaxB * kWP;
#pragma unroll
                    for (int i = tid; i < kMaxB * (kKC / 4); i += kT) {
                        const int row = i >> 3, j = i & 7;
                        const unsigned dst = (unsigned)__cvta_generic_to_shared(sbuf + row * kWP + 4 * j);
                        const float* src = a.tbuf + (long long)(row < B ? row : B - 1) * H + kc * kKC + 4 * j;
                        const int nbytes = row < B ? 16 : 0;           // rows past the batch: zero fill
                        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(nbytes) : "memory");
                    }
#pragma unroll
                    for (int i = tid; i < kTileN * (kKC / 4); i += kT) {
                        const int col = i >> 3, j = i & 7;
                        const int gc = col0 + col;
                        const unsigned dst = (unsigned)__cvta_generic_to_shared(wbuf + col * kWP + 4 * j);
                        const float* src = a.w_out + (long long)(gc < a.V ? gc : a.V - 1) * H + kc * kKC + 4 * j;
                        const int nbytes = gc < a.V ? 16 : 0;          // columns past V: zero fill
                        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(nbytes) : "memory");
                    }
                };
                float acc[4][8];
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
#pragma unroll
                for (int s = 0; s < kStages - 1; ++s) {
                    if (s < nk) issue(s);
                    asm volatile("cp.async.commit_group;" ::: "memory");
                }
                for (int kc = 0; kc < nk; ++kc) {
                    asm volatile("cp.async.wait_group %0;" ::"n"(kStages - 2) : "memory");
                    __syncthreads();              // chunk kc landed for everyone; everyone is done with chunk kc - 1
                    if (kc + kStages - 1 < nk) issue(kc + kStages - 1);
                    asm volatile("cp.async.commit_group;" ::: "memory");
                    const float* sb = U + (kc % kStages) * kStageFloats;
                    const float* wb = sb + kMaxB * kWP;
#pragma unroll
                    for (int k4 = 0; k4 < kKC / 4; ++k4) {
                        float4 s[4], w[8];
#pragma unroll
                        for (int i = 0; i < 4; ++i) s[i] = *reinterpret_cast<const float4*>(sb + (4 * ty + i) * kWP + 4 * k4);
#pragma unroll
                        for (int j = 0; j < 8; ++j) w[j] = *reinterpret_cast<const float4*>(wb + (tx + 16 * j) * kWP + 4 * k4);
#pragma unroll
                        for (int i = 0; i < 4; ++i)
#pragma unroll
                            for (int j = 0; j < 8; ++j) acc[i][j] = dot4(s[i], w[j], acc[i][j]);
                    }
                }
                __syncthreads();                  // ring free again (next tile's prologue / next step's h staging)
                if constexpr (kBeamMode) {
                    // per row: the tile's top K by K rounds of (best untaken column of the thread -> argmax over the 16
                    // lanes of the row), then the tile's sum exp(logit - max) by a fixed butterfly
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const int row = 4 * ty + i;
                        float lv[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const int col = col0 + tx + 16 * j;
                            lv[j] = col < a.V ? acc[i][j] + __ldg(a.b_out + col) : -INFINITY;
                        }
                        unsigned taken = 0u;
                        float mx = 0.f;
                        for (int k = 0; k < a.K; ++k) {
                            float best = -INFINITY;
                            int bi = INT_MAX;
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                const int col = col0 + tx + 16 * j;
                                if (!((taken >> j) & 1u) && col < a.V && better(lv[j], col, best, bi)) { best = lv[j]; bi = col; }
                            }
#pragma unroll
                            for (int o = 8; o > 0; o >>= 1) {
                                const float ov = __shfl_xor_sync(0xffffffffu, best, o);
                                const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
                                if (better(ov, oi, best, bi)) { best = ov; bi = oi; }
                            }
                            if (k == 0) mx = best;
                            if (bi != INT_MAX && ((bi - col0) & 15) == tx) taken |= 1u << ((bi - col0) >> 4);
                            if (tx == 0 && row < B)
                                __stcg(a.bcand + ((long long)row * a.ntiles + tile) * a.K + k, make_float2(best, __int_as_float(bi)));
                        }
                        float se = 0.f;
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                            if (col0 + tx + 16 * j < a.V) se += expf(lv[j] - mx);
#pragma unroll
                        for (int o = 8; o > 0; o >>= 1) se += __shfl_xor_sync(0xffffffffu, se, o);
                        if (tx == 0 && row < B) __stcg(a.bstat + (long long)row * a.ntiles + tile, make_float2(mx, se));
                    }
                } else if constexpr (kTrunc) {
                    // the select phase behind the next barrier needs whole rows: the tile's logits go to the stash
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const int row = 4 * ty + i;
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const int col = col0 + tx + 16 * j;
                            if (row < B && col < a.V) __stcg(a.stash + (long long)row * a.V + col, acc[i][j] + __ldg(a.b_out + col));
                        }
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        float best = -INFINITY;
                        int bi = INT_MAX;
                        if constexpr (kSample) {
                            // columns col0 + tx + 16j of a lane quad (tx >> 2) share one Philox block per j: lane q = tx & 3
                            // computes the blocks of j = q and j = q + 4, and the quad hands word q of every block to lane q
                            const int q = tx & 3, quad = (threadIdx.x & 31) & ~3;
                            const unsigned long long seed = __ldg(a.seed);
                            const uint32_t v4 = (uint32_t)(col0 >> 2) + (uint32_t)(tx >> 2) + 4u * q;
                            const uint32_t grow = (uint32_t)(a.row_offset + 4 * ty + i);
                            const Philox4 blk[2] = {philox4x32_10(v4, (uint32_t)t, grow, 0u, (uint32_t)seed, (uint32_t)(seed >> 32)),
                                                    philox4x32_10(v4 + 16u, (uint32_t)t, grow, 0u, (uint32_t)seed, (uint32_t)(seed >> 32))};
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                uint32_t w[4];
#pragma unroll
                                for (int k = 0; k < 4; ++k) w[k] = __shfl_sync(0xffffffffu, blk[j >> 2].w[k], quad | (j & 3));
                                const uint32_t x = q == 0 ? w[0] : q == 1 ? w[1] : q == 2 ? w[2] : w[3];
                                const int col = col0 + tx + 16 * j;
                                if (col < a.V) {
                                    const float v = (acc[i][j] + __ldg(a.b_out + col)) / a.temperature + gumbel_of_bits(x);
                                    if (v > best) { best = v; bi = col; }
                                }
                            }
                        } else {
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                const int col = col0 + tx + 16 * j;
                                if (col < a.V) {
                                    const float v = acc[i][j] + __ldg(a.b_out + col);
                                    if (v > best) { best = v; bi = col; }
                                }
                            }
                        }
#pragma unroll
                        for (int o = 8; o > 0; o >>= 1) {
                            const float ov = __shfl_xor_sync(0xffffffffu, best, o);
                            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
                            if (better(ov, oi, best, bi)) { best = ov; bi = oi; }
                        }
                        const int row = 4 * ty + i;
                        if (tx == 0 && row < B) {
                            __stcg(a.cand + (long long)row * a.ntiles + tile, make_float2(best, __int_as_float(bi)));
                        }
                    }
                }
            }
        }
        grid.sync();
        if constexpr (kBeamMode) {
            merge_beams<kStop>(a, t, U);
            grid.sync();
        } else if constexpr (kTrunc) {
            select_words(a, t, U);
            grid.sync();
        }
    }
    if constexpr (kBeamMode) {
        // backtrack: column t of every row's (word, parent) is read before any thread overwrites it with the word of the path
        if (blockIdx.x == 0) {
            int cur = tid;
            for (int t = (kStop ? t_run : a.T) - 1; t >= 0; --t) {
                long long p = 0;
                if (tid < B) p = __ldcg(a.tokens + (long long)cur * a.T + t);
                __syncthreads();
                if (tid < B) {
                    a.tokens[(long long)tid * a.T + t] = p & 0xffffffffll;
                    cur = (int)(p >> 32);
                }
            }
            if (tid < B) a.scores[tid] = __ldcg(a.bscore + tid);
            if constexpr (kStop)
                if (tid < B)
                    for (int t = t_run; t < a.T; ++t) a.tokens[(long long)tid * a.T + t] = a.pad_token;
        }
    } else if (blockIdx.x == 0) {
        if constexpr (kStop) {
            if (t_run == a.T) {
                if constexpr (kTrunc) {
                    if (tid < B) TOK[tid] = __ldcg(a.words + tid);
                } else pick_words(a, TOK);
                __syncthreads();
                if (tid < B) a.tokens[(long long)tid * a.T + a.T - 1] = FIN[tid] ? a.pad_token : TOK[tid];
            } else if (tid < B) {
                for (int t = t_run; t < a.T; ++t) a.tokens[(long long)tid * a.T + t] = a.pad_token;
            }
        } else {
            if constexpr (kTrunc) {
                if (tid < B) TOK[tid] = __ldcg(a.words + tid);
            } else pick_words(a, TOK);
            __syncthreads();
            if (tid < B) a.tokens[(long long)tid * a.T + a.T - 1] = TOK[tid];
        }
    }
}

}  // namespace decode
}  // namespace pcd

namespace pcd {
namespace decode {

// the kernel of one (mode, stop) pair; its first call reads the SM count and sets the kernel's shared-memory limit
template <int kMode, bool kStop, bool kTrunc = false>
static const void* kernel_of(int& sms_out, LaunchState& L) {
    static int sms = 0;                                     // per instantiation: each one sets its own smem attribute
    if (!sms) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
            cudaFuncSetAttribute(decode_kernel<kMode, kStop, kTrunc>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess) {
            sms = 0;
            snprintf(L.last_err, sizeof L.last_err, "decode setup: %s", cudaGetErrorString(cudaGetLastError()));
            return nullptr;
        }
    }
    sms_out = sms;
    return (const void*)decode_kernel<kMode, kStop, kTrunc>;
}

// a call that passed validate(): alignment, shared memory, grid, then one cooperative launch
static int run(const pcd_decode_args& p, void* stream) {
    const int B = p.B * p.K, H = p.H, E = p.E, V = p.V;   // B counts rows: items x K for the beam decode
    if ((((uintptr_t)p.emb) | ((uintptr_t)p.w_ih) | ((uintptr_t)p.w_hh) | ((uintptr_t)p.h0) | ((uintptr_t)p.w_out) | ((uintptr_t)p.work)) & 15) return PCD_ERR_ALIGN;
    if (p.mode == kSampled && ((uintptr_t)p.seed) & 7) return PCD_ERR_ALIGN;
    LaunchState& L = launch_state();
    const size_t smem = ((size_t)16 * (H + 4) + (size_t)16 * (E + 4) + (size_t)u_floats(H) + kMaxB + 64 * kMaxB +
                         (p.mode == kBeam || p.stop ? kMaxB : 0)) * sizeof(float);
    if (smem > 227 * 1024) return PCD_ERR_UNSUPPORTED;
    using KernelOf = const void* (*)(int&, LaunchState&);
    static const KernelOf kernels[3][2] = {{kernel_of<kGreedy, false>, kernel_of<kGreedy, true>},
                                           {kernel_of<kSampled, false>, kernel_of<kSampled, true>},
                                           {kernel_of<kBeam, false>, kernel_of<kBeam, true>}};
    static const KernelOf truncating[2] = {kernel_of<kSampled, false, true>, kernel_of<kSampled, true, true>};
    const bool trunc = p.mode == kSampled && p.truncate;
    int sms = 0;
    const void* kernel = trunc ? truncating[p.stop ? 1 : 0](sms, L) : kernels[p.mode][p.stop ? 1 : 0](sms, L);
    if (!kernel) return PCD_ERR_CUDA;
    const int ntiles = tiles_of(V);
    int grid = ntiles < sms ? ntiles : sms;                 // one block per SM: all of them co-resident (cooperative launch)
    if (grid < H / kUnits) grid = H / kUnits;
    if (grid > sms) return PCD_ERR_UNSUPPORTED;
    const Work w = work_of(p.mode, p.B, p.K, H, V, trunc);
    Args a;
    a.T = p.T; a.B = B; a.H = H; a.E = E; a.V = V; a.start = p.start_token; a.ntiles = ntiles;
    a.emb = p.emb; a.w_ih = p.w_ih; a.w_hh = p.w_hh; a.b_ih = p.b_ih; a.b_hh = p.b_hh; a.h0 = p.h0; a.c0 = p.c0;
    a.w_out = p.w_out; a.b_out = p.b_out;
    a.tokens = p.tokens;
    a.hbuf = p.work;
    a.tbuf = p.work + w.tbuf;
    a.cand = reinterpret_cast<float2*>(p.work + w.cand);
    a.seed = p.seed; a.temperature = p.temperature; a.row_offset = p.row_offset;
    a.K = p.K;
    a.cbuf = p.work + w.cbuf;
    a.bcand = reinterpret_cast<float2*>(p.work + w.bcand);
    a.bstat = reinterpret_cast<float2*>(p.work + w.bstat);
    a.bscore = p.work + w.bscore;
    a.scores = p.scores;
    a.end_token = p.end_token; a.pad_token = p.pad_token; a.length_penalty = p.length_penalty;
    a.blen = reinterpret_cast<int*>(p.work + w.blen);
    a.top_k = p.top_k; a.top_p = p.top_p;
    a.stash = p.work + w.stash;
    a.words = reinterpret_cast<int*>(p.work + w.words);
    void* args[] = {&a};
    cudaError_t e = cudaLaunchCooperativeKernel(kernel, dim3(grid), dim3(kT), args, smem, (cudaStream_t)stream);
    count_launch(L);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) {
        snprintf(L.last_err, sizeof L.last_err, "cooperative launch decode: %s", cudaGetErrorString(e));
        return PCD_ERR_CUDA;
    }
    return PCD_OK;
}

}  // namespace decode
}  // namespace pcd

#else   // ---- CPU emulation build (tests only) ----------------------------------------------------------------------

#include <math.h>
#include <algorithm>
#include <vector>

static inline float sigm_(float x) { return 1.f / (1.f + expf(-x)); }

namespace pcd {
namespace decode {

// one LSTM step of a row from (h, c) on the input word, and the vocabulary logits of the new state, with the kernel's
// arithmetic: fp64 gate and vocabulary sums rounded to fp32.  c_out may be c; h_out is not h
static void step_emu(const pcd_decode_args& a, int word, int t, const float* h, const float* c, float* h_out, float* c_out,
                     float* logits) {
    const int H = a.H, E = a.E;
    std::vector<float> x((size_t)E), s((size_t)H);
    for (int k = 0; k < E; ++k) x[k] = t ? a.emb[(long long)word * E + k] : tanhf(a.emb[(long long)word * E + k]);
    for (int j = 0; j < H; ++j) {
        float g[4];
        for (int q = 0; q < 4; ++q) {
            double acc = (double)a.b_ih[q * H + j] + a.b_hh[q * H + j];
            for (int k = 0; k < E; ++k) acc += (double)x[k] * a.w_ih[(long long)(q * H + j) * E + k];
            for (int k = 0; k < H; ++k) acc += (double)h[k] * a.w_hh[(long long)(q * H + j) * H + k];
            g[q] = (float)acc;
        }
        const float gi = sigm_(g[0]), gf = sigm_(g[1]), gg = tanhf(g[2]), go = sigm_(g[3]);
        c_out[j] = gf * c[j] + gi * gg;
        h_out[j] = go * tanhf(c_out[j]);
    }
    for (int j = 0; j < H; ++j) s[j] = tanhf(h_out[j]);
    for (int v = 0; v < a.V; ++v) {
        double acc = a.b_out[v];
        for (int k = 0; k < H; ++k) acc += (double)s[k] * a.w_out[(long long)v * H + k];
        logits[v] = (float)acc;
    }
}

// truncated sampling: the smallest order key of the kept set S of a row's logits (pcdarts_sm100.h), by sorting where the
// kernel runs a radix select; the masses are the kernel's integers
static unsigned long long kept_boundary(const pcd_decode_args& a, const float* logit) {
    const int V = a.V;
    std::vector<unsigned long long> key((size_t)V);
    float lmax = -INFINITY;
    for (int v = 0; v < V; ++v) { key[v] = order_key(logit[v], v); lmax = logit[v] > lmax ? logit[v] : lmax; }
    std::vector<int> order((size_t)V);
    for (int v = 0; v < V; ++v) order[v] = v;
    std::sort(order.begin(), order.end(), [&](int x, int y) { return key[x] > key[y]; });
    int n = a.top_k > 0 && a.top_k < V ? a.top_k : V;
    if (a.top_p < 1.f) {
        const float scale = ldexpf(1.f, mass_shift(V));
        unsigned long long Z = 0, acc = 0;
        for (int i = 0; i < n; ++i) Z += mass_of(logit[order[i]], lmax, a.temperature, scale);
        const unsigned long long tgt = nucleus_target(Z, a.top_p);
        int i = 0;
        while ((acc += mass_of(logit[order[i]], lmax, a.temperature, scale)) < tgt) ++i;
        n = i + 1;
    }
    return key[order[n - 1]];
}

// greedy / sampled: argmax of the fp32 logit (greedy) or of logit / T + G(seed, t, row_offset + b, v) (sampled); ties go
// to the lowest index.  truncate: the sampled argmax runs over the kept set only.  stop: after end_token a row's remaining
// positions are pad_token (rows are independent, so the row simply ends there)
static int decode_emu(const pcd_decode_args& a) {
    const int T = a.T, B = a.B, H = a.H, V = a.V;
    const bool sample = a.mode == kSampled, trunc = sample && a.truncate;
    const unsigned long long key = sample ? *a.seed : 0ull;
    std::vector<float> h(a.h0, a.h0 + (size_t)B * H), c(a.c0, a.c0 + (size_t)B * H), hn((size_t)H), logit((size_t)V);
    for (int b = 0; b < B; ++b) {
        int word = a.start_token;
        float* hb = h.data() + (size_t)b * H;
        float* cb = c.data() + (size_t)b * H;
        for (int t = 0; t < T; ++t) {
            step_emu(a, word, t, hb, cb, hn.data(), cb, logit.data());
            std::copy(hn.begin(), hn.end(), hb);
            const unsigned long long lo = trunc ? kept_boundary(a, logit.data()) : 0ull;
            float best = -INFINITY;
            int bi = 0;
            for (int v = 0; v < V; ++v) {
                if (trunc && order_key(logit[v], v) < lo) continue;
                const float score = sample ? logit[v] / a.temperature + decode_gumbel(key, t, a.row_offset + b, v) : logit[v];
                if (score > best) { best = score; bi = v; }
            }
            word = bi;
            a.tokens[(long long)b * T + t] = bi;
            if (a.stop && bi == a.end_token) {
                for (int tt = t + 1; tt < T; ++tt) a.tokens[(long long)b * T + tt] = a.pad_token;
                break;
            }
        }
    }
    return PCD_OK;
}

// beam decode: lambda = logit - lse in fp32 (lse from fp64 sums), candidate score s_k + lambda in fp32, ties to the lower
// beam, then the lower word.  stop: finished beams contribute (k, pad_token), candidates are ranked by key with the raw
// scores beside them, and the loop ends once every row has finished
static int beam_emu(const pcd_decode_args& a) {
    const int T = a.T, B = a.B, K = a.K, H = a.H, V = a.V, R = B * K;
    const float alpha = a.stop ? a.length_penalty : 0.f;
    auto rank_key = [alpha](float sc, int L) { return alpha != 0.f ? sc / powf((float)L, alpha) : sc; };
    std::vector<float> h((size_t)R * H), c((size_t)R * H), hn((size_t)R * H), cn((size_t)R * H);
    std::vector<float> lam((size_t)R * V), score((size_t)R), nscore((size_t)R);
    std::vector<int> word((size_t)R, a.start_token), hist_w((size_t)T * R), hist_p((size_t)T * R);
    std::vector<int> len((size_t)R, 0), nlen((size_t)R, 0);     // stop: frozen length of a finished beam, 0 while live
    for (int r = 0; r < R; ++r) {
        std::copy(a.h0 + (size_t)(r / K) * H, a.h0 + (size_t)(r / K + 1) * H, h.begin() + (size_t)r * H);
        std::copy(a.c0 + (size_t)(r / K) * H, a.c0 + (size_t)(r / K + 1) * H, c.begin() + (size_t)r * H);
        score[r] = r % K ? -INFINITY : 0.f;
    }
    int t_run = T;
    for (int t = 0; t < T; ++t) {
        for (int r = 0; r < R; ++r) {
            if (len[r]) continue;                         // finished: its state is never used again
            float* lr = lam.data() + (size_t)r * V;
            step_emu(a, word[r], t, h.data() + (size_t)r * H, c.data() + (size_t)r * H, hn.data() + (size_t)r * H,
                     cn.data() + (size_t)r * H, lr);
            float mx = -INFINITY;
            for (int v = 0; v < V; ++v) mx = lr[v] > mx ? lr[v] : mx;
            double se = 0.0;
            for (int v = 0; v < V; ++v) se += exp((double)lr[v] - mx);
            const float lse = (float)(mx + log(se));
            for (int v = 0; v < V; ++v) lr[v] = lr[v] - lse;
        }
        for (int b = 0; b < B; ++b) {                     // top K of the item's candidates by key, best first
            std::vector<float> bs(K, -INFINITY), braw(K, -INFINITY);
            std::vector<int> bk(K, INT_MAX);
            auto insert = [&](float sc, int key, float raw) {
                for (int q = 0; q < K; ++q)
                    if (sc > bs[q] || (sc == bs[q] && key < bk[q])) {
                        std::swap(sc, bs[q]); std::swap(key, bk[q]); std::swap(raw, braw[q]);
                    }
            };
            for (int k = 0; k < K; ++k) {
                const int r = b * K + k;
                if (len[r]) {                             // a finished beam: the one candidate (k, pad_token), score unchanged
                    insert(rank_key(score[r], len[r]), k * V + a.pad_token, score[r]);
                    continue;
                }
                for (int v = 0; v < V; ++v) {
                    const float raw = score[r] + lam[(size_t)r * V + v];
                    insert(a.stop ? rank_key(raw, t + 1) : raw, k * V + v, raw);
                }
            }
            for (int j = 0; j < K; ++j) {
                const int r = b * K + j, parent = b * K + bk[j] / V, v = bk[j] % V;
                hist_w[(size_t)t * R + r] = v;
                hist_p[(size_t)t * R + r] = parent;
                word[r] = v;
                nscore[r] = braw[j];
                nlen[r] = len[parent] ? len[parent] : (a.stop && v == a.end_token ? t + 1 : 0);
                std::copy(hn.begin() + (size_t)parent * H, hn.begin() + (size_t)(parent + 1) * H, h.begin() + (size_t)r * H);
                std::copy(cn.begin() + (size_t)parent * H, cn.begin() + (size_t)(parent + 1) * H, c.begin() + (size_t)r * H);
            }
        }
        score.swap(nscore);
        len.swap(nlen);
        if (std::all_of(len.begin(), len.end(), [](int l) { return l > 0; })) { t_run = t + 1; break; }
    }
    for (int r = 0; r < R; ++r) {
        int cur = r;
        for (int t = t_run - 1; t >= 0; --t) {
            a.tokens[(long long)r * T + t] = hist_w[(size_t)t * R + cur];
            cur = hist_p[(size_t)t * R + cur];
        }
        for (int t = t_run; t < T; ++t) a.tokens[(long long)r * T + t] = a.pad_token;
        a.scores[r] = score[r];
    }
    return PCD_OK;
}

static int run(const pcd_decode_args& a, void*) { return a.mode == kBeam ? beam_emu(a) : decode_emu(a); }

}  // namespace decode
}  // namespace pcd

#endif

extern "C" int pcd_decode(const pcd_decode_args* a, void* stream) {
    const int rc = pcd::decode::validate(a);
    return rc != PCD_OK ? rc : pcd::decode::run(*a, stream);
}
