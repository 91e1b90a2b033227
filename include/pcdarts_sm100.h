/*
 * pcdarts_sm100.h — C ABI of libpcdarts_sm100.so (hand-written sm_100a CUDA).
 *
 * Drop-in boundary for ONE hot path of aahamed/LCT-VQA: forward + backward of the PC-DARTS search
 * network (MixedOp / Cell / Network).  Every entry point replaces the ATen/cuDNN dispatch sequence
 * of one reference module's forward (and the autograd backward of that sequence); the reference
 * interface each one stands in for is cited as path:line under the upstream repo.
 *
 * Conventions (all entry points)
 *   - plain C: raw device pointers, sizes, a cudaStream_t passed as void*; no torch types.
 *   - tensors are fp32, logical NCHW, W contiguous, channel stride = H*W; the batch stride is
 *     explicit where a tensor may be a channel slice of a larger one.
 *   - the library never allocates, frees, retains pointers or synchronises; every workspace is
 *     caller-owned; all work is enqueued on `stream` (CUDA-graph capturable).
 *   - return value: 0 on success, a negative pcd_status otherwise; never throws, never exits.
 *   - callable from the forward (Python main) thread and the backward (autograd worker) thread of one process: the compute
 *     entry points keep no state between calls.  Process-global state is limited to: idempotent cudaFuncSetAttribute
 *     calls; an atomic launch counter (pcd_launch_count); the last CUDA error string (pcd_last_cuda_error, diagnostics
 *     only); the opt-in weight-gradient overlap (pcd_set_overlap: one library-owned low-priority stream + two events, set
 *     outside capture, used by one backward at a time); and the opt-in event profiler (pcd_profile_*: a single-threaded
 *     measurement mode).
 *   - BatchNorm is training-mode (batch statistics, running stats updated in place,
 *     unbiased variance, num_batches_tracked += 1), eps/momentum as given, except in the `*_eval`
 *     entry points, which use the running statistics and write none of them.
 */
#ifndef PCDARTS_SM100_H
#define PCDARTS_SM100_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PCD_VERSION 100          /* 0.1.0 */
#define PCD_NUM_PRIMITIVES 8     /* genotypes.py:5-14 */
#define PCD_MAX_STEPS 4
#define PCD_MAX_EDGES 14         /* sum_{i<4} (2+i), model_search.py:76-81 */

typedef enum pcd_status {
    PCD_OK = 0,
    PCD_ERR_ARG = -1,            /* null pointer / inconsistent sizes */
    PCD_ERR_UNSUPPORTED = -2,    /* shape outside the compiled template set */
    PCD_ERR_CUDA = -3,           /* launch failed; see pcd_last_cuda_error() */
    PCD_ERR_ALIGN = -4           /* pointer not 16-byte aligned where required */
} pcd_status;

int pcd_version(void);
const char* pcd_strerror(int status);
/* 1 when the library was compiled by nvcc for sm_100a, 0 for the CPU emulation build used only by
 * tests/ (tests/emu): the product loader refuses a library that returns 0. */
int pcd_is_cuda_build(void);
const char* pcd_last_cuda_error(void);

/* Measurement hooks (bench.py): number of kernels this library has launched since it was loaded, and an
 * optional per-launch CUDA-event profiler (events are recorded on the launching stream around every
 * kernel while enabled; collect() synchronises them and accumulates milliseconds per kernel id). */
long long pcd_launch_count(void);
int pcd_profile_enable(int on);
int pcd_profile_num_kernels(void);
const char* pcd_profile_kernel_name(int id);
int pcd_profile_collect(double* ms, long long* count, int max_kernels);

/* ------------------------------------------------------------------------------------------------
 * channel_shuffle(x, groups)                     darts_vqa/pcdarts/model_search.py:14-28
 * out[:, j*groups + g] = in[:, g*(C/groups) + j]   — bit-exact copy.
 * ---------------------------------------------------------------------------------------------- */
int pcd_channel_shuffle(const float* x, float* y, int batch, int channels, int hw, int groups,
                        void* stream);

/* ------------------------------------------------------------------------------------------------
 * Cell(steps=4, multiplier=4, C_pp, C_p, C, reduction, reduction_prev).forward(s0, s1, weights,
 * weights2)                                      darts_vqa/pcdarts/model_search.py:61-94
 * including its 14 MixedOp.forward (model_search.py:44-58), the candidate ops of operations.py:4-104,
 * the partial-channel slice / 2x2 max-pool bypass / channel_shuffle, the beta-weighted node sums and
 * the preprocess ReLUConvBN / FactorizedReduce.
 *
 * A MixedOp on its own (MixedOp(C, stride).forward(x, weights)) is the degenerate cell
 * `pcd_mixedop_*` below: one edge, beta = 1, no preprocess.
 * ---------------------------------------------------------------------------------------------- */
typedef struct pcd_cell_shape {
    int32_t batch;            /* B */
    int32_t c_prev_prev;      /* channels of s0 */
    int32_t c_prev;           /* channels of s1 */
    int32_t channels;         /* C: channels of every state inside the cell (multiple of 16) */
    int32_t height, width;    /* spatial size of s1 (s0 is 2x that when reduction_prev) */
    int32_t reduction;        /* edges from s0/s1 have stride 2 */
    int32_t reduction_prev;   /* preprocess0 is FactorizedReduce */
    int32_t steps;            /* must be 4 */
    float bn_eps;             /* 1e-5 */
    float bn_momentum;        /* 0.1 */
} pcd_cell_shape;

/* Sizes of the caller-owned arenas, in elements. */
typedef struct pcd_cell_sizes {
    int64_t param_floats;     /* weights, registration order of Cell.named_parameters() */
    int64_t running_floats;   /* BN running_mean/running_var pairs, registration order */
    int64_t nbt_int64;        /* BN num_batches_tracked, registration order */
    int64_t out_floats;       /* B * 4C * Ho * Wo */
    int64_t saved_floats;     /* activations kept for backward */
    int64_t stats_doubles;    /* forward BN sums (kept for backward) */
    int64_t bwd_work_floats;  /* backward scratch */
    int64_t bwd_stats_doubles;/* backward reduction scratch */
    int32_t out_height, out_width;
} pcd_cell_sizes;

int pcd_cell_sizes_of(const pcd_cell_shape* shape, pcd_cell_sizes* out);

typedef struct pcd_cell_fwd_args {
    pcd_cell_shape shape;
    const float* s0;          /* (B, C_pp, H0, W0) contiguous */
    const float* s1;          /* (B, C_p, H, W) contiguous */
    const float* weights;     /* (14, 8) softmax(alphas) rows, device */
    const float* weights2;    /* (14,) grouped softmax(betas), device */
    const float* params;      /* param arena */
    float* running;           /* running-stat arena (updated) */
    int64_t* nbt;             /* num_batches_tracked arena (updated) */
    float* out;               /* (B, 4C, Ho, Wo) contiguous */
    float* saved;             /* saved arena */
    double* stats;            /* stats arena (zeroed by the call) */
    int32_t skip_dw_outputs;  /* 1: the backward of this forward will not ask for parameter gradients (the two
                                 finite-difference passes of the Hessian-vector product, architect_vqa.py:109,114): the
                                 saved depthwise outputs, which only the weight-gradient jobs read, are not written
                                 (pcd_cell_backward must then be called with need_param_grads == 0).  0: everything saved */
} pcd_cell_fwd_args;

int pcd_cell_forward(const pcd_cell_fwd_args* a, void* stream);

typedef struct pcd_cell_bwd_args {
    pcd_cell_shape shape;
    const float* s0;
    const float* s1;
    const float* weights;
    const float* weights2;
    const float* params;
    const float* out;         /* forward output (the node tensors live in it) */
    const float* saved;
    const double* stats;
    const float* grad_out;    /* (B, 4C, Ho, Wo) contiguous */
    float* grad_s0;           /* written */
    float* grad_s1;           /* written */
    float* grad_weights;      /* (14, 8) written */
    float* grad_weights2;     /* (14,) written */
    float* grad_params;       /* param-arena shaped; zeroed then accumulated; may be NULL when
                                 need_param_grads == 0 (the HVP passes, architect_vqa.py:110,115) */
    float* work;              /* bwd_work_floats */
    double* bstats;           /* bwd_stats_doubles (zeroed by the call) */
    int32_t need_param_grads;
    int32_t need_input_grads; /* grad_s0/grad_s1 wanted */
} pcd_cell_bwd_args;

int pcd_cell_backward(const pcd_cell_bwd_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * MixedOp(C, stride).forward(x, weights)         darts_vqa/pcdarts/model_search.py:30-58
 * ---------------------------------------------------------------------------------------------- */
typedef struct pcd_mixedop_shape {
    int32_t batch, channels, height, width, stride;
    float bn_eps, bn_momentum;
} pcd_mixedop_shape;

typedef struct pcd_mixedop_sizes {
    int64_t param_floats, running_floats, nbt_int64, out_floats, saved_floats, stats_doubles,
            bwd_work_floats, bwd_stats_doubles;
    int32_t out_height, out_width;
} pcd_mixedop_sizes;

int pcd_mixedop_sizes_of(const pcd_mixedop_shape* shape, pcd_mixedop_sizes* out);

typedef struct pcd_mixedop_fwd_args {
    pcd_mixedop_shape shape;
    const float* x;           /* (B, C, H, W) contiguous */
    const float* weights;     /* (8,) */
    const float* params;
    float* running;
    int64_t* nbt;
    float* out;               /* (B, C, H/stride, W/stride) */
    float* saved;
    double* stats;
} pcd_mixedop_fwd_args;

int pcd_mixedop_forward(const pcd_mixedop_fwd_args* a, void* stream);

typedef struct pcd_mixedop_bwd_args {
    pcd_mixedop_shape shape;
    const float* x;
    const float* weights;
    const float* params;
    const float* saved;
    const double* stats;
    const float* grad_out;
    float* grad_x;
    float* grad_weights;      /* (8,) */
    float* grad_params;
    float* work;
    double* bstats;
    int32_t need_param_grads;
} pcd_mixedop_bwd_args;

int pcd_mixedop_backward(const pcd_mixedop_bwd_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Network.stem = Conv2d(3, 3C, 3, padding=1, bias=False) + BatchNorm2d(3C) (affine)
 *                                                darts_vqa/pcdarts/model_search.py:110-113,150-151
 * params arena: conv weight (Cout,3,3,3), bn weight (Cout), bn bias (Cout).
 * saved: pre-BN conv output z (B,Cout,H,W).  stats: 2*Cout doubles.  bstats: 2*Cout doubles.
 * ---------------------------------------------------------------------------------------------- */
typedef struct pcd_stem_args {
    int32_t batch, c_out, height, width;
    float bn_eps, bn_momentum;
    const float* x;           /* (B,3,H,W) contiguous (the reference expands 1-channel input first) */
    const float* params;
    float* running;           /* mean(Cout), var(Cout) */
    int64_t* nbt;
    float* out;               /* fwd: written.  bwd: read */
    float* saved_z;           /* fwd: written.  bwd: read */
    double* stats;            /* fwd: written.  bwd: read */
    /* backward only */
    const float* grad_out;
    float* grad_x;            /* may be NULL */
    float* grad_params;       /* zeroed then accumulated; may be NULL */
    double* bstats;
} pcd_stem_args;

int pcd_stem_forward(const pcd_stem_args* a, void* stream);
int pcd_stem_backward(const pcd_stem_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * ReLUConvBN(C_in, C_out, 1, 1, 0, affine=False)   darts_vqa/pcdarts/operations.py:22-33
 * FactorizedReduce(C_in, C_out, affine=False)      darts_vqa/pcdarts/operations.py:90-104
 * (the Cell preprocess ops, model_search.py:67-71, when used on their own)
 * weight: [C_out][C_in]; for FactorizedReduce conv_1 rows then conv_2 rows, back to back.
 * y holds the normalised output; stats (2*C_out doubles) is kept for backward.
 * ---------------------------------------------------------------------------------------------- */
typedef struct pcd_pre_args {
    int32_t batch, c_in, c_out, height, width;   /* input spatial size */
    int32_t factorized;                          /* 1 => FactorizedReduce (output is H/2 x W/2) */
    float bn_eps, bn_momentum;
    const float* x;
    const float* weight;
    float* running;          /* mean(C_out), var(C_out); fwd only */
    int64_t* nbt;            /* fwd only */
    float* y;                /* fwd: written.  bwd: read */
    double* stats;           /* fwd: written.  bwd: read */
    /* backward only */
    const float* grad_y;
    float* grad_x;           /* may be NULL */
    float* grad_weight;      /* zeroed then accumulated; may be NULL */
    double* bstats;          /* 2*C_out doubles scratch */
} pcd_pre_args;

int pcd_preprocess_forward(const pcd_pre_args* a, void* stream);
int pcd_preprocess_backward(const pcd_pre_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * The candidate operations as STAND-ALONE ops on all channels of a tensor — what `OPS[name](C, stride, affine)` modules
 * run when they are called on their own and what a network derived from a genotype (SURVEY.md 8f-4; the reference stops at
 * Network.genotype(), model_search.py:218-263) is made of.  Training-mode BatchNorm only.  H, W <= 64.
 *   DilConv  (operations.py:35-47):  dwconv(relu) -> pwconv (+stats) -> bn_apply
 *   SepConv  (operations.py:50-66):  that unit twice, the first with the stride
 *   AvgPool2d(3, stride, 1, count_include_pad=False) / MaxPool2d(3, stride, 1)   (operations.py:6-7)
 * Buffers are the caller's; grad_weight buffers are zeroed by the call and then accumulated.
 * ---------------------------------------------------------------------------------------------- */
typedef struct pcd_dwconv_args {
    int32_t batch, channels, height, width;      /* input size */
    int32_t kernel, stride, padding, dilation;   /* kernel 3, 5 or 7; stride 1 or 2 */
    int32_t relu_input;                          /* 1 => the conv reads relu(x) (and grad_x is masked by x > 0) */
    const float* x;            /* (B, C, H, W) */
    const float* weight;       /* (C, 1, k, k) */
    float* out;                /* fwd: (B, C, Ho, Wo) */
    const float* grad_out;     /* bwd */
    float* grad_x;             /* bwd, may be NULL */
    float* grad_weight;        /* bwd, may be NULL */
} pcd_dwconv_args;
int pcd_dwconv_forward(const pcd_dwconv_args* a, void* stream);
int pcd_dwconv_backward(const pcd_dwconv_args* a, void* stream);

typedef struct pcd_pwconv_args {
    int32_t batch, c_in, c_out, hw;              /* channels multiples of 4 (<= 128), hw a multiple of 4 */
    float bn_eps;
    const float* x;            /* (B, c_in, hw) */
    const float* weight;       /* (c_out, c_in) */
    float* z;                  /* fwd: pre-BatchNorm output, written.  bwd: read */
    double* stats;             /* fwd: sum[c_out], sumsq[c_out], zeroed then accumulated.  bwd: read */
    const float* grad_y;       /* bwd: gradient w.r.t. the BatchNorm OUTPUT gamma * yhat + beta */
    const float* gamma;        /* bwd: NULL => 1 */
    const double* bstats;      /* bwd: sum grad_y [c_out], sum grad_y * yhat [c_out]  (pcd_bn_backward_stats) */
    float* grad_x;             /* bwd, may be NULL */
    float* grad_weight;        /* bwd, may be NULL */
} pcd_pwconv_args;
int pcd_pwconv_forward(const pcd_pwconv_args* a, void* stream);
int pcd_pwconv_backward(const pcd_pwconv_args* a, void* stream);

typedef struct pcd_bn_args {
    int32_t batch, channels, hw;
    float bn_eps, bn_momentum;
    const float* z;            /* pre-BatchNorm tensor */
    const double* stats;       /* sum, sumsq of z per channel (pcd_pwconv_forward) */
    const float* gamma;        /* NULL => 1 */
    const float* beta;         /* NULL => 0 */
    float* running;            /* apply: mean(C), var(C) updated like nn.BatchNorm2d; may be NULL */
    int64_t* nbt;              /* apply: num_batches_tracked += 1; may be NULL iff running is */
    float* y;                  /* apply: gamma * (z - mean) * rstd + beta */
    const float* grad_y;       /* backward_stats */
    double* bstats;            /* backward_stats: sum grad_y, sum grad_y * yhat (zeroed by the call) = d beta, d gamma */
} pcd_bn_args;
int pcd_bn_apply(const pcd_bn_args* a, void* stream);
int pcd_bn_backward_stats(const pcd_bn_args* a, void* stream);

typedef struct pcd_pool_args {
    int32_t batch, channels, height, width, stride, is_max;
    const float* x;
    float* y;                  /* fwd */
    const float* grad_y;       /* bwd */
    float* grad_x;             /* bwd */
} pcd_pool_args;
int pcd_pool3x3_forward(const pcd_pool_args* a, void* stream);
int pcd_pool3x3_backward(const pcd_pool_args* a, void* stream);

/* y[n][c][p] = scale[c] * x[n][c][p] + shift[c]  (NULL => 1 / 0): the affine half of BatchNorm(affine=True) behind the
 * preprocess kernels' normalised output */
int pcd_channel_affine(const float* x, const float* scale, const float* shift, float* y, int batch, int channels, int hw,
                       void* stream);

/* ------------------------------------------------------------------------------------------------
 * Eval mode (module.eval(), BatchNorm from running statistics), forward only.
 * Every BatchNorm is the per-channel affine map y = scale * z + shift with scale = gamma / sqrt(running_var + eps) and
 * shift = beta - running_mean * scale (gamma = 1, beta = 0 without affine).  The calls read the same parameter and
 * running-stat arenas, at the same offsets, as the training-mode calls above, and write nothing but their outputs
 * (and `work`): no statistics, no running-stat updates, no num_batches_tracked, no saved activations.
 * A node of a cell is ONE launch (every incoming edge, all 8 candidate ops, alpha / beta weighting, bypass channels and
 * channel shuffle).  Shape envelope as in training mode.
 * ---------------------------------------------------------------------------------------------- */
typedef struct pcd_cell_eval_args {
    pcd_cell_shape shape;
    const float* s0;          /* (B, C_pp, H0, W0) contiguous */
    const float* s1;          /* (B, C_p, H, W) contiguous */
    const float* weights;     /* (14, 8) softmax(alphas) rows, device */
    const float* weights2;    /* (14,) grouped softmax(betas), device */
    const float* params;      /* param arena (pcd_cell_sizes_of) */
    const float* running;     /* running-stat arena, read only */
    float* out;               /* (B, 4C, Ho, Wo) contiguous */
    float* work;              /* pcd_cell_eval_work_floats: the two preprocessed states */
} pcd_cell_eval_args;

int pcd_cell_eval_work_floats(const pcd_cell_shape* shape, int64_t* work_floats);
int pcd_cell_forward_eval(const pcd_cell_eval_args* a, void* stream);

typedef struct pcd_mixedop_eval_args {
    pcd_mixedop_shape shape;
    const float* x;           /* (B, C, H, W) contiguous */
    const float* weights;     /* (8,) */
    const float* params;
    const float* running;     /* read only */
    float* out;               /* (B, C, H/stride, W/stride) */
} pcd_mixedop_eval_args;

int pcd_mixedop_forward_eval(const pcd_mixedop_eval_args* a, void* stream);

/* ReLUConvBN(C_in, C_out, 1, 1, 0) / FactorizedReduce: C_out a multiple of 16 (32 for FactorizedReduce) */
typedef struct pcd_pre_eval_args {
    int32_t batch, c_in, c_out, height, width;   /* input spatial size */
    int32_t factorized;
    float bn_eps;
    const float* x;
    const float* weight;      /* as pcd_pre_args.weight */
    const float* running;     /* mean(C_out), var(C_out) */
    const float* gamma;       /* NULL => 1 (affine=False) */
    const float* beta;        /* NULL => 0 */
    float* y;                 /* (B, C_out, Ho, Wo) */
} pcd_pre_eval_args;

int pcd_preprocess_forward_eval(const pcd_pre_eval_args* a, void* stream);

typedef struct pcd_stem_eval_args {
    int32_t batch, c_out, height, width;
    float bn_eps;
    const float* x;           /* (B,3,H,W) contiguous */
    const float* params;      /* conv weight (Cout,3,3,3), bn weight (Cout), bn bias (Cout) */
    const float* running;     /* mean(Cout), var(Cout) */
    float* out;               /* (B,Cout,H,W) */
} pcd_stem_eval_args;

int pcd_stem_forward_eval(const pcd_stem_eval_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Network.global_pooling = AdaptiveAvgPool2d(7) followed by flatten
 *                                                darts_vqa/pcdarts/model_search.py:129,176-178
 * ---------------------------------------------------------------------------------------------- */
int pcd_adaptive_avgpool_forward(const float* x, float* y, int batch, int channels, int h, int w,
                                 int oh, int ow, void* stream);
int pcd_adaptive_avgpool_backward(const float* gy, float* gx, int batch, int channels, int h, int w,
                                  int oh, int ow, void* stream);

/* Overlap of the deferred weight-gradient jobs with the rest of the backward pass.  With overlap on,
 * pcd_cell_backward enqueues them on a library-owned low-priority stream (forked with an event: no host
 * synchronisation; CUDA-graph capturable) and returns without joining: grad_params and every buffer passed to that
 * call must stay alive and unread until pcd_overlap_join(stream) has been enqueued on the consuming stream.
 * Call pcd_set_overlap outside stream capture.  Default off. */
int pcd_set_overlap(int on);
int pcd_overlap_join(void* stream);

/* ------------------------------------------------------------------------------------------------
 * Dense fp32 contraction on the tcgen05 tensor cores (3xTF32 split, fp32 accumulation in tensor memory):
 *     C[M][N] = A[M][K] * B[N][K]^T (+ bias[N])        row-major, K contiguous in A and B
 * Replaces the cuBLAS SGEMMs behind nn.Linear for the question decoder's vocabulary projection
 * (darts_vqa/vqa_model.py:192-194, fc1 over B*30 rows) and its backward products.
 * A, B: 16-byte aligned, lda / ldb multiples of 4.  split_k > 1: K is split over blockIdx.z and partial sums are
 * added atomically into a zeroed C (done here).  bias may be NULL.
 * ---------------------------------------------------------------------------------------------- */
int pcd_gemm_tn_3xtf32(const float* A, long long lda, const float* B, long long ldb, float* C, long long ldc,
                       int M, int N, int K, const float* bias, int split_k, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Small dense products in exact fp32 (FMA): C[i][j] = sum_l A[i*a_i + l*a_l] * B[j*b_j + l*b_l] (+ bias[j]).  The generic strides
 * express y = x W^T + b, dx = dy W and dW = dy^T x of an nn.Linear without operand transposes.  Used for the answer head
 * (darts_vqa/vqa_model.py:308-316) and the question encoder's fc2 (:186-190) at batch 64 instead of a library SGEMM.
 * ---------------------------------------------------------------------------------------------- */
int pcd_gemm_small_f32(const float* A, long long a_i, long long a_l, const float* B, long long b_j, long long b_l, float* C,
                       long long ldc, int I, int J, int L, const float* bias, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Cross-entropy over the vocabulary logits, in the padded-pitch layout the projection GEMM writes
 * (darts_vqa/vqa_model.py:356-358: CE(qst_out[:, :-1], qst[:, 1:]); rows with a negative target are ignored).
 *   forward : lse[r] = logsumexp(logits[r, :V]);  loss_rows[r] = lse[r] - logits[r, target[r]]  (0 if ignored)
 *   backward: dlogits[r, c] = scale * (softmax(logits[r])[c] - [c == target[r]])  (0 for ignored rows and pad columns);
 *             `scale` is a device scalar (upstream grad / number of valid rows)
 * pcd_transpose_pad: dst[c][r] = src[r][c] (r < R, c < C), dst columns [R, ld_d) zero — the K-major operands of the
 * backward GEMMs (dlogits^T, W^T, h^T).
 * ---------------------------------------------------------------------------------------------- */
int pcd_ce_forward(const float* logits, long long ld, int M, int V, const long long* targets, float* lse,
                   float* loss_rows, void* stream);
int pcd_ce_backward(const float* logits, long long ld, int M, int V, const long long* targets, const float* lse,
                    const float* scale, float* dlogits, void* stream);
int pcd_transpose_pad(const float* src, long long ld_s, int R, int C, float* dst, long long ld_d, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Single-layer LSTM recurrence of the question encoder (darts_vqa/vqa_model.py:165,176-184: nn.LSTM(300, 512, 1), T = 30,
 * h0 = c0 = image embedding) as persistent cooperative kernels (one grid barrier per time step).  PyTorch gate order
 * i, f, g, o.  gx = x W_ih^T + b_ih + b_hh ([T][B][4H], from pcd_gemm_tn_3xtf32).  Forward saves the gate activations
 * `act`, the cell states `cs` and the outputs `hs`; backward turns (dhs, dhT, dcT) into dgates ([T][B][4H]; the weight /
 * input gradients are GEMMs over it), dh0 and dc0.  B <= 64, H a power of two in [16, 512].  pbuf: scratch of
 * pcd_lstm_pbuf_floats(B, H) floats.
 * ---------------------------------------------------------------------------------------------- */
size_t pcd_lstm_pbuf_floats(int B, int H);
int pcd_lstm_forward(int T, int B, int H, const float* gx, const float* w_hh, const float* h0, const float* c0,
                     float* act, float* cs, float* hs, void* stream);
int pcd_lstm_backward(int T, int B, int H, const float* dhs, const float* dhT, const float* dcT, const float* act,
                      const float* cs, const float* c0, const float* w_hh, float* dgates, float* dh0, float* dc0,
                      float* pbuf, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Question decode: replaces QstEncoder.generate's 30-iteration loop of embedding -> nn.LSTM step -> tanh -> Linear(H, V)
 * -> argmax (darts_vqa/vqa_model.py:103-136, basic_vqa/models_lct.py:124-157) with one persistent cooperative kernel, in
 * one of three modes, each with or without end-of-sequence decoding.  One pcd_decode_args describes a call; the struct is
 * a HOST pointer read at the call, every pointer in it is device memory.
 *
 * Every mode: h = h0[row], c = c0[row]; the first input is tanh(emb[start_token]), later inputs emb[previous word] (no tanh:
 * vqa_model.py:133); gate order i, f, g, o; logits l = tanh(h_t) w_out^T + b_out.
 *   PCD_DECODE_GREEDY (deterministic sampling): word t of row b is argmax_v l_v, ties to the lowest index.
 *              tokens: [B][T] int64.
 *   PCD_DECODE_SAMPLED (QstEncoder.generate with deterministic=False: every word drawn from softmax(logits / temperature),
 *              darts_vqa/vqa_model.py:87-92), by the Gumbel-max trick: word t of row b is
 *                  argmax_v ( logit_v / temperature + G(seed, t, row_offset + b, v) )
 *              with G a standard Gumbel variable from Philox4x32-10:  key = {seed & 0xffffffff, seed >> 32}, counter =
 *              {v >> 2, t, row, 0}, x = word (v & 3) of the block, u = ((float)(x >> 9) + 0.5f) * 2^-23, G = -logf(-logf(u)).
 *              The noise depends only on (seed, t, row, v): a batch decoded in slices (row_offset = first row of the slice)
 *              draws what one call would.  `seed` is a DEVICE pointer to one 8-byte-aligned uint64, read by the kernel (a
 *              CUDA graph replays the seed the buffer holds at replay time).  The distribution equals torch.multinomial's;
 *              the random stream does not.  tokens: [B][T] int64.
 *   PCD_DECODE_BEAM (QstEncoder.generate with deterministic=True and beam_size = K > 1): items b = 0..B-1, beams
 *              k = 0..K-1, rows r = b*K + k.
 *     t = 0:     every row of item b starts from h = h0[b], c = c0[b] with input tanh(emb[start_token]); the beam scores start
 *                at (0, -inf, ..., -inf), so only beam 0 of an item contributes candidates.
 *     each step: per row one LSTM step gives (h_t, c_t) and the logits l_r; log-probabilities lambda_r = l_r - logsumexp(l_r)
 *                (temperature 1).  The candidates of item b are the pairs (k, v) scored s_{b,k} + lambda_{b,k}[v]; the K
 *                highest become the new beams j = 0..K-1 in descending order, exact ties going to the lower k, then the
 *                lower v.  Beam j takes over the (h_t, c_t) of its parent row, and its next input is emb[v_j] (no tanh, as
 *                the greedy decode after the start token).
 *     output:    tokens [B][K][T] int64, the words on beam j's path (backtracked through the parent pointers); scores
 *                [B][K] fp32, the cumulative log-probability of that path; beams best first.  tokens is also used as
 *                scratch until the kernel ends.
 * Without the stop (stop = 0) every row has exactly T words, and beams have no length penalty.
 *
 * End-of-sequence decoding (stop = 1): a stop word E = end_token, a padding word P = pad_token and, for beams, a length
 * penalty alpha = length_penalty.
 *   greedy, sampled: every word is chosen exactly as without the stop; once a row has emitted E, every later position is P
 *              (E itself stays).  A stopped decode therefore equals the unstopped one truncated after the first E and filled
 *              with P, bit for bit (rows are independent, the sampled noise depends on (seed, t, row, v) only).
 *   beam:      a beam is finished once its last word is E.  A live beam k contributes the candidates (k, v) for every v, raw
 *              score s_k + lambda_k[v]; a finished beam contributes exactly one, (k, P), with its raw score s_k unchanged.
 *              Candidates are ranked by the key s / powf((float)L, alpha) in fp32 (s itself when alpha = 0), L the
 *              hypothesis length counting E: t + 1 for a live candidate at step t, the frozen length for a finished beam.
 *              Ties as without the stop (lower k, then lower v).  scores returns the raw cumulative log-probability of
 *              each path up to and including E (P adds 0); beams come out best first by key.  With alpha = 0 and E never
 *              emitted the result is bit-equal to the decode without the stop.
 *   early exit: once every row of the launch has finished, the kernel leaves its time loop and the remaining positions are
 *              P (beams: the backtrack starts from the last step run).
 *
 * Truncated sampling (sampled mode, truncate = 1; HF-style order: temperature, then top-k, then top-p renormalised over the
 * top-k set).  l is a row's fp32 logits (as above), T the temperature.
 *   order:     v precedes w iff l_v > l_w, or l_v = l_w and v < w (ties to the lower word, as the greedy argmax; -0 = +0).
 *   top-k:     S_k = the first min(top_k, V) words in that order; top_k = 0 (or >= V): all V words.
 *   nucleus:   q_v = expf((l_v - l_max) / T) in fp32, rounded to an integer multiple of 2^-s with s = 63 - (bit length
 *              of V); these masses are summed exactly in 64-bit integers, so any summation order gives the same sums.
 *              Z = sum of q over S_k; the target is ceil(top_p * Z) with Z rounded to fp64 and the product in fp64 (at
 *              most Z).  S = the shortest prefix of S_k, in order, whose mass reaches the target: never empty (the first
 *              word has q = 1).  top_p = 1: S = S_k, with no mass computed.
 *   draw:      word t of row b = argmax over v in S of (l_v / T + G(seed, t, row_offset + b, v)), the score and noise of
 *              untruncated sampling, ties to the lower word: distributed as softmax(l / T) restricted to S and renormalised.
 *   So top_k = 0 with top_p = 1 gives the untruncated words bit for bit, and top_k = 1, or a top_p below 1/V, the greedy
 *   words.  stop = 1 combines as with plain sampling.  The kernel keeps each step's logits in the workspace (rows x V
 *   floats) and finds S by radix select behind one more grid barrier per step.
 *
 * Envelope: H a multiple of 32 up to 512, E a multiple of 4, start_token in [0, V); greedy and sampled: B <= 64 rows; beam:
 * 1 <= K <= 8, K <= V, B*K <= 64 rows.  PCD_ERR_UNSUPPORTED outside it.
 * PCD_ERR_ARG, before any shape check: a mode outside the three; K != 1 outside beam mode; a null emb .. b_out, tokens or
 * work, or a null scores in beam mode; sampled: a null seed, a negative row_offset or a temperature that is not finite and
 * > 0; stop: an E or P outside [0, V) or an alpha that is not finite; truncate = 1 outside sampled mode, a negative
 * top_k, or a top_p that is not finite or lies outside (0, 1].
 * PCD_ERR_ALIGN: emb, w_ih, w_hh, h0, w_out and work must be 16-byte aligned, the seed 8-byte aligned.
 * work: pcd_decode_work_floats(a) floats (it reads mode, B, K, H, V and truncate; truncation adds B x V + B floats).
 * The call only uses caller-owned memory and
 * neither synchronises nor allocates (CUDA-graph capturable).  All reductions run in a fixed order: equal inputs give
 * bit-equal outputs.
 * ---------------------------------------------------------------------------------------------- */
enum { PCD_DECODE_GREEDY = 0, PCD_DECODE_SAMPLED = 1, PCD_DECODE_BEAM = 2 };

typedef struct pcd_decode_args {
    int mode;                         /* PCD_DECODE_* */
    int T, B, K, H, E, V;             /* B: rows (greedy, sampled) or items (beam); K: beams per item, 1 outside beam mode */
    int start_token;
    int stop;                         /* 1: end-of-sequence decoding */
    int end_token, pad_token;         /* stop only */
    float length_penalty;             /* beam with stop only */
    float temperature;                /* sampled only */
    int row_offset;                   /* sampled only: global index of row 0 */
    int truncate;                     /* sampled only, 1: top-k / nucleus truncation (0: sample from every word) */
    int top_k;                        /* truncate only: 0 = no top-k limit */
    float top_p;                      /* truncate only: in (0, 1], 1 = no nucleus */
    const unsigned long long* seed;   /* sampled only */
    const float *emb, *w_ih, *w_hh, *b_ih, *b_hh, *h0, *c0, *w_out, *b_out;
    long long* tokens;                /* [B][T]; beam [B][K][T] */
    float* scores;                    /* beam only: [B][K] */
    float* work;
} pcd_decode_args;

size_t pcd_decode_work_floats(const pcd_decode_args* a);
int pcd_decode(const pcd_decode_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Drop-path node sum of the derived network's cells (pcdarts/model.py; DARTS's drop_path on every non-Identity op output):
 *     forward : out[b]     = d1(b) * h1[b] + d2(b) * h2[b]
 *     backward: grad_h1[b] = d1(b) * grad_out[b],  grad_h2[b] = d2(b) * grad_out[b]     (either output may be NULL)
 * h1, h2, out, grad_* are (batch, sample_numel) fp32, contiguous.  d_i(b) x = x when drop_i is 0, else (x / keep) * m_i(b) with
 * IEEE division (DARTS's x.div_(keep_prob).mul_(mask), bit for bit for the same mask); the sum is one fp32 add, so with both
 * flags off, or keep = 1, out is bit-equal to h1 + h2.  m_i(b) in {0, 1} is a pure function (pcd_philox.cuh):
 *     x = Philox4x32-10(counter = {sample_offset + b, cell, 2 * node + i, 0x44504154}, key = {seed & 0xffffffff, seed >> 32}).word[0]
 *     m = ((x >> 8) * 2^-24 < keep)
 * so a sample's mask depends on its global index only: data-parallel shards (sample_offset = rank * local batch) draw what one
 * process would draw on the whole batch.  `seed` (one uint64) and `keep` (one float) are DEVICE pointers read when the kernel
 * runs (CUDA-graph capturable: a replay uses the values they hold then).  The backward recomputes the masks.
 * PCD_ERR_ARG for a null seed or keep while a drop flag is set, a negative sample_offset (or sample_offset + batch >= 2^31),
 * or a null tensor pointer; PCD_OK without a launch for an empty tensor.
 * ---------------------------------------------------------------------------------------------- */
typedef struct pcd_droppath_args {
    int batch;
    long long sample_numel;   /* C*H*W */
    int drop1, drop2;         /* input i is subject to drop-path */
    int cell, node;           /* position of the node in the network: counter words of the mask */
    int sample_offset;        /* global index of sample 0 */
    const unsigned long long* seed;
    const float* keep;        /* 1 - drop_path_prob */
    const float* h1;          /* forward */
    const float* h2;
    float* out;
    const float* grad_out;    /* backward */
    float* grad_h1;
    float* grad_h2;
} pcd_droppath_args;

int pcd_droppath_sum_forward(const pcd_droppath_args* a, void* stream);
int pcd_droppath_sum_backward(const pcd_droppath_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Optimizer-side elementwise operations over a short table of flat runs.  The search step updates all 732 parameter
 * tensors several times per step outside the network — w' = w - eta * dL/dw (darts_vqa/pcdarts/architect_vqa.py:35-38),
 * w +- R v of the finite-difference Hessian-vector product (:106-118), clip_grad_norm_ and Adam
 * (darts_vqa/experiment.py:196-198).  The search network's parameters sit back to back in one arena and their gradients
 * come back as one flat buffer per cell, so those tensors are a few dozen contiguous runs: `n` runs (<= pcd_flat_max_runs()),
 * sizes[i] elements each, one device pointer per run and operand (HOST arrays of device pointers).
 *   pcd_flat_axpy  : y += (alpha_dev ? alpha * *alpha_dev : alpha) * x
 *   pcd_flat_scale : y *= *scale_dev
 *   pcd_flat_sumsq : *out += sum of squares (the caller zeroes *out); deterministic (fixed reduction order, no atomics: every
 *                    data-parallel rank must derive the same clip coefficient); work: pcd_flat_sumsq_work(elements) doubles
 *   pcd_flat_adam  : torch.optim.Adam's update (L2-style weight decay); *step_dev = step count AFTER the increment
 * ---------------------------------------------------------------------------------------------- */
int pcd_flat_max_runs(void);
int pcd_flat_axpy(int n, const long long* sizes, float* const* y, float* const* x, const float* alpha_dev, float alpha, void* stream);
int pcd_flat_scale(int n, const long long* sizes, float* const* y, const float* scale_dev, void* stream);
long long pcd_flat_sumsq_work(long long total_elements);
int pcd_flat_sumsq(int n, const long long* sizes, float* const* x, double* out, double* work, void* stream);
int pcd_flat_adam(int n, const long long* sizes, float* const* p, float* const* g, float* const* m, float* const* v, float lr,
                  float beta1, float beta2, float eps, float weight_decay, const float* step_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PCDARTS_SM100_H */
