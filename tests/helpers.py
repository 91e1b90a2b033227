"""Shared test helpers (tolerances, golden loading)."""
import os

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
REL_TOL = 1e-4     # north_star: "within rel 1e-4 (fp32)"


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False)
    return {k: (torch.from_numpy(z[k]) if z[k].dtype.kind in "fiu" else z[k]) for k in z.files}


def rel_err(a, b):
    """max|a-b| / max(|b|_inf, tiny) — the per-tensor metric of SURVEY.md §7.1 step 0."""
    a = torch.as_tensor(a).double().cpu()
    b = torch.as_tensor(b).double().cpu()
    assert a.shape == b.shape, (a.shape, b.shape)
    if a.numel() == 0:
        return 0.0
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-12)).item()


def assert_close(a, b, tol=REL_TOL, what=""):
    e = rel_err(a, b)
    assert e <= tol, f"{what}: rel err {e:.3e} > {tol:.1e}"


# ---- pcd_gemm_tn_3xtf32: shapes of the envelope sweep and the accuracy criterion that separates 3xTF32 from fewer terms ----
# (M, N, K, lda, ldc, split_k, bias).  Every K (4 and 10 / 17 below one k-block, 10 / 17 ragged and read through a wider
# row pitch, 4100 = many k-blocks) meets every split (1, 3, more than there are k-blocks: clamped) with and without bias;
# the (M, N) pairs walk all of M in {1, 127, 128, 129, 300} x N in {4, 129, 255, 256, 257}; ldc > N on two of three cases.
# The last two have more than 3 x 148 work items for every tile configuration: a persistent CTA walks >= 3 tiles, so
# both tensor-memory accumulator buffers wrap their mbarrier phase.
def _gemm_cases():
    mn = [(m, n) for m in (1, 127, 128, 129, 300) for n in (4, 129, 255, 256, 257)]
    cases = []
    i = 0
    for k, lda in ((4, 4), (10, 12), (16, 16), (17, 20), (300, 300), (4100, 4100)):
        for split in (1, 3, 1 << 20):
            for bias in (False, True):
                m, n = mn[(7 * i) % len(mn)]
                ldc = (n, n + 3, n + (-n) % 4 + 8)[i % 3]
                cases.append((m, n, k, lda, ldc, split, bias))
                i += 1
    cases += [(300, 40000, 68, 68, 40004, 1, True), (300, 40000, 68, 72, 40001, 3, True)]
    return cases


GEMM_CASES = _gemm_cases()

# Accept a product when its error (max |C - exact| / max |exact|) is within F32_FACTOR of a plain fp32 product's on the same
# operands AND below a TF32_DIVISOR-th of the error of the 1xTF32 product (operands truncated to 10 mantissa bits, exact
# accumulation).  The fp32 error is floored at 2^-21, the relative error 3xTF32 keeps per product by design (the dropped
# lo*lo term and the truncated lo operand, <= 2^-22 each): with 4 outputs the fp32 maximum alone can be 2^-24 by luck.
# Calibrated on a B200 (1000 W) over GEMM_CASES x the four tile configurations x both kernels: the kernel's error reaches
# 66x the (floored) fp32 error and 0.045x the 1xTF32 error; the products missing one correction term reach no less than
# 279x and 0.26x.  The kernel's worst cases are the longest accumulations (K = 4100 in one split: 3.5e-5, ~100x the
# error of the same 3-term product accumulated exactly; 1.1e-5 with three splits; 3e-6 at K = 300): the error grows
# linearly with the k-blocks per split, as it does when each MMA's sum is truncated into the fp32 tensor-memory
# accumulator rather than rounded.
F32_FACTOR = 128.0
TF32_DIVISOR = 10.0
F32_FLOOR = 2.0 ** -21


def trunc_tf32(x):
    """x with the low 13 mantissa bits cleared: the operand kind::tf32 multiplies (float32 in, float32 out)."""
    return (x.float().contiguous().view(torch.int32) & -8192).view(torch.float32)


def gemm_errors(c, a, b, bias=None):
    """(err of c, err of the fp32 product, err of the 1xTF32 product) against the float64 product of a (M, K), b (N, K)."""
    def err(x, ref):
        return ((x.double() - ref).abs().max() / ref.abs().max().clamp_min(1e-300)).item()
    a64, b64 = a.double(), b.double()
    bias64 = 0.0 if bias is None else bias.double()
    ref = a64 @ b64.T + bias64
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        c32 = a.float() @ b.float().T + (0.0 if bias is None else bias.float())
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    c1 = trunc_tf32(a).double() @ trunc_tf32(b).double().T + bias64
    return err(c, ref), err(c32, ref), err(c1, ref)


def accept_3xtf32(err, err32, err1):
    return err <= F32_FACTOR * max(err32, F32_FLOOR) and err <= err1 / TF32_DIVISOR
