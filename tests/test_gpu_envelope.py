"""The GPU-only kernels across everything their launchers accept.

pcd_gemm_sm100.cu, pcd_pre_tc.cu and pcd_ce.cu have no emulated body (their CPU build is a plain reference loop or
PCD_ERR_UNSUPPORTED), so these cases are the only evidence that the tensor-core GEMM, the tensor-core preprocess and the
cross-entropy kernels are right at the edges of their envelope.  Each case shows that it reached the kernel it targets:
the GEMM is called through the C ABI, the preprocess cases read the library profiler's kernel names, and the MixedOp /
cell cases assert that the production edge kernels (fwdB4_*, bwdA4_*) ran and the generic ones did not.

GEMM accuracy: helpers.accept_3xtf32 (CPU-checked to reject 1- and 2-term split products at every shape of the sweep).
Measured on a B200 (1000 W power limit), worst over GEMM_CASES per tile configuration, identical on both kernels: error /
floored fp32 error 58 / 52 / 66 / 56 and error / 1xTF32 error 0.045 / 0.035 / 0.044 / 0.040 for configurations 1-4.
The whole file takes about 16 s of test time on that GPU.
"""
import os
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F

import parity_cases as P
from helpers import F32_FLOOR, GEMM_CASES, accept_3xtf32, gemm_errors

pytestmark = pytest.mark.gpu
DEV = "cuda"
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def _lib():
    import pcd_native
    return pcd_native.load_cuda()


def _profiled(fn):
    """Run fn() with the library's launch profiler on; -> (result, {kernel name: launches})."""
    import pcd_native
    lib = _lib()
    lib.pcd_profile_enable(1)
    try:
        out = fn()
        torch.cuda.synchronize()
        names = {k: v[1] for k, v in pcd_native.profile_collect(lib).items()}
    finally:
        lib.pcd_profile_enable(0)
    return out, names


# ---------------------------------------------------------------------------------------------------------------------
# A. pcd_gemm_tn_3xtf32 through the C ABI
# ---------------------------------------------------------------------------------------------------------------------
def _gemm_case(lib, case, seed):
    """One call on NaN-guarded buffers -> (err, err fp32, err 1xTF32).  A and B carry NaN in their pad columns [K, lda)
    (TMA must not read past K); C is (M + 1) x ldc of NaN and only its M x N window may change."""
    m, n, k, lda, ldc, split, has_bias = case
    g = torch.Generator().manual_seed(seed)
    a = torch.full((m, lda), float("nan"))
    b = torch.full((n, lda), float("nan"))
    a[:, :k] = torch.randn(m, k, generator=g)
    b[:, :k] = torch.randn(n, k, generator=g)
    bias = torch.randn(n, generator=g).to(DEV) if has_bias else None
    a, b = a.to(DEV), b.to(DEV)
    c = torch.full((m + 1, ldc), float("nan"), device=DEV)
    rc = lib.pcd_gemm_tn_3xtf32(a.data_ptr(), lda, b.data_ptr(), lda, c.data_ptr(), ldc, m, n, k,
                                None if bias is None else bias.data_ptr(), split, torch.cuda.current_stream().cuda_stream)
    assert rc == 0, (case, lib.pcd_strerror(rc), lib.pcd_last_cuda_error())
    torch.cuda.synchronize()
    assert torch.isnan(c[m]).all(), (case, "row M written")
    assert torch.isnan(c[:m, n:]).all(), (case, "columns [N, ldc) written")
    win = c[:m, :n]
    assert torch.isfinite(win).all(), (case, "window not fully written")
    return gemm_errors(win, a[:, :k], b[:, :k], bias)


def gemm_sweep():
    """Every tile configuration x every case of helpers.GEMM_CASES; -> report lines.  Raises on the first failure."""
    lib = _lib()
    lines = []
    try:
        for cfg in (1, 2, 3, 4):
            lib.pcd_gemm_debug_cfg(cfg)
            worst32 = worst1 = 0.0
            for i, case in enumerate(GEMM_CASES):
                err, err32, err1 = _gemm_case(lib, case, 1000 * cfg + i)
                assert accept_3xtf32(err, err32, err1), (cfg, case, err, err32, err1)
                worst32 = max(worst32, err / max(err32, F32_FLOOR))
                worst1 = max(worst1, err / err1)
            lines.append(f"cfg {cfg}: worst err / fp32 err {worst32:.2f}, worst err / 1xTF32 err {worst1:.2e}")
    finally:
        lib.pcd_gemm_debug_cfg(0)
    return lines


def _gemm_kernel_names():
    """CUDA kernel names launched by one small pcd_gemm_tn_3xtf32 call (torch profiler)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        _gemm_case(_lib(), (129, 257, 68, 68, 260, 1, True), 5)
        torch.cuda.synchronize()
    return {e.key for e in prof.key_averages() if "gemm_tn_3xtf32" in e.key}


@pytest.fixture
def gemm_cfg_restored():
    yield
    _lib().pcd_gemm_debug_cfg(0)


def test_gemm_3xtf32_envelope_persistent(gemm_cfg_restored):
    """The persistent kernel (the default) at all four tile configurations: see helpers.GEMM_CASES for the shapes."""
    names = _gemm_kernel_names()
    assert names and all("persist" in s for s in names), names
    print("\n".join(gemm_sweep()))


def test_gemm_3xtf32_envelope_one_tile_per_cta():
    """The same sweep on the one-tile-per-CTA kernel.  PCD_GEMM_PERSIST is read once per process, so this arm runs in a
    child process that exits (or is killed at the timeout) before the test returns."""
    env = dict(os.environ, PCD_GEMM_PERSIST="0",
               PYTHONPATH=os.pathsep.join([HERE, os.path.join(ROOT, "lct-vqa_b200"), ROOT, os.environ.get("PYTHONPATH", "")]))
    r = subprocess.run([sys.executable, "-s", os.path.abspath(__file__), "--gemm-one-tile-per-cta"], env=env, cwd=ROOT,
                       capture_output=True, text=True, timeout=600)
    print(r.stdout)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    assert "one-tile-per-cta sweep ok" in r.stdout


def test_gemm_3xtf32_rejects_bad_arguments():
    """Misaligned operands / pitches are refused (PCD_ERR_ALIGN), never run."""
    lib = _lib()
    a = torch.randn(8, 20, device=DEV)
    c = torch.zeros(8, 8, device=DEV)
    st = torch.cuda.current_stream().cuda_stream
    for args in ((a.data_ptr(), 18, a.data_ptr(), 20, c.data_ptr(), 8, 8, 8, 16, None, 1, st),      # lda % 4
                 (a.data_ptr() + 4, 20, a.data_ptr(), 20, c.data_ptr(), 8, 8, 8, 16, None, 1, st),  # A not 16-byte aligned
                 (a.data_ptr(), 12, a.data_ptr(), 20, c.data_ptr(), 8, 8, 8, 16, None, 1, st),      # lda < K
                 (a.data_ptr(), 20, a.data_ptr(), 20, c.data_ptr(), 7, 8, 8, 16, None, 1, st)):     # ldc < N
        assert lib.pcd_gemm_tn_3xtf32(*args) != 0, args


# ---------------------------------------------------------------------------------------------------------------------
# B. tensor-core preprocess across pre_tc_supported
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("c_in,c_out,H,W,B", [
    (16, 16, 8, 16, 1),        # one 128-pixel tile; dW k-split clamped to 1
    (32, 32, 64, 128, 2),      # W = 128: one image row per tile
    (48, 16, 32, 128, 3),
    (64, 32, 128, 64, 2),      # H = 2W
    (96, 64, 16, 32, 4),       # H = W/2; 128 tensor-memory columns
    (80, 16, 32, 32, 3),       # 128 columns, C_in not a power of two
    (192, 64, 16, 16, 5),      # ragged second dW m-tile (the tile reads 64 channels of the next image)
    (240, 32, 8, 16, 1),       # ragged second dW m-tile at the end of the tensor (TMA zero fill)
    (144, 16, 32, 16, 2),      # 256 columns
])
def test_preprocess_tensor_core_envelope(c_in, c_out, H, W, B, monkeypatch):
    """pre_tc_fwd (PCD_PRE_TC_FWD=1), pre_tc_dx and pre_tc_dw against BN(conv1x1(relu(x))) in float64, next to the FP32-FMA
    kernels (PCD_NO_PRE_TC=1) on the same tensors; a shape that quietly fell back to the FMA kernels fails."""
    import config
    config.DEVICE = DEV
    from pcdarts.operations import ReLUConvBN
    torch.manual_seed(c_in + c_out + H + W + B)
    m = ReLUConvBN(c_in, c_out, 1, 1, 0, affine=False).to(DEV).train()
    x = torch.randn(B, c_in, H, W, device=DEV)
    G = torch.randn(B, c_out, H, W, device=DEV)

    def run():
        xx = x.clone().requires_grad_(True)
        m.zero_grad()
        y = m(xx)
        (y * G).sum().backward()
        return y.detach().clone(), xx.grad.clone(), m.op[1].weight.grad.clone()
    xd = x.double().requires_grad_(True)
    wd = m.op[1].weight.detach().double().requires_grad_(True)
    yd = F.batch_norm(F.conv2d(F.relu(xd), wd), None, None, training=True, eps=1e-5)
    (yd * G.double()).sum().backward()
    ref = (yd.detach(), xd.grad, wd.grad)
    monkeypatch.setenv("PCD_PRE_TC_FWD", "1")
    got, names = _profiled(run)
    for k in ("pre_tc_fwd", "pre_tc_dx", "pre_tc_dw"):
        assert names.get(k, 0) >= 1, (k, names)
    monkeypatch.setenv("PCD_NO_PRE_TC", "1")
    fma, names = _profiled(run)
    assert not any(k.startswith("pre_tc") for k in names), names
    rep = {n: dict(tc=P.rel_err(a_, r), fma=P.rel_err(c_, r)) for n, r, a_, c_ in zip(("y", "dx", "dW"), ref, got, fma)}
    print("preprocess tc / fma vs fp64:", rep)
    for n, v in rep.items():
        assert v["tc"] <= 2e-5, (n, rep)


# ---------------------------------------------------------------------------------------------------------------------
# C. cross-entropy rows and transpose_pad
# ---------------------------------------------------------------------------------------------------------------------
def _ce_reference(logits, V, tg, scale):
    """float64 on the CPU: lse of every row; loss and dlogits of the rows with 0 <= target < V (the others are 0)."""
    l64 = logits[:, :V].double().cpu()
    t = tg.cpu()
    valid = (t >= 0) & (t < V)
    lse = torch.logsumexp(l64, 1)
    loss = torch.zeros_like(lse)
    dl = torch.softmax(l64, 1)
    rows = valid.nonzero().flatten()
    loss[rows] = lse[rows] - l64[rows, t[rows]]
    dl[rows, t[rows]] -= 1.0
    dl[~valid] = 0.0
    return lse, loss, scale * dl


@pytest.mark.parametrize("V,M,spread", [(1, 5, 1.0), (3, 7, 1.0), (4, 6, 1.0), (5, 9, 80.0), (1027, 33, 80.0),
                                        (1027, 8, 1.0)])
def test_ce_kernels_edge_rows(V, M, spread):
    """pcd_ce_forward / pcd_ce_backward called directly on a buffer with pitch ld > V whose pad columns hold NaN: targets
    negative, in range and >= V; logits up to +-spread; a row whose maximum dominates, placed in the scalar tail
    c >= 4 * (V / 4) when V % 4 != 0.  lse against float64 logsumexp, dlogits exact 0 in ignored rows and pad columns."""
    lib = _lib()
    ld = V + (-V) % 4 + 8
    g = torch.Generator().manual_seed(V + M)
    logits = torch.full((M, ld), float("nan"))
    logits[:, :V] = spread * (2 * torch.rand(M, V, generator=g) - 1)
    logits[0, V - 1] = spread + 40.0                       # dominant logit in the last column (the tail when V % 4)
    tg = torch.randint(0, V, (M,), generator=g)
    tg[0] = V - 1
    tg[1] = V                                              # out of range: ignored
    tg[2] = -100
    tg[M - 1] = V + 1000
    logits, tgd = logits.to(DEV), tg.to(DEV)
    lse = torch.empty(M, device=DEV)
    rows = torch.empty(M, device=DEV)
    dl = torch.full((M, ld), float("nan"), device=DEV)
    scale = torch.tensor([0.37], device=DEV)
    st = torch.cuda.current_stream().cuda_stream
    assert lib.pcd_ce_forward(logits.data_ptr(), ld, M, V, tgd.data_ptr(), lse.data_ptr(), rows.data_ptr(), st) == 0
    assert lib.pcd_ce_backward(logits.data_ptr(), ld, M, V, tgd.data_ptr(), lse.data_ptr(), scale.data_ptr(), dl.data_ptr(), st) == 0
    torch.cuda.synchronize()
    lse_r, loss_r, dl_r = _ce_reference(logits, V, tg, 0.37)
    valid = (tg >= 0) & (tg < V)
    assert (rows.cpu()[~valid] == 0).all() and (dl.cpu()[~valid] == 0).all()
    assert (dl[:, V:] == 0).all(), "pad columns of dlogits must be exactly 0"
    assert ((lse.double().cpu() - lse_r).abs() <= 2e-6 * lse_r.abs().clamp_min(1.0)).all(), (lse, lse_r)
    assert ((rows.double().cpu() - loss_r).abs() <= 2e-6 * lse_r.abs().clamp_min(1.0)).all(), (rows, loss_r)
    P.assert_close(dl[:, :V].double().cpu(), dl_r, 1e-5, "dlogits")


def test_ce_all_rows_ignored():
    """No valid row: nvalid clamps to 1, the loss is 0 and every gradient is exactly 0."""
    from pcd_ops import vocab_cross_entropy
    g = torch.Generator().manual_seed(3)
    x = torch.randn(4, 5, 32, generator=g).to(DEV).requires_grad_(True)
    w = torch.randn(41, 32, generator=g).to(DEV).requires_grad_(True)
    b = torch.randn(41, generator=g).to(DEV).requires_grad_(True)
    tg = torch.tensor([-100, 41, 1000, -1, 41] * 4).reshape(4, 5).to(DEV)
    loss = vocab_cross_entropy(x, w, b, tg)
    loss.backward()
    assert loss.item() == 0.0
    for t in (x, w, b):
        assert (t.grad == 0).all()


def test_vocab_cross_entropy_targets_out_of_range():
    """Rows with a target >= V are ignored and left out of the mean's denominator, like negative targets; the float64
    reference masks those rows itself on the CPU (an out-of-range target is never handed to F.cross_entropy)."""
    from pcd_ops import vocab_cross_entropy
    B, T, K, V = 6, 9, 64, 1027
    g = torch.Generator().manual_seed(11)
    x = torch.randn(B, T, K, generator=g)
    w = torch.randn(V, K, generator=g) / K ** 0.5
    b = 0.1 * torch.randn(V, generator=g)
    tg = torch.randint(0, V, (B, T), generator=g)
    tg[:, -1] = -100
    tg[0, 2], tg[3, 4], tg[5, 0] = V, V + 7, 1 << 40
    xd, wd, bd = (t.to(DEV).requires_grad_(True) for t in (x, w, b))
    loss = vocab_cross_entropy(xd, wd, bd, tg.to(DEV))
    (2.0 * loss).backward()
    keep = ((tg >= 0) & (tg < V)).flatten()
    xr, wr, br = (t.double().requires_grad_(True) for t in (x, w, b))
    ref = F.cross_entropy(F.linear(xr, wr, br).flatten(end_dim=1)[keep], tg.flatten()[keep])
    (2.0 * ref).backward()
    P.assert_close(loss.double().cpu(), ref, 1e-5, "loss")
    for got, r, name in ((xd.grad, xr.grad, "dx"), (wd.grad, wr.grad, "dw"), (bd.grad, br.grad, "db")):
        P.assert_close(got.double().cpu(), r, 5e-5, name)


@pytest.mark.parametrize("R,C,ld_s,ld_d", [(1, 1, 1, 4), (33, 45, 47, 40), (70, 31, 31, 100), (129, 257, 260, 132)])
def test_transpose_pad(R, C, ld_s, ld_d):
    """dst[c][r] = src[r][c] bit-exact, dst[c][R:ld_d] exactly 0 over a NaN-filled destination; source pad never read."""
    lib = _lib()
    src = torch.full((R, ld_s), float("nan"))
    src[:, :C] = torch.randn(R, C, generator=torch.Generator().manual_seed(R + C))
    src = src.to(DEV)
    dst = torch.full((C + 1, ld_d), float("nan"), device=DEV)
    assert lib.pcd_transpose_pad(src.data_ptr(), ld_s, R, C, dst.data_ptr(), ld_d, torch.cuda.current_stream().cuda_stream) == 0
    torch.cuda.synchronize()
    assert torch.equal(dst[:C, :R], src[:, :C].T)
    assert (dst[:C, R:] == 0).all()
    assert torch.isnan(dst[C]).all()


# ---------------------------------------------------------------------------------------------------------------------
# D. production MixedOp / cell kernels on non-square inputs
# ---------------------------------------------------------------------------------------------------------------------
def _assert_production(names):
    """The v4 forward and the v4 stage-A backward ran; no generic edge kernel did."""
    assert any(k.startswith("fwdB4_") for k in names), names
    assert any(k.startswith("bwdA4_") for k in names), names
    assert not any(k.startswith("fwdB_") or k.startswith("bwdA_") for k in names), names


@pytest.mark.parametrize("C,stride,H,W", [(16, 1, 32, 64), (16, 1, 16, 64), (32, 2, 128, 64), (32, 1, 64, 32), (32, 1, 16, 32),
                                          (64, 2, 64, 32), (64, 1, 32, 16), (64, 1, 48, 16), (32, 2, 32, 64)])
@pytest.mark.parametrize("jobs", ["1", "2"])
def test_mixed_op_production_non_square(C, stride, H, W, jobs, monkeypatch):
    monkeypatch.setenv("PCD_V4_JOBS", jobs)
    _, names = _profiled(lambda: P.mixed_vs_oracle(C, stride, 2, H, DEV, W=W))
    _assert_production(names)


@pytest.mark.parametrize("cpp,cp,C,red,rp,H,W", [(48, 48, 16, False, False, 128, 64), (48, 64, 32, True, False, 128, 64),
                                                 (64, 128, 64, True, True, 64, 32), (128, 256, 64, False, True, 32, 16),
                                                 (128, 256, 64, False, True, 48, 16)])
@pytest.mark.parametrize("act_only", [False, True])
def test_cell_production_non_square(cpp, cp, C, red, rp, H, W, act_only):
    _, names = _profiled(lambda: P.cell_vs_oracle(cpp, cp, C, red, rp, 2, H, DEV, act_only=act_only, W=W))
    _assert_production(names)


def test_network_non_square_vs_oracle():
    """The search network on 128 x 64 images at batch 4: every cell on the production kernels."""
    (worst, within), names = _profiled(lambda: P.network_vs_oracle(4, 128, DEV, W=64))
    _assert_production(names)
    print("worst weight-grad error over the four cells:", worst, "share within 1e-4:", within)


if __name__ == "__main__" and sys.argv[1:] == ["--gemm-one-tile-per-cta"]:
    assert os.environ.get("PCD_GEMM_PERSIST") == "0"
    names = _gemm_kernel_names()
    assert names and not any("persist" in s for s in names), names
    print("\n".join(gemm_sweep()))
    print("one-tile-per-cta sweep ok")
