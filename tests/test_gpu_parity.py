"""GPU parity: the sm_100a kernels, called through the C ABI, against the reference goldens and the
CPU oracle.  rel 1e-4 on outputs / weight grads / alpha-beta grads, bit-exact channel indexing."""
import pytest
import torch

import parity_cases as P

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.mark.parametrize("name,C,stride", P.MIXED)
def test_mixed_op_golden(name, C, stride):
    P.mixed_case(name, C, stride, DEV)


@pytest.mark.parametrize("name,cpp,cp,C,red,rp", P.CELLS)
def test_cell_golden(name, cpp, cp, C, red, rp):
    P.cell_case(name, cpp, cp, C, red, rp, DEV)


def test_network_golden():
    P.network_case(DEV)


def test_network_full_size_vs_oracle():
    """BASELINE.json configuration: C=16, 4 cells, 64x64 images, batch 64 — output, then every cell's backward replayed
    through the oracle on the tensors it actually received."""
    worst, within = P.network_vs_oracle(64, 64, DEV)
    print("worst weight-grad error over the four cells:", worst, "share within 1e-4:", within)
    print("fp64 yardstick:", P.network_vs_oracle.evidence)


def test_shuffle_bit_exact():
    P.shuffle_case(DEV)


# the five production edge shapes of SURVEY.md §8(a) at a batch the oracle finishes in seconds; then two non-square inputs
# at a production width whose output height is not a multiple of 16: they run the generic kernels
@pytest.mark.parametrize("C,stride,B,H", [(16, 1, 4, 64), (32, 2, 4, 64), (32, 1, 4, 32), (64, 2, 4, 32), (64, 1, 8, 16),
                                          pytest.param(32, 2, 4, (48, 64), id="32-2-4-48x64"),
                                          pytest.param(64, 2, 4, (16, 32), id="64-2-4-16x32")])
@pytest.mark.parametrize("jobs", ["auto", "1", "2"])
def test_mixed_op_production_shapes_vs_oracle(C, stride, B, H, jobs, monkeypatch):
    # jobs: the v4 forward kernels' two block layouts (all stage-A jobs in one block | split over two), forced either way
    if jobs != "auto":
        monkeypatch.setenv("PCD_V4_JOBS", jobs)
    H, W = H if isinstance(H, tuple) else (H, H)
    P.mixed_vs_oracle(C, stride, B, H, DEV, W=W)


@pytest.mark.parametrize("C,stride,B,H", [(16, 1, 4, 64), (32, 2, 4, 64), (32, 1, 4, 32), (64, 2, 4, 32), (64, 1, 8, 16)])
def test_mixed_op_exact_ties(C, stride, B, H):
    """Inputs on a 0.5 grid: 3x3 and 2x2 max-pool windows full of exact ties (ATen routes the gradient to the first maximum
    in scan order), ReLU inputs exactly 0 (zero sub-gradient)."""
    P.mixed_vs_oracle(C, stride, B, H, DEV, quantized=True)


# the eight production preprocess shapes (SURVEY.md §8a) at reduced batch, plus shapes that make one block loop over
# several input-channel chunks (many pixel tiles) and shapes that split the chunks over blockIdx.z (few tiles)
@pytest.mark.parametrize("c_in,c_out,fr,B,H", [
    (48, 16, False, 4, 64), (48, 32, False, 4, 64), (64, 32, False, 4, 64), (64, 64, True, 4, 64),
    (128, 64, False, 4, 32), (128, 64, True, 4, 32), (256, 64, False, 4, 16), (256, 64, False, 40, 64),
    (128, 64, True, 40, 64), (64, 32, True, 2, 8), (48, 16, False, 1, 9)])
def test_preprocess_vs_oracle(c_in, c_out, fr, B, H):
    P.pre_vs_oracle(c_in, c_out, fr, B, H, DEV)


@pytest.mark.parametrize("c_in,c_out,H", [(48, 16, 64), (48, 32, 64), (64, 32, 64), (128, 64, 32), (256, 64, 16)])
def test_preprocess_tensor_core_path_full_batch(c_in, c_out, H, monkeypatch):
    """The tcgen05 preprocess kernels at the production shapes and FULL batch (64) against a float64 evaluation on the GPU,
    next to the FP32-FMA kernels (PCD_NO_PRE_TC=1) on the same tensors: there are no ReLU / max-pool decisions inside this
    op's backward and its forward ReLU acts on the given input, so no tie flips to excuse — plain rel 2e-5 (3xTF32)."""
    import config
    import torch.nn.functional as F
    config.DEVICE = DEV
    from pcdarts.operations import ReLUConvBN
    torch.manual_seed(c_in + c_out + H)
    m = ReLUConvBN(c_in, c_out, 1, 1, 0, affine=False).to(DEV).train()
    x = torch.randn(64, c_in, H, H, device=DEV)
    G = torch.randn(64, c_out, H, H, device=DEV)

    def run():
        xx = x.clone().requires_grad_(True)
        m.zero_grad()
        y = m(xx)
        (y * G).sum().backward()
        return y.detach().clone(), xx.grad.clone(), m.op[1].weight.grad.clone()
    monkeypatch.setenv("PCD_PRE_TC_FWD", "1")          # the forward kernel is opt-in (see run_pre_forward in pcd_api.cu)
    xd = x.double().requires_grad_(True)
    wd = m.op[1].weight.detach().double().requires_grad_(True)
    yd = F.batch_norm(F.conv2d(F.relu(xd), wd), None, None, training=True, eps=1e-5)
    (yd * G.double()).sum().backward()
    ref = (yd.detach(), xd.grad, wd.grad)
    got = run()
    again = run()
    monkeypatch.setenv("PCD_NO_PRE_TC", "1")
    fma = run()
    rep = {}
    for name, r, a_, b_, c_ in zip(("y", "dx", "dW"), ref, got, again, fma):
        rep[name] = dict(tc_vs_fp64=P.rel_err(a_, r), fma_vs_fp64=P.rel_err(c_, r), tc_run_to_run=P.rel_err(b_, a_))
    print("preprocess tc vs fma vs fp64:", rep)
    for name, v in rep.items():
        assert v["tc_run_to_run"] <= 2e-6, (name, rep)          # only the order of the statistics / dW atomics may differ
        assert v["tc_vs_fp64"] <= 2e-5, (name, rep)


# the four production cells (C=16@64, reduce C=32 64->32, reduce C=64 32->16, C=64@16) at batch 2: production backward kernels
# with the cell-wide deferred weight-gradient launch; once more with frozen weights (activation-only backward, HVP passes)
@pytest.mark.parametrize("cpp,cp,C,red,rp,H", [(48, 48, 16, False, False, 64), (48, 64, 32, True, False, 64),
                                               (64, 128, 64, True, True, 32), (128, 256, 64, False, True, 16)])
@pytest.mark.parametrize("act_only", [False, True])
def test_cell_production_geometry_vs_oracle(cpp, cp, C, red, rp, H, act_only):
    P.cell_vs_oracle(cpp, cp, C, red, rp, 2, H, DEV, act_only=act_only)


def test_w_step_with_wgrad_overlap_matches_golden():
    """Weight-grad jobs on the library's low-priority stream (joined in the stem backward): same w-step as the golden."""
    import pcd_ops
    pcd_ops.set_wgrad_overlap(True)
    try:
        P.wstep_case(DEV)
        P.network_case(DEV)
    finally:
        pcd_ops.overlap_join(torch.zeros(1, device=DEV))
        pcd_ops.set_wgrad_overlap(False)


@pytest.mark.parametrize("cpp,cp,C,red,rp,H,B", [(48, 48, 16, False, False, 64, 5), (64, 128, 64, True, True, 32, 7),
                                                 (128, 256, 64, False, True, 16, 9), (48, 64, 32, True, False, 64, 1)])
def test_cell_production_geometry_ragged_batch(cpp, cp, C, red, rp, H, B):
    """Batches that do not divide the kernels' image groups (weight-grad jobs walk 4 images per block, source-grad / stem
    blocks take several): the last group is partial."""
    P.cell_vs_oracle(cpp, cp, C, red, rp, B, H, DEV, act_only=False)


@pytest.mark.parametrize("M,K,N", [(1920, 512, 17858), (64, 512, 1000), (120, 36, 70), (256, 1024, 512), (64, 12544, 512),
                                   (64, 1000, 1000), (6, 16, 12)])
def test_linear_3xtf32_vs_fp64(M, K, N, monkeypatch):
    """Linear3xTF32Function (nn.Linear drop-in) vs an fp64 reference: forward, dX (split-K), dW, db, ragged tiles.  The
    size threshold is lifted so that the products linear_3xtf32 would send to the FMA kernel (covered by
    test_small_linear_vs_fp64) run on the tcgen05 GEMM as well."""
    import torch.nn.functional as F
    import pcd_ops
    from pcd_ops import linear_3xtf32
    monkeypatch.setattr(pcd_ops, "_TC_MIN_FLOP", 0.0)
    g = torch.Generator().manual_seed(M + K + N)
    L = 4 if M % 4 == 0 else 2
    x = torch.randn(M // L, L, K, generator=g).to(DEV).requires_grad_(True)
    w = (torch.randn(N, K, generator=g) / K ** 0.5).to(DEV).requires_grad_(True)
    b = torch.randn(N, generator=g).to(DEV).requires_grad_(True)
    G = torch.randn(M // L, L, N, generator=g).to(DEV)
    y = linear_3xtf32(x, w, b)
    (y * G).sum().backward()
    xr, wr, br = (t.detach().double().requires_grad_(True) for t in (x, w, b))
    yr = F.linear(xr, wr, br)
    (yr * G.double()).sum().backward()
    for got, ref, name in ((y, yr, "y"), (x.grad, xr.grad, "dx"), (w.grad, wr.grad, "dw"), (b.grad, br.grad, "db")):
        P.assert_close(got.double(), ref, 5e-5, name)


@pytest.mark.parametrize("M,K,N", [(64, 512, 1000), (64, 1000, 1000), (64, 1024, 512), (5, 36, 70), (130, 10, 33)])
def test_small_linear_vs_fp64(M, K, N):
    """pcd_gemm_small_f32: the answer head / question fc2 products in exact fp32 (no library GEMM), strides instead of transposes."""
    import torch.nn.functional as F
    from pcd_ops import SmallLinearFunction
    g = torch.Generator().manual_seed(M + K + N)
    x = torch.randn(M, K, generator=g).to(DEV).requires_grad_(True)
    w = (torch.randn(N, K, generator=g) / K ** 0.5).to(DEV).requires_grad_(True)
    b = torch.randn(N, generator=g).to(DEV).requires_grad_(True)
    G = torch.randn(M, N, generator=g).to(DEV)
    y = SmallLinearFunction.apply(x, w, b)
    (y * G).sum().backward()
    xr, wr, br = (t.detach().double().requires_grad_(True) for t in (x, w, b))
    yr = F.linear(xr, wr, br)
    (yr * G.double()).sum().backward()
    for got, ref, name in ((y, yr, "y"), (x.grad, xr.grad, "dx"), (w.grad, wr.grad, "dw"), (b.grad, br.grad, "db")):
        P.assert_close(got.double(), ref, 2e-6, name)


# fused vocabulary projection + cross-entropy (ignored rows, padded pitch) vs an fp64 reference
@pytest.mark.parametrize("B,T,K,V", [(64, 30, 512, 17858), (6, 30, 16, 41), (4, 5, 32, 1000)])
def test_vocab_cross_entropy_vs_fp64(B, T, K, V):
    import torch.nn.functional as F
    from pcd_ops import vocab_cross_entropy
    g = torch.Generator().manual_seed(B + T + K + V)
    x = torch.randn(B, T, K, generator=g).to(DEV).requires_grad_(True)
    w = (torch.randn(V, K, generator=g) / K ** 0.5).to(DEV).requires_grad_(True)
    b = (0.1 * torch.randn(V, generator=g)).to(DEV).requires_grad_(True)
    q = torch.randint(0, V, (B, T), generator=g).to(DEV)
    tg = torch.cat((q[:, 1:], q.new_full((B, 1), -100)), 1)
    loss = vocab_cross_entropy(x, w, b, tg)
    (3.0 * loss).backward()
    xr, wr, br = (t.detach().double().requires_grad_(True) for t in (x, w, b))
    ref = F.cross_entropy(F.linear(xr, wr, br)[:, :-1].flatten(end_dim=1), q[:, 1:].flatten())
    (3.0 * ref).backward()
    P.assert_close(loss.double(), ref, 1e-5, "loss")
    for got, r, name in ((x.grad, xr.grad, "dx"), (w.grad, wr.grad, "dw"), (b.grad, br.grad, "db")):
        P.assert_close(got.double(), r, 5e-5, name)


# persistent-kernel LSTM (tcgen05 projections + cooperative recurrence kernels) vs nn.LSTM in fp64
@pytest.mark.parametrize("T,B,E,H", [(30, 64, 300, 512), (5, 3, 8, 16), (7, 64, 12, 64), (30, 256, 300, 512), (6, 130, 12, 64),
                                     (5, 20, 12, 128), (4, 33, 8, 256), (3, 17, 8, 32)])
def test_lstm_vs_fp64(T, B, E, H):
    from pcd_ops import lstm_forward
    g = torch.Generator().manual_seed(T + B + E + H)
    lstm = torch.nn.LSTM(E, H, 1).to(DEV)
    x = torch.randn(T, B, E, generator=g).to(DEV).requires_grad_(True)
    h0 = (0.5 * torch.randn(1, B, H, generator=g)).to(DEV).requires_grad_(True)
    G1, G2, G3 = (torch.randn(*s, generator=g).to(DEV) for s in ((T, B, H), (1, B, H), (1, B, H)))
    out, (h, c) = lstm_forward(lstm, x, h0, h0)
    ((out * G1).sum() + (h * G2).sum() + (c * G3).sum()).backward()
    got = [out, h, c, x.grad, h0.grad] + [p.grad for p in lstm.parameters()]
    ref_lstm = torch.nn.LSTM(E, H, 1).to(DEV).double()
    ref_lstm.load_state_dict({k: v.double() for k, v in lstm.state_dict().items()})
    xr, hr = x.detach().double().requires_grad_(True), h0.detach().double().requires_grad_(True)
    outr, (h_r, c_r) = ref_lstm(xr, (hr, hr))
    ((outr * G1.double()).sum() + (h_r * G2.double()).sum() + (c_r * G3.double()).sum()).backward()
    ref = [outr, h_r, c_r, xr.grad, hr.grad] + [p.grad for p in ref_lstm.parameters()]
    for a_, b_, name in zip(got, ref, ("out", "hT", "cT", "dx", "dh0", "dW_ih", "dW_hh", "db_ih", "db_hh")):
        P.assert_close(a_.double(), b_, 5e-5, name)


def test_architect_lct_golden():
    """3-stage LCT alpha-step (architect_lct.py:32-92): EF passes on the sm_100a kernels, W = VGG19 in stock torch."""
    P.architect_lct_case(DEV)


def test_vqa_model_golden():
    P.vqa_case(DEV)


@pytest.mark.parametrize("unrolled", [False, True])
def test_architect_step_golden(unrolled):
    P.architect_case(DEV, unrolled)


def test_architect_step_golden_concurrent_hvp():
    """Hessian-vector product with its two passes on two streams (model | twin): same golden step."""
    P.architect_case(DEV, True, concurrent_hvp=True)


def test_w_step_golden():
    P.wstep_case(DEV)


def _graph_pair(unrolled):
    from argparse import Namespace
    from pcdarts.architect_vqa import Architect
    from search import GraphedSearchStep, SearchStep

    def make():
        m = P.make_vqa(DEV)
        arch = Architect(m, Namespace(arch_learn_rate=0.0, arch_wt_decay=0.0, qst_only=False))
        arch.optimizer = torch.optim.Adam(m.arch_parameters(), lr=0.0, betas=(0.5, 0.999), capturable=True)
        arch.unrolled_model().dropout.p = 0.0
        arch.device_scalars = True
        return m, SearchStep(m, arch, torch.optim.Adam(m.parameters(), lr=0.0, capturable=True))
    batches = [(P.vqa_batch(31, DEV), P.vqa_batch(32, DEV)), (P.vqa_batch(41, DEV), P.vqa_batch(42, DEV))]
    m1, eager = make()
    m2, st = make()
    graphed = GraphedSearchStep(st, *batches[0], 1e-3, unrolled=unrolled, warmup=2)      # the warm-up steps are undone
    return m1, eager, m2, graphed, batches


def test_graphed_search_step_matches_eager():
    """CUDA-graph replay of the whole search step == the eager step (first-order alpha-step + w-step).
    Learning rates are 0, so both models hold bit-identical weights and must agree on the loss, the
    alpha/beta grads and every weight grad; the second batch exercises the copy into the static inputs."""
    from helpers import assert_close
    m1, eager, m2, graphed, batches = _graph_pair(unrolled=False)
    for train, valid in batches:
        loss_e = eager.step(train, valid, 1e-3, unrolled=False)
        loss_g = graphed(train, valid)
        torch.cuda.synchronize()
        assert_close(loss_g, loss_e, 1e-6, "loss")
        for x, y in zip(m2.arch_parameters(), m1.arch_parameters()):
            assert_close(x.grad, y.grad, 1e-5, "arch grad")
        for (k, x), y in zip(m2.named_parameters(), m1.parameters()):
            assert_close(x.grad, y.grad, 1e-4, k)
    k = "img_encoder.darts.stem.1.num_batches_tracked"       # BN side effects advance identically
    assert int(m2.state_dict()[k]) == int(m1.state_dict()[k])


def test_graphed_unrolled_step_runs():
    """The unrolled (HVP) step also captures and replays.  Its w +- R v updates leave one-ulp residue in the
    weights that depends on fp32 atomic ordering, and with 2-sample tensors a single ReLU input within 1e-6 of
    zero then moves a gradient by ~1e-3 (see DESIGN.md §2), so only the loss and the alpha/beta grads are
    compared, loosely."""
    from helpers import assert_close
    m1, eager, m2, graphed, batches = _graph_pair(unrolled=True)
    for train, valid in batches:
        loss_e = eager.step(train, valid, 1e-3, unrolled=True)
        loss_g = graphed(train, valid)
        torch.cuda.synchronize()
        assert_close(loss_g, loss_e, 1e-4, "loss")
        for x, y in zip(m2.arch_parameters(), m1.arch_parameters()):
            assert_close(x.grad, y.grad, 2e-2, "arch grad")      # a smoke test at 2 samples; parity lives in the full-size test


def test_graphed_lct_step_matches_eager():
    """ArchitectLct.step replayed from a CUDA graph (search.GraphedLctStep) == the eager step.  The architecture learning
    rate is 0 so both copies stay at the same alphas; the finite-difference stages are compared at their own noise level."""
    import config
    from helpers import assert_close
    from search import GraphedLctStep
    lr0, wd0 = config.ARCH_LEARNING_RATE, config.ARCH_WEIGHT_DECAY
    config.ARCH_LEARNING_RATE, config.ARCH_WEIGHT_DECAY = 0.0, 0.0
    try:
        ef1, w1, eager = P.make_lct(DEV)
        ef2, w2, arch2 = P.make_lct(DEV)
    finally:
        config.ARCH_LEARNING_RATE, config.ARCH_WEIGHT_DECAY = lr0, wd0
    tr, va = P.lct_batch(21, DEV), P.lct_batch(22, DEV)
    import pcd_ops
    pcd_ops.set_wgrad_overlap(True)          # deferred weight-grad jobs on the side stream must be joined inside the capture
    try:
        graphed = GraphedLctStep(arch2, tr, va, 1e-3, 1e-3, warmup=2)
    finally:
        pcd_ops.set_wgrad_overlap(False)
    for _ in range(2):
        eager.step(*tr, *va, 1e-3, 1e-3)
    for train, valid in ((tr, va), (P.lct_batch(23, DEV), P.lct_batch(24, DEV))):
        eager.step(*train, *valid, 1e-3, 1e-3)
        graphed(train, valid)
        torch.cuda.synchronize()
        Le, Lg = eager.last, arch2.last
        assert_close(Lg["unrolled_loss"], Le["unrolled_loss"], 1e-5, "W' validation loss")
        assert_close(Lg["grad_wprime_norm"], Le["grad_wprime_norm"], 1e-4, "|grad W'|")
        for key in ("kappa_p", "kappa_n"):
            ne = torch.cat([t.reshape(-1) for t in Le[key]]).norm()
            ng = torch.cat([t.reshape(-1) for t in Lg[key]]).norm()
            assert_close(ng, ne, 1e-4, key)
        for i in range(4):
            assert_close(Lg["gamma_p"][i], Le["gamma_p"][i], 1e-3, f"gamma_p{i}")
            assert_close(Lg["gamma_n"][i], Le["gamma_n"][i], 1e-3, f"gamma_n{i}")


@pytest.mark.parametrize("B,H,E,V,T", [(64, 512, 300, 17858, 30), (5, 32, 12, 300, 7), (37, 128, 64, 1000, 12), (64, 256, 300, 129, 5),
                                       (130, 512, 300, 17858, 6)])
def test_greedy_decode(B, H, E, V, T):
    """Persistent greedy-decode kernel vs the reference loop in fp64 (production size first; ragged vocabulary tiles, partial
    batches, fewer gate blocks than vocabulary tiles and the reverse)."""
    P.decode_case(DEV, B, H, E, V, T)


def test_generate_uses_decode_kernel():
    """QstEncoder.generate (both packages) == its own stock-torch loop, and it goes through the native decode."""
    import pcd_native
    from vqa_model import QstEncoder
    torch.manual_seed(5)
    q = QstEncoder(700, 20, 64, 1, 64).to(DEV)
    img = torch.randn(6, 64, device=DEV) * 0.5
    lib = pcd_native.load_cuda()
    n0 = lib.pcd_launch_count()
    fast = q.generate(img)
    assert lib.pcd_launch_count() == n0 + 1
    q.deterministic = None            # falsy but argmax in sample(): forces the torch loop
    q.sample = lambda prob: torch.argmax(prob, 2)
    slow = q.generate(img)
    assert (fast == slow).float().mean().item() >= 0.98


def test_native_library_is_the_one_running():
    import pcd_native
    lib = pcd_native.load_cuda()
    assert lib.pcd_is_cuda_build() == 1
    maps = open("/proc/self/maps").read()
    assert "libpcdarts_sm100.so" in maps


def test_generate_golden():
    """The persistent decode kernel reproduces the words the unmodified reference generated (tests/golden/generate.npz);
    steps whose reference top-2 margin is within 1e-4 of a tie (and what follows them in that row) are not compared."""
    P.generate_golden_case(DEV, tie=1e-4)


# ---- the benchmarked configuration itself (B = 64, 64x64, V = 17858, hidden 512): one whole search step vs the oracle ----
@pytest.mark.parametrize("graphed", [False, True])
@pytest.mark.parametrize("unrolled", [True, False])
def test_search_step_full_size_vs_oracle(unrolled, graphed):
    """alpha-step (unrolled with the finite-difference HVP, or first-order) + w-step exactly as bench.py runs them — eagerly
    and replayed from the CUDA graph — against oracle.architect_step + oracle.w_step on the same tensors: L_val(w'), |v|,
    g+, g- (rel 1e-4), the raw HVP (cancellation-aware bound), d alpha / d beta (1e-4), alphas after Adam (1e-5), the w-step
    loss (1e-5), every clipped weight gradient (1e-4; search-network tensors with the tie-flip criterion), BN side effects."""
    rep = P.search_step_vs_oracle(DEV, unrolled, graphed)
    print("full-size search step:", rep)


# stand-alone candidate operations on all channels (SURVEY.md §8f-4): native op kernels vs the same layers in float64
@pytest.mark.parametrize("name,C,stride,affine,B,H", P.OPS_CASES + [
    ("sep_conv_3x3", 16, 1, True, 8, 64), ("sep_conv_5x5", 32, 2, True, 8, 64), ("dil_conv_5x5", 64, 1, True, 16, 16),
    ("dil_conv_3x3", 64, 2, True, 8, 32), ("max_pool_3x3", 32, 2, True, 8, 64), ("avg_pool_3x3", 64, 1, True, 16, 16),
    ("skip_connect", 64, 2, True, 8, 32), ("sep_conv_7x7", 16, 1, True, 4, 32)])
def test_op_vs_stock(name, C, stride, affine, B, H):
    P.op_vs_stock(name, C, stride, affine, B, H, DEV)


@pytest.mark.parametrize("name,stride", [("max_pool_3x3", 1), ("max_pool_3x3", 2), ("sep_conv_3x3", 1)])
def test_op_exact_ties(name, stride):
    P.op_vs_stock(name, 8, stride, True, 2, 12, DEV, quantized=True)


@pytest.mark.parametrize("B,img", [(2, 32), (8, 64)])
def test_derived_network_vs_stock(B, img):
    """The network a genotype describes (pcdarts/model.py): stem, 4 derived cells, pooling; forward + every weight gradient."""
    ok, worst = P.derived_vs_stock(DEV, B=B, img=img)
    print(f"derived network B={B} img={img}: share within 1e-4 = {ok:.3f}, worst {worst}")


@pytest.mark.parametrize("B,H,W", [(64, 64, 64), (5, 32, 32), (2, 10, 20), (1, 9, 9)])
def test_stem_vs_torch(B, H, W):
    P.stem_vs_torch(DEV, B, H, W)
