"""CPU checks of the CUDA kernel SOURCES: the same .cuh bodies compiled with -DPCD_EMU (phases run as
host loops) against the reference goldens.  This validates index arithmetic / math of the kernels
where no GPU exists; it is test infrastructure, not a product path (see pcd_native.enable_emulation).
"""
import pytest
import torch

import parity_cases as P


@pytest.fixture(scope="module", autouse=True)
def emulation():
    import pcd_build
    import pcd_native
    pcd_native.enable_emulation(pcd_build.build_emu())
    yield
    pcd_native._emu_lib = None


@pytest.mark.parametrize("name,C,stride", P.MIXED)
def test_mixed_op_emulated(name, C, stride):
    P.mixed_case(name, C, stride, "cpu")


@pytest.mark.parametrize("name,cpp,cp,C,red,rp", P.CELLS)
def test_cell_emulated(name, cpp, cp, C, red, rp):
    P.cell_case(name, cpp, cp, C, red, rp, "cpu")


# the five production edge geometries (v4 forward, production backward kernels), one image each; then two non-square
# inputs at a production width whose output height is not a multiple of 16: they run the generic kernels
@pytest.mark.parametrize("C,stride,B,H", [(16, 1, 1, 64), (32, 2, 1, 64), (32, 1, 2, 32), (64, 2, 1, 32), (64, 1, 2, 16),
                                          pytest.param(32, 2, 1, (48, 64), id="32-2-1-48x64"),
                                          pytest.param(64, 2, 1, (16, 32), id="64-2-1-16x32")])
@pytest.mark.parametrize("jobs", ["1", "2"])
def test_mixed_op_fixed_tiles_emulated(C, stride, B, H, jobs, monkeypatch):
    # v4 forward kernels: one block runs every stage-A job (large waves) | jobs split over two blocks (small waves)
    monkeypatch.setenv("PCD_V4_JOBS", jobs)
    H, W = H if isinstance(H, tuple) else (H, H)
    P.mixed_vs_oracle(C, stride, B, H, "cpu", W=W)


@pytest.mark.parametrize("C,stride,B,H", [(16, 1, 1, 64), (32, 2, 1, 64), (64, 2, 1, 32), (64, 1, 2, 16)])
def test_mixed_op_exact_ties_emulated(C, stride, B, H):
    """Max-pool windows full of exact ties, ReLU inputs exactly 0: first-maximum routing / zero sub-gradient as in ATen."""
    P.mixed_vs_oracle(C, stride, B, H, "cpu", quantized=True)


# preprocess 1x1 GEMM kernels: ragged pixel tiles, FactorizedReduce (fast and generic loads), partial channel chunks
@pytest.mark.parametrize("c_in,c_out,fr,B,H", [(48, 16, False, 2, 16), (48, 32, False, 1, 20), (64, 64, True, 2, 16),
                                                 (128, 64, False, 1, 18), (64, 32, True, 1, 12), (40, 16, False, 1, 9),
                                                 (256, 64, False, 1, 16)])
def test_preprocess_emulated(c_in, c_out, fr, B, H):
    P.pre_vs_oracle(c_in, c_out, fr, B, H, "cpu")


# a production-geometry cell (production backward kernels + deferred weight-grad launch), one image
@pytest.mark.parametrize("cpp,cp,C,red,rp,H", [(128, 256, 64, False, True, 16), (64, 128, 64, True, True, 32)])
def test_cell_production_geometry_emulated(cpp, cp, C, red, rp, H):
    P.cell_vs_oracle(cpp, cp, C, red, rp, 1, H, "cpu")


def test_network_emulated():
    P.network_case("cpu")


def test_shuffle_emulated():
    P.shuffle_case("cpu")


def test_vqa_model_emulated():
    P.vqa_case("cpu")


@pytest.mark.parametrize("unrolled", [False, True])
def test_architect_emulated(unrolled):
    P.architect_case("cpu", unrolled)


def test_architect_concurrent_hvp_emulated():
    """The two finite-difference passes on two module copies (model at w + R v, twin at w - R v) instead of one after the other on
    the model: same g+, g-, alpha/beta gradients and BatchNorm side effects as the reference's golden step."""
    P.architect_case("cpu", True, concurrent_hvp=True)


def test_w_step_emulated():
    P.wstep_case("cpu")


def test_architect_lct_emulated():
    P.architect_lct_case("cpu")


def test_product_refuses_cpu_without_emulation():
    import pcd_native
    keep, pcd_native._emu_lib = pcd_native._emu_lib, None
    try:
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            pcd_native.lib_for(torch.zeros(1))
    finally:
        pcd_native._emu_lib = keep


@pytest.mark.parametrize("B,H,E,V,T", [(5, 32, 12, 300, 7), (3, 64, 8, 128, 4)])
def test_greedy_decode(B, H, E, V, T):
    """Host side of the greedy decode (argument marshalling, token layout, <start>/tanh convention) on the emulation build."""
    P.decode_case("cpu", B, H, E, V, T)


def test_generate_golden():
    """QstEncoder.generate through the decode entry point == the words of the unmodified reference's generate()."""
    assert P.generate_golden_case("cpu") == 5 * 30 + 9 * 12


def test_generate_outside_the_kernel_envelope_is_loud():
    """Hidden sizes the decode kernel does not take (not a multiple of 32) RAISE unless stock ops were opted in; sampled
    (non-deterministic) decoding is the reference's own module loop by design.  Both give (B, max_length) int64 words."""
    import pcd_ops
    from pcd_ops import decode_supported
    from vqa_model import QstEncoder
    torch.manual_seed(3)
    q = QstEncoder(90, 8, 48, 1, 48, max_length=6)           # H = 48
    img = 0.3 * torch.randn(4, 48)
    assert not decode_supported(img, q.lstm, q.word2vec, q.fc1)
    with pytest.raises(RuntimeError, match="PCD_ERR_UNSUPPORTED"):
        q.generate(img)
    pcd_ops.allow_stock_ops(True)
    words = q.generate(img)
    assert words.shape == (4, 6) and words.dtype == torch.long and int(words.max()) < 90
    pcd_ops.allow_stock_ops(False)
    q2 = QstEncoder(90, 8, 32, 1, 32, deterministic=False, max_length=5)
    img2 = 0.3 * torch.randn(3, 32)
    assert decode_supported(img2, q2.lstm, q2.word2vec, q2.fc1)      # the shape is fine, the sampling mode is not
    words2 = q2.generate(img2)
    assert words2.shape == (3, 5) and int(words2.min()) >= 0 and int(words2.max()) < 90


def test_lstm_outside_the_envelope_raises_and_any_linear_is_native():
    import pcd_ops
    y = pcd_ops.linear_3xtf32(torch.ones(3, 10), torch.ones(5, 10), None)        # depth 10: the FMA kernel takes it
    assert torch.allclose(y, torch.full((3, 5), 10.0))
    lstm = torch.nn.LSTM(10, 16, 1)
    with pytest.raises(RuntimeError, match="PCD_ERR_UNSUPPORTED"):
        pcd_ops.lstm_forward(lstm, torch.randn(4, 2, 10), torch.zeros(1, 2, 16), torch.zeros(1, 2, 16))


def test_lstm_and_decode_tile_batches_above_64():
    """B = 70 runs as two launches over contiguous slices and equals the one-launch result on each slice."""
    import pcd_ops
    torch.manual_seed(1)
    lstm = torch.nn.LSTM(8, 32, 1)
    x = torch.randn(5, 70, 8, requires_grad=True)
    h0 = 0.3 * torch.randn(1, 70, 32)
    out, (h, c) = pcd_ops.lstm_forward(lstm, x, h0, h0)
    ref, (hr, cr) = lstm(x, (h0, h0))
    assert torch.allclose(out, ref, atol=2e-5) and torch.allclose(h, hr, atol=2e-5) and torch.allclose(c, cr, atol=2e-5)
    out.sum().backward()
    gx = x.grad.clone()
    x.grad = None
    ref.sum().backward()
    assert torch.allclose(gx, x.grad, atol=2e-5)
    emb = torch.nn.Embedding(50, 8)
    proj = torch.nn.Linear(32, 50)
    tok = pcd_ops.decode_greedy(h0[0], lstm, emb, proj, 4)
    assert tok.shape == (70, 4)
    assert torch.equal(tok[:64], pcd_ops.decode_greedy(h0[0, :64], lstm, emb, proj, 4))
    assert torch.equal(tok[64:], pcd_ops.decode_greedy(h0[0, 64:], lstm, emb, proj, 4))


def test_lstm_bias_grads_do_not_share_a_buffer():
    """b_ih and b_hh get equal gradients in SEPARATE tensors.  One shared buffer is touched twice by every in-place consumer:
    under data parallelism the flat clip kernel then scaled it from two thread blocks at once and 4 replicas drifted apart
    (profiles/r02_bench_dp4_drift.json; profiles/tools/dp_drift.py pinned it to these two parameters)."""
    import pcd_ops
    torch.manual_seed(2)
    lstm = torch.nn.LSTM(8, 32, 1)
    x = torch.randn(4, 3, 8)
    h0 = 0.3 * torch.randn(1, 3, 32)
    out, _ = pcd_ops.lstm_forward(lstm, x, h0, h0)
    g_ih, g_hh = torch.autograd.grad(out.sum(), [lstm.bias_ih_l0, lstm.bias_hh_l0])
    assert torch.equal(g_ih, g_hh) and g_ih.data_ptr() != g_hh.data_ptr()


def test_activation_only_passes_skip_parameter_products():
    """Inside pcd_ops.weight_grads(False) (the architect's alpha-only passes, architect_vqa.py:110,115) the dense Functions
    return the data gradients unchanged and no weight / bias gradient at all."""
    import pcd_ops
    torch.manual_seed(3)
    lin = torch.nn.Linear(8, 12)
    lstm = torch.nn.LSTM(8, 32, 1)
    x = torch.randn(5, 3, 8, requires_grad=True)
    h0 = (0.3 * torch.randn(1, 3, 32)).requires_grad_(True)
    tgt = torch.randint(0, 12, (15,))

    def run():
        out, _ = pcd_ops.lstm_forward(lstm, x, h0, h0)
        proj = torch.nn.Linear(32, 8)
        proj.load_state_dict({"weight": torch.ones(8, 32) / 32, "bias": torch.zeros(8)})
        y = pcd_ops.linear_3xtf32(pcd_ops.linear_3xtf32(out, proj.weight, proj.bias), lin.weight, lin.bias)
        loss = pcd_ops.vocab_cross_entropy(y.reshape(15, 12), torch.eye(12), None, tgt) + y.square().mean()
        params = [lin.weight, lin.bias] + list(lstm.parameters())
        return torch.autograd.grad(loss, [x, h0] + params, allow_unused=True)
    full = run()
    with pcd_ops.weight_grads(False):
        act = run()
    assert torch.equal(full[0], act[0]) and torch.equal(full[1], act[1])
    assert all(g is not None for g in full[2:]) and all(g is None for g in act[2:])


@pytest.mark.parametrize("B,H,W", [(2, 64, 64), (3, 16, 32), (2, 10, 20), (1, 9, 9), (2, 8, 128)])
def test_stem_vs_torch_emulated(B, H, W):
    P.stem_vs_torch("cpu", B, H, W)


def test_make_capturable_moves_adam_step_counters():
    """search.make_capturable flips an optimizer that has already stepped (host-side `step` counters) to the capturable form."""
    from search import make_capturable
    p = torch.nn.Parameter(torch.ones(3))
    opt = torch.optim.Adam([p], lr=1e-3)
    p.grad = torch.ones(3)
    opt.step()
    make_capturable(opt)
    assert opt.param_groups[0]["capturable"] is True
    assert torch.is_tensor(opt.state[p]["step"]) and opt.state[p]["step"].device == p.device


@pytest.mark.parametrize("unrolled", [True, False])
def test_search_step_vs_oracle_emulated(unrolled):
    """The logic of the full-size GPU test (tests/test_gpu_parity.py::test_search_step_full_size_vs_oracle) at a size the
    emulation finishes in seconds: one alpha-step + w-step of SearchStep against oracle.architect_step + oracle.w_step."""
    P.search_step_vs_oracle("cpu", unrolled, graphed=False, B=2, V=40, img=32, dims=dict(P.VQA_DIMS, qst_vocab_size=None))


def test_skip_stage2_architect_runs_an_unrolled_step():
    """config.SKIP_STAGE2: get_architect hands the darts_vqa-flavour Architect an EF model whose _loss takes the
    reference's three arguments (basic_vqa/pcdarts/architect.py:25,62,98); its unrolled step must run (ADVICE r01)."""
    import config
    from architect_factory import get_architect
    ef, w, _ = P.make_lct("cpu")
    keep = config.SKIP_STAGE2
    config.SKIP_STAGE2 = True
    try:
        arch = get_architect(ef, w, None, None)
    finally:
        config.SKIP_STAGE2 = keep
    assert type(arch).__name__ == "Architect"
    before = [a.detach().clone() for a in ef.arch_parameters()]
    arch.unrolled_model()
    for mod in arch.unrolled_model().modules():
        if isinstance(mod, torch.nn.Dropout):
            mod.p = 0.0
    arch.step(*P.lct_batch(21, "cpu"), *P.lct_batch(22, "cpu"), 1e-3, None, unrolled=True)
    assert all(a.grad is not None and torch.isfinite(a.grad).all() for a in ef.arch_parameters())
    assert any(not torch.equal(a.detach(), b) for a, b in zip(ef.arch_parameters(), before))
    twin = ef.img_encoder.darts.new()           # Network.new() keeps the owning-model back reference (basic_vqa model_search.py:139-141)
    assert twin._vqa_model() is ef.img_encoder.darts._vqa_model()


def test_graph_warmup_state_is_restored():
    """search._TrainingState: what GraphedSearchStep uses to undo its warm-up steps (weights, buffers, alphas, Adam state)."""
    from search import _TrainingState
    lin = torch.nn.Linear(3, 2)
    bn = torch.nn.BatchNorm1d(2)
    mod = torch.nn.Sequential(lin, bn)
    alpha = torch.zeros(4, requires_grad=True)
    opt = torch.optim.Adam(list(mod.parameters()) + [alpha], lr=0.1)
    snap = _TrainingState([mod], [alpha], [opt])
    ref = [t.clone() for t in snap.tensors]
    for _ in range(2):
        opt.zero_grad()
        (mod(torch.randn(5, 3)).sum() + alpha.sum()).backward()
        opt.step()
    assert int(bn.num_batches_tracked) == 2
    snap.restore()
    assert all(torch.equal(a, b) for a, b in zip(snap.tensors, ref))
    assert int(bn.num_batches_tracked) == 0
    for st in opt.state.values():
        assert float(st["step"]) == 0 and float(st["exp_avg"].abs().max()) == 0 and float(st["exp_avg_sq"].abs().max()) == 0


def test_graph_warmup_restore_survives_arena_rebinding():
    """The first forward re-binds every parameter's .data to a view of the flat arena (pcd_ops.Arena); a snapshot taken
    before it must still restore into the live storage (found on the GPU: the graph used to start two steps late)."""
    from search import _TrainingState
    m = P.make_vqa("cpu")
    opt = torch.optim.Adam(m.parameters(), lr=1e-2)
    snap = _TrainingState([m], m.arch_parameters(), [opt])
    before = [p.detach().clone() for p in m.parameters()]
    ptr_before = next(iter(m.img_encoder.darts.cells.parameters())).data_ptr()
    img, qst, lbl = P.vqa_batch(11, "cpu")
    m._loss(img, qst, lbl).backward()
    opt.step()
    assert next(iter(m.img_encoder.darts.cells.parameters())).data_ptr() != ptr_before      # storage was re-bound
    assert any(not torch.equal(a, b) for a, b in zip(m.parameters(), before))
    snap.restore()
    assert all(torch.equal(a.detach(), b) for a, b in zip(m.parameters(), before))


def test_flat_optimizer_ops_match_torch():
    """pcd_flat: runs found across the parameter arena, axpy / norm / clip / Adam == the torch reference (foreach / per-tensor)."""
    import pcd_flat
    torch.manual_seed(0)
    arena = torch.randn(1000)
    ps = [arena[0:10].view(2, 5), arena[10:250].view(240), arena[250:1000].view(30, 25), torch.randn(7, 3), torch.randn(5)]
    garena = torch.randn(240 + 750)
    gs = [torch.randn(2, 5), garena[0:240], garena[240:990].view(30, 25), torch.randn(7, 3), torch.randn(5)]
    sizes, ptrs = pcd_flat.co_runs(ps, gs)
    assert sizes == [10, 990, 21, 5]                      # p contiguous over 0..2, g only over 1..2
    ref = [p.clone() for p in ps]
    pcd_flat.axpy_(ps, gs, alpha=-0.25)
    for a, b, g in zip(ps, ref, gs):
        assert torch.allclose(a, b - 0.25 * g, rtol=0, atol=1e-6)
    R = torch.tensor([0.5])
    pcd_flat.axpy_(ps, gs, alpha=2.0, alpha_dev=R)
    for a, b, g in zip(ps, ref, gs):
        assert torch.allclose(a, b + 0.75 * g, rtol=0, atol=1e-6)
    total = torch.sqrt(sum((g.double() ** 2).sum() for g in gs))
    assert abs(float(pcd_flat.norm(gs)) - float(total)) <= 1e-6 * float(total)
    # clip + Adam against torch over three steps
    params = [torch.nn.Parameter(p.clone()) for p in ps]
    mine = [torch.nn.Parameter(p.clone()) for p in ps]
    opt_t = torch.optim.Adam(params, lr=1e-2, weight_decay=1e-3)
    opt_m = pcd_flat.FlatAdam(mine, lr=1e-2, weight_decay=1e-3)
    for step in range(3):
        for p, q, g in zip(params, mine, gs):
            p.grad = (g * (step + 1)).clone()
            q.grad = (g * (step + 1)).clone()
        n_t = torch.nn.utils.clip_grad_norm_(params, 5.0)
        n_m = pcd_flat.clip_grad_norm_(mine, 5.0)
        assert abs(float(n_t) - float(n_m)) <= 1e-5 * float(n_t)
        for p, q in zip(params, mine):
            assert torch.allclose(p.grad, q.grad, rtol=1e-5, atol=1e-7)
        opt_t.step()
        opt_m.step()
        for p, q in zip(params, mine):
            assert torch.allclose(p, q, rtol=1e-5, atol=1e-6), (step, (p - q).abs().max())


@pytest.mark.parametrize("M,K,N", [(64, 512, 1000), (5, 36, 70), (64, 1024, 512), (3, 16, 12)])
def test_small_linear_matches_torch(M, K, N):
    """pcd_gemm_small_f32 (exact-fp32 FMA GEMM of the answer head / question fc2): y, dx, dW, db against F.linear in fp64."""
    import torch.nn.functional as F
    from pcd_ops import SmallLinearFunction
    g = torch.Generator().manual_seed(M + K + N)
    x = torch.randn(M, K, generator=g, requires_grad=True)
    w = (torch.randn(N, K, generator=g) / K ** 0.5).requires_grad_(True)
    b = torch.randn(N, generator=g, requires_grad=True)
    G = torch.randn(M, N, generator=g)
    y = SmallLinearFunction.apply(x, w, b)
    (y * G).sum().backward()
    xr, wr, br = (t.detach().double().requires_grad_(True) for t in (x, w, b))
    yr = F.linear(xr, wr, br)
    (yr * G.double()).sum().backward()
    for got, ref, name in ((y, yr, "y"), (x.grad, xr.grad, "dx"), (w.grad, wr.grad, "dw"), (b.grad, br.grad, "db")):
        P.assert_close(got.double(), ref, 2e-6, name)


def test_arena_verify_detects_a_rebound_parameter():
    """Arena.verify (run once per w-step): a parameter whose .data was re-bound in the MIDDLE of the arena is reported (the
    cheap per-forward check only looks at the ends of each group)."""
    from pcdarts.model_search import Cell
    m = Cell(4, 4, 48, 48, 16, False, False).train()
    P._fill(m, 3)
    s0, s1 = torch.randn(1, 48, 8, 8), torch.randn(1, 48, 8, 8)
    w, w2 = torch.softmax(torch.randn(14, 8), -1), torch.softmax(torch.randn(14), 0)
    m(s0, s1, w, w2)
    ar = m._arena()
    ar.verify()
    mid = ar.params[len(ar.params) // 2]
    mid.data = mid.data.clone()
    ar.ensure()                              # ends unchanged: not noticed here
    with pytest.raises(RuntimeError, match="left its flat arena"):
        ar.verify()


def test_vocab_cross_entropy_out_of_range_targets_emulated():
    """Targets < 0 or >= V are ignored rows: loss 0, gradient 0, not counted in the mean (the GPU kernels' rule, emulated);
    the float64 reference drops those rows itself."""
    import torch.nn.functional as F
    import pcd_ops
    g = torch.Generator().manual_seed(4)
    V = 13
    x = torch.randn(3, 5, 8, generator=g)
    w, b = torch.randn(V, 8, generator=g), torch.randn(V, generator=g)
    tg = torch.randint(0, V, (3, 5), generator=g)
    tg[0, 1], tg[1, 3], tg[2, 0], tg[2, 4] = V, -100, V + 5, 1 << 40
    xe, we, be = (t.clone().requires_grad_(True) for t in (x, w, b))
    loss = pcd_ops.vocab_cross_entropy(xe, we, be, tg)
    loss.backward()
    keep = ((tg >= 0) & (tg < V)).flatten()
    xr, wr, br = (t.double().requires_grad_(True) for t in (x, w, b))
    ref = F.cross_entropy(F.linear(xr, wr, br).flatten(end_dim=1)[keep], tg.flatten()[keep])
    ref.backward()
    P.assert_close(loss, ref, 1e-6, "loss")
    for got, r, name in ((xe.grad, xr.grad, "dx"), (we.grad, wr.grad, "dw"), (be.grad, br.grad, "db")):
        P.assert_close(got, r, 1e-5, name)
