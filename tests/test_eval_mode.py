"""Eval mode (BatchNorm from running statistics, forward only) of MixedOp, Cell, Network, VqaModel and the derived network,
against the oracle with training=False.  CPU cases run the eval kernels' sources through the -DPCD_EMU build; GPU cases
run the sm_100a library at the benchmark's sizes.

Running statistics are set to distinct seeded values spread wide (mean of order 1, variance 0.05 .. 20), so a kernel that
reads another BatchNorm's slot, swaps mean and variance or ignores the statistics fails.  Every case also checks that the
forward writes no parameter, running statistic, num_batches_tracked or arch weight, and that eval mode with autograd
recording raises NotImplementedError.
"""
import copy
import math

import pytest
import torch

import parity_cases as P
from helpers import REL_TOL, assert_close, load_golden, rel_err
from oracle import pcdarts_oracle as O


@pytest.fixture(scope="module")
def emulation():
    import pcd_build
    import pcd_native
    pcd_native.enable_emulation(pcd_build.build_emu())
    yield
    pcd_native._emu_lib = None


def _spread_stats_(module, seed):
    """Distinct running statistics per BatchNorm and channel: mean ~ U(-1.5, 1.5), variance log-uniform in [0.05, 20]."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for m in module.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                n = m.running_mean.numel()
                m.running_mean.copy_(3.0 * torch.rand(n, generator=g) - 1.5)
                m.running_var.copy_(torch.exp(math.log(0.05) + math.log(400.0) * torch.rand(n, generator=g)))
                m.num_batches_tracked.fill_(7)


def _snapshot(module, extra=()):
    return [t.detach().clone() for t in list(module.state_dict().values()) + list(extra)]


def _assert_unchanged(before, module, extra=()):
    after = list(module.state_dict().values()) + list(extra)
    assert len(before) == len(after)
    for a, b in zip(before, after):
        assert torch.equal(a, b.detach().to(a.device)), "eval forward wrote a parameter / buffer / arch weight"


def _oracle_state(module, dtype=None):
    sd = {k: v.detach().clone().cpu() for k, v in module.state_dict().items()}
    if dtype is not None:
        sd = {k: (v.to(dtype) if v.is_floating_point() else v) for k, v in sd.items()}
    return O.split_state(sd)


# ---- MixedOp -----------------------------------------------------------------------------------------------------
def mixed_eval_case(C, stride, x, w, device, seed):
    import config
    config.DEVICE = device
    from pcdarts.model_search import MixedOp
    m = MixedOp(C, stride)
    P._fill(m, seed)
    _spread_stats_(m, seed)
    m.eval()
    par, buf = _oracle_state(m)
    yr = O.mixed_op(par, O.BNState(buf), "_ops.", x, w, stride, training=False)
    m.to(device)
    xd, wd = x.to(device), w.to(device)
    before = _snapshot(m)
    with torch.no_grad():
        y = m(xd, wd)
    _assert_unchanged(before, m)
    assert_close(y, yr, REL_TOL, "MixedOp eval")
    c = C // 4
    mp = xd[:, c:] if stride == 1 else torch.nn.functional.max_pool2d(xd[:, c:], 2, 2)
    for q in range(1, 4):            # bypass channels: exact copies
        assert torch.equal(y[:, q::4], mp[:, (q - 1) * c:q * c])
    with pytest.raises(NotImplementedError, match="no_grad"):
        m(xd.requires_grad_(True), wd)


@pytest.mark.parametrize("name,C,stride", P.MIXED)
def test_mixed_op_eval_emulated(emulation, name, C, stride):
    g = load_golden("mixed_" + name)
    mixed_eval_case(C, stride, g["x"], g["w"], "cpu", 100 + C + stride)


@pytest.mark.parametrize("B", [1, 3])
def test_mixed_op_eval_batch_sizes_emulated(emulation, B):
    gen = torch.Generator().manual_seed(B)
    mixed_eval_case(32, 2, torch.randn(B, 32, 14, 14, generator=gen), torch.softmax(torch.randn(8, generator=gen), 0), "cpu", 5)


# ---- Cell --------------------------------------------------------------------------------------------------------
def cell_eval_case(cpp, cp, C, red, rp, B, H, device, seed=13):
    import config
    config.DEVICE = device
    from pcdarts.model_search import Cell
    m = Cell(4, 4, cpp, cp, C, red, rp)
    P._fill(m, seed)
    _spread_stats_(m, seed)
    m.eval()
    gen = torch.Generator().manual_seed(seed)
    s0 = torch.randn(B, cpp, 2 * H if rp else H, 2 * H if rp else H, generator=gen)
    s1 = torch.randn(B, cp, H, H, generator=gen)
    w = torch.softmax(torch.randn(14, 8, generator=gen), -1)
    w2 = torch.softmax(torch.randn(14, generator=gen), 0)
    par, buf = _oracle_state(m)
    yr = O.cell_forward(par, O.BNState(buf), "", s0, s1, w, w2, red, rp, training=False)
    m.to(device)
    ins = [t.to(device) for t in (s0, s1, w, w2)]
    before = _snapshot(m, ins[2:])
    with torch.no_grad():
        y = m(*ins)
    _assert_unchanged(before, m, ins[2:])
    assert_close(y, yr, REL_TOL, "Cell eval")
    with pytest.raises(NotImplementedError):
        m(*ins)                      # grad enabled and the parameters require grad


@pytest.mark.parametrize("name,cpp,cp,C,red,rp", P.CELLS)
def test_cell_eval_emulated(emulation, name, cpp, cp, C, red, rp):
    cell_eval_case(cpp, cp, C, red, rp, 2, 8, "cpu")


# the production spatial sizes of the 4-cell network at 64 x 64 input (64^2 / 32^2 / 16^2), one image each, one odd batch
@pytest.mark.parametrize("name,cpp,cp,C,red,rp,B,H", [("normal", 48, 48, 16, False, False, 1, 64),
                                                    ("reduce", 48, 64, 32, True, False, 1, 64),
                                                    ("reduce_rp", 64, 128, 64, True, True, 1, 32),
                                                    ("normal_rp", 128, 256, 64, False, True, 3, 16)])
def test_cell_eval_production_sizes_emulated(emulation, name, cpp, cp, C, red, rp, B, H):
    cell_eval_case(cpp, cp, C, red, rp, B, H, "cpu")


# ---- Network -----------------------------------------------------------------------------------------------------
def network_eval_case(B, H, device, seed=17, dtype_ref=torch.float32, tol=REL_TOL, trained_stats=False):
    import config
    config.DEVICE = device
    from pcdarts.model_search import Network
    net = Network(16, 10, 4)
    P._fill(net, seed)
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(B, 3, H, H, generator=gen)
    arch = [1e-1 * torch.randn(s, generator=gen) for s in ((14, 8), (14, 8), (14,), (14,))]
    net.to(device)
    for a, v in zip(net.arch_parameters(), arch):
        a.data.copy_(v)
    if trained_stats:                # running statistics written by native training-mode forwards
        net.train()
        with torch.no_grad():
            for k in range(2):
                net(torch.randn(B, 3, H, H, generator=gen).to(device) + k)
    else:
        _spread_stats_(net, seed)
    net.eval()
    par, buf = _oracle_state(net, dtype_ref)
    yr = O.network_forward(par, O.BNState(buf), [a.to(dtype_ref) for a in arch], x.to(dtype_ref), training=False)
    before = _snapshot(net, net.arch_parameters())
    with torch.no_grad():
        y = net(x.to(device))
    _assert_unchanged(before, net, net.arch_parameters())
    assert_close(y.double().cpu(), yr.double(), tol, "Network eval")
    with pytest.raises(NotImplementedError):
        net(x.to(device))            # the arch weights require grad
    return net, y


def test_network_eval_emulated(emulation):
    network_eval_case(2, 32, "cpu")


def test_network_eval_after_native_training_forwards_emulated(emulation):
    network_eval_case(3, 16, "cpu", trained_stats=True)


# ---- VqaModel ----------------------------------------------------------------------------------------------------
def _oracle_generate(par, feat, T=30, start=2):
    """Greedy decode of QstEncoder.generate in the oracle's terms: (tokens, top-2 logit margins)."""
    h = c = feat
    word = torch.full((feat.shape[0],), start, dtype=torch.long)
    toks, margins = [], []
    for t in range(T):
        emb = torch.nn.functional.embedding(word, par["qst_encoder.word2vec.weight"])
        emb = torch.tanh(emb) if t == 0 else emb          # the reference squashes only the <start> embedding
        _, h, c = O.lstm_forward(par, "qst_encoder.lstm.", emb[None], h, c)
        logits = torch.nn.functional.linear(torch.tanh(h), par["qst_encoder.fc1.weight"], par["qst_encoder.fc1.bias"])
        top = logits.topk(2, dim=1).values
        word = logits.argmax(1)
        toks.append(word)
        margins.append(top[:, 0] - top[:, 1])
    return torch.stack(toks, 1), torch.stack(margins, 1)


def vqa_eval_case(m, img, qst, lbl, dims_kw, tol=REL_TOL, tie=1e-5):
    """m in eval mode; every output against the oracle with training=False (dropout off in eval mode)."""
    par, buf = _oracle_state(m, torch.float64)
    arch = [a.detach().cpu().double() for a in m.arch_parameters()]
    imgc, qstc, lblc = img.cpu().double(), qst.cpu(), lbl.cpu()
    ans_r, qout_r = O.vqa_forward(par, O.BNState(buf), arch, imgc, qstc, training=False, **dims_kw)
    loss_r = O.vqa_loss(par, O.BNState(buf), arch, imgc, qstc, lblc, training=False, **dims_kw)
    before = _snapshot(m, m.arch_parameters())
    with torch.no_grad():
        ans, qout = m(img, qst)
        loss = m._loss(img, qst, lbl)
        toks, _ = m.generate(img)
    _assert_unchanged(before, m, m.arch_parameters())
    assert_close(ans.double().cpu(), ans_r, tol, "answer logits")
    assert_close(qout.double().cpu(), qout_r, tol, "question logits")
    assert_close(loss.double().cpu(), loss_r, tol, "loss")
    feat = O.network_forward(par, O.BNState(buf), arch, imgc, pre="img_encoder.darts.", training=False, **dims_kw)
    feat = torch.nn.functional.linear(feat, par["img_encoder.fc.weight"], par["img_encoder.fc.bias"])
    feat = feat / feat.norm(p=2, dim=1, keepdim=True)
    ref, margin = _oracle_generate(par, feat, toks.shape[1])
    compared = 0
    for b in range(ref.shape[0]):
        for t in range(ref.shape[1]):
            if float(margin[b, t]) < tie:
                break
            assert int(toks[b, t]) == int(ref[b, t]), (b, t)
            compared += 1
    assert compared > 0
    with pytest.raises(NotImplementedError):
        m(img, qst)


def test_vqa_model_eval_emulated(emulation):
    m = P.make_vqa("cpu")
    _spread_stats_(m, 400)
    m.eval()
    img, qst, lbl = P.vqa_batch(11, "cpu", B=3)
    vqa_eval_case(m, img, qst, lbl, {})


# ---- derived network ---------------------------------------------------------------------------------------------
def derived_eval_case(device, B=3, img=32, C=16, layers=4, tol=1e-4):
    from pcdarts.genotypes import Genotype
    from pcdarts.model import NetworkDerived
    torch.manual_seed(11)
    geno = Genotype(normal=P.TEST_GENOTYPE["normal"], normal_concat=range(2, 6), reduce=P.TEST_GENOTYPE["reduce"],
                    reduce_concat=range(2, 6))
    net = NetworkDerived(C, layers, geno)
    with torch.no_grad():
        for m in net.modules():
            if isinstance(m, torch.nn.BatchNorm2d) and m.affine:
                m.weight.copy_(1.0 + 0.2 * torch.randn_like(m.weight))
                m.bias.copy_(0.2 * torch.randn_like(m.bias))
    _spread_stats_(net, 23)
    net.eval()
    ref = copy.deepcopy(net).double()
    net = net.to(device)
    x = torch.randn(B, 3, img, img)
    before = _snapshot(net)
    with torch.no_grad():
        y = net(x.to(device))
        yr = ref(x.double(), stock=True)
    _assert_unchanged(before, net)
    assert_close(y.double().cpu(), yr, tol, "derived network eval")
    with pytest.raises(NotImplementedError):
        net(x.to(device))


def test_derived_network_eval_emulated(emulation):
    derived_eval_case("cpu")


def test_op_modules_eval_emulated(emulation):
    """Stand-alone op modules and preprocess ops in eval mode against their stock layers in float64."""
    from pcdarts.operations import OPS, FactorizedReduce, ReLUConvBN
    mods = [(OPS["sep_conv_3x3"](16, 2, True), 16), (OPS["dil_conv_5x5"](8, 1, False), 8), (ReLUConvBN(48, 16, 1, 1, 0), 48),
            (ReLUConvBN(48, 32, 1, 1, 0, affine=False), 48), (FactorizedReduce(32, 64), 32)]
    for i, (m, cin) in enumerate(mods):
        _spread_stats_(m, 40 + i)
        m.eval()
        x = torch.randn(3, cin, 12, 12)
        ref = copy.deepcopy(m).double()
        before = _snapshot(m)
        with torch.no_grad():
            y = m(x)
            yr = ref.stock_forward(x.double())
        _assert_unchanged(before, m)
        assert_close(y.double(), yr, 1e-5, type(m).__name__)
        with pytest.raises(NotImplementedError):
            m(x)


# ---- GPU: benchmark sizes ----------------------------------------------------------------------------------------
def _shuffle_on_device(x, groups=4):
    """oracle.channel_shuffle with its index on x's device (the oracle builds it on the CPU)."""
    return x.index_select(1, torch.from_numpy(O.shuffle_perm(x.shape[1], groups)).to(x.device))


def _cuda_fp32_oracle():
    prev = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    return prev


@pytest.mark.gpu
def test_network_eval_full_size_vs_float64_gpu(monkeypatch):
    """B = 64, 64 x 64: the output and every cell's output within rel 1e-4 of the oracle evaluated in float64 on the GPU
    (the fp32 oracle on the GPU, TF32 off, is reported beside it)."""
    import config
    config.DEVICE = "cuda"
    from pcdarts.model_search import Network
    monkeypatch.setattr(O, "channel_shuffle", _shuffle_on_device)
    prev = _cuda_fp32_oracle()
    try:
        net = Network(16, 10, 4)
        P._fill(net, 17)
        _spread_stats_(net, 17)
        gen = torch.Generator().manual_seed(17)
        x = torch.randn(64, 3, 64, 64, generator=gen)
        arch = [1e-1 * torch.randn(s, generator=gen) for s in ((14, 8), (14, 8), (14,), (14,))]
        net.to("cuda").eval()
        for a, v in zip(net.arch_parameters(), arch):
            a.data.copy_(v)
        import pcd_ops
        cells_out, cell_eval = [], pcd_ops.cell_forward_eval
        monkeypatch.setattr(pcd_ops, "cell_forward_eval", lambda *a: cells_out.append(cell_eval(*a)) or cells_out[-1])
        before = _snapshot(net, net.arch_parameters())
        with torch.no_grad():
            y = net(x.cuda())
        assert len(cells_out) == 4
        _assert_unchanged(before, net, net.arch_parameters())
        errs = {}
        for dt in (torch.float64, torch.float32):
            sd = {k: (v.detach().to(dt) if v.is_floating_point() else v.detach()) for k, v in net.state_dict().items()}
            par, buf = O.split_state(sd)
            with torch.no_grad():
                xr = x.cuda().to(dt)
                z = torch.nn.functional.conv2d(xr, par["stem.0.weight"], padding=1)
                s0 = s1 = O.batch_norm(par, O.BNState(buf), "stem.1.", z, training=False)
                ref_cells = []
                for i, (_, _, _, red, rp) in enumerate(O.cell_plan(16, 4)):
                    wts, wts2 = O.arch_weights(arch[1].cuda().to(dt), arch[3].cuda().to(dt)) if red else \
                        O.arch_weights(arch[0].cuda().to(dt), arch[2].cuda().to(dt))
                    # every cell replayed on the very inputs ours received: the error of one cell is not compounded
                    ins = (s0, s1) if i == 0 else ((cells_out[i - 2] if i >= 2 else s1).to(dt), cells_out[i - 1].to(dt))
                    ref_cells.append(O.cell_forward(par, O.BNState(buf), f"cells.{i}.", ins[0], ins[1], wts, wts2, red, rp,
                                                    training=False))
                yr = torch.nn.functional.adaptive_avg_pool2d(cells_out[-1].to(dt), 7).flatten(1)
                yfull = O.network_forward(par, O.BNState(buf), [a.cuda().to(dt) for a in arch], xr, training=False)
            errs[dt] = ([rel_err(o, r) for o, r in zip(cells_out, ref_cells)], rel_err(y, yr), rel_err(y, yfull))
        cell64, pool64, full64 = errs[torch.float64]
        assert max(cell64) <= 1e-4, errs
        assert pool64 <= 1e-4 and full64 <= 1e-4, errs
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = prev


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 130])
def test_network_eval_batch_sizes_gpu(B):
    network_eval_case(B, 64, "cuda", dtype_ref=torch.float64)


@pytest.mark.gpu
def test_network_eval_after_native_training_forwards_gpu():
    network_eval_case(8, 64, "cuda", dtype_ref=torch.float64, trained_stats=True)


@pytest.mark.gpu
@pytest.mark.parametrize("name,C,stride", P.MIXED)
def test_mixed_op_eval_gpu(name, C, stride):
    g = load_golden("mixed_" + name)
    mixed_eval_case(C, stride, g["x"], g["w"], "cuda", 100 + C + stride)


@pytest.mark.gpu
def test_vqa_model_eval_benchmark_dims_gpu():
    import config
    config.DEVICE = "cuda"
    from vqa_model import VqaModel
    V = 17858
    m = VqaModel(img_encoder_type="darts", qst_vocab_size=V, **P.FULL_DIMS)
    P._fill(m, 400)
    _spread_stats_(m, 400)
    m.to("cuda").eval()
    for i, a in enumerate(m.arch_parameters()):
        a.data.copy_(0.5 * torch.randn(a.shape, generator=torch.Generator().manual_seed(30 + i)))
    img, qst, lbl = P.full_batch(5, 64, V, 64)
    prev = _cuda_fp32_oracle()
    try:
        vqa_eval_case(m, img.cuda(), qst.cuda(), lbl.cuda(), {})
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = prev


@pytest.mark.gpu
def test_derived_network_eval_gpu():
    derived_eval_case("cuda", B=5, img=64)
