"""Stand-alone candidate operations (SURVEY.md §8f-4) — the op kernels' SOURCES compiled with -DPCD_EMU, against the same
layers in stock torch at float64, plus the pin of that stock path to the reference's own modules."""
import sys

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


@pytest.mark.parametrize("name,C,stride,affine,B,H", P.OPS_CASES)
def test_op_vs_stock_emulated(name, C, stride, affine, B, H):
    P.op_vs_stock(name, C, stride, affine, B, H, "cpu")


@pytest.mark.parametrize("name,stride", [("max_pool_3x3", 1), ("max_pool_3x3", 2), ("sep_conv_3x3", 1), ("dil_conv_5x5", 2)])
def test_op_exact_ties_emulated(name, stride):
    """Pool windows full of equal values (first maximum in scan order takes the gradient, like ATen), ReLU inputs exactly 0."""
    P.op_vs_stock(name, 8, stride, True, 2, 12, "cpu", quantized=True)


@pytest.mark.parametrize("cpb", ["2", "3"])
def test_pointwise_backward_walks_several_chunks(cpb, monkeypatch):
    """pw_bwd blocks that walk several 128-pixel chunks (what large batches use): 20 x 20 planes = 3 full chunks + a ragged one."""
    monkeypatch.setenv("PCD_PW_CPB", cpb)
    P.op_vs_stock("dil_conv_3x3", 8, 1, True, 2, 20, "cpu")
    P.op_vs_stock("sep_conv_3x3", 16, 2, True, 1, 32, "cpu")


def test_unsupported_ops_raise():
    from pcdarts.operations import OPS
    op = OPS["conv_7x1_1x7"](8, 1, True)
    with pytest.raises(RuntimeError, match="PCD_ERR_UNSUPPORTED"):
        op(torch.randn(1, 8, 8, 8))
    with pytest.raises(RuntimeError, match="PCD_ERR_UNSUPPORTED"):
        OPS["sep_conv_3x3"](6, 1, True)(torch.randn(1, 6, 8, 8))           # channels not a multiple of 4
    with pytest.raises(RuntimeError, match="PCD_ERR_UNSUPPORTED"):
        OPS["max_pool_3x3"](4, 1, True)(torch.randn(1, 4, 80, 80))         # planes above 64 x 64
    with pytest.raises(NotImplementedError):
        OPS["dil_conv_3x3"](8, 1, True).eval()(torch.randn(1, 8, 8, 8))    # eval-mode BatchNorm is out of scope


_STOCK_MIXED = {}


def _stock_mixed(name, C, stride):
    """MixedOp of the reference (model_search.py:44-58) composed from this repo's OPS modules' `stock_forward`, with the
    weights, input, arch weights and output gradient its golden generator used (tests/golden/make_golden.py mixed_case).
    One thread, like the generator: the weight-gradient sums then come out in the same order."""
    if name not in _STOCK_MIXED:
        import config
        from oracle import pcdarts_oracle as O
        from pcdarts.model_search import MixedOp
        from helpers import load_golden
        config.DEVICE = torch.device("cpu")
        g = load_golden("mixed_" + name)
        m = MixedOp(C, stride).train()
        P._fill(m, 100 + C + stride)
        x = g["x"].clone().requires_grad_(True)
        w = g["w"].clone().requires_grad_(True)
        c = C // 4
        threads = torch.get_num_threads()
        torch.set_num_threads(1)
        try:
            acc = 0
            for k, op in enumerate(m._ops):          # python sum() order of the reference: ((0 + w0 o0) + w1 o1) + ...
                if isinstance(op, torch.nn.Sequential):      # pool candidate + BatchNorm2d(affine=False)
                    o = op[1](op[0].stock_forward(x[:, :c]))
                else:
                    o = op.stock_forward(x[:, :c]) if hasattr(op, "stock_forward") else op(x[:, :c])
                acc = acc + w[k] * o
            rest = x[:, c:] if stride == 1 else torch.nn.functional.max_pool2d(x[:, c:], 2, 2)
            y = O.channel_shuffle(torch.cat([acc, rest], dim=1))
            (y * g["G"]).sum().backward()
        finally:
            torch.set_num_threads(threads)
        _STOCK_MIXED[name] = (m, y.detach(), x.grad, w.grad, g)
    return _STOCK_MIXED[name]


@pytest.mark.parametrize("primitive", ["none", "max_pool_3x3", "avg_pool_3x3", "skip_connect", "sep_conv_3x3", "sep_conv_5x5",
                                       "dil_conv_3x3", "dil_conv_5x5"])
@pytest.mark.parametrize("name,C,stride", P.MIXED)
def test_stock_forward_is_the_reference_module(name, C, stride, primitive):
    """`stock_forward` (the yardstick of the op parity tests) against what the reference's own OPS[primitive] modules computed
    inside its MixedOp (tests/golden/mixed_*.npz): the MixedOp output and input / arch-weight gradients, and this primitive's
    weight gradients and BatchNorm buffers.  Bit-equal on the generator's thread count; 1e-6 leaves room for a CPU whose
    vector width orders the weight-gradient sums differently."""
    from pcdarts.genotypes import PRIMITIVES
    from helpers import assert_close
    m, y, dx, dw, g = _stock_mixed(name, C, stride)
    for got, k in ((y, "y"), (dx, "dx"), (dw, "dw")):
        assert_close(got, g[k], 1e-6, k)
    pre = f"_ops.{PRIMITIVES.index(primitive)}."
    for k, p in m.named_parameters():
        if k.startswith(pre):
            assert_close(p.grad, g["grad." + k], 1e-6, k)
    for k, v in m.state_dict().items():
        if k.startswith(pre) and ("running" in k or "tracked" in k):
            assert_close(v.double(), g["buf." + k].double(), 1e-6, k)


def test_derived_network_vs_stock_emulated():
    """NetworkDerived (pcdarts/model.py) end to end: stem, 4 derived cells (2 reductions), pooling — forward, all weight grads."""
    P.derived_vs_stock("cpu")


def test_derive_from_search_network():
    import config
    config.DEVICE = torch.device("cpu")
    from pcdarts.model import derive
    from pcdarts.model_search import Network
    torch.manual_seed(0)
    search = Network(16, 10, 4)
    net = derive(search)
    g = search.genotype()
    assert net.genotype() == g and len(net.cells) == 4 and net.output_ch == search.output_ch
    assert [type(c.preprocess0).__name__ for c in net.cells] == [type(c.preprocess0).__name__ for c in search.cells]
    names = [n for n, _ in g.normal]
    assert all(n in ("max_pool_3x3", "avg_pool_3x3", "skip_connect", "sep_conv_3x3", "sep_conv_5x5", "dil_conv_3x3", "dil_conv_5x5") for n in names)
