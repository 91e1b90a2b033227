"""Host-side logic that needs neither kernels nor the reference tree: genotype derivation against the reference's golden."""
import os

import torch


def test_genotype_matches_reference_golden():
    """Network.genotype() against the unmodified reference (tests/golden/make_golden_genotype.py): 'none' never chosen, the two
    strongest edges per node, ties resolved like the reference's sorted() / argmax."""
    import numpy as np
    import config
    config.DEVICE = torch.device("cpu")
    from pcdarts.model_search import Network
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "genotype.npz"))
    net = Network(16, 10, 4)
    for case in range(6):
        with torch.no_grad():
            for t, k in zip(net.arch_parameters(), ("alphas_normal", "alphas_reduce", "betas_normal", "betas_reduce")):
                t.copy_(torch.from_numpy(z[f"c{case}_{k}"]))
        g = net.genotype()
        assert [f"{n}:{j}" for n, j in g.normal] == [str(s) for s in z[f"c{case}_normal"]], case
        assert [f"{n}:{j}" for n, j in g.reduce] == [str(s) for s in z[f"c{case}_reduce"]], case
        assert list(g.normal_concat) + list(g.reduce_concat) == [int(v) for v in z[f"c{case}_concat"]]


def test_auto_split_fills_whole_rounds():
    """pcd_ops._auto_split: K splits for the persistent GEMM's round-robin schedule (one CTA per SM, 148 SMs)."""
    import pcd_ops
    f = pcd_ops._auto_split
    assert f(1920, 17858, 512) == 1                    # 1050 tiles: more than enough work items
    assert f(17858, 512, 1920) == 1
    s = f(1920, 512, 17860)                            # vocabulary dX: 30 tiles
    assert 2 <= s <= 32 and (30 * s) % 148 > 110 or (30 * s) <= 148      # the last round is nearly full
    assert f(1920, 300, 2048) == 4                     # 30 tiles x 4 = 120 items: one round (5 would be two)
    assert f(64, 512, 12544) == 32                     # 2 tiles: as many splits as the cap allows
    for m, n, k in ((64, 64, 64), (128, 256, 100), (5, 1000, 129), (300, 300, 300)):
        s = f(m, n, k)
        bk = 16 if n >= 256 else 32
        assert 1 <= s <= max(1, min(32, -(-k // bk) // 8))


def test_3xtf32_acceptance_rejects_fewer_terms():
    """The criterion the GPU sweep of pcd_gemm_tn_3xtf32 applies (helpers.accept_3xtf32) can fail: at every shape of that
    sweep it accepts the 3-term split product hi*hi + hi*lo + lo*hi (operands truncated as kind::tf32 truncates them) and
    rejects the 1-term product and both 2-term products (either correction dropped)."""
    from helpers import GEMM_CASES, accept_3xtf32, gemm_errors, trunc_tf32
    g = torch.Generator().manual_seed(0)
    for m, n, k, _, _, _, has_bias in GEMM_CASES:
        a, b = torch.randn(m, k, generator=g), torch.randn(n, k, generator=g)
        bias = torch.randn(n, generator=g) if has_bias else None
        ah, bh = trunc_tf32(a), trunc_tf32(b)
        al, bl = trunc_tf32(a - ah).double(), trunc_tf32(b - bh).double()
        ah, bh = ah.double(), bh.double()
        bias64 = 0.0 if bias is None else bias.double()
        terms = {"hi*hi": ah @ bh.T, "hi*lo": ah @ bl.T, "lo*hi": al @ bh.T}
        for kept, want in ((("hi*hi",), False), (("hi*hi", "hi*lo"), False), (("hi*hi", "lo*hi"), False),
                           (("hi*hi", "hi*lo", "lo*hi"), True)):
            c = sum(terms[t] for t in kept) + bias64
            errs = gemm_errors(c, a, b, bias)
            assert accept_3xtf32(*errs) == want, (m, n, k, kept, errs)
