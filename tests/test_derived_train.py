"""Training the derived architecture: the drop-path node sum (pcd_droppath_sum_*) against its numpy restatement
(droppath_oracle.py), drop-path in NetworkDerived against the float64 stock layers carrying the oracle's masks, derive_vqa,
data-parallel masks, and GraphedTrainStep.  CPU cases run the kernel source's -DPCD_EMU build; `gpu` cases the sm_100a kernel."""
import copy
import ctypes
import os

import numpy as np
import pytest
import torch

import droppath_oracle as O
import parity_cases as P
from helpers import assert_close, rel_err

SEEDS = (0x0123456789ABCDEF, 7, 0xFFFFFFFFFFFFFFFF)
DIMS = dict(embed_size=512, ans_vocab_size=1000, word_embed_size=300, num_layers=1, hidden_size=512)


@pytest.fixture(scope="module")
def emulation():
    import pcd_build
    import pcd_native
    pcd_native.enable_emulation(pcd_build.build_emu())
    yield pcd_native._emu_lib
    pcd_native._emu_lib = None


def seed_tensor(seed, device):
    s = int(seed) & (2 ** 64 - 1)
    return torch.tensor([s - 2 ** 64 if s >= 2 ** 63 else s], dtype=torch.int64, device=device)


def keep_tensor(p, device):
    return torch.full((1,), 1.0 - p, dtype=torch.float32, device=device)


def node_case(device, shape, seed, cell, node, offset, drop=(True, True), p=0.3, h1=None, h2=None):
    """One forward + backward of pcd_ops.droppath_sum against the oracle, bit for bit."""
    from pcd_ops import droppath_sum
    g = torch.Generator().manual_seed(cell * 31 + node + offset)
    h1 = torch.randn(shape, generator=g) if h1 is None else h1
    h2 = torch.randn(shape, generator=g) if h2 is None else h2
    gy = torch.randn(shape, generator=g)
    a, b = h1.clone().to(device).requires_grad_(), h2.clone().to(device).requires_grad_()
    keep = keep_tensor(p, device)
    y = droppath_sum(a, b, drop[0], drop[1], keep, seed_tensor(seed, device), cell, node, offset)
    ga, gb = torch.autograd.grad(y, (a, b), gy.to(device))
    k32 = np.float32(1.0 - p)
    ref, m1, m2 = O.node_sum(h1.numpy(), h2.numpy(), drop[0], drop[1], k32, seed, cell, node, offset)
    r1, r2 = O.node_sum_backward(gy.numpy(), drop[0], drop[1], k32, seed, cell, node, offset)
    assert torch.equal(y.cpu(), torch.from_numpy(ref))
    assert torch.equal(ga.cpu(), torch.from_numpy(r1)) and torch.equal(gb.cpu(), torch.from_numpy(r2))
    return m1, m2


# ---- the kernel against the oracle -------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(4, 4, 8, 8), (3, 3, 5, 7), (5, 1, 1, 3), (2, 16, 6, 6)])
@pytest.mark.parametrize("seed", SEEDS)
def test_kernel_matches_oracle_emulated(emulation, shape, seed):
    for cell, node, offset in ((0, 0, 0), (3, 2, 5), (7, 3, 1000)):
        for drop in ((True, True), (True, False), (False, True)):
            node_case("cpu", shape, seed, cell, node, offset, drop)


def test_kernel_unaligned_inputs_emulated(emulation):
    """Views that do not start on a 16-byte boundary take the scalar path, with the same result."""
    g = torch.Generator().manual_seed(5)
    buf1, buf2 = torch.randn(3 * 4 * 5 * 5 + 1, generator=g), torch.randn(3 * 4 * 5 * 5 + 3, generator=g)
    node_case("cpu", (3, 4, 5, 5), SEEDS[0], 1, 1, 2, h1=buf1[1:].view(3, 4, 5, 5), h2=buf2[3:].view(3, 4, 5, 5))


def test_keep_one_and_no_flags_are_plain_sum_emulated(emulation):
    from pcd_ops import droppath_sum
    g = torch.Generator().manual_seed(1)
    h1, h2, gy = (torch.randn(3, 4, 5, 7, generator=g) for _ in range(3))
    for drop, p in (((True, True), 0.0), ((False, False), 0.5)):
        a, b = h1.clone().requires_grad_(), h2.clone().requires_grad_()
        y = droppath_sum(a, b, *drop, keep_tensor(p, "cpu"), seed_tensor(9, "cpu"), 2, 1, 0)
        assert torch.equal(y, h1 + h2)
        ga, gb = torch.autograd.grad(y, (a, b), gy)
        assert torch.equal(ga, gy) and torch.equal(gb, gy)
    y = droppath_sum(h1, h2, False, False, None, None, 0, 0)        # nothing dropped: no seed or keep needed
    assert torch.equal(y, h1 + h2)


def test_masks_do_not_depend_on_sharding_emulated(emulation):
    from pcd_ops import droppath_sum
    g = torch.Generator().manual_seed(2)
    h1, h2 = torch.randn(4, 3, 4, 5, generator=g), torch.randn(4, 3, 4, 5, generator=g)
    args = (True, True, keep_tensor(0.5, "cpu"), seed_tensor(SEEDS[0], "cpu"), 1, 2)
    whole = droppath_sum(h1, h2, *args, 0)
    halves = torch.cat([droppath_sum(h1[:2], h2[:2], *args, 0), droppath_sum(h1[2:], h2[2:], *args, 2)])
    assert torch.equal(whole, halves)
    # and p = 0.5 does drop something here, differently for the two inputs
    _, m1, m2 = O.node_sum(h1.numpy(), h2.numpy(), True, True, np.float32(0.5), SEEDS[0], 1, 2)
    assert 0 < m1.sum() + m2.sum() < 8 and not np.array_equal(m1, m2)


def test_entry_points_reject_bad_arguments(emulation):
    import pcd_native as N
    lib = emulation
    x = torch.zeros(2, 8)
    out = torch.empty(2, 8)
    seed, keep = seed_tensor(1, "cpu"), keep_tensor(0.2, "cpu")

    def args(drop=1, offset=0, seed_p=seed, keep_p=keep, batch=2, numel=8):
        return N.DropPathArgs(batch, numel, drop, 0, 0, 0, offset, N.ptr(seed_p), N.ptr(keep_p), N.ptr(x), N.ptr(x), N.ptr(out),
                              N.ptr(x), N.ptr(out), None)
    for fn in (lib.pcd_droppath_sum_forward, lib.pcd_droppath_sum_backward):
        assert fn(ctypes.byref(args()), None) == 0
        assert fn(ctypes.byref(args(seed_p=None)), None) == -1
        assert fn(ctypes.byref(args(keep_p=None)), None) == -1
        assert fn(ctypes.byref(args(offset=-1)), None) == -1
        assert fn(ctypes.byref(args(drop=0, seed_p=None, keep_p=None)), None) == 0       # nothing dropped: none needed
        assert fn(ctypes.byref(args(batch=0)), None) == 0
        assert fn(ctypes.byref(args(numel=0)), None) == 0
        assert fn(None, None) == -1
    from pcd_ops import droppath_sum
    with pytest.raises(ValueError):
        droppath_sum(x, x, True, False, None, seed, 0, 0)
    with pytest.raises(ValueError):
        droppath_sum(x, x, True, False, keep, seed, 0, 0, -2)


# ---- drop-path in the derived network ----------------------------------------------------------------------------
def _net(C=16, layers=4):
    from pcdarts.genotypes import Genotype
    from pcdarts.model import NetworkDerived
    torch.manual_seed(11)
    geno = Genotype(normal=P.TEST_GENOTYPE["normal"], normal_concat=range(2, 6), reduce=P.TEST_GENOTYPE["reduce"],
                    reduce_concat=range(2, 6))
    net = NetworkDerived(C, layers, geno).train()
    with torch.no_grad():
        for m in net.modules():
            if isinstance(m, torch.nn.BatchNorm2d) and m.affine:
                m.weight.copy_(1.0 + 0.2 * torch.randn_like(m.weight))
                m.bias.copy_(0.2 * torch.randn_like(m.bias))
    return net


def derived_droppath_vs_stock(device, B=2, img=32, p=0.3, seed=SEEDS[0], offset=0, tol=1e-4, share=0.97):
    """NetworkDerived in training mode with drop-path against the same modules as stock torch layers in float64 (and in fp32,
    the yardstick) applying the oracle's masks: output, every weight gradient, BatchNorm buffers; the bars of
    parity_cases.derived_vs_stock."""
    net = _net()
    net.drop_path_prob = p
    net.drop_path_offset = offset
    ref = copy.deepcopy(net).double()
    ref32 = copy.deepcopy(net).to(device)
    net = net.to(device)
    net.drop_path_seed = seed_tensor(seed, device)
    k32 = np.float32(1.0 - p)
    rows = range(offset, offset + B)
    masks = lambda cell, node, inp: torch.from_numpy(O.masks(seed, rows, cell, 2 * node + inp, k32))
    x = torch.randn(B, 3, img, img)
    y = net(x.to(device))
    yr = ref(x.double(), stock=True, drop_masks=masks)
    y32 = ref32(x.to(device), stock=True, drop_masks=masks)
    gy = torch.randn(yr.shape)
    got = torch.autograd.grad(y, list(net.parameters()), gy.to(device))
    exp = torch.autograd.grad(yr, list(ref.parameters()), gy.double())
    g32 = torch.autograd.grad(y32, list(ref32.parameters()), gy.to(device))
    assert_close(y.double().cpu(), yr, tol, "derived network output with drop-path")
    errs = sorted(((rel_err(a_.double().cpu(), b_), n) for a_, b_, (n, _) in zip(got, exp, net.named_parameters())), reverse=True)
    yard = sorted((rel_err(a_.double().cpu(), b_) for a_, b_ in zip(g32, exp)), reverse=True)
    ok = sum(e <= tol for e, _ in errs) / len(errs)
    ok32 = sum(e <= tol for e in yard) / len(yard)
    med, med32 = errs[len(errs) // 2][0], yard[len(yard) // 2]
    assert ok >= min(share, ok32 - 0.05), (ok, ok32, errs[:5])
    assert med <= max(1e-5, 2 * med32), (med, med32)
    assert errs[0][0] <= max(50 * tol, 3 * yard[0]), (errs[:5], yard[:3])
    for (k, b1), (_, b2) in zip(net.named_buffers(), ref.named_buffers()):
        if k.endswith("num_batches_tracked"):
            assert int(b1) == int(b2), k
        else:
            assert_close(b1.double().cpu(), b2, 1e-4, k)
    # the masks did drop paths: a run without drop-path gives another output
    ref.drop_path_prob = 0.0
    assert rel_err(ref(x.double(), stock=True), yr) > 1e-3
    return ok


def test_derived_network_droppath_vs_stock_emulated(emulation):
    derived_droppath_vs_stock("cpu", B=3, offset=6)


def test_identity_edges_are_never_dropped(emulation, monkeypatch):
    import pcd_ops
    from pcdarts.operations import Identity
    net = _net()
    net.drop_path_prob = 0.5
    seen = []
    real = pcd_ops.droppath_sum

    def spy(h1, h2, drop1, drop2, *rest):
        seen.append((drop1, drop2))
        return real(h1, h2, drop1, drop2, *rest)
    monkeypatch.setattr(pcd_ops, "droppath_sum", spy)
    net(torch.randn(2, 3, 32, 32))
    expect = [(not isinstance(c._ops[2 * i], Identity), not isinstance(c._ops[2 * i + 1], Identity))
              for c in net.cells for i in range(c._steps)]
    assert seen == expect
    assert not all(d for pair in seen for d in pair)                  # the test genotype has Identity edges ...
    flat = [d for pair in seen for d in pair]
    assert sum(flat) > len(flat) // 2                                 # ... and FactorizedReduce ones, which are dropped
    # an Identity input passes through unscaled, whatever the mask
    h = torch.randn(4, 2, 3, 3)
    y = real(h, torch.zeros_like(h), False, True, keep_tensor(0.5, "cpu"), seed_tensor(3, "cpu"), 0, 0)
    assert torch.equal(y, h)


def test_eval_mode_and_zero_prob_are_todays_path(emulation, monkeypatch):
    """In eval mode drop_path_prob is ignored, and at p = 0 in training mode nothing is dropped: both bit-equal to the plain
    node sum h1 + h2."""
    import pcd_ops
    x = torch.randn(2, 3, 32, 32)
    plain = _net()
    drop = copy.deepcopy(plain)
    drop.drop_path_prob = 0.0
    y_drop = drop(x)
    with monkeypatch.context() as mp_:
        mp_.setattr(pcd_ops, "droppath_sum", lambda h1, h2, *a: h1 + h2)
        y_plain = plain(x)
    assert torch.equal(y_drop, y_plain)
    for m in (plain, drop):
        m.eval()
    drop.drop_path_prob = 0.6
    with torch.no_grad():
        y_drop = drop(x)
        with monkeypatch.context() as mp_:
            mp_.setattr(pcd_ops, "droppath_sum", lambda h1, h2, *a: h1 + h2)
            y_plain = plain(x)
    assert torch.equal(y_drop, y_plain)


def test_drop_path_prob_setter():
    net = _net(layers=3)
    assert net.drop_path_prob == 0.0
    net.drop_path_prob = 0.2
    assert net.drop_path_prob == 0.2 and float(net._drop_keep) == np.float32(0.8)
    for bad in (-0.1, 1.0, 1.5):
        with pytest.raises(ValueError):
            net.drop_path_prob = bad
    assert net.drop_path_prob == 0.2
    with pytest.raises(ValueError):         # the yardstick needs the masks it should apply
        net(torch.randn(1, 3, 16, 16), stock=True)


# ---- derive_vqa -----------------------------------------------------------------------------------------------------
def test_derive_vqa_runs_and_keeps_the_heads(emulation):
    from vqa_model import DerivedEncoder, derive_vqa
    from pcdarts.model import NetworkDerived
    search = P.make_vqa("cpu")
    torch.manual_seed(3)
    m = derive_vqa(search)
    assert isinstance(m.img_encoder, DerivedEncoder) and isinstance(m.img_encoder.darts, NetworkDerived)
    assert m.genotype() == search.genotype() and m.arch_parameters() == []
    keys = lambda mod: [k for k in mod.state_dict() if not k.startswith("img_encoder.")]
    assert keys(m) == keys(search)
    for k in keys(m):
        assert m.state_dict()[k].shape == search.state_dict()[k].shape
    assert "img_encoder.fc.weight" in m.state_dict()
    m.img_encoder.darts.drop_path_prob = 0.2
    img, qst, lbl = P.vqa_batch(7, "cpu")
    loss = m._loss(img, qst, lbl)
    assert torch.isfinite(loss)
    loss.backward()
    assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in m.img_encoder.parameters())
    words, ans = m.generate(img)
    assert words.shape == (img.shape[0], m.qst_encoder.max_length) and ans.shape == (img.shape[0], P.VQA_DIMS["ans_vocab_size"])
    m.eval()
    with torch.no_grad():
        a1, q1 = m(img, qst)
    assert torch.isfinite(a1).all() and torch.isfinite(q1).all()
    with pytest.raises(ValueError):
        m.new()


# ---- data parallel (gloo, world size 2, emulated kernels) --------------------------------------------------------
DP_SEED = 0x5EED5EED12345678


def _derived_vqa_dp():
    import pcd_ops
    from vqa_model import derive_vqa
    search = P.make_vqa("cpu")
    torch.manual_seed(21)
    m = derive_vqa(search)
    pcd_ops.allow_stock_ops(True)
    m.dropout.p = 0.0
    m.img_encoder.darts.drop_path_prob = 0.3
    m.img_encoder.darts.drop_path_seed = seed_tensor(DP_SEED, "cpu")
    return m


def _worker_derived(rank, world, port, out_dir):
    from test_dist_gloo import _setup
    _setup()
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    import pcd_dist
    from search import SearchStep
    pcd_dist.init_from_env("gloo")
    m = _derived_vqa_dp()
    step = SearchStep(m, None, torch.optim.Adam(m.parameters(), lr=1e-3), reducer=pcd_dist.GradReducer())
    loss = step.w_step(*P.vqa_batch(100 + rank, "cpu"))
    torch.save({"params": [p.detach().clone() for p in m.parameters()], "grads": [p.grad.clone() for p in m.parameters()],
                "loss": loss}, os.path.join(out_dir, f"derived_rank{rank}.pt"))
    dist.barrier()
    dist.destroy_process_group()


def test_dp_derived_wstep_matches_hand_averaged(tmp_path):
    import torch.multiprocessing as mp
    from test_dist_gloo import _free_port, _setup
    _setup()
    mp.spawn(_worker_derived, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    r0, r1 = (torch.load(os.path.join(tmp_path, f"derived_rank{r}.pt")) for r in range(2))
    for a, b in zip(r0["params"], r1["params"]):
        assert torch.equal(a, b)                     # replicas stay bit-identical
    # one process, the two shards with their global sample offsets, gradients averaged by hand, clipped as w_step does
    grads = []
    for rank in range(2):
        m = _derived_vqa_dp()
        m.img_encoder.darts.drop_path_offset = rank * 2
        loss = m._loss(*P.vqa_batch(100 + rank, "cpu"))
        grads.append(torch.autograd.grad(loss, list(m.parameters())))
    avg = [(a + b) / 2 for a, b in zip(*grads)]
    norm = torch.norm(torch.stack([g.norm() for g in avg]))
    coef = min(1.0, 5.0 / (float(norm) + 1e-6))
    for g, ref in zip(r0["grads"], avg):
        assert_close(g, ref * coef, 1e-5, "averaged derived w-grad")
    # the shard offsets matter: rank 1's masks are not rank 0's
    m = _derived_vqa_dp()
    other = torch.autograd.grad(m._loss(*P.vqa_batch(101, "cpu")), list(m.parameters()))
    assert max(rel_err(a, b) for a, b in zip(other, grads[1])) > 1e-3


# ---- GPU -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(128, 64, 64, 64), (7, 3, 5, 9), (130, 16, 31, 31), (2, 1, 1, 1)])
def test_kernel_matches_oracle_gpu(shape):
    for seed, cell, node, offset in ((SEEDS[0], 0, 0, 0), (SEEDS[2], 5, 3, 384)):
        for drop in ((True, True), (False, True)):
            node_case("cuda", shape, seed, cell, node, offset, drop, p=0.2)


@pytest.mark.gpu
def test_mask_statistics_gpu():
    """Keep rate at p = 0.2 over 1.2e5 draws per input: two-sided binomial test; the two inputs of a node: 2x2 chi-square."""
    from scipy import stats
    from pcd_ops import droppath_sum
    B, p = 60000, 0.2
    keep = keep_tensor(p, "cuda")
    ones = torch.ones(B, 1, 1, 1, device="cuda")
    m1s, m2s = [], []
    for cell in (0, 1):
        y = droppath_sum(ones, 2 * ones, True, True, keep, seed_tensor(SEEDS[0] + cell, "cuda"), cell, 1, 0)
        code = torch.round(y.flatten() * keep).long().cpu()          # m1 + 2 m2
        m1s.append(code % 2)
        m2s.append(code // 2)
    m1, m2 = torch.cat(m1s).numpy(), torch.cat(m2s).numpy()
    k = float(keep)
    for m in (m1, m2):
        assert stats.binomtest(int(m.sum()), len(m), k).pvalue > 1e-3, (m.mean(), k)
    table = np.array([[np.sum((m1 == a) & (m2 == b)) for b in (0, 1)] for a in (0, 1)])
    assert stats.chi2_contingency(table)[1] > 1e-3, table


@pytest.mark.gpu
def test_derived_network_droppath_vs_stock_gpu():
    ok = derived_droppath_vs_stock("cuda", B=64, img=64, offset=128)
    print(f"derived network with drop-path, B=64, 64x64: share within 1e-4 = {ok:.3f}")


def _derived_bench_model(seed=10):
    """A derived VqaModel at the benchmark dimensions (V = 17858, 1000 answers, hidden 512, 64x64 images)."""
    from vqa_model import VqaModel, derive_vqa
    torch.manual_seed(seed)
    search = VqaModel(qst_vocab_size=17858, img_encoder_type="darts", **DIMS).cuda().train()
    torch.manual_seed(seed + 1)
    return derive_vqa(search)


def _batch(B, seed=3):
    g = torch.Generator().manual_seed(seed)
    img = torch.randn(B, 3, 64, 64, generator=g)
    qst = torch.randint(0, 17858, (B, 30), generator=g)
    qst[:, 0] = 2
    return [img.cuda(), qst.cuda(), torch.randint(0, 1000, (B,), generator=g).cuda()]


@pytest.mark.gpu
def test_graphed_train_step_first_replay_equals_eager_gpu():
    import pcd_flat
    from search import GraphedTrainStep, SearchStep
    m = _derived_bench_model()
    m.dropout.p = 0.0
    m.img_encoder.darts.drop_path_prob = 0.2
    m.img_encoder.darts.drop_path_seed = seed_tensor(SEEDS[0], "cuda")
    twin = copy.deepcopy(m)
    batch = _batch(32)
    eager = SearchStep(twin, None, pcd_flat.FlatAdam(twin.parameters(), lr=1e-3))
    loss_e = eager.w_step(*batch)
    graphed = GraphedTrainStep(SearchStep(m, None, pcd_flat.FlatAdam(m.parameters(), lr=1e-3)), batch)
    loss_g = graphed().clone()
    torch.cuda.synchronize()
    assert_close(loss_g, loss_e, 1e-5, "loss")
    for (k, a), b in zip(m.named_buffers(), twin.buffers()):
        if k.endswith("num_batches_tracked"):
            assert int(a) == int(b), k
        else:
            assert_close(a, b, 1e-4, k)
    errs = sorted(rel_err(a, b) for a, b in zip(m.parameters(), twin.parameters()))
    assert errs[len(errs) // 2] <= 1e-6 and errs[-1] <= 1e-3, errs[-5:]


@pytest.mark.gpu
def test_graphed_train_step_reads_seed_and_prob_at_replay_gpu():
    """lr = 0 keeps the weights fixed, so two replays on one batch differ only through the masks."""
    import pcd_flat
    from search import GraphedTrainStep, SearchStep
    m = _derived_bench_model()
    m.dropout.p = 0.0
    net = m.img_encoder.darts
    net.drop_path_prob = 0.3
    batch = _batch(16)
    step = GraphedTrainStep(SearchStep(m, None, pcd_flat.FlatAdam(m.parameters(), lr=0.0)), batch)
    differ = lambda a, b: abs(a - b) > 1e-5 * abs(b)
    l1, l2 = float(step()), float(step())
    assert differ(l1, l2), (l1, l2)          # a drawn seed: new masks on every replay
    net.drop_path_prob = 0.0                 # no re-capture
    l3, l4 = float(step()), float(step())
    assert abs(l3 - l4) <= 1e-6 * abs(l4), (l3, l4)
    with torch.no_grad():
        ref = float(m._loss(*batch))         # eager, p = 0: nothing dropped
    assert abs(l3 - ref) <= 1e-5 * abs(ref), (l3, ref)
    net.drop_path_prob = 0.3
    assert differ(float(step()), l3)


@pytest.mark.gpu
def test_graphed_derived_vqa_trains_at_benchmark_size_gpu():
    import pcd_flat
    from search import GraphedTrainStep, SearchStep
    m = _derived_bench_model()
    m.img_encoder.darts.drop_path_prob = 0.2
    step = GraphedTrainStep(SearchStep(m, None, pcd_flat.FlatAdam(m.parameters(), lr=1e-3)), _batch(128))
    losses = [float(step()) for _ in range(5)]
    assert all(np.isfinite(losses)), losses
    assert all(torch.isfinite(p).all() for p in m.parameters())
