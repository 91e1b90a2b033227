"""Beam-search question decode (pcd_decode_beam, pcd_ops.decode_beam, QstEncoder(beam_size=K)) against the float64 beam search
of beam_oracle.py.  CPU cases run the kernel source's -DPCD_EMU build; `gpu` cases run the sm_100a kernel.

Comparison rule.  fp32 can reorder near-ties, so the search is compared margin-aware.  TAU bounds the fp32 error one step adds
to a cumulative beam score: the score is a running fp32 sum of lambda = logit - lse with |score| < 512 over 30 words, so its
rounding adds at most half an ulp of 256..512 (1.5e-5) per step, and the fp32 logit and log-sum-exp add ~1e-6 per step at
|logit| < 10 (H = 512 terms).  5e-5 covers both with margin; test_beam_decode_production prints the error it measures (on a
B200 at 1000 W: at most 1.9e-6 per step, K in {2, 4, 8}).  After
t + 1 steps two candidate scores can each be off by (t + 1) TAU, so
  - an item whose every decision margin at step t exceeds 2 (t + 1) TAU must come out with the oracle's tokens exactly;
  - otherwise the kernel's best beam, re-scored in float64, must be no worse than T TAU below the oracle's best.
Independently of the search, every returned score must equal the float64 teacher-forced log-probability of its sequence
within T TAU."""
import pytest
import torch

import beam_oracle as BO
import parity_cases as P

TAU = 5e-5


@pytest.fixture(scope="module")
def emulation():
    import pcd_build
    import pcd_native
    pcd_native.enable_emulation(pcd_build.build_emu())
    yield pcd_native._emu_lib
    pcd_native._emu_lib = None


def _modules(B, H, E, V, seed=3):
    """Embedding, LSTM, projection and h0, seeded independently of module init; the projection is scaled so that the logits
    spread over a few units (log-probabilities far from uniform, as in a trained decoder)."""
    g = torch.Generator().manual_seed(seed)
    emb, lstm, proj = torch.nn.Embedding(V, E), torch.nn.LSTM(E, H, 1), torch.nn.Linear(H, V)
    with torch.no_grad():
        for p in list(emb.parameters()) + list(lstm.parameters()) + list(proj.parameters()):
            p.copy_(torch.randn(p.shape, generator=g) * (0.5 if p.dim() > 1 else 0.1) / (p.shape[-1] ** 0.5 if p.dim() > 1 else 1.0))
        emb.weight.mul_(E ** 0.5)
        proj.weight.mul_(6.0)
    h0 = torch.randn(B, H, generator=g) * 0.5
    return emb, lstm, proj, h0


def check_beams(tokens, scores, mods, h0, T, K, items=None):
    """The rules of the module docstring on the items `items` (default: all).  Returns (share of items decided by margins,
    largest per-step score error)."""
    tokens, scores = tokens.cpu(), scores.cpu()
    B = h0.shape[0]
    V = mods[2].out_features
    assert tokens.shape == (B, K, T) and tokens.dtype == torch.long and scores.shape == (B, K) and scores.dtype == torch.float32
    assert int(tokens.min()) >= 0 and int(tokens.max()) < V
    items = torch.arange(B) if items is None else torch.as_tensor(items)
    tokens, scores, h0 = tokens[items], scores[items], h0[items]
    Pm = BO.params64(*mods)
    ref = BO.sequence_logprob(Pm, h0, tokens)
    err = (scores.double() - ref).abs().max().item()
    assert err <= T * TAU, (err, T * TAU)
    assert bool((scores[:, :-1] >= scores[:, 1:]).all()), scores            # best first
    for b in range(len(items)):                                              # distinct paths
        assert len({tuple(x) for x in tokens[b].tolist()}) == K
    o_tok, o_s, margins = BO.beam_search(Pm, h0, T, K)
    clear = (margins > 2 * TAU * torch.arange(1, T + 1, dtype=torch.float64)).all(1)
    for b in range(len(items)):
        if clear[b]:
            assert torch.equal(tokens[b], o_tok[b]), (b, tokens[b], o_tok[b], scores[b], o_s[b])
        else:
            assert ref[b, 0] >= o_s[b, 0] - T * TAU, (b, ref[b, 0], o_s[b, 0])
    return clear.double().mean().item(), err / T


def beam_case(device, B, K, H, E, V, T, seed=3, items=None):
    from pcd_ops import decode_beam
    emb, lstm, proj, h0 = _modules(B, H, E, V, seed)
    mods = [m.to(device) for m in (emb, lstm, proj)]
    tokens, scores = decode_beam(h0.to(device), mods[1], mods[0], mods[2], T, K)
    assert tokens.device.type == torch.device(device).type
    return check_beams(tokens, scores, (emb, lstm, proj), h0, T, K, items), (tokens, scores, mods, h0)


class _Counting:
    """Stands in for one ctypes function of the loaded library: counts the calls and forwards them."""

    def __init__(self, fn):
        self.fn, self.calls = fn, 0

    def __call__(self, *args):
        self.calls += 1
        return self.fn(*args)


# ---- CPU: the emulated kernel source ---------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [1, 2, 4, 8])
@pytest.mark.parametrize("B,H,E,V,T", [(1, 32, 8, 50, 1), (3, 64, 12, 300, 5), (16, 32, 12, 1000, 5), (3, 32, 8, 1000, 30),
                                       (16, 64, 8, 50, 5), (1, 64, 12, 300, 30)])
def test_beam_decode_emulated(emulation, B, H, E, V, T, K):
    """Every value of B in {1, 3, 16}, K in {1, 2, 4, 8}, H in {32, 64}, E in {8, 12}, V in {50, 300, 1000} (one tile, several,
    a partial last tile) and T in {1, 5, 30}; B = 16 with K = 8 is two launches."""
    decided, _ = beam_case("cpu", B, K, H, E, V, T)[0]
    if T <= 5:                                  # short runs: most items are decided by clear margins (the token check bites)
        assert decided >= 0.5, decided


def test_beam_width_one_is_greedy(emulation):
    """K = 1 gives the greedy decode's words wherever the oracle's top-2 gap exceeds rounding (with K = 1 the decision
    margin is the gap between the two best logits)."""
    from pcd_ops import decode_beam, decode_greedy
    B, H, E, V, T = 12, 32, 8, 300, 12
    emb, lstm, proj, h0 = _modules(B, H, E, V, seed=6)
    tokens, _ = decode_beam(h0, lstm, emb, proj, T, 1)
    greedy = decode_greedy(h0, lstm, emb, proj, T)
    _, _, margins = BO.beam_search(BO.params64(emb, lstm, proj), h0, T, 1)
    clear = (margins > 2 * TAU * torch.arange(1, T + 1, dtype=torch.float64)).all(1)
    assert int(clear.sum()) >= B // 2
    assert torch.equal(tokens[clear, 0], greedy[clear])


def test_batch_slicing_does_not_change_the_result(emulation):
    """B = 20 items at K = 4 run as launches of 16 and 4 items; decoding every item on its own gives the same bits."""
    from pcd_ops import decode_beam
    emb, lstm, proj, h0 = _modules(20, 32, 8, 200, seed=4)
    tokens, scores = decode_beam(h0, lstm, emb, proj, 6, 4)
    for b in (0, 15, 16, 19):
        t1, s1 = decode_beam(h0[b:b + 1], lstm, emb, proj, 6, 4)
        assert torch.equal(t1[0], tokens[b]) and torch.equal(s1[0], scores[b])


def test_generate_routes_beam_search_to_the_kernel(emulation, monkeypatch):
    """beam_size = 1 never reaches pcd_decode_beam; beam_size > 1 does (both packages) and returns beam 0 as (B, T)."""
    import models_lct
    import pcd_ops
    import vqa_model
    lib = emulation
    beam, greedy = _Counting(lib.pcd_decode_beam), _Counting(lib.pcd_decode_greedy)
    monkeypatch.setattr(lib, "pcd_decode_beam", beam)
    monkeypatch.setattr(lib, "pcd_decode_greedy", greedy)
    torch.manual_seed(3)
    img = 0.3 * torch.randn(3, 32)
    for mod in (vqa_model, models_lct):
        q = mod.QstEncoder(90, 8, 32, 1, 32, max_length=5)
        assert q.beam_size == 1
        n, g = beam.calls, greedy.calls
        q.generate(img)
        assert beam.calls == n and greedy.calls == g + 1
        q.beam_size = 3
        words = q.generate(img)
        assert beam.calls == n + 1 and greedy.calls == g + 1
        proj = q.fc1 if mod is vqa_model else q.fc2
        tokens, _ = pcd_ops.decode_beam(img, q.lstm, q.word2vec, proj, 5, 3)
        assert words.shape == (3, 5) and words.dtype == torch.long and torch.equal(words, tokens[:, 0])
        q.deterministic = False
        with pytest.raises(ValueError, match="deterministic"):
            q.generate(img)
    positional = vqa_model.QstEncoder(90, 8, 32, 1, 32, True, 0.1, 5, 2)     # the new keyword trails the old ones
    assert positional.max_length == 5 and positional.beam_size == 2
    q48 = vqa_model.QstEncoder(90, 8, 48, 1, 48, max_length=4, beam_size=2)  # H = 48: no stock beam loop, even when allowed
    prev = pcd_ops.allow_stock_ops(True)
    try:
        with pytest.raises(RuntimeError, match="PCD_ERR_UNSUPPORTED"):
            q48.generate(0.3 * torch.randn(2, 48))
    finally:
        pcd_ops.allow_stock_ops(prev)


def test_bad_arguments(emulation):
    from pcd_ops import decode_beam
    emb, lstm, proj, h0 = _modules(2, 32, 8, 6)
    for bad in (0, -1, 9, 7, 2.5, True):                           # 7 > V = 6
        with pytest.raises(ValueError, match="beam_size"):
            decode_beam(h0, lstm, emb, proj, 3, bad)
    lib = emulation
    ops = [emb.weight, lstm.weight_ih_l0, lstm.weight_hh_l0, lstm.bias_ih_l0, lstm.bias_hh_l0, h0, h0, proj.weight, proj.bias]
    ptrs = [t.detach().data_ptr() for t in ops]
    tokens = torch.empty(64 * 3, dtype=torch.long)
    scores = torch.empty(64)
    work = torch.empty(int(lib.pcd_decode_beam_work_floats(8, 8, 32, 6)))

    def call(B=2, K=2, V=6, T=3, start=2, ptrs=ptrs, out=(tokens.data_ptr(), scores.data_ptr(), work.data_ptr())):
        return lib.pcd_decode_beam(T, B, K, 32, 8, V, start, *ptrs, *out, None)

    assert call() == 0
    for kw in (dict(K=0), dict(K=9), dict(K=7), dict(B=9, K=8), dict(B=33, K=2), dict(B=0), dict(T=0), dict(start=6)):
        assert call(**kw) == -2, kw                  # PCD_ERR_UNSUPPORTED
    for i in range(len(ptrs)):
        assert call(ptrs=ptrs[:i] + [None] + ptrs[i + 1:]) == -1, i         # PCD_ERR_ARG
    for i in range(3):
        out = [tokens.data_ptr(), scores.data_ptr(), work.data_ptr()]
        out[i] = None
        assert call(out=tuple(out)) == -1, i


def test_unrolled_twin_keeps_the_beam_width():
    """ArchitectLct generates its pseudo questions with the unrolled twin (model.new()): it must search as wide as the model."""
    ef, _, _ = P.make_lct("cpu")
    ef.qst_encoder.beam_size = 4
    assert ef.new().qst_encoder.beam_size == 4


# ---- GPU --------------------------------------------------------------------------------------------------------------
PROD = dict(H=512, E=300, V=17858, T=30)


@pytest.mark.gpu
@pytest.mark.parametrize("K", [2, 4, 8])
def test_beam_decode_production(K):
    """B = 64 at the benchmark's decoder dimensions (K = 8: eight launches of 8 items = 64 rows, the envelope's edge); the
    float64 oracle runs on 8 of the items to bound its CPU time."""
    (decided, step_err), _ = beam_case("cuda", 64, K, PROD["H"], PROD["E"], PROD["V"], PROD["T"], seed=11,
                                       items=[0, 7, 8, 21, 34, 47, 56, 63])
    print(f"K={K}: {decided:.2f} of the items decided by margins, largest score error per step {step_err:.2e}")


@pytest.mark.gpu
@pytest.mark.parametrize("B,K,H,E,V,T", [(130, 4, 128, 64, 1000, 12), (5, 3, 32, 12, 300, 7), (8, 8, 256, 300, 129, 5)])
def test_beam_decode_shapes(B, K, H, E, V, T):
    """B = 130 at K = 4 is nine launches (16 items each, 2 in the last); V = 1000 and 129 leave a partial last tile (129: one
    column), fewer gate blocks than tiles and the reverse; slicing does not change the bits."""
    from pcd_ops import decode_beam
    (decided, _), (tokens, scores, mods, h0) = beam_case("cuda", B, K, H, E, V, T, seed=12)
    # the exact-token rule must have compared whole items.  How many stay clear of 2 (t + 1) TAU over the run is a property of
    # the seeded data (the float64 oracle's margins), not of the kernel: 57 / 130, 5 / 5 and 4 / 8 for these three cases
    assert round(decided * B) >= min(4, B), decided
    hd = h0.to("cuda")
    for b0 in (0, B - 2):
        t1, s1 = decode_beam(hd[b0:b0 + 2], mods[1], mods[0], mods[2], T, K)
        assert torch.equal(t1, tokens[b0:b0 + 2]) and torch.equal(s1, scores[b0:b0 + 2])


@pytest.mark.gpu
def test_beam_decode_is_deterministic():
    from pcd_ops import decode_beam
    emb, lstm, proj, h0 = _modules(64, PROD["H"], PROD["E"], PROD["V"], seed=13)
    mods = [m.to("cuda") for m in (emb, lstm, proj)]
    hd = h0.to("cuda")
    a = decode_beam(hd, mods[1], mods[0], mods[2], PROD["T"], 4)
    b = decode_beam(hd, mods[1], mods[0], mods[2], PROD["T"], 4)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@pytest.mark.gpu
def test_beam_width_one_against_the_greedy_kernel():
    """K = 1 runs the same fp32 logits as pcd_decode_greedy; the words agree wherever the oracle's top-2 gap exceeds rounding."""
    from pcd_ops import decode_beam, decode_greedy
    B, T = 64, PROD["T"]
    emb, lstm, proj, h0 = _modules(B, PROD["H"], PROD["E"], PROD["V"], seed=14)
    mods = [m.to("cuda") for m in (emb, lstm, proj)]
    hd = h0.to("cuda")
    tokens, _ = decode_beam(hd, mods[1], mods[0], mods[2], T, 1)
    greedy = decode_greedy(hd, mods[1], mods[0], mods[2], T)
    _, _, margins = BO.beam_search(BO.params64(emb, lstm, proj), h0, T, 1)
    clear = (margins > 2 * TAU * torch.arange(1, T + 1, dtype=torch.float64)).all(1)
    assert int(clear.sum()) >= 4             # the comparison covers whole items: 20 of 64 for this seed (oracle margins only)
    assert torch.equal(tokens.cpu()[clear, 0], greedy.cpu()[clear])


@pytest.mark.gpu
def test_misaligned_operand_is_rejected():
    import pcd_native
    lib = pcd_native.load_cuda()
    emb, lstm, proj, h0 = _modules(2, 32, 8, 40)
    ops = [t.detach().to("cuda").contiguous() for t in (emb.weight, lstm.weight_ih_l0, lstm.weight_hh_l0, lstm.bias_ih_l0,
                                                         lstm.bias_hh_l0, h0, h0, proj.weight, proj.bias)]
    tokens = torch.empty(2 * 2 * 3, dtype=torch.long, device="cuda")
    scores = torch.empty(4, device="cuda")
    work = torch.empty(int(lib.pcd_decode_beam_work_floats(2, 2, 32, 40)) + 4, device="cuda")
    ptrs = [t.data_ptr() for t in ops]
    assert lib.pcd_decode_beam(3, 2, 2, 32, 8, 40, 2, *ptrs, tokens.data_ptr(), scores.data_ptr(), work.data_ptr() + 4,
                               None) == -4          # PCD_ERR_ALIGN: nothing launched
    assert lib.pcd_decode_beam(3, 2, 2, 32, 8, 40, 2, *ptrs, tokens.data_ptr(), scores.data_ptr(), work.data_ptr(), None) == 0
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_beam_generate_in_a_cuda_graph():
    """generate() with beam_size = 4 captured in a CUDA graph replays the eager words."""
    import vqa_model
    torch.manual_seed(5)
    q = vqa_model.QstEncoder(500, 12, 64, 1, 64, max_length=6, beam_size=4).cuda()
    img = 0.5 * torch.randn(20, 64, device="cuda")
    eager = q.generate(img)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        q.generate(img)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        words = q.generate(img)
    for _ in range(2):
        words.zero_()
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(words, eager)


@pytest.mark.gpu
def test_graphed_lct_step_with_beam_search(monkeypatch):
    """search.GraphedLctStep with beam_size = 4 on the EF model (and so on its unrolled twin): the three generate() calls of
    ArchitectLct.step run on pcd_decode_beam, the replays give finite losses and the first replay equals the eager step."""
    import math
    import config
    import pcd_native
    from helpers import assert_close
    from search import GraphedLctStep
    monkeypatch.setitem(P.LCT_DIMS, "hidden_size", 32)        # inside the decode envelope (embed = hidden: h0 is the image
    monkeypatch.setitem(P.LCT_DIMS, "embed_size", 32)         # embedding)
    lr0, wd0 = config.ARCH_LEARNING_RATE, config.ARCH_WEIGHT_DECAY
    config.ARCH_LEARNING_RATE, config.ARCH_WEIGHT_DECAY = 0.0, 0.0
    try:
        ef1, _, eager = P.make_lct("cuda")
        ef2, _, arch2 = P.make_lct("cuda")
    finally:
        config.ARCH_LEARNING_RATE, config.ARCH_WEIGHT_DECAY = lr0, wd0
    ef1.qst_encoder.beam_size = ef2.qst_encoder.beam_size = 4
    lib = pcd_native.load_cuda()
    beam, greedy = _Counting(lib.pcd_decode_beam), _Counting(lib.pcd_decode_greedy)
    monkeypatch.setattr(lib, "pcd_decode_beam", beam)
    monkeypatch.setattr(lib, "pcd_decode_greedy", greedy)
    tr, va = P.lct_batch(21, "cuda"), P.lct_batch(22, "cuda")
    graphed = GraphedLctStep(arch2, tr, va, 1e-3, 1e-3, warmup=2)
    assert beam.calls == 3 * 3 and greedy.calls == 0           # two warm-up steps + the captured step
    for _ in range(2):
        eager.step(*tr, *va, 1e-3, 1e-3)
    eager.step(*tr, *va, 1e-3, 1e-3)
    graphed(tr, va)
    torch.cuda.synchronize()
    assert_close(arch2.last["unrolled_loss"], eager.last["unrolled_loss"], 1e-5, "W' validation loss")
    losses = [float(graphed(tr, va)) for _ in range(2)]
    torch.cuda.synchronize()
    assert all(math.isfinite(x) for x in losses), losses
