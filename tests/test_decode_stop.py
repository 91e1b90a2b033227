"""End-of-sequence decoding (pcd_decode with stop = 1, the end_token / pad_token / length_penalty keywords of pcd_ops and
QstEncoder).  CPU cases run the kernel source's -DPCD_EMU build; `gpu` cases run the sm_100a kernel.

Greedy and sampled rows are independent and choose every word as without the stop, so a stopped decode must equal the
unstopped one truncated after the first end word and filled with the pad word, bit for bit.  Beams are compared with the
float64 search of stop_oracle.py under the margin rule of test_decode_beam.py applied to the ranking keys s / L^alpha: the
key of a hypothesis of length L >= 1 carries at most the error of its raw score (alpha >= 0), so the same TAU bounds it."""
import copy
import ctypes

import pytest
import torch

import beam_oracle as BO
import parity_cases as P
import stop_oracle as SO
from pcd_native import DECODE_BEAM, DECODE_GREEDY, DECODE_SAMPLED
from test_decode_beam import PROD, TAU, _Decodes, _decode_args, _modules

END, PAD = 3, 0                  # the vocabulary's <end> and <pad>


@pytest.fixture(scope="module")
def emulation():
    import pcd_build
    import pcd_native
    pcd_native.enable_emulation(pcd_build.build_emu())
    yield pcd_native._emu_lib
    pcd_native._emu_lib = None


def _stop_modules(B, H, E, V, seed=3, end_bias=None, end=END):
    """_modules with the end word's output bias set: rows then end at a spread of lengths (None leaves the bias as drawn)."""
    emb, lstm, proj, h0 = _modules(B, H, E, V, seed)
    if end_bias is not None:
        with torch.no_grad():
            proj.bias[end] = end_bias
    return emb, lstm, proj, h0


def _key32(scores, lengths, alpha):
    """The kernel's fp32 ranking key of each returned beam."""
    return scores / torch.pow(lengths.float(), alpha) if alpha != 0 else scores


def check_stop_beams(tokens, scores, mods, h0, T, K, alpha, end=END, pad=PAD, items=None):
    """The margin rule on keys, the raw scores against the float64 teacher-forced log-probability up to the end word,
    padding after it, distinct paths best first by key.  Returns (share of items decided by margins, beams that finished)."""
    tokens, scores = tokens.cpu(), scores.cpu()
    B = h0.shape[0]
    assert tokens.shape == (B, K, T) and tokens.dtype == torch.long and scores.shape == (B, K) and scores.dtype == torch.float32
    items = torch.arange(B) if items is None else torch.as_tensor(items)
    tokens, scores, h0 = tokens[items], scores[items], h0[items]
    assert torch.equal(tokens, SO.truncate(tokens, end, pad))                 # pad after the first end word
    Pm = BO.params64(*mods)
    ref = SO.sequence_logprob_stop(Pm, h0, tokens, end)
    err = (scores.double() - ref).abs().max().item()
    assert err <= T * TAU, (err, T * TAU)
    lengths = SO.lengths_of(tokens, end)
    keys = _key32(scores, lengths, alpha)
    assert bool((keys[:, :-1] >= keys[:, 1:] - 1e-6 * keys[:, 1:].abs()).all()), keys      # best first by key
    for b in range(len(items)):
        assert len({tuple(x) for x in tokens[b].tolist()}) == K                         # distinct paths
    o_tok, _, o_key, _, margins = SO.beam_search_stop(Pm, h0, T, K, end, pad, alpha)
    clear = (margins > 2 * TAU * torch.arange(1, T + 1, dtype=torch.float64)).all(1)
    ref_key = SO._key(ref, lengths, alpha)
    for b in range(len(items)):
        if clear[b]:
            assert torch.equal(tokens[b], o_tok[b]), (b, tokens[b], o_tok[b], scores[b])
        else:
            assert ref_key[b, 0] >= o_key[b, 0] - T * TAU, (b, ref_key[b, 0], o_key[b, 0])
    return clear.double().mean().item(), int((tokens == end).any(-1).sum())


def _decode_all(device, mods, h0, T, mode, stop, K=4, alpha=0.0, seed=77, pad=PAD):
    from pcd_ops import decode_beam, decode_greedy, decode_sample
    emb, lstm, proj = mods
    kw = dict(end_token=END, pad_token=pad) if stop else {}
    if mode == "greedy":
        return decode_greedy(h0, lstm, emb, proj, T, **kw)
    if mode == "sampled":
        return decode_sample(h0, lstm, emb, proj, T, 0.7, seed=seed, **kw)
    if stop:
        kw["length_penalty"] = alpha
    return decode_beam(h0, lstm, emb, proj, T, K, **kw)


# ---- CPU: the emulated kernel source ---------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["greedy", "sampled"])
@pytest.mark.parametrize("B,H,E,V,T,end_bias,pad", [(6, 32, 8, 50, 12, 1.0, 0), (3, 64, 12, 300, 20, 2.0, 1),
                                                    (16, 32, 12, 1000, 9, 2.5, 0), (70, 32, 8, 40, 6, 0.5, 7)])
def test_stopped_equals_truncated_emulated(emulation, mode, B, H, E, V, T, end_bias, pad):
    """B = 70 is two launches; the end bias spreads the rows' lengths."""
    mods = _stop_modules(B, H, E, V, seed=5, end_bias=end_bias)
    h0 = mods[3]
    full = _decode_all("cpu", mods[:3], h0, T, mode, False)
    stopped = _decode_all("cpu", mods[:3], h0, T, mode, True, pad=pad)
    assert torch.equal(stopped, SO.truncate(full, END, pad))
    ended = (full == END).any(1)
    assert 0 < int(ended.sum()), "no row emitted the end word: the case does not test the stop"


@pytest.mark.parametrize("mode", ["greedy", "sampled", "beam"])
def test_end_never_emitted_is_bit_equal_emulated(emulation, mode):
    """An end word whose logit is far below the rest is never chosen: every mode equals its call without the stop (beams at
    alpha = 0)."""
    emb, lstm, proj, h0 = _stop_modules(9, 32, 8, 300, seed=6, end_bias=-1e4)
    a = _decode_all("cpu", (emb, lstm, proj), h0, 10, mode, False)
    b = _decode_all("cpu", (emb, lstm, proj), h0, 10, mode, True)
    if mode == "beam":
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    else:
        assert torch.equal(a, b)


@pytest.mark.parametrize("alpha", [0.0, 0.7, 1.0])
@pytest.mark.parametrize("B,K,H,E,V,T", [(3, 4, 32, 8, 300, 12), (8, 2, 64, 12, 50, 20), (16, 8, 32, 12, 1000, 8)])
def test_beam_stop_emulated(emulation, alpha, B, K, H, E, V, T):
    from pcd_ops import decode_beam
    emb, lstm, proj, h0 = _stop_modules(B, H, E, V, seed=7, end_bias=2.0)
    tokens, scores = decode_beam(h0, lstm, emb, proj, T, K, end_token=END, pad_token=PAD, length_penalty=alpha)
    decided, finished = check_stop_beams(tokens, scores, (emb, lstm, proj), h0, T, K, alpha)
    assert finished > 0
    assert round(decided * B) >= min(2, B), decided


def test_every_row_ends_at_step_zero_emulated(emulation):
    """An end word made certain by its bias: greedy and sampled rows are [E, P, P, ...]; the best beam too, and the other
    beams end one step later (the kernel leaves its loop after two steps)."""
    from pcd_ops import decode_beam
    emb, lstm, proj, h0 = _stop_modules(5, 32, 8, 60, seed=8, end_bias=50.0)
    row = torch.tensor([END] + [PAD] * 7)
    for mode in ("greedy", "sampled"):
        assert torch.equal(_decode_all("cpu", (emb, lstm, proj), h0, 8, mode, True), row.expand(5, 8))
    tokens, scores = decode_beam(h0, lstm, emb, proj, 8, 3, end_token=END, pad_token=PAD, length_penalty=0.5)
    assert torch.equal(tokens[:, 0], row.expand(5, 8))
    assert bool((tokens[:, 1:, 1] == END).all()) and bool((tokens[:, 1:, 2:] == PAD).all())
    check_stop_beams(tokens, scores, (emb, lstm, proj), h0, 8, 3, 0.5)


def test_batch_slicing_does_not_change_the_result(emulation):
    """B = 20 items at K = 4 run as launches of 16 and 4 items; decoding items on their own gives the same bits."""
    from pcd_ops import decode_beam
    emb, lstm, proj, h0 = _stop_modules(20, 32, 8, 200, seed=4, end_bias=2.0)
    tokens, scores = decode_beam(h0, lstm, emb, proj, 10, 4, end_token=END, length_penalty=0.7)
    assert int((tokens == END).sum()) > 0
    for b in (0, 15, 16, 19):
        t1, s1 = decode_beam(h0[b:b + 1], lstm, emb, proj, 10, 4, end_token=END, length_penalty=0.7)
        assert torch.equal(t1[0], tokens[b]) and torch.equal(s1[0], scores[b])


def test_generate_routes_to_the_stop_mode(emulation, monkeypatch):
    """end_token=None decodes without the stop; a set end_token decodes with it (both packages, all three modes)."""
    import models_lct
    import pcd_ops
    import vqa_model
    lib = emulation
    rec = _Decodes(lib.pcd_decode)
    monkeypatch.setattr(lib, "pcd_decode", rec)
    calls = lambda: tuple(rec.count(mode, stop) for stop in (0, 1) for mode in (DECODE_GREEDY, DECODE_SAMPLED, DECODE_BEAM))
    torch.manual_seed(3)
    img = 0.3 * torch.randn(3, 32)
    for mod in (vqa_model, models_lct):
        q = mod.QstEncoder(90, 8, 32, 1, 32, max_length=5)
        assert q.end_token is None and q.length_penalty == 0.0
        proj = q.fc1 if mod is vqa_model else q.fc2
        for det, beam, i in ((True, 1, 0), (False, 1, 1), (True, 3, 2)):
            q.deterministic, q.beam_size, q.end_token, q.length_penalty = det, beam, None, 0.0
            n = calls()
            q.generate(img)
            assert calls() == tuple(c + (j == i) for j, c in enumerate(n)), (det, beam)
            q.end_token, q.length_penalty = END, 0.5
            n = calls()
            words = q.generate(img)
            assert calls() == tuple(c + (j == i + 3) for j, c in enumerate(n)), (det, beam)
            assert words.shape == (3, 5) and words.dtype == torch.long
            if det and beam == 1:
                assert torch.equal(words, pcd_ops.decode_greedy(img, q.lstm, q.word2vec, proj, 5, end_token=END))
            if beam > 1:
                tokens, _ = pcd_ops.decode_beam(img, q.lstm, q.word2vec, proj, 5, 3, end_token=END, length_penalty=0.5)
                assert torch.equal(words, tokens[:, 0])
    positional = vqa_model.QstEncoder(90, 8, 32, 1, 32, True, 0.1, 5, 2, 3, 0.6)     # the new keywords trail the old ones
    assert positional.beam_size == 2 and positional.end_token == 3 and positional.length_penalty == 0.6


def test_outside_the_envelope_raises_even_with_stock_ops(emulation):
    """H = 48: no stock loop decodes with an end word, whatever the mode."""
    import models_lct
    import vqa_model
    prev = __import__("pcd_ops").allow_stock_ops(True)
    try:
        for mod in (vqa_model, models_lct):
            for det, beam in ((True, 1), (False, 1), (True, 2)):
                q = mod.QstEncoder(90, 8, 48, 1, 48, deterministic=det, max_length=4, beam_size=beam, end_token=END)
                with pytest.raises(RuntimeError, match="PCD_ERR_UNSUPPORTED"):
                    q.generate(0.3 * torch.randn(2, 48))
    finally:
        __import__("pcd_ops").allow_stock_ops(prev)


def test_bad_stop_arguments(emulation):
    from pcd_ops import decode_beam, decode_greedy, decode_sample
    import pcd_native
    emb, lstm, proj, h0 = _modules(2, 32, 8, 6)
    for kw in (dict(end_token=6), dict(end_token=-1), dict(end_token=2.5), dict(end_token=True), dict(end_token=3, pad_token=6),
               dict(end_token=3, pad_token=-1)):
        with pytest.raises(ValueError, match="_token"):
            decode_greedy(h0, lstm, emb, proj, 3, **kw)
        with pytest.raises(ValueError, match="_token"):
            decode_sample(h0, lstm, emb, proj, 3, 1.0, **kw)
        with pytest.raises(ValueError, match="_token"):
            decode_beam(h0, lstm, emb, proj, 3, 2, **kw)
    for alpha in (float("nan"), float("inf"), 1e39):
        with pytest.raises(ValueError, match="length_penalty"):
            decode_beam(h0, lstm, emb, proj, 3, 2, end_token=3, length_penalty=alpha)
        # without end_token every hypothesis has max_length words: the penalty is not used, so it is not checked either
        assert torch.equal(decode_beam(h0, lstm, emb, proj, 3, 2, length_penalty=alpha)[0], decode_beam(h0, lstm, emb, proj, 3, 2)[0])
    lib = emulation
    ops = [emb.weight, lstm.weight_ih_l0, lstm.weight_hh_l0, lstm.bias_ih_l0, lstm.bias_hh_l0, h0, h0, proj.weight, proj.bias]
    ptrs = [t.detach().data_ptr() for t in ops]
    tokens = torch.empty(64 * 3, dtype=torch.long)
    scores = torch.empty(64)
    work = torch.empty(int(lib.pcd_decode_work_floats(ctypes.byref(pcd_native.DecodeArgs(mode=DECODE_BEAM, B=8, K=8, H=32,
                                                                                          V=6)))))
    seed = torch.tensor([5], dtype=torch.int64)

    def calls(stop):
        """the three modes with the stop (end_token, pad_token, length_penalty); None: a null pcd_decode_args"""
        if stop is None:
            return (lib.pcd_decode(None, None),) * 3
        end, pad, alpha = stop
        common = dict(T=3, H=32, E=8, V=6, start_token=2, stop=1, end_token=end, pad_token=pad, length_penalty=alpha,
                      tokens=tokens.data_ptr(), work=work.data_ptr())
        return tuple(lib.pcd_decode(ctypes.byref(_decode_args(ptrs, **common, **kw)), None) for kw in (
            dict(mode=DECODE_GREEDY, B=2, K=1),
            dict(mode=DECODE_SAMPLED, B=2, K=1, temperature=1.0, seed=seed.data_ptr()),
            dict(mode=DECODE_BEAM, B=2, K=2, scores=scores.data_ptr())))

    assert calls((3, 0, 0.5)) == (0, 0, 0)
    for bad in (None, (6, 0, 0.0), (-1, 0, 0.0), (3, 6, 0.0), (3, -1, 0.0), (3, 0, float("nan")), (3, 0, float("inf"))):
        assert calls(bad) == (-1, -1, -1), bad                       # PCD_ERR_ARG


def test_unrolled_twin_keeps_the_stop():
    """ArchitectLct generates its pseudo questions with the unrolled twin (model.new()): it must stop as the model does."""
    ef, _, _ = P.make_lct("cpu")
    ef.qst_encoder.end_token, ef.qst_encoder.length_penalty = END, 0.7
    twin = ef.new().qst_encoder
    assert twin.end_token == END and twin.length_penalty == 0.7


# ---- GPU --------------------------------------------------------------------------------------------------------------
def _prod(seed, end_bias, B=64):
    emb, lstm, proj, h0 = _stop_modules(B, PROD["H"], PROD["E"], PROD["V"], seed=seed, end_bias=end_bias)
    return (emb, lstm, proj), h0, [m.to("cuda") for m in (emb, lstm, proj)], h0.to("cuda")


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["greedy", "sampled"])
def test_stopped_equals_truncated_production(mode):
    """B = 64 at the benchmark's decoder dimensions: the stopped kernel equals the unstopped kernel truncated, bit for bit."""
    _, _, mods, hd = _prod(21, 3.0)
    full = _decode_all("cuda", mods, hd, PROD["T"], mode, False).cpu()
    stopped = _decode_all("cuda", mods, hd, PROD["T"], mode, True).cpu()
    assert torch.equal(stopped, SO.truncate(full, END, PAD))
    ended = (full == END).any(1)
    print(f"{mode}: {int(ended.sum())} of 64 rows ended, lengths {sorted(SO.lengths_of(full, END).tolist())}")
    assert 0 < int(ended.sum())


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["greedy", "sampled", "beam"])
def test_end_never_emitted_is_bit_equal_production(mode):
    _, _, mods, hd = _prod(22, -1e4)
    a = _decode_all("cuda", mods, hd, PROD["T"], mode, False)
    b = _decode_all("cuda", mods, hd, PROD["T"], mode, True)
    if mode == "beam":
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    else:
        assert torch.equal(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("alpha", [0.0, 0.7, 1.0])
def test_beam_stop_production(alpha):
    """K = 4, B = 64 items (four launches); the float64 oracle runs on 8 of them; a rerun gives the same bits."""
    from pcd_ops import decode_beam
    cpu_mods, h0, mods, hd = _prod(23, 3.0)
    tokens, scores = decode_beam(hd, mods[1], mods[0], mods[2], PROD["T"], 4, end_token=END, length_penalty=alpha)
    again = decode_beam(hd, mods[1], mods[0], mods[2], PROD["T"], 4, end_token=END, length_penalty=alpha)
    assert torch.equal(tokens, again[0]) and torch.equal(scores, again[1])
    decided, finished = check_stop_beams(tokens, scores, cpu_mods, h0, PROD["T"], 4, alpha,
                                         items=[0, 7, 8, 21, 34, 47, 56, 63])
    print(f"alpha={alpha}: {decided:.2f} of the items decided by margins, {finished} of 32 beams finished")
    assert finished > 0


@pytest.mark.gpu
def test_slicing_at_b130():
    """B = 130: greedy in launches of 64, 64 and 2 rows, beams (K = 4) in nine launches; slices decoded alone agree."""
    from pcd_ops import decode_beam, decode_greedy
    _, _, mods, hd = _stop_modules_cuda(130)
    g = decode_greedy(hd, mods[1], mods[0], mods[2], 12, end_token=END)
    t, s = decode_beam(hd, mods[1], mods[0], mods[2], 12, 4, end_token=END, length_penalty=0.7)
    assert int((g == END).sum()) > 0 and int((t == END).sum()) > 0
    for b0 in (0, 63, 128):
        g1 = decode_greedy(hd[b0:b0 + 2], mods[1], mods[0], mods[2], 12, end_token=END)
        t1, s1 = decode_beam(hd[b0:b0 + 2], mods[1], mods[0], mods[2], 12, 4, end_token=END, length_penalty=0.7)
        assert torch.equal(g1, g[b0:b0 + 2]) and torch.equal(t1, t[b0:b0 + 2]) and torch.equal(s1, s[b0:b0 + 2])


def _stop_modules_cuda(B):
    emb, lstm, proj, h0 = _stop_modules(B, 128, 64, 1000, seed=24, end_bias=2.5)
    return (emb, lstm, proj), h0, [m.to("cuda") for m in (emb, lstm, proj)], h0.to("cuda")


@pytest.mark.gpu
def test_early_exit_production():
    """The end word made certain by its bias: every row finishes at step 0 (beams: the best at step 0, the rest at step 1),
    the kernel leaves its loop and the remaining positions are the pad word."""
    from pcd_ops import decode_beam
    cpu_mods, h0, mods, hd = _prod(25, 50.0)
    row = torch.tensor([END] + [PAD] * (PROD["T"] - 1))
    for mode in ("greedy", "sampled"):
        assert torch.equal(_decode_all("cuda", mods, hd, PROD["T"], mode, True).cpu(), row.expand(64, -1))
    tokens, scores = decode_beam(hd, mods[1], mods[0], mods[2], PROD["T"], 4, end_token=END, length_penalty=0.5)
    tokens = tokens.cpu()
    assert torch.equal(tokens[:, 0], row.expand(64, -1))
    assert bool((tokens[:, 1:, 1] == END).all()) and bool((tokens[:, 1:, 2:] == PAD).all())
    check_stop_beams(tokens, scores, cpu_mods, h0, PROD["T"], 4, 0.5, items=[0, 31, 63])


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["greedy", "beam"])
def test_early_exit_leaves_the_time_loop(mode):
    """The same stopped call on two end biases: +50 ends every row at step 0 (beams: all beams by step 1), -1e4 never lets the
    end word be chosen.  Both write the same number of padded columns, so only the early exit can make the first much faster:
    it runs 1 (beams: 2) of the 30 steps, the second all 30.  The bound 0.5 leaves room for launch overheads."""
    cpu_mods, _, mods, hd = _prod(26, 50.0, B=64 if mode == "greedy" else 16)
    proj_never = copy.deepcopy(mods[2])
    with torch.no_grad():
        proj_never.bias[END] = -1e4

    def run(proj):
        if mode == "greedy":
            return _decode_all("cuda", (mods[0], mods[1], proj), hd, PROD["T"], "greedy", True)
        return _decode_all("cuda", (mods[0], mods[1], proj), hd, PROD["T"], "beam", True, K=4)

    def ms(proj, n=10):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            run(proj)
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / n

    for p in (mods[2], proj_never):
        run(p)
    torch.cuda.synchronize()
    early = min(ms(mods[2]) for _ in range(3))
    full = min(ms(proj_never) for _ in range(3))
    print(f"{mode}: {early:.3f} ms with every row ended at step 0, {full:.3f} ms with none ending")
    assert early < 0.5 * full, (early, full)


@pytest.mark.gpu
@pytest.mark.parametrize("beam_size,deterministic", [(1, True), (1, False), (4, True)])
def test_stop_generate_in_a_cuda_graph(beam_size, deterministic):
    """generate() with end_token captured in a CUDA graph replays the eager words (sampled: with a fixed seed the replay
    draws a fresh seed, so it is checked for the stop rule only)."""
    import vqa_model
    torch.manual_seed(5)
    q = vqa_model.QstEncoder(500, 12, 64, 1, 64, deterministic=deterministic, max_length=12, beam_size=beam_size,
                             end_token=END, length_penalty=0.7).cuda()
    with torch.no_grad():
        q.fc1.bias[END] = 2.5
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
        w = words.cpu()
        assert torch.equal(w, SO.truncate(w, END, PAD)) and int((w == END).sum()) > 0
        if deterministic:
            assert torch.equal(words, eager)


@pytest.mark.gpu
def test_graphed_lct_step_decodes_beams_with_the_stop(monkeypatch):
    """search.GraphedLctStep with end_token = 3 and beam_size = 4 on the EF model and its unrolled twin: the three generate()
    calls of ArchitectLct.step run on pcd_decode in beam mode with the stop, the replays give finite losses and the first
    equals the eager step."""
    import math
    import config
    import pcd_native
    from helpers import assert_close
    from search import GraphedLctStep
    monkeypatch.setitem(P.LCT_DIMS, "hidden_size", 32)
    monkeypatch.setitem(P.LCT_DIMS, "embed_size", 32)
    lr0, wd0 = config.ARCH_LEARNING_RATE, config.ARCH_WEIGHT_DECAY
    config.ARCH_LEARNING_RATE, config.ARCH_WEIGHT_DECAY = 0.0, 0.0
    try:
        ef1, _, eager = P.make_lct("cuda")
        ef2, _, arch2 = P.make_lct("cuda")
    finally:
        config.ARCH_LEARNING_RATE, config.ARCH_WEIGHT_DECAY = lr0, wd0
    for ef in (ef1, ef2):
        ef.qst_encoder.beam_size, ef.qst_encoder.end_token, ef.qst_encoder.length_penalty = 4, END, 0.7
    lib = pcd_native.load_cuda()
    rec = _Decodes(lib.pcd_decode)
    monkeypatch.setattr(lib, "pcd_decode", rec)
    tr, va = P.lct_batch(21, "cuda"), P.lct_batch(22, "cuda")
    graphed = GraphedLctStep(arch2, tr, va, 1e-3, 1e-3, warmup=2)
    assert rec.count(DECODE_BEAM, 1) == 3 * 3 and len(rec.seen) == 3 * 3       # two warm-up steps + the captured step
    for _ in range(2):
        eager.step(*tr, *va, 1e-3, 1e-3)
    eager.step(*tr, *va, 1e-3, 1e-3)
    graphed(tr, va)
    torch.cuda.synchronize()
    assert_close(arch2.last["unrolled_loss"], eager.last["unrolled_loss"], 1e-5, "W' validation loss")
    losses = [float(graphed(tr, va)) for _ in range(2)]
    torch.cuda.synchronize()
    assert all(math.isfinite(x) for x in losses), losses
