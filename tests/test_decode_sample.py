"""Sampled question decode (QstEncoder.generate with deterministic=False) on the persistent decode kernel: Gumbel-max over
Philox noise (pcd_decode in sampled mode) against the float64 restatement in sample_oracle.py.  CPU cases run the kernel
source's -DPCD_EMU build; `gpu` cases run the sm_100a kernel."""
import ctypes
import math

import numpy as np
import pytest
import torch

import parity_cases as P
import sample_oracle as S
from pcd_native import DECODE_GREEDY, DECODE_SAMPLED, DecodeArgs
from test_decode_beam import _Decodes, _decode_args

SEED = 0x0123456789ABCDEF         # both key words non-zero


@pytest.fixture(scope="module")
def emulation():
    import pcd_build
    import pcd_native
    pcd_native.enable_emulation(pcd_build.build_emu())
    yield pcd_native._emu_lib
    pcd_native._emu_lib = None


def _modules(B, H, E, V, seed=3, same_h0=False):
    """Embedding, LSTM, projection and h0 filled as in parity_cases.decode_case (seeded, independent of module init)."""
    g = torch.Generator().manual_seed(seed)
    emb, lstm, proj = torch.nn.Embedding(V, E), torch.nn.LSTM(E, H, 1), torch.nn.Linear(H, V)
    with torch.no_grad():
        for p in list(emb.parameters()) + list(lstm.parameters()) + list(proj.parameters()):
            p.copy_(torch.randn(p.shape, generator=g) * (0.5 if p.dim() > 1 else 0.1) / (p.shape[-1] ** 0.5 if p.dim() > 1 else 1.0))
        emb.weight.mul_(E ** 0.5)
    h0 = torch.randn(1 if same_h0 else B, H, generator=g) * 0.5
    return emb, lstm, proj, h0.expand(B, H).contiguous()


def _oracle(emb, lstm, proj, h0, T, temperature, seed, force=None, row_offset=0):
    d = lambda t: t.detach().cpu().double().numpy()
    return S.decode_sampled(d(emb.weight), d(lstm.weight_ih_l0), d(lstm.weight_hh_l0), d(lstm.bias_ih_l0), d(lstm.bias_hh_l0),
                            d(proj.weight), d(proj.bias), d(h0), T, temperature, seed, start_token=2, row_offset=row_offset,
                            force=force)


def check_against_oracle(tokens, mods, h0, T, temperature, seed):
    """The kernel's words, teacher-forced through the float64 oracle: every word must be a best score up to fp32 rounding
    (scores are logit / T + G, so the bound scales with the largest score), and >= 98 % must be THE best."""
    tokens = tokens.cpu().numpy()
    B = h0.shape[0]
    assert tokens.shape == (B, T) and tokens.min() >= 0 and tokens.max() < mods[2].out_features
    _, scores = _oracle(*mods, h0, T, temperature, seed, force=tokens)
    exact = 0
    for t in range(T):
        top = scores[t].max(1)
        mine = scores[t][np.arange(B), tokens[:, t]]
        scale = np.abs(scores[t]).max()
        assert (top - mine).max() <= 2e-5 * scale, (t, (top - mine).max(), scale)
        exact += int((scores[t].argmax(1) == tokens[:, t]).sum())
    assert exact >= 0.98 * B * T, (exact, B * T)
    return exact / (B * T)


def sample_case(device, B, H, E, V, T, temperature, seed=SEED):
    from pcd_ops import decode_sample, decode_supported
    emb, lstm, proj, h0 = _modules(B, H, E, V)
    mods = [m.to(device) for m in (emb, lstm, proj)]
    assert decode_supported(h0.to(device), mods[1], mods[0], mods[2])
    tokens = decode_sample(h0.to(device), mods[1], mods[0], mods[2], T, temperature, start_token=2, seed=seed)
    assert tokens.dtype == torch.long and tokens.device.type == torch.device(device).type
    return check_against_oracle(tokens, (emb, lstm, proj), h0, T, temperature, seed)


# ---- CPU: the oracle's noise ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("counter,key,expect", [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0), (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))])
def test_philox_known_answers(counter, key, expect):
    """The Random123 known-answer vectors of Philox4x32-10."""
    assert tuple(int(w) for w in S.philox4x32_10(counter, key)) == expect


def test_gumbel_is_finite_at_the_extreme_bits():
    u = S.uniform_of_bits([0, 0xFFFFFFFF])
    assert u[0] == np.float32(2.0 ** -24) and u[1] == np.float32(1 - 2.0 ** -24)
    for dt in (np.float32, np.float64):
        G = S.gumbel_of_bits([0, 0xFFFFFFFF], dt)
        assert np.isfinite(G).all() and -2.82 < G[0] < -2.81 and 16.6 < G[1] < 16.7


# ---- CPU: the emulated kernel source -------------------------------------------------------------------------------
@pytest.mark.parametrize("temperature", [1.0, 0.1])
@pytest.mark.parametrize("B,H,E,V,T", [(5, 32, 12, 300, 7), (3, 64, 8, 128, 4), (70, 32, 8, 50, 3)])
def test_sampled_decode_emulated(emulation, B, H, E, V, T, temperature):
    """Argument marshalling, noise indexing (t, global row, v) and the temperature on the emulation build; B = 70 is decoded
    as two slices, the second with row_offset 64."""
    sample_case("cpu", B, H, E, V, T, temperature)


def test_seed_fixes_the_words(emulation):
    from pcd_ops import decode_sample
    emb, lstm, proj, h0 = _modules(16, 32, 8, 200)
    a = decode_sample(h0, lstm, emb, proj, 6, 1.0, seed=11)
    assert torch.equal(a, decode_sample(h0, lstm, emb, proj, 6, 1.0, seed=11))
    assert torch.equal(a, decode_sample(h0, lstm, emb, proj, 6, 1.0, seed=torch.tensor([11])))
    assert not torch.equal(a, decode_sample(h0, lstm, emb, proj, 6, 1.0, seed=12))
    torch.manual_seed(4)
    b = decode_sample(h0, lstm, emb, proj, 6, 1.0)
    torch.manual_seed(4)
    assert torch.equal(b, decode_sample(h0, lstm, emb, proj, 6, 1.0))       # seed=None: torch's generator


def test_generate_routes_sampling_to_the_sampled_mode(emulation, monkeypatch):
    """deterministic=False inside the envelope goes through the sampled mode of pcd_decode (both packages); deterministic=None
    with an overridden sample() (the stock-loop reference arm of the timing tools and GPU tests) and H outside the envelope
    do not."""
    import models_lct
    import vqa_model
    lib = emulation
    rec = _Decodes(lib.pcd_decode)
    monkeypatch.setattr(lib, "pcd_decode", rec)
    sample, greedy = lambda: rec.count(DECODE_SAMPLED), lambda: rec.count(DECODE_GREEDY)
    torch.manual_seed(3)
    img = 0.3 * torch.randn(3, 32)
    for mod in (vqa_model, models_lct):
        q = mod.QstEncoder(90, 8, 32, 1, 32, deterministic=False, temperature=0.5, max_length=5)
        n = sample()
        words = q.generate(img)
        assert sample() == n + 1 and greedy() == 0
        assert words.shape == (3, 5) and words.dtype == torch.long and 0 <= int(words.min()) and int(words.max()) < 90
        q.deterministic = None
        q.sample = lambda prob: torch.argmax(prob, 2)
        assert q.generate(img).shape == (3, 5)
        assert sample() == n + 1 and greedy() == 0
    q48 = vqa_model.QstEncoder(90, 8, 48, 1, 48, deterministic=False, max_length=4)     # H = 48: stock loop, no raise
    assert q48.generate(0.3 * torch.randn(2, 48)).shape == (2, 4)
    assert sample() == 2


def test_sampled_generate_matches_the_oracle_with_the_drawn_seed(emulation):
    """generate() draws its seed from torch's generator; the words are the oracle's for the seed that was drawn."""
    import vqa_model
    torch.manual_seed(9)
    q = vqa_model.QstEncoder(120, 8, 32, 1, 32, deterministic=False, temperature=0.7, max_length=4)
    img = 0.5 * torch.randn(4, 32)
    state = torch.get_rng_state()
    words = q.generate(img)
    torch.set_rng_state(state)
    seed = int(torch.empty(1, dtype=torch.int64).random_(-2 ** 63, None))
    check_against_oracle(words, (q.word2vec, q.lstm, q.fc1), img, 4, 0.7, seed)


def test_bad_temperature_and_decode_args(emulation):
    from pcd_ops import decode_sample
    emb, lstm, proj, h0 = _modules(2, 32, 8, 40)
    for bad in (0.0, -1.0, float("nan"), float("inf"), 1e-50):
        with pytest.raises(ValueError, match="temperature"):
            decode_sample(h0, lstm, emb, proj, 3, bad, seed=1)
    lib = emulation
    seed = torch.tensor([1])
    ops = [emb.weight, lstm.weight_ih_l0, lstm.weight_hh_l0, lstm.bias_ih_l0, lstm.bias_hh_l0, h0, h0, proj.weight, proj.bias]
    ptrs = [t.detach().data_ptr() for t in ops]
    tokens = torch.empty(2, 3, dtype=torch.long)
    work = torch.empty(int(lib.pcd_decode_work_floats(ctypes.byref(DecodeArgs(mode=DECODE_SAMPLED, B=2, K=1, H=32, V=40)))))

    def call(row_offset=0, temperature=1.0, seed_ptr=seed.data_ptr(), T=3, K=1):
        a = _decode_args(ptrs, mode=DECODE_SAMPLED, T=T, B=2, K=K, H=32, E=8, V=40, start_token=2, row_offset=row_offset,
                         temperature=temperature, seed=seed_ptr, tokens=tokens.data_ptr(), work=work.data_ptr())
        return lib.pcd_decode(ctypes.byref(a), None)

    assert call() == 0
    for kw in (dict(temperature=0.0), dict(temperature=-2.0), dict(temperature=float("nan")), dict(temperature=float("inf")),
               dict(seed_ptr=None), dict(row_offset=-1), dict(K=2)):
        assert call(**kw) == -1, kw                  # PCD_ERR_ARG
        assert call(T=0, **kw) == -1, kw             # before the shape check
    assert call(T=0) == -2                           # PCD_ERR_UNSUPPORTED


def test_unrolled_twin_keeps_the_sampling_configuration():
    """ArchitectLct generates its pseudo questions with the unrolled twin (model.new()): it must decode like the model."""
    ef, _, _ = P.make_lct("cpu")
    ef.qst_encoder.deterministic, ef.qst_encoder.temperature = False, 0.25
    twin = ef.new()
    assert twin.qst_encoder.deterministic is False and twin.qst_encoder.temperature == 0.25
    assert ef.new().qst_encoder.max_length == ef.qst_encoder.max_length


# ---- GPU --------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("B,H,E,V,T,temperature", [(64, 512, 300, 17858, 30, 0.1), (5, 32, 12, 300, 7, 0.1),
                                                   (37, 128, 64, 1000, 12, 0.1), (64, 256, 300, 129, 5, 0.1),
                                                   (130, 512, 300, 17858, 6, 0.1), (37, 128, 64, 1000, 12, 1.0)])
def test_sampled_decode(B, H, E, V, T, temperature):
    """Production size first; ragged vocabulary tiles, partial batches, fewer gate blocks than vocabulary tiles and the
    reverse; B = 130 is three slices (row offsets 64 and 128)."""
    sample_case("cuda", B, H, E, V, T, temperature)


@pytest.mark.gpu
@pytest.mark.parametrize("temperature", [1.0, 0.1])
def test_sampled_words_follow_the_softmax(temperature):
    """One step, 64 identical rows x 100 fixed seeds = 6400 draws of the first word, against softmax(logits / T) of the
    float64 oracle: chi-square with bins of expected count < 5 pooled."""
    from scipy.stats import chi2
    from pcd_ops import decode_sample
    B, H, E, V = 64, 64, 12, 300
    emb, lstm, proj, h0 = _modules(B, H, E, V, seed=8, same_h0=True)
    mods = [m.to("cuda") for m in (emb, lstm, proj)]
    hd = h0.to("cuda")
    draws = torch.cat([decode_sample(hd, mods[1], mods[0], mods[2], 1, temperature, seed=1000 + s)[:, 0] for s in range(100)])
    counts = np.bincount(draws.cpu().numpy(), minlength=V).astype(np.float64)
    if temperature == 1.0:
        first = decode_sample(hd, mods[1], mods[0], mods[2], 1, 1.0, seed=1000)[:, 0]
        assert len(set(first.tolist())) > 1               # identical rows draw independently within one call
    _, scores = _oracle(emb, lstm, proj, h0[:1], 1, temperature, 0)
    logits = (scores[0, 0] - S.gumbel_noise(0, 0, [0], V)[0]) * temperature
    p = np.exp(logits / temperature - (logits / temperature).max())
    expected = p / p.sum() * len(draws)
    order = np.argsort(expected)
    obs, exp, acc_o, acc_e = [], [], 0.0, 0.0
    for i in order:                                       # pool the rarest words until each bin expects >= 5
        acc_o += counts[i]
        acc_e += expected[i]
        if acc_e >= 5:
            obs.append(acc_o); exp.append(acc_e); acc_o = acc_e = 0.0
    if acc_e > 0:
        obs[-1] += acc_o; exp[-1] += acc_e
    obs, exp = np.array(obs), np.array(exp)
    stat = ((obs - exp) ** 2 / exp).sum()
    pval = chi2.sf(stat, len(obs) - 1)
    print(f"T={temperature}: {len(obs)} bins, chi2 {stat:.1f}, p {pval:.3g}")
    assert len(obs) >= 2 and pval > 1e-4


@pytest.mark.gpu
def test_sampled_decode_in_a_cuda_graph():
    """A captured seed draw + decode_sample(seed=that buffer): each replay samples with the seed it drew."""
    from pcd_ops import decode_sample
    B, H, E, V, T = 16, 64, 12, 500, 6
    emb, lstm, proj, h0 = _modules(B, H, E, V, seed=5)
    mods = [m.to("cuda") for m in (emb, lstm, proj)]
    hd = h0.to("cuda")
    seed = torch.zeros(1, dtype=torch.int64, device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        decode_sample(hd, mods[1], mods[0], mods[2], T, 1.0, seed=seed)          # warm-up (kernel attributes) outside capture
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        seed.random_(-2 ** 63, None)
        tokens = decode_sample(hd, mods[1], mods[0], mods[2], T, 1.0, seed=seed)
    runs = []
    for _ in range(2):
        graph.replay()
        torch.cuda.synchronize()
        runs.append((int(seed.item()), tokens.clone()))
    assert runs[0][0] != runs[1][0] and not torch.equal(runs[0][1], runs[1][1])
    for sd, tok in runs:
        check_against_oracle(tok, (emb, lstm, proj), h0, T, 1.0, sd)


@pytest.mark.gpu
def test_graphed_lct_step_decodes_in_sampled_mode(monkeypatch):
    """search.GraphedLctStep with a sampling EF model: the three generate() calls of ArchitectLct.step run on
    the sampled mode of pcd_decode (counted while capturing: replays do not call the library) and the replays give finite
    losses."""
    import pcd_native
    from search import GraphedLctStep
    monkeypatch.setitem(P.LCT_DIMS, "hidden_size", 32)        # inside the decode envelope (embed = hidden: h0 is the image
    monkeypatch.setitem(P.LCT_DIMS, "embed_size", 32)         # embedding)
    ef, _, arch = P.make_lct("cuda")
    ef.qst_encoder.deterministic = False
    lib = pcd_native.load_cuda()
    rec = _Decodes(lib.pcd_decode)
    monkeypatch.setattr(lib, "pcd_decode", rec)
    tr, va = P.lct_batch(21, "cuda"), P.lct_batch(22, "cuda")
    graphed = GraphedLctStep(arch, tr, va, 1e-3, 1e-3, warmup=1)
    assert rec.count(DECODE_SAMPLED) == 3 * 2 and rec.count(DECODE_GREEDY) == 0       # one warm-up step + the captured step
    losses = []
    for _ in range(2):
        losses.append(float(graphed(tr, va)))
        torch.cuda.synchronize()
    assert rec.count(DECODE_SAMPLED) == 6 and all(math.isfinite(x) for x in losses), losses
