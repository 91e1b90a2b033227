"""Top-k and nucleus (top-p) truncation of the sampled question decode (pcd_decode in sampled mode with truncate = 1,
pcd_ops.decode_sample(top_k=, top_p=), QstEncoder(top_k=, top_p=)) against the float64 restatement in truncate_oracle.py.
CPU cases run the kernel source's -DPCD_EMU build; `gpu` cases run the sm_100a kernel.

Comparison rule.  The kernel's logits are fp32 sums over H <= 512 products, so a word whose logit lies within the logit
error of the boundary of the kept set S, or whose nucleus mass lies within the matching mass tolerance of the target, can
fall on either side.  DELTA bounds that logit error: the beam tests measure at most 1.9e-6 per step for the score, which
contains the logit (B200, 1000 W), and test_logit_error_is_far_below_delta measures the logits themselves here.  DELTA =
2e-5 leaves a factor of ten above either.  With it:
  - every word must lie in the oracle's kept set widened by DELTA (the words some decoder with errors <= DELTA could keep);
  - its oracle score must be no more than fp32 rounding below the best score over the set narrowed by DELTA (the words
    every such decoder keeps);
  - where both boundary margins clear DELTA (logit gap > 2 DELTA, nucleus log-ratio > 4 DELTA / T), or where the best
    score over the widened set is also the best over the narrowed one (then no boundary within DELTA changes the draw),
    at least 98 % of the words must be exactly the oracle's.
The identities of the header (no truncation, top_k = 1, top_p < 1/V) hold bit for bit, against the kernel's own modes."""
import ctypes
import math

import numpy as np
import pytest
import torch

import parity_cases as P
import sample_oracle as S
import truncate_oracle as TO
from pcd_native import DECODE_BEAM, DECODE_GREEDY, DECODE_SAMPLED, DecodeArgs
from test_decode_beam import _Decodes, _decode_args

DELTA = 2e-5
SEED = 0x0123456789ABCDEF
PROD = dict(H=512, E=300, V=17858)


@pytest.fixture(scope="module")
def emulation():
    import pcd_build
    import pcd_native
    pcd_native.enable_emulation(pcd_build.build_emu())
    yield pcd_native._emu_lib
    pcd_native._emu_lib = None


class _TruncDecodes(_Decodes):
    """_Decodes that also records whether each sampled call truncated."""

    def __call__(self, args, stream):
        self.truncated = getattr(self, "truncated", []) + [args._obj.truncate]
        return super().__call__(args, stream)


def _modules(B, H, E, V, seed=3, same_h0=False):
    """Embedding, LSTM, projection and h0, seeded independently of module init; the projection is scaled so that the logits
    spread over a few units, as in a trained decoder (a flat distribution would make every nucleus nearly all of V)."""
    g = torch.Generator().manual_seed(seed)
    emb, lstm, proj = torch.nn.Embedding(V, E), torch.nn.LSTM(E, H, 1), torch.nn.Linear(H, V)
    with torch.no_grad():
        for p in list(emb.parameters()) + list(lstm.parameters()) + list(proj.parameters()):
            p.copy_(torch.randn(p.shape, generator=g) * (0.5 if p.dim() > 1 else 0.1) / (p.shape[-1] ** 0.5 if p.dim() > 1 else 1.0))
        emb.weight.mul_(E ** 0.5)
        proj.weight.mul_(4.0)
    h0 = torch.randn(1 if same_h0 else B, H, generator=g) * 0.5
    return emb, lstm, proj, h0.expand(B, H).contiguous()


def _d(t):
    return t.detach().cpu().double().numpy()


def _oracle(mods, h0, T, temperature, seed, top_k, top_p, force=None):
    emb, lstm, proj = mods
    return TO.decode_truncated(_d(emb.weight), _d(lstm.weight_ih_l0), _d(lstm.weight_hh_l0), _d(lstm.bias_ih_l0),
                               _d(lstm.bias_hh_l0), _d(proj.weight), _d(proj.bias), _d(h0), T, temperature, seed, top_k,
                               top_p, DELTA, force=force)


def check_truncated(tokens, mods, h0, T, temperature, seed, top_k, top_p):
    """The rules of the module docstring.  Returns (words checked exactly, share of them equal to the oracle's)."""
    tokens = tokens.cpu().numpy()
    B = h0.shape[0]
    assert tokens.shape == (B, T) and tokens.min() >= 0 and tokens.max() < mods[2].out_features
    _, scores, kept, wide, narrow, margins = _oracle(mods, h0, T, temperature, seed, top_k, top_p, force=tokens)
    eps = TO.mass_tolerance(DELTA, temperature)
    rows = np.arange(B)
    clear_n = exact = 0
    for t in range(T):
        w = tokens[:, t]
        assert wide[t, rows, w].all(), (t, np.flatnonzero(~wide[t, rows, w]))
        mine = scores[t][rows, w]
        best_narrow = np.where(narrow[t], scores[t], -np.inf).max(1)
        scale = np.abs(scores[t]).max()
        assert (best_narrow - mine).max() <= 2e-5 * scale, (t, (best_narrow - mine).max(), scale)
        clear = (margins[t, :, 0] > 2 * DELTA) & (margins[t, :, 1] > eps)
        clear |= np.where(wide[t], scores[t], -np.inf).argmax(1) == np.where(narrow[t], scores[t], -np.inf).argmax(1)
        own = np.where(kept[t], scores[t], -np.inf).argmax(1)
        clear_n += int(clear.sum())
        exact += int((own == w)[clear].sum())
    assert clear_n >= B * T // 2, (clear_n, B * T)            # the exact rule bites on most words
    assert exact >= 0.98 * clear_n, (exact, clear_n)
    return clear_n, exact / clear_n


def truncate_case(device, B, H, E, V, T, temperature, top_k, top_p, seed=SEED, mseed=3):
    from pcd_ops import decode_sample
    emb, lstm, proj, h0 = _modules(B, H, E, V, seed=mseed)
    mods = [m.to(device) for m in (emb, lstm, proj)]
    tokens = decode_sample(h0.to(device), mods[1], mods[0], mods[2], T, temperature, seed=seed, top_k=top_k, top_p=top_p)
    assert tokens.dtype == torch.long and tokens.device.type == torch.device(device).type
    return check_truncated(tokens, (emb, lstm, proj), h0, T, temperature, seed, top_k, top_p)


def _identities(device, B, H, E, V, T, temperature, seed=SEED):
    """The header's identities, bit for bit: truncation with top_k = 0, top_p = 1 (and top_k >= V) is the untruncated
    decode; top_k = 1 and a top_p below 1 / V are greedy; the stopped truncated decode is the unstopped one cut after <end>;
    reruns repeat."""
    import pcd_native as N
    import pcd_ops
    emb, lstm, proj, h0 = (m.to(device) for m in _modules(B, H, E, V, seed=7))
    args = (h0, lstm, emb, proj, T)
    plain = pcd_ops.decode_sample(*args, temperature, seed=seed)
    on = pcd_ops._decode(N.DECODE_SAMPLED, h0, lstm, emb, proj, T, 2, temperature=temperature,
                         seed=torch.tensor([seed - 2 ** 64 if seed >= 2 ** 63 else seed], device=device), truncation=(0, 1.0))[0]
    assert torch.equal(on, plain)
    assert torch.equal(pcd_ops.decode_sample(*args, temperature, seed=seed, top_k=V), plain)
    assert torch.equal(pcd_ops.decode_sample(*args, temperature, seed=seed, top_k=V + 5, top_p=1.0), plain)
    greedy = pcd_ops.decode_greedy(*args)
    assert torch.equal(pcd_ops.decode_sample(*args, temperature, seed=seed, top_k=1), greedy)
    assert 1e-6 < 1.0 / V
    assert torch.equal(pcd_ops.decode_sample(*args, temperature, seed=seed, top_p=1e-6), greedy)
    assert torch.equal(pcd_ops.decode_sample(*args, temperature, seed=seed, top_k=1, top_p=0.3), greedy)
    for kw in (dict(top_k=5), dict(top_p=0.9), dict(top_k=20, top_p=0.5)):
        full = pcd_ops.decode_sample(*args, temperature, seed=seed, **kw)
        assert torch.equal(full, pcd_ops.decode_sample(*args, temperature, seed=seed, **kw))        # reruns
        end = int(full[0, min(2, T - 1)])                   # a word some row emits
        stopped = pcd_ops.decode_sample(*args, temperature, seed=seed, end_token=end, pad_token=0, **kw)
        expect = full.clone()
        for b in range(B):
            hit = (full[b] == end).nonzero()
            if len(hit):
                expect[b, int(hit[0]) + 1:] = 0
        assert torch.equal(stopped, expect), kw


# ---- CPU: the oracle -------------------------------------------------------------------------------------------------
def test_oracle_kept_sets():
    """Top-k ties go to the lower word, the nucleus is the shortest prefix reaching top_p, and both together take the
    nucleus within the top k."""
    l = np.array([[1.0, 3.0, 3.0, 0.5, 2.0]])
    kept = lambda k, p: np.flatnonzero(TO.kept_sets(l, 1.0, k, p)[0][0]).tolist()
    assert kept(2, 1.0) == [1, 2] and kept(1, 1.0) == [1] and kept(4, 1.0) == [0, 1, 2, 4] and kept(0, 1.0) == list(range(5))
    q = np.exp(np.array([3.0, 3.0, 2.0, 1.0, 0.5]) - 3.0)
    p_two = q[:2].sum() / q.sum()
    assert kept(0, p_two - 1e-9) == [1, 2] and kept(0, p_two + 1e-9) == [1, 2, 4] and kept(0, 1e-3) == [1]
    p_in3 = q[:2].sum() / q[:3].sum()
    assert kept(3, p_in3 + 1e-9) == [1, 2, 4] and kept(3, p_in3 - 1e-9) == [1, 2]
    k, w, n, m = TO.kept_sets(l, 1.0, 2, 1.0, delta=0.4)          # gap 1.0 to word 4 > 2 delta: S is certain
    assert m[0, 0] == 1.0 and w[0].tolist() == n[0].tolist() == k[0].tolist() == [False, True, True, False, False]
    k, w, n, m = TO.kept_sets(l, 1.0, 2, 1.0, delta=0.6)          # < 2 delta: word 4 may overtake either of 1, 2
    assert w[0].tolist() == [False, True, True, False, True] and not n[0].any()


# ---- CPU: the emulated kernel source -------------------------------------------------------------------------------
@pytest.mark.parametrize("temperature", [1.0, 0.1])
@pytest.mark.parametrize("top_k,top_p", [(1, 1.0), (5, 1.0), (50, 1.0), (0, 0.5), (0, 0.9), (5, 0.9), (50, 0.5)])
@pytest.mark.parametrize("B,H,E,V,T", [(5, 32, 12, 300, 6), (37, 32, 8, 129, 4), (70, 32, 8, 1000, 3)])
def test_truncated_decode_emulated(emulation, B, H, E, V, T, temperature, top_k, top_p):
    """The oracle rule on the emulation build; B = 70 is decoded as two slices, the second with row_offset 64."""
    truncate_case("cpu", B, H, E, V, T, temperature, top_k, top_p)


@pytest.mark.parametrize("temperature", [1.0, 0.1])
def test_identities_emulated(emulation, temperature):
    _identities("cpu", 9, 32, 8, 300, 5, temperature)


def test_generate_routes_truncation_to_the_truncating_mode(emulation, monkeypatch):
    """deterministic=False with top_k / top_p goes through the truncating sampled mode in both packages; the defaults go
    through the untruncated mode with today's workspace."""
    import models_lct
    import vqa_model
    lib = emulation
    rec = _TruncDecodes(lib.pcd_decode)
    monkeypatch.setattr(lib, "pcd_decode", rec)
    torch.manual_seed(3)
    img = 0.3 * torch.randn(3, 32)
    for mod in (vqa_model, models_lct):
        for kw, flag in ((dict(top_k=5), 1), (dict(top_p=0.8), 1), (dict(top_k=3, top_p=0.5), 1), ({}, 0)):
            q = mod.QstEncoder(90, 8, 32, 1, 32, deterministic=False, temperature=0.5, max_length=5, **kw)
            n = rec.count(DECODE_SAMPLED)
            words = q.generate(img)
            assert rec.count(DECODE_SAMPLED) == n + 1 and rec.truncated[-1] == flag, kw
            assert words.shape == (3, 5) and 0 <= int(words.min()) and int(words.max()) < 90
    assert rec.count(DECODE_GREEDY) == 0 and rec.count(DECODE_BEAM) == 0
    base = dict(mode=DECODE_SAMPLED, B=5, K=1, H=32, V=300)
    plain = lib.pcd_decode_work_floats(ctypes.byref(DecodeArgs(**base)))
    assert plain == lib.pcd_decode_work_floats(ctypes.byref(DecodeArgs(**base, truncate=0, top_k=7, top_p=0.5)))
    assert lib.pcd_decode_work_floats(ctypes.byref(DecodeArgs(**base, truncate=1))) == plain + 5 * 300 + 5


def test_truncation_needs_sampling(emulation):
    import vqa_model
    img = 0.3 * torch.randn(2, 32)
    for det in (True, None):
        for kw in (dict(top_k=5), dict(top_p=0.9)):
            with pytest.raises(ValueError, match="deterministic=False"):
                vqa_model.QstEncoder(90, 8, 32, 1, 32, deterministic=det, max_length=3, **kw).generate(img)
    with pytest.raises(ValueError, match="deterministic=False"):
        vqa_model.QstEncoder(90, 8, 32, 1, 32, deterministic=True, beam_size=2, max_length=3, top_k=5).generate(img)


def test_outside_the_envelope_raises_even_with_stock_ops(emulation):
    """H = 48: no stock loop truncates."""
    import models_lct
    import vqa_model
    prev = __import__("pcd_ops").allow_stock_ops(True)
    try:
        for mod in (vqa_model, models_lct):
            for kw in (dict(top_k=5), dict(top_p=0.9)):
                q = mod.QstEncoder(90, 8, 48, 1, 48, deterministic=False, max_length=4, **kw)
                with pytest.raises(RuntimeError, match="PCD_ERR_UNSUPPORTED"):
                    q.generate(0.3 * torch.randn(2, 48))
            assert mod.QstEncoder(90, 8, 48, 1, 48, deterministic=False, max_length=4).generate(
                0.3 * torch.randn(2, 48)).shape == (2, 4)            # untruncated: the stock loop, as before
    finally:
        __import__("pcd_ops").allow_stock_ops(prev)


def test_bad_truncation_arguments(emulation):
    from pcd_ops import decode_sample
    emb, lstm, proj, h0 = _modules(2, 32, 8, 40)
    for bad in (-1, 1.5, 2.0, True, "3", None):
        with pytest.raises(ValueError, match="top_k"):
            decode_sample(h0, lstm, emb, proj, 3, 1.0, seed=1, top_k=bad)
    for bad in (0.0, -0.5, 1.5, 1.0001, float("nan"), float("inf"), 1e-50):
        with pytest.raises(ValueError, match="top_p"):
            decode_sample(h0, lstm, emb, proj, 3, 1.0, seed=1, top_p=bad)
    assert decode_sample(h0, lstm, emb, proj, 3, 1.0, seed=1, top_p=1.0 + 1e-9).shape == (2, 3)     # 1 in fp32
    lib = emulation
    seed = torch.tensor([1])
    ops = [emb.weight, lstm.weight_ih_l0, lstm.weight_hh_l0, lstm.bias_ih_l0, lstm.bias_hh_l0, h0, h0, proj.weight, proj.bias]
    ptrs = [t.detach().data_ptr() for t in ops]
    tokens = torch.empty(2, 2, 3, dtype=torch.long)
    scores = torch.empty(2, 2)
    work = torch.empty(int(lib.pcd_decode_work_floats(ctypes.byref(DecodeArgs(mode=DECODE_BEAM, B=2, K=2, H=32, V=40)))) +
                       int(lib.pcd_decode_work_floats(ctypes.byref(DecodeArgs(mode=DECODE_SAMPLED, B=2, K=1, H=32, V=40,
                                                                              truncate=1)))))

    def call(mode=DECODE_SAMPLED, truncate=1, top_k=3, top_p=0.9, T=3, K=1):
        a = _decode_args(ptrs, mode=mode, T=T, B=2, K=K, H=32, E=8, V=40, start_token=2, temperature=1.0,
                         seed=seed.data_ptr(), truncate=truncate, top_k=top_k, top_p=top_p, tokens=tokens.data_ptr(),
                         scores=scores.data_ptr(), work=work.data_ptr())
        return lib.pcd_decode(ctypes.byref(a), None)

    assert call() == 0 and call(top_k=0, top_p=1.0) == 0 and call(top_k=1000) == 0
    assert call(truncate=0, top_k=-4, top_p=float("nan")) == 0            # unused without truncation
    for kw in (dict(mode=DECODE_GREEDY), dict(mode=DECODE_BEAM, K=2), dict(top_k=-1), dict(top_p=0.0), dict(top_p=-0.5),
               dict(top_p=1.5), dict(top_p=float("nan")), dict(top_p=float("inf"))):
        assert call(**kw) == -1, kw                  # PCD_ERR_ARG
        assert call(T=0, **kw) == -1, kw             # before the shape check
    assert call(T=0) == -2                           # PCD_ERR_UNSUPPORTED


def test_unrolled_twin_keeps_the_truncation():
    """ArchitectLct generates its pseudo questions with the unrolled twin (model.new()): it must sample like the model."""
    ef, _, _ = P.make_lct("cpu")
    ef.qst_encoder.deterministic, ef.qst_encoder.top_k, ef.qst_encoder.top_p = False, 40, 0.85
    twin = ef.new().qst_encoder
    assert twin.deterministic is False and twin.top_k == 40 and twin.top_p == 0.85


# ---- GPU --------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("temperature", [0.1, 1.0])
@pytest.mark.parametrize("top_k,top_p", [(50, 1.0), (0, 0.9), (50, 0.9)])
def test_truncated_decode_production(temperature, top_k, top_p):
    clear, share = truncate_case("cuda", 64, PROD["H"], PROD["E"], PROD["V"], 30, temperature, top_k, top_p)
    print(f"T={temperature} top_k={top_k} top_p={top_p}: {clear} words clear of the boundary, {share:.4f} exact")


@pytest.mark.gpu
@pytest.mark.parametrize("B,H,E,V,T,temperature,top_k,top_p", [
    (5, 32, 12, 300, 7, 0.1, 5, 1.0), (37, 128, 64, 1000, 12, 1.0, 1, 1.0), (64, 256, 300, 129, 5, 1.0, 0, 0.5),
    (130, 512, 300, 17858, 6, 1.0, 5, 0.5), (37, 128, 64, 1000, 12, 0.1, 50, 0.9), (64, 32, 8, 30000, 4, 1.0, 50, 0.9),
    (64, 32, 8, 30000, 4, 0.1, 0, 0.5)])
def test_truncated_decode_ragged(B, H, E, V, T, temperature, top_k, top_p):
    """Ragged vocabulary tiles, partial batches, fewer blocks than rows (H = 32, V = 129: 8 blocks for 64 rows), B = 130 in
    three slices, and V = 30000 at H = 32, above the shared-memory staging capacity: the select passes read L2."""
    truncate_case("cuda", B, H, E, V, T, temperature, top_k, top_p)


@pytest.mark.gpu
@pytest.mark.parametrize("temperature", [1.0, 0.1])
def test_identities_gpu(temperature):
    _identities("cuda", 64, PROD["H"], PROD["E"], PROD["V"], 8, temperature)
    _identities("cuda", 37, 32, 8, 30000, 4, temperature)


@pytest.mark.gpu
def test_logit_error_is_far_below_delta():
    """The logits the kernel keeps in its workspace (the last step's, after teacher-forced words) against float64: the
    measured error must stay ten times below DELTA."""
    import pcd_native as N
    import pcd_ops
    B, T = 64, 6
    emb, lstm, proj, h0 = _modules(B, PROD["H"], PROD["E"], PROD["V"], seed=11)
    mods = [m.to("cuda") for m in (emb, lstm, proj)]
    lib = N.load_cuda()
    V = PROD["V"]
    ops = [pcd_ops._f32c(t) for t in (mods[0].weight, mods[1].weight_ih_l0, mods[1].weight_hh_l0, mods[1].bias_ih_l0,
                                      mods[1].bias_hh_l0, proj.weight.cuda(), proj.bias.cuda())]
    hd = h0.cuda()
    seed = torch.tensor([SEED], device="cuda")
    tokens = torch.empty(B, T, dtype=torch.long, device="cuda")
    a = _decode_args([o.data_ptr() for o in ops[:5]] + [hd.data_ptr(), hd.data_ptr()] + [o.data_ptr() for o in ops[5:]],
                     mode=DECODE_SAMPLED, T=T, B=B, K=1, H=PROD["H"], E=PROD["E"], V=V, start_token=2, temperature=1.0,
                     seed=seed.data_ptr(), truncate=1, top_k=20, top_p=0.9, tokens=tokens.data_ptr())
    work = torch.empty(int(lib.pcd_decode_work_floats(ctypes.byref(a))), device="cuda")
    a.work = work.data_ptr()
    N.check(lib, lib.pcd_decode(ctypes.byref(a), None), "pcd_decode")
    torch.cuda.synchronize()
    stash = work[-(B * V + B):-B].view(B, V).double().cpu().numpy()          # the header's layout: logits, then words
    p = [_d(x) for x in (emb.weight, lstm.weight_ih_l0, lstm.weight_hh_l0, lstm.bias_ih_l0, lstm.bias_hh_l0, proj.weight,
                         proj.bias)]
    _, scores, *_ = TO.decode_truncated(*p, _d(h0), T, 1.0, SEED, 20, 0.9, DELTA, force=tokens.cpu().numpy())
    logits = scores[T - 1] - S.gumbel_noise(SEED, T - 1, np.arange(B), V)
    err = np.abs(stash - logits).max()
    print(f"logit error {err:.3g} (|logit| <= {np.abs(logits).max():.2f}), DELTA {DELTA}")
    assert err <= DELTA / 10, err


def _draw_test(top_k, top_p, temperature=1.0):
    from scipy.stats import chi2
    from pcd_ops import decode_sample
    B, H, E, V = 64, 64, 12, 300
    emb, lstm, proj, h0 = _modules(B, H, E, V, seed=8, same_h0=True)
    mods = [m.to("cuda") for m in (emb, lstm, proj)]
    hd = h0.to("cuda")
    draws = torch.cat([decode_sample(hd, mods[1], mods[0], mods[2], 1, temperature, seed=1000 + s, top_k=top_k,
                                     top_p=top_p)[:, 0] for s in range(100)]).cpu().numpy()
    _, scores, kept, wide, _, margins = _oracle((emb, lstm, proj), h0[:1], 1, temperature, 0, top_k, top_p)
    assert margins[0, 0, 0] > 2 * DELTA and margins[0, 0, 1] > TO.mass_tolerance(DELTA, temperature)   # an unambiguous S
    kept = kept[0, 0]
    assert kept[draws].all(), np.unique(draws[~kept[draws]])
    logits = (scores[0, 0] - S.gumbel_noise(0, 0, [0], V)[0]) * temperature
    p = np.where(kept, np.exp(logits / temperature - (logits / temperature).max()), 0.0)
    expected = p / p.sum() * len(draws)
    counts = np.bincount(draws, minlength=V).astype(np.float64)
    obs, exp, acc_o, acc_e = [], [], 0.0, 0.0
    for i in np.argsort(expected):
        if not kept[i]:
            continue
        acc_o += counts[i]
        acc_e += expected[i]
        if acc_e >= 5:                                    # pool the rarest kept words until each bin expects >= 5
            obs.append(acc_o); exp.append(acc_e); acc_o = acc_e = 0.0
    if acc_e > 0:
        obs[-1] += acc_o; exp[-1] += acc_e
    obs, exp = np.array(obs), np.array(exp)
    stat = ((obs - exp) ** 2 / exp).sum()
    pval = chi2.sf(stat, len(obs) - 1)
    print(f"top_k={top_k} top_p={top_p}: {int(kept.sum())} kept words, {len(obs)} bins, chi2 {stat:.1f}, p {pval:.3g}")
    assert len(obs) >= 2 and pval > 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("top_k,top_p", [(20, 1.0), (0, 0.8)])
def test_truncated_words_follow_the_truncated_softmax(top_k, top_p):
    """One step, 64 identical rows x 100 seeds = 6400 draws of the first word: none outside the kept set, and a chi-square
    test against softmax(logits / T) restricted to it and renormalised."""
    _draw_test(top_k, top_p)


@pytest.mark.gpu
def test_truncated_decode_in_a_cuda_graph():
    """A captured seed draw + a truncated decode_sample(seed=that buffer): each replay draws new words, the oracle's for its
    seed."""
    from pcd_ops import decode_sample
    B, H, E, V, T = 16, 64, 12, 500, 6
    emb, lstm, proj, h0 = _modules(B, H, E, V, seed=5)
    mods = [m.to("cuda") for m in (emb, lstm, proj)]
    hd = h0.to("cuda")
    seed = torch.zeros(1, dtype=torch.int64, device="cuda")
    kw = dict(top_k=40, top_p=0.9)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        decode_sample(hd, mods[1], mods[0], mods[2], T, 1.0, seed=seed, **kw)      # warm-up (kernel attributes)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        seed.random_(-2 ** 63, None)
        tokens = decode_sample(hd, mods[1], mods[0], mods[2], T, 1.0, seed=seed, **kw)
    runs = []
    for _ in range(2):
        graph.replay()
        torch.cuda.synchronize()
        runs.append((int(seed.item()), tokens.clone()))
    assert runs[0][0] != runs[1][0] and not torch.equal(runs[0][1], runs[1][1])
    for sd, tok in runs:
        check_truncated(tok, (emb, lstm, proj), h0, T, 1.0, sd, **kw)


@pytest.mark.gpu
def test_graphed_lct_step_decodes_in_the_truncating_mode(monkeypatch):
    """search.GraphedLctStep with a truncating EF model: the three generate() calls of ArchitectLct.step run on the
    truncating sampled mode (counted while capturing) and the replays give finite losses."""
    import pcd_native
    from search import GraphedLctStep
    monkeypatch.setitem(P.LCT_DIMS, "hidden_size", 32)
    monkeypatch.setitem(P.LCT_DIMS, "embed_size", 32)
    ef, _, arch = P.make_lct("cuda")
    ef.qst_encoder.deterministic, ef.qst_encoder.top_k, ef.qst_encoder.top_p = False, 20, 0.9
    lib = pcd_native.load_cuda()
    rec = _TruncDecodes(lib.pcd_decode)
    monkeypatch.setattr(lib, "pcd_decode", rec)
    tr, va = P.lct_batch(21, "cuda"), P.lct_batch(22, "cuda")
    graphed = GraphedLctStep(arch, tr, va, 1e-3, 1e-3, warmup=1)
    assert rec.count(DECODE_SAMPLED) == 3 * 2 and rec.count(DECODE_GREEDY) == 0 and all(rec.truncated)
    losses = []
    for _ in range(2):
        losses.append(float(graphed(tr, va)))
        torch.cuda.synchronize()
    assert rec.count(DECODE_SAMPLED) == 6 and all(math.isfinite(x) for x in losses), losses
