"""float64 restatement of truncated sampling in the question decode (pcd_decode in sampled mode with truncate = 1; the rule is
stated in include/pcdarts_sm100.h).  Per row and step, with l the logits and T the temperature:
    order    v before w iff l_v > l_w, or l_v = l_w and v < w
    S_k      the first min(top_k, V) words in that order (top_k = 0: all)
    S        the shortest prefix of S_k whose mass sum exp((l - l_max) / T) reaches top_p times the mass of S_k (top_p = 1: S_k)
    word     argmax over v in S of l_v / T + G(seed, t, row, v), the noise of sample_oracle.py
The kernel computes l in fp32 and sums integer-quantised fp32 masses, so a word near the boundary of S can fall on either
side of it.  kept_sets therefore also returns, for a logit tolerance delta, the set every kernel within delta of these
logits could keep (wide), the set it must keep (narrow) and the two margins of the boundary.
"""
import numpy as np

import sample_oracle as S


def mass_tolerance(delta, temperature):
    """Log-ratio by which a prefix mass over the top-k mass can move when every logit moves by at most delta: each mass
    exp((l - l_max) / T) moves by a factor within exp(+-2 delta / T), numerator and denominator both; 1e-6 covers fp32
    expf and the 2^-47 quantisation of the kernel's masses."""
    return 4.0 * delta / temperature + 1e-6


def kept_sets(logits, temperature, top_k, top_p, delta=0.0):
    """logits (B, V) float64 -> (kept, wide, narrow) (B, V) bool and margins (B, 2): kept is S; wide holds every word a
    decoder with logit errors <= delta could keep, narrow only words it must keep; margins[:, 0] is the logit gap between
    the last kept word and the first dropped one (inf when S is all V words) and margins[:, 1] the log-ratio distance of
    the nucleus boundary from the target (inf without a nucleus)."""
    B, V = logits.shape
    kept, wide, narrow = (np.zeros((B, V), dtype=bool) for _ in range(3))
    margins = np.full((B, 2), np.inf)
    eps = mass_tolerance(delta, temperature)
    nk = top_k if 0 < top_k < V else V
    for b in range(B):
        l = logits[b]
        order = np.lexsort((np.arange(V), -l))
        ls = l[order]
        n = n_lo = n_hi = nk
        if top_p < 1.0:
            cum = np.cumsum(np.exp((ls[:nk] - ls[0]) / temperature))
            Z = cum[-1]
            first = lambda r: min(nk, int(np.searchsorted(cum, r * Z, side="left")) + 1)
            n, n_lo, n_hi = first(top_p), first(top_p * np.exp(-eps)), first(min(1.0, top_p * np.exp(eps)))
            hi = np.log(cum[n - 1] / (top_p * Z))
            lo = np.log(top_p * Z / cum[n - 2]) if n >= 2 else np.inf
            margins[b, 1] = min(hi, lo)
        kept[b, order[:n]] = True
        if n < V:
            margins[b, 0] = ls[n - 1] - ls[n]
        wide[b] = l >= ls[n_hi - 1] - 2 * delta
        narrow[b] = l > ls[n_lo] + 2 * delta if n_lo < V else True
    return kept, wide, narrow, margins


def _sigmoid(x):
    return 1.0 / (1.0 + np.exp(-x))


def decode_truncated(emb, w_ih, w_hh, b_ih, b_hh, w_out, b_out, h0, T, temperature, seed, top_k, top_p, delta=0.0,
                     start_token=2, row_offset=0, force=None):
    """float64 truncated sampled decode: h0 = c0 = h0 (B, H), first input tanh(emb[start_token]), later inputs emb[previous
    word].  Returns (tokens (B, T), scores (T, B, V), kept, wide, narrow (T, B, V) bool, margins (T, B, 2)) with scores =
    logits / temperature + G(seed, t, row_offset + b, v).  The words are the argmax of the scores over kept, or `force`
    (B, T) when given (teacher forcing with another decoder's words)."""
    emb, w_ih, w_hh, b_ih, b_hh, w_out, b_out, h0 = (np.asarray(a, dtype=np.float64)
                                                     for a in (emb, w_ih, w_hh, b_ih, b_hh, w_out, b_out, h0))
    B, H = h0.shape
    V = w_out.shape[0]
    rows = np.arange(row_offset, row_offset + B)
    h, c = h0.copy(), h0.copy()
    x = np.tanh(np.repeat(emb[start_token][None, :], B, 0))
    tokens = np.zeros((B, T), dtype=np.int64)
    scores = np.empty((T, B, V))
    kept, wide, narrow = (np.empty((T, B, V), dtype=bool) for _ in range(3))
    margins = np.empty((T, B, 2))
    for t in range(T):
        gates = x @ w_ih.T + h @ w_hh.T + b_ih + b_hh
        i, f, g, o = (gates[:, k * H:(k + 1) * H] for k in range(4))
        c = _sigmoid(f) * c + _sigmoid(i) * np.tanh(g)
        h = _sigmoid(o) * np.tanh(c)
        logits = np.tanh(h) @ w_out.T + b_out
        scores[t] = logits / temperature + S.gumbel_noise(seed, t, rows, V)
        kept[t], wide[t], narrow[t], margins[t] = kept_sets(logits, temperature, top_k, top_p, delta)
        own = np.where(kept[t], scores[t], -np.inf).argmax(1)
        tokens[:, t] = own if force is None else np.asarray(force)[:, t]
        x = emb[tokens[:, t]]
    return tokens, scores, kept, wide, narrow, margins
