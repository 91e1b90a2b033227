"""float64 end-of-sequence beam search of the question decoder, written from the semantics of pcd_decode in beam
mode with the stop (include/pcdarts_sm100.h), on the LSTM step of beam_oracle.py.

A beam is finished once its last word is `end`.  A live beam k contributes the candidates (k, v) for every v with raw score
s_k + lambda_k[v]; a finished beam contributes only (k, pad) with its raw score unchanged.  Candidates are ranked by the key
s / L^alpha (s for alpha = 0), L the hypothesis length counting `end`: t + 1 for a live candidate at step t, the frozen length
of a finished beam.  Exact ties go to the lower k, then the lower v (a stable sort over k*V + v).  Once every beam of every
item has finished the search ends and the remaining positions are `pad`.

As beam_oracle.beam_search, every step records the item's decision margin, here between keys: the smallest gap between
consecutive selected candidates and between the K-th and the (K+1)-th (inf for steps after the search ended).
"""
import torch

from beam_oracle import _step


def _key(raw, L, alpha):
    return raw / L.double() ** alpha if alpha != 0 else raw


def beam_search_stop(P, h0, T, K, end, pad, alpha, start_token=2):
    """-> tokens (B, K, T) int64, raw scores (B, K) float64, keys (B, K) float64, lengths (B, K) int64, margins (B, T)."""
    h0 = h0.detach().cpu().double()
    B, V = h0.shape[0], P["w_out"].shape[0]
    R = B * K
    h = h0.repeat_interleave(K, 0)
    c = h.clone()
    x = torch.tanh(P["emb"][start_token]).expand(R, -1)
    s = torch.full((B, K), float("-inf"), dtype=torch.float64)
    s[:, 0] = 0.0
    L = torch.zeros(B, K, dtype=torch.long)                  # frozen length of a finished beam, 0 while live
    words, parents = torch.empty(T, B, K, dtype=torch.long), torch.empty(T, B, K, dtype=torch.long)
    margins = torch.full((B, T), float("inf"), dtype=torch.float64)
    t_run = T
    for t in range(T):
        h, c, lam = _step(P, x, h, c)
        fin = L > 0
        raw = s[:, :, None] + lam.reshape(B, K, V)
        raw = torch.where(fin[:, :, None], torch.tensor(float("-inf"), dtype=torch.float64), raw)
        raw[:, :, pad] = torch.where(fin, s, raw[:, :, pad])
        Lc = torch.where(fin, L, torch.full_like(L, t + 1))
        key = _key(raw, Lc[:, :, None], alpha).reshape(B, K * V)
        srt, idx = torch.sort(key, dim=1, descending=True, stable=True)
        top = srt[:, :K + 1]
        gaps = top[:, :-1] - top[:, 1:] if top.shape[1] > 1 else torch.full((B, 1), float("inf"), dtype=torch.float64)
        margins[:, t] = torch.nan_to_num(gaps, nan=float("inf")).min(1).values
        sel = idx[:, :K]
        k, v = sel // V, sel % V
        s = raw.reshape(B, K * V).gather(1, sel)
        Lp = L.gather(1, k)
        L = torch.where(Lp > 0, Lp, torch.where(v == end, torch.full_like(v, t + 1), torch.zeros_like(v)))
        rows = (torch.arange(B)[:, None] * K + k).reshape(R)
        h, c, x = h[rows], c[rows], P["emb"][v.reshape(R)]
        words[t], parents[t] = v, k
        if bool((L > 0).all()):
            t_run = t + 1
            break
    tokens = torch.full((B, K, T), pad, dtype=torch.long)
    cur = torch.arange(K).expand(B, K).clone()
    for t in range(t_run - 1, -1, -1):
        tokens[:, :, t] = words[t].gather(1, cur)
        cur = parents[t].gather(1, cur)
    lengths = torch.where(L > 0, L, torch.full_like(L, T))
    return tokens, s, _key(s, lengths, alpha), lengths, margins


def lengths_of(tokens, end):
    """Hypothesis length counting the first `end` (the full length where there is none), for tokens (..., T)."""
    T = tokens.shape[-1]
    hit = tokens == end
    first = torch.where(hit.any(-1), hit.long().argmax(-1), torch.full(tokens.shape[:-1], T - 1))
    return first + 1


def sequence_logprob_stop(P, h0, tokens, end, start_token=2):
    """float64 teacher-forced log-probability of every sequence in tokens (B, K, T) up to and including its first `end`."""
    h0 = h0.detach().cpu().double()
    tokens = torch.as_tensor(tokens).cpu()
    B, K, T = tokens.shape
    flat = tokens.reshape(B * K, T)
    n = lengths_of(flat, end)
    h = h0.repeat_interleave(K, 0)
    c = h.clone()
    x = torch.tanh(P["emb"][start_token]).expand(B * K, -1)
    total = torch.zeros(B * K, dtype=torch.float64)
    for t in range(T):
        h, c, lam = _step(P, x, h, c)
        total += torch.where(t < n, lam.gather(1, flat[:, t:t + 1])[:, 0], torch.zeros((), dtype=torch.float64))
        x = P["emb"][flat[:, t]]
    return total.reshape(B, K)


def truncate(tokens, end, pad):
    """The unstopped decode truncated after each row's first `end` and filled with `pad`."""
    hit = (tokens == end).long()
    after = (hit.cumsum(-1) - hit) > 0
    return torch.where(after, torch.full_like(tokens, pad), tokens)
