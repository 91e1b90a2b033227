"""float64 beam search of the question decoder, written from the semantics of pcd_decode_beam (include/pcdarts_sm100.h).

Items b, beams k, rows r = b*K + k, exactly T words.  Every row of item b starts from h = c = h0[b] with input
tanh(emb[start]); beam scores start at (0, -inf, ..., -inf).  Per step and row: one LSTM step, logits
l = tanh(h) w_out^T + b_out, lambda = log_softmax(l).  The candidates of item b are the pairs (k, v) scored s_k + lambda_k[v];
the K best (exact ties to the lower k, then the lower v: a stable sort over the flat index k*V + v) become the new beams,
each continuing its parent's (h, c) with input emb[v].

Besides the words and scores, every step records the item's decision margin: the smallest of the gaps between consecutive
selected beams and between the K-th and the (K+1)-th candidate.  A decoder whose scores carry an error below half that
margin makes the same choice.
"""
import torch


def params64(emb, lstm, proj):
    d = lambda t: t.detach().cpu().double()
    return dict(emb=d(emb.weight), w_ih=d(lstm.weight_ih_l0), w_hh=d(lstm.weight_hh_l0), b=d(lstm.bias_ih_l0) + d(lstm.bias_hh_l0),
                w_out=d(proj.weight), b_out=d(proj.bias))


def _step(P, x, h, c):
    gates = x @ P["w_ih"].T + h @ P["w_hh"].T + P["b"]
    i, f, g, o = gates.chunk(4, 1)
    c = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(g)
    h = torch.sigmoid(o) * torch.tanh(c)
    return h, c, torch.log_softmax(torch.tanh(h) @ P["w_out"].T + P["b_out"], dim=1)


def beam_search(P, h0, T, K, start_token=2):
    """-> tokens (B, K, T) int64, scores (B, K) float64, margins (B, T) float64."""
    h0 = h0.detach().cpu().double()
    B, V = h0.shape[0], P["w_out"].shape[0]
    R = B * K
    h = h0.repeat_interleave(K, 0)
    c = h.clone()
    x = torch.tanh(P["emb"][start_token]).expand(R, -1)
    s = torch.full((B, K), float("-inf"), dtype=torch.float64)
    s[:, 0] = 0.0
    words, parents = torch.empty(T, B, K, dtype=torch.long), torch.empty(T, B, K, dtype=torch.long)
    margins = torch.empty(B, T, dtype=torch.float64)
    for t in range(T):
        h, c, lam = _step(P, x, h, c)
        cand = (s.reshape(R, 1) + lam).reshape(B, K * V)
        srt, idx = torch.sort(cand, dim=1, descending=True, stable=True)
        top = srt[:, :K + 1]
        gaps = top[:, :-1] - top[:, 1:] if top.shape[1] > 1 else torch.full((B, 1), float("inf"), dtype=torch.float64)
        margins[:, t] = torch.nan_to_num(gaps, nan=float("inf")).min(1).values     # -inf - -inf: no decision there
        sel = idx[:, :K]
        k, v = sel // V, sel % V
        rows = (torch.arange(B)[:, None] * K + k).reshape(R)
        h, c, x = h[rows], c[rows], P["emb"][v.reshape(R)]
        s = srt[:, :K]
        words[t], parents[t] = v, k
    tokens = torch.empty(B, K, T, dtype=torch.long)
    cur = torch.arange(K).expand(B, K).clone()
    for t in range(T - 1, -1, -1):
        tokens[:, :, t] = words[t].gather(1, cur)
        cur = parents[t].gather(1, cur)
    return tokens, s, margins


def sequence_logprob(P, h0, tokens, start_token=2):
    """float64 teacher-forced log-probability of every sequence in tokens (B, K, T), the path starting from h0[b]."""
    h0 = h0.detach().cpu().double()
    tokens = torch.as_tensor(tokens).cpu()
    B, K, T = tokens.shape
    flat = tokens.reshape(B * K, T)
    h = h0.repeat_interleave(K, 0)
    c = h.clone()
    x = torch.tanh(P["emb"][start_token]).expand(B * K, -1)
    total = torch.zeros(B * K, dtype=torch.float64)
    for t in range(T):
        h, c, lam = _step(P, x, h, c)
        total += lam.gather(1, flat[:, t:t + 1])[:, 0]
        x = P["emb"][flat[:, t]]
    return total.reshape(B, K)
