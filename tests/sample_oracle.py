"""numpy restatement of the sampled question decode (pcd_decode in sampled mode; the noise is lct-vqa_b200/csrc/pcd_philox.cuh).

By the Gumbel-max trick the kernel draws word t of row b as argmax_v (logit_v / T + G(seed, t, row, v)), which is distributed
as softmax(logit / T), the distribution QstEncoder.sample draws from with torch.multinomial.  G is a pure function of
(seed, t, global row, v):
    key = {seed & 0xffffffff, seed >> 32},  counter = {v >> 2, t, row, 0},  x = Philox4x32-10(counter, key).word[v & 3]
    u = ((float)(x >> 9) + 0.5f) * 2^-23  (exact in fp32),  G = -log(-log(u))
Here G is evaluated in float64 from the same u; the kernel's fp32 logf differs from it by rounding only.
"""
import numpy as np

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
_MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(counter, key):
    """Philox4x32-10 (Salmon et al., SC'11; the Random123 reference).  counter (..., 4), key (..., 2), unsigned 32-bit
    words, broadcast against each other -> (..., 4) uint32."""
    counter = np.asarray(counter, dtype=np.uint64)
    key = np.asarray(key, dtype=np.uint64)
    c0, c1, c2, c3 = (counter[..., i] for i in range(4))
    k0, k1 = key[..., 0], key[..., 1]
    for _ in range(10):
        p0, p1 = _M0 * c0, _M1 * c2                     # 32 x 32 -> 64 bits: exact in uint64
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & _MASK, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & _MASK
        k0, k1 = (k0 + _W0) & _MASK, (k1 + _W1) & _MASK
    return np.stack(np.broadcast_arrays(c0, c1, c2, c3), -1).astype(np.uint32)


def uniform_of_bits(x):
    """The kernel's u in fp32: ((float)(x >> 9) + 0.5f) * 2^-23, in [2^-24, 1 - 2^-24]."""
    x = np.asarray(x, dtype=np.uint32)
    return ((x >> np.uint32(9)).astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -23)


def gumbel_of_bits(x, dtype=np.float64):
    u = uniform_of_bits(x).astype(dtype)
    return -np.log(-np.log(u))


def seed_key(seed):
    s = int(seed) & (2 ** 64 - 1)
    return np.array([s & 0xFFFFFFFF, s >> 32], dtype=np.uint64)


def gumbel_noise(seed, t, rows, V):
    """G(seed, t, row, v) for every row in `rows` (global batch indices) and v < V -> (len(rows), V) float64."""
    rows = np.asarray(rows, dtype=np.uint64)
    nblk = (V + 3) // 4
    ctr = np.zeros((len(rows), nblk, 4), dtype=np.uint64)
    ctr[..., 0] = np.arange(nblk, dtype=np.uint64)[None, :]
    ctr[..., 1] = t
    ctr[..., 2] = rows[:, None]
    words = philox4x32_10(ctr, seed_key(seed))           # word (v & 3) of block (v >> 2) is column v
    return gumbel_of_bits(words.reshape(len(rows), 4 * nblk)[:, :V])


def _sigmoid(x):
    return 1.0 / (1.0 + np.exp(-x))


def decode_sampled(emb, w_ih, w_hh, b_ih, b_hh, w_out, b_out, h0, T, temperature, seed, start_token=2, row_offset=0,
                   force=None):
    """float64 sampled decode of QstEncoder.generate (vqa_model.py:103-136 with deterministic=False): h0 = c0 = h0 (B, H),
    first input tanh(emb[start_token]), later inputs emb[previous word], logits = tanh(h_t) w_out^T + b_out.
    Returns (tokens (B, T), scores (T, B, V)) with scores = logits / temperature + G(seed, t, row_offset + b, v); the words are
    the argmax of the scores, or `force` (B, T) when given (teacher forcing with another decoder's words)."""
    emb, w_ih, w_hh, b_ih, b_hh, w_out, b_out, h0 = (np.asarray(a, dtype=np.float64)
                                                     for a in (emb, w_ih, w_hh, b_ih, b_hh, w_out, b_out, h0))
    B, H = h0.shape
    V = w_out.shape[0]
    rows = np.arange(row_offset, row_offset + B)
    h, c = h0.copy(), h0.copy()
    x = np.tanh(np.repeat(emb[start_token][None, :], B, 0))
    tokens = np.zeros((B, T), dtype=np.int64)
    scores = np.empty((T, B, V))
    for t in range(T):
        gates = x @ w_ih.T + h @ w_hh.T + b_ih + b_hh
        i, f, g, o = (gates[:, k * H:(k + 1) * H] for k in range(4))
        c = _sigmoid(f) * c + _sigmoid(i) * np.tanh(g)
        h = _sigmoid(o) * np.tanh(c)
        scores[t] = (np.tanh(h) @ w_out.T + b_out) / temperature + gumbel_noise(seed, t, rows, V)
        tokens[:, t] = scores[t].argmax(1) if force is None else np.asarray(force)[:, t]
        x = emb[tokens[:, t]]
    return tokens, scores
