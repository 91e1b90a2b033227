"""numpy restatement of the drop-path node sum (pcd_droppath_sum_*; the masks are lct-vqa_b200/csrc/pcd_philox.cuh), on the
Philox of sample_oracle.py:
    x = Philox4x32-10(counter = {global_sample, cell, 2 * node + input, 0x44504154}, key = seed).word[0]
    u = (x >> 8) * 2^-24,  m = 1 iff u < keep
    node = d1 * h1 + d2 * h2,  d_i h = (h / keep) * m_i  (fp32, IEEE division) for a dropped input, else h
"""
import numpy as np

import sample_oracle as S

DPAT = 0x44504154


def masks(seed, samples, cell, slot, keep):
    """m(seed, sample, cell, slot) for every global sample index in `samples` -> float32 array of 0 / 1."""
    samples = np.asarray(samples, dtype=np.uint64)
    ctr = np.zeros((len(samples), 4), dtype=np.uint64)
    ctr[:, 0] = samples
    ctr[:, 1] = cell
    ctr[:, 2] = slot
    ctr[:, 3] = DPAT
    x = S.philox4x32_10(ctr, S.seed_key(seed))[:, 0]
    u = (x >> np.uint32(8)).astype(np.float32) * np.float32(2.0 ** -24)
    return (u < np.float32(keep)).astype(np.float32)


def _scaled(h, drop, keep, m):
    if not drop:
        return h
    return (h / np.float32(keep)) * m.reshape((-1,) + (1,) * (h.ndim - 1))


def node_sum(h1, h2, drop1, drop2, keep, seed, cell, node, offset=0):
    """float32 forward of one node: (node, m1, m2)."""
    h1, h2 = np.asarray(h1, dtype=np.float32), np.asarray(h2, dtype=np.float32)
    rows = np.arange(offset, offset + h1.shape[0])
    m1, m2 = masks(seed, rows, cell, 2 * node, keep), masks(seed, rows, cell, 2 * node + 1, keep)
    return _scaled(h1, drop1, keep, m1) + _scaled(h2, drop2, keep, m2), m1, m2


def node_sum_backward(g, drop1, drop2, keep, seed, cell, node, offset=0):
    """float32 (grad_h1, grad_h2) = (d1 * g, d2 * g)."""
    g = np.asarray(g, dtype=np.float32)
    rows = np.arange(offset, offset + g.shape[0])
    m1, m2 = masks(seed, rows, cell, 2 * node, keep), masks(seed, rows, cell, 2 * node + 1, keep)
    return _scaled(g, drop1, keep, m1), _scaled(g, drop2, keep, m2)
