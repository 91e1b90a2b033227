// pcd_philox.cuh — the Gumbel noise of the sampled question decode (sampled pcd_decode), shared by the sm_100a kernel and
// the -DPCD_EMU build so that both (and the numpy restatement in tests/sample_oracle.py) draw the same numbers.
//
// By the Gumbel-max trick, argmax_v (logit_v / T + G_v) with independent standard Gumbel G_v is distributed as
// softmax(logit / T).  G is a pure function of (seed, step t, global batch row, vocabulary index v):
//     key     = { seed & 0xffffffff, seed >> 32 }
//     counter = { v >> 2, t, row, 0 }
//     x       = Philox4x32-10(counter, key).word[v & 3]                      (Salmon et al., SC'11; Random123)
//     u       = ((float)(x >> 9) + 0.5f) * 2^-23                             exact in fp32, u in [2^-24, 1 - 2^-24]
//     G       = -logf(-logf(u))                                              finite, in [-2.82, 16.7]
// u is built from 23 bits so that it never rounds to 1 (24 bits + 0.5 would: G = +inf).
//
// The drop-path masks of the derived network's node sum (pcd_droppath_sum_*, csrc/pcd_droppath.cu) come from the same
// generator, one Bernoulli(keep) draw per (sample, cell, node input):
//     counter = { global_sample, cell, 2 * node + input, 0x44504154 }        'DPAT': disjoint from the decode noise (c3 = 0)
//     x       = Philox4x32-10(counter, key = seed).word[0]
//     u       = (x >> 8) * 2^-24                                             exact in fp32, u in [0, 1 - 2^-24]
//     m       = 1 iff u < keep                                               keep = 1 never drops
#pragma once
#include "pcd_common.cuh"

namespace pcd {

struct Philox4 { uint32_t w[4]; };

PCD_HOSTDEV Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const unsigned long long p0 = (unsigned long long)0xD2511F53u * c0, p1 = (unsigned long long)0xCD9E8D57u * c2;
        const uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0, hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
        c0 = hi1 ^ c1 ^ k0;
        c1 = lo1;
        c2 = hi0 ^ c3 ^ k1;
        c3 = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    Philox4 o;
    o.w[0] = c0; o.w[1] = c1; o.w[2] = c2; o.w[3] = c3;
    return o;
}

// one 32-bit Philox word -> standard Gumbel variable
PCD_HOSTDEV float gumbel_of_bits(uint32_t x) {
    const float u = ((float)(x >> 9) + 0.5f) * 0x1p-23f;
    return -logf(-logf(u));
}

// the noise G(seed, t, row, v) itself (one Philox block per call: the kernel shares each block between four lanes instead)
PCD_HOSTDEV float decode_gumbel(unsigned long long seed, int t, int row, int v) {
    const Philox4 r = philox4x32_10((uint32_t)v >> 2, (uint32_t)t, (uint32_t)row, 0u, (uint32_t)seed, (uint32_t)(seed >> 32));
    return gumbel_of_bits(r.w[v & 3]);
}

constexpr uint32_t kDropPathStream = 0x44504154u;     // 'DPAT'

// the drop-path mask m(seed, global sample, cell, slot = 2 * node + input) for keep probability `keep`: 1.f or 0.f
PCD_HOSTDEV float droppath_mask(unsigned long long seed, int sample, int cell, int slot, float keep) {
    const Philox4 r = philox4x32_10((uint32_t)sample, (uint32_t)cell, (uint32_t)slot, kDropPathStream, (uint32_t)seed,
                                    (uint32_t)(seed >> 32));
    return (float)(r.w[0] >> 8) * 0x1p-24f < keep ? 1.f : 0.f;
}

}  // namespace pcd
