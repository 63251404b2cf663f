"""Host restatement of the in-kernel noise of sample_kernel and remask_kernel (csrc/elementwise.cuh), in numpy uint64 arithmetic.

Philox4x32-10 (Salmon et al., SC'11; the Random123 constants) with key = (seed_lo, seed_hi) and the counters
  sample:  (ctr_lo, g, step, ctr_hi)               ctr = philox_row(seq0, b, t) * Q + q; word j of group g = i*32 + lane is column 4 g + j
  remask:  (ctr_lo, 0x52454d41, step, ctr_hi)      ctr = philox_row(seq0, b, t); word x
philox_row(seq0, b, t) = (seq0 + b) T_b + t (seq_layout.cuh), i.e. the target row index of a uniform batch at seq0 = 0.
The Gumbel value of a word takes its top 24 bits k to u = float32(k + 1/2) 2^-24, exactly as the kernel rounds it (k = 2^24 - 1 gives
the largest float below 1), and then g = -log(-log(u)) in float64 from that u."""
from __future__ import annotations

import numpy as np

M0, M1 = 0xD2511F53, 0xCD9E8D57
W0, W1 = 0x9E3779B9, 0xBB67AE85
REMASK_WORD = 0x52454D41
_MASK = np.uint64(0xFFFFFFFF)
U_MAX = np.float32(1.0 - 2.0 ** -24)

# Sample draws whose top 24 bits k lie in [0xFFFFF0, 0xFFFFFF] (step 0, uniform batch with Q = 1, so the counter is the row):
# k -> (seed, row, column), the first hit over seeds 0, 1, ... and rows 0..63. The u == 1 case of the unclamped formula is 0xFFFFFF.
SAMPLE_TAIL = {
    0xFFFFF0: (287, 2, 871), 0xFFFFF1: (84, 48, 276), 0xFFFFF2: (247, 63, 710), 0xFFFFF3: (216, 5, 825), 0xFFFFF4: (196, 58, 659),
    0xFFFFF5: (7, 0, 571), 0xFFFFF6: (2, 6, 695), 0xFFFFF7: (177, 58, 554), 0xFFFFF8: (146, 22, 378), 0xFFFFF9: (57, 11, 994),
    0xFFFFFA: (211, 36, 542), 0xFFFFFB: (46, 26, 182), 0xFFFFFC: (95, 42, 175), 0xFFFFFD: (2, 53, 545), 0xFFFFFE: (165, 9, 783),
    0xFFFFFF: (1, 34, 106),
}
# re-masking draw with k = 0xFFFFFF: (seed, step, row of a B = 1, T = 4096 batch)
REMASK_U1 = (2747, 0, 1531)


def philox4x32_10(ctr, key):
    """ctr: 4 words, key: 2 words, each an int or an integer array (broadcast together). Returns uint32 [..., 4]."""
    c = [np.asarray(w, dtype=np.uint64) & _MASK for w in ctr]
    k0, k1 = (np.asarray(w, dtype=np.uint64) & _MASK for w in key)
    for _ in range(10):
        p0 = np.uint64(M0) * c[0]
        p1 = np.uint64(M1) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & _MASK, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & _MASK]
        k0 = (k0 + np.uint64(W0)) & _MASK
        k1 = (k1 + np.uint64(W1)) & _MASK
    return np.stack(np.broadcast_arrays(*c), -1).astype(np.uint32)


def _key(seed):
    seed = int(seed)
    return seed & 0xFFFFFFFF, seed >> 32


def sample_counter(b, t, q, T, Q, seq0=0):
    """Counter of level q of target row t of sequence b (uniform batch of T targets, Q levels per row)."""
    return ((seq0 + np.asarray(b, dtype=np.int64)) * T + np.asarray(t, dtype=np.int64)) * Q + np.asarray(q, dtype=np.int64)


def sample_bits(ctr, seed, step):
    """uint32 [..., 1024]: the word each column of a row with counter `ctr` draws."""
    ctr = np.asarray(ctr, dtype=np.uint64)[..., None]
    g = np.arange(256, dtype=np.uint64)
    words = philox4x32_10((ctr & _MASK, g, step, ctr >> np.uint64(32)), _key(seed))  # [..., 256, 4]
    return words.reshape(*words.shape[:-2], 1024)


def remask_bits(ctr, seed, step):
    """uint32 [...]: the word (x) the re-masking draws for a target row with counter `ctr`."""
    ctr = np.asarray(ctr, dtype=np.uint64)
    return philox4x32_10((ctr & _MASK, REMASK_WORD, step, ctr >> np.uint64(32)), _key(seed))[..., 0]


def uniform(bits):
    """float32 u in (0, 1) of each word, rounded as the kernel rounds it."""
    k = np.asarray(bits, dtype=np.uint32) >> np.uint32(8)
    u = (k.astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -24)
    return np.where(k == 0xFFFFFF, U_MAX, u).astype(np.float32)


def gumbel(bits):
    """float64 g = -log(-log(u)) of each word (u - 1 is exact in float64, so log1p keeps the tail near u = 1)."""
    u = uniform(bits).astype(np.float64)
    return -np.log(-np.log1p(u - 1.0))


def sample_gumbel(ctr, seed, step):
    return gumbel(sample_bits(ctr, seed, step))


def remask_gumbel(ctr, seed, step):
    return gumbel(remask_bits(ctr, seed, step))
