"""The host Philox / Gumbel reference of tests/philox_ref.py on its own: Random123's known answers, the draws the GPU sampling tests
lean on (pinned here so that they cannot drift), and the u -> g mapping over every 24-bit input."""
import numpy as np

from tests import philox_ref as P
from tests.philox_ref import REMASK_U1, SAMPLE_TAIL

# Random123 kat_vectors, philox4x32 with 10 rounds: (counter, key, result)
KAT = [
    ((0x00000000, 0x00000000, 0x00000000, 0x00000000), (0x00000000, 0x00000000), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF), (0xFFFFFFFF, 0xFFFFFFFF), (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0), (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
]


def test_known_answers():
    for ctr, key, want in KAT:
        assert tuple(int(w) for w in P.philox4x32_10(ctr, key)) == want
    # vectorised over a counter array: each element equals its scalar evaluation
    ctrs = np.array([0, 1, 0xFFFFFFFF, 0x123456789])
    got = P.philox4x32_10((ctrs & 0xFFFFFFFF, 7, 3, ctrs >> 32), (5, 9))
    for i, c in enumerate(ctrs):
        assert np.array_equal(got[i], P.philox4x32_10((int(c) & 0xFFFFFFFF, 7, 3, int(c) >> 32), (5, 9)))


def test_counter_layout():
    """Column 4 g + j takes word j of group g (g = i*32 + lane covers columns i*128 + lane*4 + j); the counter's high word and the
    key's high word both reach the bits."""
    bits = P.sample_bits(np.array([5, 5 + 2 ** 32]), 2 ** 32 + 3, 7)
    for g in (0, 1, 31, 32, 255):
        assert np.array_equal(bits[0, 4 * g:4 * g + 4], P.philox4x32_10((5, g, 7, 0), (3, 1)))
        assert np.array_equal(bits[1, 4 * g:4 * g + 4], P.philox4x32_10((5, g, 7, 1), (3, 1)))
    assert P.remask_bits(5, 2 ** 32 + 3, 7) == P.philox4x32_10((5, 0x52454D41, 7, 0), (3, 1))[0]
    assert int(P.sample_counter(1, 3, 2, T=40, Q=11)) == (1 * 40 + 3) * 11 + 2
    assert int(P.sample_counter(0, 3, 0, T=64, Q=1, seq0=2 ** 26)) == 2 ** 32 + 3


def test_pinned_tail_draws():
    for k, (seed, row, col) in SAMPLE_TAIL.items():
        assert int(P.sample_bits(row, seed, 0)[col]) >> 8 == k, hex(k)
    seed, step, row = REMASK_U1
    assert int(P.remask_bits(row, seed, step)) >> 8 == 0xFFFFFF
    # the exact tail value the GPU tail test grades (u = 1 - 2^-23)
    seed, row, col = SAMPLE_TAIL[0xFFFFFE]
    assert P.uniform(P.sample_bits(row, seed, 0)[col]) == np.float32(1 - 2.0 ** -23)
    assert abs(P.sample_gumbel(row, seed, 0)[col] - 15.942385) < 1e-6


def test_uniform_and_gumbel_over_every_k():
    k = np.arange(2 ** 24, dtype=np.uint32)
    # without the clamp the top k rounds to u == 1 (k + 1/2 needs 25 bits, ties go to even)
    raw = (k.astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -24)
    assert np.flatnonzero(raw >= 1).tolist() == [0xFFFFFF]
    u = P.uniform(k << np.uint32(8))
    assert u.dtype == np.float32 and (u > 0).all() and (u < 1).all()
    assert np.array_equal(u[:-1], raw[:-1]) and u[-1] == np.float32(1 - 2.0 ** -24)
    assert (np.diff(u) >= 0).all()
    g = P.gumbel(k << np.uint32(8))
    assert np.isfinite(g).all()
    assert abs(g.max() - 16.6355) < 1e-3 and abs(g.min() + 2.8525) < 1e-3
    # the low 8 bits do not matter
    assert np.array_equal(P.uniform((k << np.uint32(8)) | np.uint32(0xFF)), u)
