"""Packing plan of the DAC decoder batch (edm_tts_b200/varlen.py, used by DACDecoder.forward_batch), on CPU: utterances packed along
time with zero gap rows, every gap wide enough for the widest one-sided conv read into its stage, and the chunk cut."""
import random

import pytest

from edm_tts_b200 import varlen

RATES = [(8, 5, 4, 2), (2, 2, 2, 2), (3, 7), (4, 5, 8)]


def _lengths(T, rates):
    """DACDecoder.lengths (a method of a GPU-backed object) restated: the time length after the first conv and each transposed conv."""
    out = [T]
    for s in rates:
        out.append(varlen.conv_transpose_length(out[-1], s))
    return out


def _check_chunk(ch, T, rates, g0):
    K = len(rates)
    reads = varlen.dac_stage_reads(rates)
    assert len(ch.rows) == len(ch.starts) == len(ch.lengths) == K + 1
    for i, t in enumerate(T):
        assert [ch.lengths[k][i] for k in range(K + 1)] == _lengths(t, rates)
    for k in range(1, K + 1):
        assert ch.rows[k] == rates[k - 1] * ch.rows[k - 1]
        assert all(a == rates[k - 1] * b for a, b in zip(ch.starts[k], ch.starts[k - 1]))
    for k in range(K + 1):
        valid = [(a, a + n) for a, n in zip(ch.starts[k], ch.lengths[k])]
        assert all(0 <= b < e <= ch.rows[k] for b, e in valid)
        assert all(valid[i][1] <= valid[i + 1][0] for i in range(len(valid) - 1))
        gaps = ch.gaps(k)
        assert all(e - b >= reads[k] for b, e in gaps), (k, gaps)
        # the gap ranges are exactly the complement of the valid ranges
        covered = sorted(valid + gaps)
        assert covered[0][0] == 0 and covered[-1][1] == ch.rows[k]
        assert all(covered[i][1] == covered[i + 1][0] for i in range(len(covered) - 1))
        assert len(gaps) == len(valid) + 1
    assert ch.starts[0][0] == g0 and ch.rows[0] == g0 * (len(T) + 1) + sum(T)


@pytest.mark.parametrize("rates", RATES)
def test_min_gap_is_smallest(rates):
    g0 = varlen.dac_min_gap(rates)
    reads = varlen.dac_stage_reads(rates)
    assert all(g >= n for g, n in zip(varlen.dac_stage_gaps(g0, rates), reads))
    assert any(g < n for g, n in zip(varlen.dac_stage_gaps(g0 - 1, rates), reads))


def test_default_rates_gaps():
    assert varlen.dac_min_gap((8, 5, 4, 2)) == 4
    assert varlen.dac_stage_gaps(4, (8, 5, 4, 2)) == [4, 32, 158, 632, 1264]
    assert varlen.dac_stage_reads((8, 5, 4, 2)) == [3, 27, 27, 27, 27]
    with pytest.raises(ValueError):
        varlen.dac_min_gap((8, 1))


@pytest.mark.parametrize("rates", RATES)
def test_pack_geometry(rates):
    g0 = varlen.dac_min_gap(rates)
    rng = random.Random(sum(rates))
    for T in ([1], [1, 2, 3], [rng.randint(1, 400) for _ in range(17)], [150, 1000, 1, 129]):
        _check_chunk(varlen.dac_pack(T, rates, g0), T, rates, g0)


@pytest.mark.parametrize("rates", RATES)
def test_plan_chunks(rates):
    g0 = varlen.dac_min_gap(rates)
    hop = 1
    for r in rates:
        hop *= r
    rng = random.Random(7)
    T = [rng.randint(1, 300) for _ in range(40)]
    one = varlen.dac_plan(T, rates, 1 << 40)
    assert len(one) == 1 and (one[0].start, one[0].stop, one[0].t0) == (0, 40, 0)
    for limit in (1, hop * 200, hop * 700, hop * 3000):
        plan = varlen.dac_plan(T, rates, limit)
        assert plan[0].start == 0 and plan[-1].stop == len(T)
        assert all(a.stop == b.start for a, b in zip(plan, plan[1:]))
        for ch in plan:
            sub = T[ch.start:ch.stop]
            assert ch.t0 == sum(T[:ch.start])
            _check_chunk(ch, sub, rates, g0)
            assert ch.rows[-1] == hop * ch.rows[0]
            # within the limit, or a single utterance that alone exceeds it
            assert ch.rows[-1] <= limit or (len(sub) == 1 and hop * (2 * g0 + sub[0]) > limit)
        # greedy: the next utterance would not have fitted
        for a, b in zip(plan, plan[1:]):
            assert hop * (g0 * (b.start - a.start + 2) + sum(T[a.start:b.start + 1])) > limit
    assert [ch.stop - ch.start for ch in varlen.dac_plan(T, rates, 1)] == [1] * len(T)
