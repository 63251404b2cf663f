"""Packing plan of the DAC encoder batch (edm_tts_b200/varlen.py, used by DACEncoder.forward_batch), on CPU: clips packed along time
with zero gap rows at hop-aligned starts, every gap wide enough for the widest one-sided conv read into its stage, the chunk cut, and
a float64 restatement of the encoder over the packed layout that reproduces every clip's single-clip encode. Also the list form of
TokenShardWriter.add_batch."""
import math
import random

import pytest
import torch
import torch.nn.functional as F

from edm_tts_b200 import varlen

RATES = [(2, 4, 5, 8), (2, 2, 2, 2), (3, 7), (4, 5, 8), (64, 2)]


def _check_chunk(ch, L, rates, g):
    K = len(rates)
    hop = math.prod(rates)
    reads = varlen.enc_stage_reads(rates)
    assert len(ch.rows) == len(ch.starts) == len(ch.lengths) == K + 1
    for i, x in enumerate(L):
        chain = [x]
        for s in rates:
            chain.append(varlen.strided_conv_length(chain[-1], s))
        assert [ch.lengths[k][i] for k in range(K + 1)] == chain
    r = 1
    for k in range(K + 1):
        assert ch.rows[k] * r == ch.rows[0] and all(a % (hop // r) == 0 and a * r == b for a, b in zip(ch.starts[k], ch.starts[0]))
        valid = [(a, a + n) for a, n in zip(ch.starts[k], ch.lengths[k])]
        assert all(0 <= b < e <= ch.rows[k] for b, e in valid)
        gaps = ch.gaps(k)
        assert all(e - b >= reads[k] for b, e in gaps), (k, gaps)
        # the gap ranges are exactly the complement of the valid ranges
        covered = sorted(valid + gaps)
        assert covered[0][0] == 0 and covered[-1][1] == ch.rows[k]
        assert all(covered[i][1] == covered[i + 1][0] for i in range(len(covered) - 1))
        assert len(gaps) == len(valid) + 1
        r *= rates[k] if k < K else 1
    assert ch.starts[0][0] == hop * g and ch.rows[-1] % 8 == 0 and ch.rows[0] == hop * ch.rows[-1]
    assert ch.rows[-1] == varlen.enc_rows(g + sum(-(-x // hop) + g for x in L))


@pytest.mark.parametrize("rates", RATES)
def test_min_gap_is_smallest(rates):
    g = varlen.enc_min_gap(rates)
    reads = varlen.enc_stage_reads(rates)
    assert all(x >= n for x, n in zip(varlen.enc_stage_gaps(g, rates), reads))
    assert any(x < n for x, n in zip(varlen.enc_stage_gaps(g - 1, rates), reads))
    # G - 1 leaves a real gap narrower than its stage's read (hop-multiple clips leave the narrowest gaps)
    hop = math.prod(rates)
    if g > 1:
        ch = varlen.enc_pack([hop * 3, hop * 2], rates, g - 1)
        assert any(e - b < reads[k] for k in range(len(rates) + 1) for b, e in ch.gaps(k)[:-1])


def test_default_rates_gaps():
    assert varlen.enc_min_gap((2, 4, 5, 8)) == 4
    assert varlen.enc_stage_gaps(4, (2, 4, 5, 8)) == [1280, 640, 160, 32, 4]
    assert varlen.enc_stage_reads((2, 4, 5, 8)) == [27, 27, 27, 27, 1]
    assert varlen.enc_stage_reads((64, 2)) == [32, 27, 1]
    with pytest.raises(ValueError):
        varlen.enc_min_gap((2, 1))


@pytest.mark.parametrize("rates", RATES)
def test_pack_geometry(rates):
    g = varlen.enc_min_gap(rates)
    hop = math.prod(rates)
    rng = random.Random(sum(rates))
    for L in ([hop], [hop, 2 * hop + 1, 3 * hop - 1], [rng.randint(hop, 300 * hop) for _ in range(17)], [150 * hop + 7, 1000 * hop, hop + 5]):
        _check_chunk(varlen.enc_pack(L, rates, g), L, rates, g)


@pytest.mark.parametrize("rates", RATES)
def test_plan_chunks(rates):
    g = varlen.enc_min_gap(rates)
    hop = math.prod(rates)
    rng = random.Random(7)
    L = [rng.randint(hop, 300 * hop) for _ in range(40)]
    one = varlen.enc_plan(L, rates, 1 << 40)
    assert len(one) == 1 and (one[0].start, one[0].stop, one[0].t0) == (0, 40, 0)
    for limit in (1, hop * 200, hop * 700, hop * 3000):
        plan = varlen.enc_plan(L, rates, limit)
        assert plan[0].start == 0 and plan[-1].stop == len(L)
        assert all(a.stop == b.start for a, b in zip(plan, plan[1:]))
        for ch in plan:
            sub = L[ch.start:ch.stop]
            assert ch.t0 == sum(L[:ch.start])
            _check_chunk(ch, sub, rates, g)
            # within the limit, or a single clip that alone exceeds it
            assert ch.rows[0] <= limit or len(sub) == 1
        # greedy: the next clip would not have fitted
        for a, b in zip(plan, plan[1:]):
            assert varlen.enc_pack(L[a.start:b.start + 1], rates, g).rows[0] > limit
    assert [ch.stop - ch.start for ch in varlen.enc_plan(L, rates, 1)] == [1] * len(L)


# ---------------------------------------------------------------------------------------------------------------------------------
# float64 restatement of the encoder over the packed layout (oracle/dac_encoder.py functions), zeroing the Snake'd operand's gap rows
# after the same launches as the CUDA path: first conv, every ResidualUnit, every strided conv. The fp32 stream keeps its gap rows.

def _packed_encode(sd, clips, rates, g):
    from oracle.dac_encoder import _conv, snake

    ch = varlen.enc_pack([c.shape[-1] for c in clips], rates, g)
    audio = torch.zeros(1, 1, ch.rows[0], dtype=torch.float64)
    for a, c in zip(ch.starts[0], clips):
        audio[0, 0, a:a + c.shape[-1]] = c[0]

    def operand(x, alpha, k):
        h = snake(x, alpha)
        for b, e in ch.gaps(k):
            h[..., b:e] = 0.0
        return h

    x = _conv(sd, "block.0", audio, padding=3)
    n = 1
    for k, stride in enumerate(rates):
        op = operand(x, sd[f"block.{n}.block.0.block.0.alpha"], k)
        for u, dilation in enumerate((1, 3, 9)):
            ru = f"block.{n}.block.{u}.block."
            h = _conv(sd, ru + "1", op, dilation=dilation, padding=3 * dilation)
            h = _conv(sd, ru + "3", snake(h, sd[ru + "2.alpha"]))
            x = x + h
            nxt = f"block.{n}.block.{u + 1}.block.0.alpha" if u < 2 else f"block.{n}.block.3.alpha"
            op = operand(x, sd[nxt], k)
        x = _conv(sd, f"block.{n}.block.4", op, stride=stride, padding=math.ceil(stride / 2))
        assert x.shape[-1] == ch.rows[k + 1]
        n += 1
    z = _conv(sd, f"block.{n + 1}", operand(x, sd[f"block.{n}.alpha"], len(rates)), padding=1)
    return [z[0, :, a:a + t] for a, t in zip(ch.starts[-1], ch.lengths[-1])]


@pytest.fixture(scope="module")
def enc_sd():
    from edm_tts_b200.synthetic import make_encoder_state_dict

    return {k: v.double() for k, v in make_encoder_state_dict(64, (2, 4, 5, 8), 1).items()}


def test_packed_emulation_matches_single_clips(enc_sd):
    from oracle.dac_encoder import encoder_forward

    rates = (2, 4, 5, 8)
    g = varlen.enc_min_gap(rates)
    gen = torch.Generator().manual_seed(3)
    lengths = [3333, 640, 4801, 2 * 320, 1999]          # hop multiples and not, a 2-frame clip
    clips = [(torch.randn(1, n, generator=gen, dtype=torch.float64) * 0.3).clamp(-1, 1) for n in lengths]
    with torch.inference_mode():
        want = [encoder_forward(enc_sd, c[None])[0] for c in clips]
        got = _packed_encode(enc_sd, clips, rates, g)
        short = _packed_encode(enc_sd, clips, rates, g - 1)
    worst = max((a - b).abs().max().item() for a, b in zip(got, want))
    assert all(a.shape == b.shape for a, b in zip(got, want)) and worst < 1e-12, worst
    # one gap frame less and the neighbouring clips leak into each other's conv padding
    assert max((a - b).abs().max().item() for a, b in zip(short, want)) > 1e-6


# ---------------------------------------------------------------------------------------------------------------------------------
def test_token_shards_from_lists(tmp_path):
    from edm_tts_b200.token_shards import TokenShardWriter, read_token_shards

    g = torch.Generator().manual_seed(1)
    T = [7, 30, 1]
    ac = [torch.randint(0, 1024, (12, t), generator=g) for t in T]
    sc = [torch.randint(0, 1024, (t,), generator=g) for t in T]
    w = TokenShardWriter(str(tmp_path), rank=0, max_files_per_output_file=2)
    w.add_batch(["a", "b", "c"], ac, sc, transcriptions=["x", "y", "z"])
    files = w.close()
    assert len(files) == 1
    d = torch.load(files[0])
    assert list(d) == ["a", "b", "c"] and d["b"]["transcription"] == "y"
    seen = [ex for _, ex in read_token_shards(str(tmp_path))]
    assert [ex["length"] for ex in seen] == T
    for ex, a, s in zip(seen, ac, sc):
        assert torch.equal(ex["acoustic_tokens"].long(), a.t()) and torch.equal(ex["semantic_tokens"][:, 0].long(), s)


def test_token_shards_list_mismatch_raises(tmp_path):
    from edm_tts_b200.token_shards import TokenShardWriter

    w = TokenShardWriter(str(tmp_path))
    ac = [torch.zeros(12, 10, dtype=torch.long), torch.zeros(12, 4, dtype=torch.long)]
    with pytest.raises(ValueError):
        w.add_batch(["a", "b"], ac, [torch.zeros(10, dtype=torch.long), torch.zeros(5, dtype=torch.long)])
    with pytest.raises(ValueError):
        w.add_batch(["a", "b"], ac, [torch.zeros(10, dtype=torch.long)])
    with pytest.raises(ValueError):
        w.add_batch(["a"], ac[:1], torch.zeros(1, 10, dtype=torch.long))       # a list and a tensor
    assert w.close() == []
