"""DAC encoder batches of different lengths (DACEncoder.forward_batch, DAC.encode_to_codes_batch): the clips are packed along time with
zero gap rows at hop-aligned starts, and the contract is bit identity with encoding each clip alone. The clip lengths give 1, 2, 15,
16, 17, 127, 128 and 129 frames (the 128-row tile edges of the latent stage), most of them not hop multiples."""
import random

import pytest
import torch

pytestmark = pytest.mark.gpu

HOP = 320
L_MIX = [HOP, 2 * HOP + 37, 15 * HOP + 100, 16 * HOP, 17 * HOP + 5, 40 * HOP + 319, 127 * HOP + 200, 128 * HOP, 129 * HOP + 11, 5001]


def _shuffled(seed=0):
    L = list(L_MIX)
    random.Random(seed).shuffle(L)
    return L


def _clips(L, seed, device="cuda", dtype=torch.float32):
    g = torch.Generator().manual_seed(seed)
    return [(torch.randn(1, n, generator=g) * 0.3).clamp(-1, 1).to(device, dtype) for n in L]


@pytest.fixture(scope="module")
def sd():
    from edm_tts_b200.synthetic import make_encoder_state_dict

    return make_encoder_state_dict(64, (2, 4, 5, 8), 1)


@pytest.fixture(scope="module")
def enc(sd):
    from edm_tts_b200.dac_encoder import DACEncoder

    return DACEncoder(sd, 64)


@pytest.fixture(scope="module")
def dac():
    from edm_tts_b200.dac import DAC
    from edm_tts_b200.synthetic import make_dac_state_dict

    return DAC(make_dac_state_dict(3))


@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_forward_batch_matches_single(sd, fused, dtype):
    from edm_tts_b200.dac_encoder import DACEncoder, code_lengths

    enc = DACEncoder(sd, 64, fused=fused)
    L = _shuffled(1)
    clips = _clips(L, 5)
    out = enc.forward_batch(clips, out_dtype=dtype)
    enc.forward_batch(_clips(L[:3], 6), out_dtype=dtype)          # the outputs of a call are not overwritten by the next one
    assert len(out) == len(L)
    assert sorted(z.shape[1] for z in out) == sorted(code_lengths(n) for n in L) and {1, 2, 15, 16, 17, 127, 128, 129} <= {z.shape[1] for z in out}
    for i, n in enumerate(L):
        one = enc(clips[i][None], out_dtype=dtype)[0]
        assert out[i].shape == (1024, code_lengths(n)) and out[i].dtype == dtype
        assert torch.equal(out[i], one), f"clip {i} (L={n})"


def test_forward_batch_converts_like_forward(enc):
    clips = _clips([3 * HOP + 7, 9000], 2, device="cpu", dtype=torch.float64) + _clips([2000], 3, dtype=torch.bfloat16)
    for z, a in zip(enc.forward_batch(clips), clips):
        assert torch.equal(z, enc(a[None])[0])


def test_encode_to_codes_batch_matches_single(dac):
    L = _shuffled(2)
    clips = _clips(L, 9)
    out = dac.encode_to_codes_batch(clips)
    flat = out[0].untyped_storage()
    for i, n in enumerate(L):
        one = dac.encode_to_codes(clips[i][None])[0]
        assert out[i].dtype == torch.int64 and out[i].is_contiguous() and out[i].untyped_storage().data_ptr() == flat.data_ptr()
        assert out[i].shape == one.shape == (12, int(dac.get_code_lengths(torch.tensor([n]))[0])), f"clip {i}"
        assert torch.equal(out[i], one), f"clip {i} (L={n})"


def test_chunking_gives_the_same_bits(sd):
    from edm_tts_b200 import varlen
    from edm_tts_b200.dac_encoder import DACEncoder

    enc = DACEncoder(sd, 64)
    L = _shuffled(3)
    clips = _clips(L, 7)
    whole = enc.forward_batch(clips)          # grows the packed workspace to the whole list: later chunks meet its stale rows
    for limit in (1, 60 * HOP):               # one clip per chunk; chunks of uneven size
        enc.max_chunk_samples = limit
        plan = varlen.enc_plan(L, enc.strides, limit)
        assert len(plan) > 1 and (limit > 1 or len(plan) == len(L))
        got = enc.forward_batch(clips)
        assert all(torch.equal(a, b) for a, b in zip(got, whole))
    # a large call, then a smaller one on the same object (the smaller chunk reads no stale row, sd's front and tail rows included)
    enc.max_chunk_samples = 1 << 23
    small = [clips[L.index(2 * HOP + 37)], clips[L.index(17 * HOP + 5)]]
    for z, a in zip(enc.forward_batch(small), small):
        assert torch.equal(z, enc(a[None])[0])


def test_permutation_permutes_outputs(enc):
    L = _shuffled(4)
    clips = _clips(L, 8)
    base = enc.forward_batch(clips)
    perm = list(range(len(L)))
    random.Random(5).shuffle(perm)
    got = enc.forward_batch([clips[p] for p in perm])
    for j, p in enumerate(perm):
        assert torch.equal(got[j], base[p])


def test_padding_changes_only_the_tail(dac):
    """The reference's Collator right-pads the list to the longest clip: every frame t < T_i - 8 keeps its codes, the last <= 8 may
    not (the padding zeros become bias / Snake(bias) after the first conv, where a clip encoded alone reads zero conv padding)."""
    L = _shuffled(5)
    clips = _clips(L, 10)
    out = dac.encode_to_codes_batch(clips)
    Lmax = max(L)
    padded = torch.stack([torch.nn.functional.pad(c, (0, Lmax - c.shape[1])) for c in clips])
    codes = dac.encode_to_codes(padded)
    changed = {}
    for i, c in enumerate(out):
        T = c.shape[1]
        head = T if L[i] == Lmax else max(0, T - 8)
        assert torch.equal(codes[i, :, :head], c[:, :head]), f"clip {i}"
        changed[L[i]] = int((codes[i, :, head:T] != c[:, head:]).any(0).sum())
    print("frames among the last 8 whose codes padding changed, per clip length:", changed)


def test_oracle_tolerance(enc, sd):
    from oracle.dac_encoder import encoder_forward
    from tests.test_gpu_dac_encoder import _check

    clips = _clips([16000 + 77, 129 * HOP], 11)
    for z, a in zip(enc.forward_batch(clips, out_dtype=torch.float32), clips):
        with torch.inference_mode():
            ref = encoder_forward(sd, a[None].cpu())
        assert z.shape == ref.shape[1:]
        _check(z, ref[0])


def test_codec_round_trip(dac):
    """encode_to_codes_batch -> decode_from_codes_batch equals, per clip, encode_to_codes -> decode_from_codes."""
    L = [17 * HOP + 5, 2 * HOP + 37, 50 * HOP]
    clips = _clips(L, 12)
    wavs = dac.decode_from_codes_batch(dac.encode_to_codes_batch(clips))
    for i, a in enumerate(clips):
        want = dac.decode_from_codes(dac.encode_to_codes(a[None]))[0]
        assert torch.equal(wavs[i], want), f"clip {i} (L={L[i]})"


def test_errors(enc, dac):
    a = torch.zeros(1, 1000, device="cuda")
    bad = [[], a, [a[0]], [torch.zeros(2, 1000, device="cuda")], [a[None]], [a, torch.zeros(1, 100, device="cuda")], [a, "audio"]]
    for audios in bad:
        with pytest.raises(ValueError):
            enc.forward_batch(audios)
        with pytest.raises(ValueError):
            dac.encode_to_codes_batch(audios)
    with pytest.raises(ValueError):
        enc.forward_batch([a], out_dtype=torch.float16)
