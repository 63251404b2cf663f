"""DAC decoder batches of different lengths (DACDecoder.forward_batch, DAC.decode_from_codes_batch): the utterances are packed along
time with zero gap rows, and the contract is bit identity with decoding each utterance alone. The lengths cross the 128-row tile
edges of the latent stage (127 / 128 / 129) and of the 8x stage (15 / 16 / 17 frames = 120 / 128 / 136 rows)."""
import random

import pytest
import torch

pytestmark = pytest.mark.gpu

T_MIX = [1, 2, 3, 15, 16, 17, 37, 127, 128, 129, 150, 400]


def _shuffled(seed=0):
    T = list(T_MIX)
    random.Random(seed).shuffle(T)
    return T


def _latents(T, seed, dtype=torch.float32):
    g = torch.Generator().manual_seed(seed)
    return [(torch.randn(1024, t, generator=g) * 0.5).to("cuda", dtype) for t in T]


@pytest.fixture(scope="module")
def dec():
    from edm_tts_b200.dac_decoder import DACDecoder
    from edm_tts_b200.synthetic import make_decoder_state_dict

    return DACDecoder(make_decoder_state_dict(1024, 1536, (8, 5, 4, 2), 2))


@pytest.fixture(scope="module")
def dac():
    from edm_tts_b200.dac import DAC
    from edm_tts_b200.synthetic import make_dac_state_dict

    return DAC(make_dac_state_dict(3))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_forward_batch_matches_single(dec, dtype):
    T = _shuffled(1)
    zs = _latents(T, 5, dtype)
    out = dec.forward_batch(zs)
    assert len(out) == len(T)
    for i, t in enumerate(T):
        one = dec(zs[i][None])[0]
        assert out[i].shape == (1, dec.lengths(t)[-1]) and out[i].dtype == torch.float32
        assert torch.equal(out[i], one), f"utterance {i} (T={t})"


def test_decode_from_codes_batch_matches_single(dac):
    T = _shuffled(2)
    g = torch.Generator().manual_seed(9)
    codes = [torch.randint(0, 1024, (12, t), generator=g).cuda() for t in T]
    lengths = [t * 320 - (7 * i) % 300 if t > 1 else None for i, t in enumerate(T)]
    out = dac.decode_from_codes_batch(codes, lengths)
    for i in range(len(T)):
        one = dac.decode_from_codes(codes[i][None], lengths[i])[0]
        assert out[i].shape == one.shape and torch.equal(out[i], one), f"utterance {i} (T={T[i]})"
    # fewer levels than the quantizer has, and a bf16 latent through decode_batch
    c4 = [c[:4] for c in codes[:3]]
    out4 = dac.decode_from_codes_batch(c4)
    for i in range(3):
        assert torch.equal(out4[i], dac.decode_from_codes(c4[i][None])[0])
    zs = _latents(T[:4], 3, torch.bfloat16)
    outz = dac.decode_batch(zs, [100, None, 5, 1000])
    for i, n in enumerate([100, None, 5, 1000]):
        assert torch.equal(outz[i], dac.decode(zs[i][None], n)["audio"][0])


def test_chunking_gives_the_same_bits(dec):
    from edm_tts_b200 import varlen

    T = _shuffled(3)
    zs = _latents(T, 7)
    whole = [a.clone() for a in dec.forward_batch(zs)]
    keep = dec.max_chunk_samples
    try:
        for limit in (1, 200 * 320):          # one utterance per chunk; chunks of uneven size
            dec.max_chunk_samples = limit
            plan = varlen.dac_plan(T, dec.rates, limit)
            assert len(plan) > 1
            got = dec.forward_batch(zs)
            assert all(torch.equal(a, b) for a, b in zip(got, whole))
    finally:
        dec.max_chunk_samples = keep


def test_permutation_permutes_outputs(dec):
    T = _shuffled(4)
    zs = _latents(T, 8)
    base = [a.clone() for a in dec.forward_batch(zs)]
    perm = list(range(len(T)))
    random.Random(5).shuffle(perm)
    got = dec.forward_batch([zs[p] for p in perm])
    for j, p in enumerate(perm):
        assert torch.equal(got[j], base[p])


def test_oracle_tolerance(dec):
    from edm_tts_b200.synthetic import make_decoder_state_dict
    from oracle.dac_decoder import decoder_forward
    from tests.test_gpu_dac_decoder import _check

    sd = make_decoder_state_dict(1024, 1536, (8, 5, 4, 2), 2)
    zs = _latents([37, 150], 11)
    out = dec.forward_batch(zs)
    for z, a in zip(zs, out):
        with torch.inference_mode():
            ref = decoder_forward(sd, z[None].cpu())
        assert a.shape == ref.shape[1:]
        _check(a, ref[0])


def test_pipeline_s2a_batch_to_waveforms():
    """S2A infer_batch -> decode_from_codes_batch equals, per utterance, infer_special(..., batch_offset=i) -> decode_from_codes."""
    from edm_tts_b200.dac import DAC
    from edm_tts_b200.synthetic import make_dac_state_dict
    from tests.parity_utils import full_model

    cfg, sd, model = full_model()
    dsd = make_dac_state_dict(0)
    for k in list(dsd):
        if k.startswith("quantizer."):
            dsd[k] = sd["acoustic_model." + k].cpu()
    dac = DAC(dsd)
    T = [50, 129, 17]
    g = torch.Generator().manual_seed(21)
    sem = [torch.randint(0, cfg.num_semantic, (t,), generator=g).cuda() for t in T]
    codes = model.infer_batch(sem, steps=4, seed=3)
    wavs = dac.decode_from_codes_batch(codes)
    for i, t in enumerate(T):
        one = model.infer_special(sem[i][None], steps=4, seed=3, batch_offset=i)
        assert torch.equal(codes[i], one[0])
        want = dac.decode_from_codes(one)[0]
        assert wavs[i].shape == (1, t * 320 + 16) and torch.equal(wavs[i], want), f"utterance {i} (T={t})"


def test_errors(dec, dac):
    z = torch.zeros(1024, 5, device="cuda")
    c = torch.zeros(12, 5, dtype=torch.int64, device="cuda")
    bad_latents = [[], [torch.zeros(1024, 5, 1, device="cuda")], [torch.zeros(512, 5, device="cuda")], [z, torch.zeros(1024, 0, device="cuda")],
                   z]
    for zs in bad_latents:
        with pytest.raises(ValueError):
            dec.forward_batch(zs)
    bad_codes = [[], [c, c[:4]], [torch.zeros(13, 5, dtype=torch.int64, device="cuda")], [c[:, :0]], [c[0]], [c.float()], c]
    for cs in bad_codes:
        with pytest.raises(ValueError):
            dac.decode_from_codes_batch(cs)
    with pytest.raises(ValueError):
        dac.decode_from_codes_batch([c, c], lengths=[100])
    with pytest.raises(ValueError):
        dac.decode_batch([z, z], lengths=[100, 200, 300])
