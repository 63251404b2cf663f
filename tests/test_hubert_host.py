"""HuBERT host side (no GPU): weight packing from a transformers HubertModel state dict, the folded positional-conv weight, frame
counts against HubertModel._get_feat_extract_output_lengths, the packed-batch plan, and the configurations that are refused."""
import pytest
import torch

from edm_tts_b200 import hubert as H
from edm_tts_b200.synthetic import hubert_config, make_hubert_state_dict


@pytest.fixture(scope="module")
def small():
    cfg = hubert_config(num_hidden_layers=3)
    return cfg, make_hubert_state_dict(0, cfg)


def test_packing_reads_exactly_the_used_keys(small):
    cfg, sd = small
    read = set()

    class Spy(dict):
        def __getitem__(self, k):
            read.add(k)
            return dict.__getitem__(self, k)

    w = H.pack_weights(Spy(sd), cfg, output_layer=2)
    assert len(w["layers"]) == 2
    used = {k for k in sd if not (k == "masked_spec_embed" or k.startswith("encoder.layer_norm.") or k.startswith("encoder.layers.2."))}
    assert read == used, read ^ used
    assert w["final_ln"] is None
    read.clear()
    w3 = H.pack_weights(Spy(sd), cfg, output_layer=3)   # the last entry of hidden_states is taken after encoder.layer_norm
    assert read == {k for k in sd if k != "masked_spec_embed"} and w3["final_ln"] is not None
    # a wrapper's prefix
    w2 = H.pack_weights({"hubert." + k: v for k, v in sd.items()}, cfg, output_layer=2, prefix="hubert.")
    assert torch.equal(w2["layers"][1]["wqkv"], w["layers"][1]["wqkv"])
    for missing in ("encoder.layers.1.attention.k_proj.bias", "feature_extractor.conv_layers.6.layer_norm.weight"):
        with pytest.raises(KeyError, match="k_proj|conv_layers"):
            H.pack_weights({k: v for k, v in sd.items() if k != missing}, cfg, output_layer=2)


def test_operand_layouts(small):
    cfg, sd = small
    w = H.pack_weights(sd, cfg, output_layer=1)
    wq, wk, wv = (sd[f"encoder.layers.0.attention.{n}_proj.weight"] for n in "qkv")
    assert torch.equal(w["layers"][0]["wqkv"].float(), torch.cat([wq, wk, wv]).bfloat16().float())
    c1 = sd["feature_extractor.conv_layers.1.conv.weight"]          # k = 3: taps (0 | 1), (2 | 0) over the [rows / 2][1024] view
    assert w["convs"][0]["taps"] == 2 and torch.equal(w["convs"][0]["w"][:, 1024 + 512:], torch.zeros(512, 512, dtype=torch.bfloat16))
    assert torch.equal(w["convs"][0]["w"][:, 512:1024].float(), c1[:, :, 1].bfloat16().float())
    assert w["convs"][5]["taps"] == 1 and w["convs"][5]["w"].shape == (512, 1024)
    assert torch.equal(w["conv0_w"], sd["feature_extractor.conv_layers.0.conv.weight"][:, 0, :].t())


def test_pos_conv_weight_fold_matches_the_module(small):
    from transformers import HubertModel

    cfg, sd = small
    m = HubertModel(cfg)
    m.load_state_dict(sd)
    w = H.pack_weights(sd, cfg, output_layer=1)
    ref = m.encoder.pos_conv_embed.conv.weight.detach().float()
    torch.testing.assert_close(w["pos_w_f32"], ref, rtol=1e-6, atol=1e-7)
    assert torch.equal(w["pos_w"].float().view(1024, 128, 64).permute(0, 2, 1), w["pos_w_f32"].bfloat16().float())


def test_frame_counts_match_transformers(small):
    from transformers import HubertModel

    m = HubertModel(small[0])
    lens = [400, 401, 719, 720, 721, 1039, 1040, 16000, 116800, 960160, 10 ** 6]
    lens += list(range(400, 5000, 37))
    ref = m._get_feat_extract_output_lengths(torch.tensor(lens)).tolist()
    assert [H.frame_count(n) for n in lens] == ref
    assert H.frame_count(960160) == 3000
    assert [H.frame_count(n) for n in (0, 1, 399)] == [0, 0, 0]


def test_packed_plan():
    lens = [400, 1000, 5000, 16000, 640, 321 * 320]
    chunks = H.plan(lens, 30000)
    assert [(c.start, c.stop) for c in chunks] == [(0, 5), (5, 6)]     # the last clip is longer than the budget: a chunk of its own
    for ch in chunks:
        L = lens[ch.start:ch.stop]
        assert ch.n_samples <= 30000 or ch.stop - ch.start == 1
        assert ch.n_samples % H.HOP == 0
        for i, (s, n) in enumerate(zip(ch.sample_starts, L)):
            assert s % H.HOP == 0
            end = ch.sample_starts[i + 1] if i + 1 < len(L) else ch.n_samples
            assert s + n <= end and end - s < n + H.HOP                   # the clip fits its slot, slots are as short as alignment allows
            assert ch.frames[i] == H.frame_count(n)
            T = ch.frames[i]
            assert ch.gather[ch.cu[i]:ch.cu[i + 1]] == list(range(s // H.HOP, s // H.HOP + T))
            p0 = ch.pad_starts[i]
            assert ch.pad_map[p0:p0 + T] == list(range(ch.cu[i], ch.cu[i + 1]))
            assert ch.pad_map[p0 - H.POS_PAD:p0] == [-1] * H.POS_PAD       # zero padding of the positional conv before ...
            assert ch.pad_map[p0 + T:p0 + T + H.POS_PAD] == [-1] * H.POS_PAD  # ... and after every sequence
        assert ch.cu[-1] == len(ch.gather) == sum(ch.frames)
        assert len(ch.pad_map) == H.POS_PAD + sum(T + H.POS_PAD for T in ch.frames)
    with pytest.raises(ValueError, match="400"):
        H.plan([1000, 399], 1 << 20)
    with pytest.raises(ValueError, match="empty"):
        H.plan([], 1 << 20)


@pytest.mark.parametrize("bad", [dict(hidden_size=768), dict(num_attention_heads=12), dict(conv_dim=(256,) * 7),
                                 dict(feat_extract_norm="group"), dict(do_stable_layer_norm=False), dict(intermediate_size=3072),
                                 dict(conv_bias=False), dict(conv_pos_batch_norm=True)])
def test_rejected_configs(bad):
    with pytest.raises(ValueError):
        H.check_config(hubert_config(**bad))
    with pytest.raises(ValueError):   # refused before any device is needed
        H.HubertFeatures(hubert_config(**bad), {}, device="cpu")


@pytest.mark.parametrize("layer", [0, 25, 18.0])
def test_rejected_output_layer(layer):
    with pytest.raises(ValueError, match="output_layer"):
        H.check_config(hubert_config(), layer)
