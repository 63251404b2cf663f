"""Deterministic synthetic weights and inputs under the reference's state-dict key names (SURVEY.md section 8b).

Used by bench.py (random-init weights of the reference architecture; there are no checkpoints offline) and, re-exported
through oracle/weights.py, by the parity tests and the golden-vector generator, so that all of them see bit-identical
tensors. Every tensor is drawn from its own torch.Generator seeded by crc32(key) ^ seed on the CPU, so the build
container (where the reference is importable) and the GPU box (where it is not) regenerate the same weights without
shipping 2 GB. Pure data generation: no model arithmetic lives here.
"""
from __future__ import annotations

import math
import zlib
from dataclasses import dataclass, field

import torch


@dataclass
class OracleConfig:
    """Dims of the S2A model + DAC quantizer. Defaults = configs/injection_conformer/base_config + configs/dac/base_config."""
    hidden: int = 1024
    heads: int = 16
    depth: int = 16
    ff_mult: int = 4
    conv_expansion: int = 2
    conv_kernel: int = 5
    injection_layers: tuple = (4, 7, 10, 13)
    num_semantic: int = 1024
    n_codebooks: int = 12
    codebook_size: int = 1024
    codebook_dim: int = 8
    latent_dim: int = 1024
    residual: bool = True
    use_injection: bool = True

    @property
    def dim_head(self) -> int:
        return self.hidden // self.heads


def _gen(key: str, seed: int) -> torch.Generator:
    g = torch.Generator(device="cpu")
    g.manual_seed((zlib.crc32(key.encode()) ^ (seed * 2654435761)) & 0x7FFFFFFF)
    return g


def _randn(key, seed, *shape, std=1.0):
    return torch.randn(*shape, generator=_gen(key, seed), dtype=torch.float32) * std


def _conformer_layer(sd: dict, p: str, d: int, ff_mult: int, conv_expansion: int, conv_kernel: int, seed: int) -> None:
    """Parameters of one ConformerBlock (edm_tts/models/conformer/conformer.py:184-235) under prefix p."""
    def linear(prefix, out_f, in_f, bias=True):
        sd[prefix + ".weight"] = _randn(prefix + ".weight", seed, out_f, in_f, std=1.0 / math.sqrt(in_f))
        if bias:
            sd[prefix + ".bias"] = _randn(prefix + ".bias", seed, out_f, std=0.05)

    def lnorm(prefix, n):
        sd[prefix + ".weight"] = 1.0 + _randn(prefix + ".weight", seed, n, std=0.1)
        sd[prefix + ".bias"] = _randn(prefix + ".bias", seed, n, std=0.05)

    inner = d * conv_expansion
    for ff in ("ff1", "ff2"):
        linear(p + ff + ".fn.fn.net.0", d * ff_mult, d)
        linear(p + ff + ".fn.fn.net.3", d, d * ff_mult)
        lnorm(p + ff + ".fn.norm", d)
    linear(p + "attn.fn.to_q", d, d, bias=False)
    linear(p + "attn.fn.to_kv", 2 * d, d, bias=False)
    linear(p + "attn.fn.to_out", d, d)
    lnorm(p + "attn.norm", d)
    lnorm(p + "conv.net.0", d)
    sd[p + "conv.net.2.weight"] = _randn(p + "conv.net.2.weight", seed, inner * 2, d, 1, std=1 / math.sqrt(d))
    sd[p + "conv.net.2.bias"] = _randn(p + "conv.net.2.bias", seed, inner * 2, std=0.05)
    sd[p + "conv.net.4.conv.weight"] = _randn(p + "conv.net.4.conv.weight", seed, inner, 1, conv_kernel, std=0.5)
    sd[p + "conv.net.4.conv.bias"] = _randn(p + "conv.net.4.conv.bias", seed, inner, std=0.05)
    sd[p + "conv.net.6.weight"] = 1.0 + _randn(p + "conv.net.6.weight", seed, 1, inner, 1, std=0.1)
    sd[p + "conv.net.7.weight"] = _randn(p + "conv.net.7.weight", seed, d, inner, 1, std=1 / math.sqrt(inner))
    sd[p + "conv.net.7.bias"] = _randn(p + "conv.net.7.bias", seed, d, std=0.05)
    lnorm(p + "post_norm", d)


@dataclass
class T2SConfig:
    """Dims of TextToSemanticWLen (edm_tts/models/text_to_semantic/configuration.py:4-86). Defaults = its base config (hidden 512,
    16 heads of 32); configs/text_to_semantic_w_length/train_config.yaml trains hidden 384, 8 heads of 48, depth 12."""
    hidden: int = 512
    text_vocab: int = 256
    semantic_vocab: int = 1024
    heads: int = 16
    depth: int = 8
    lp_heads: int = 16
    lp_depth: int = 4
    ff_mult: int = 4
    conv_expansion: int = 2
    conv_kernel: int = 5
    num_special: int = 5          # pad 0, text 1, speech 2, sep 3, mask 4
    target_length: float = 60.0   # synthetic length head: exp(bias) frames

    @property
    def dim_head(self) -> int:
        return self.hidden // self.heads

    @property
    def lp_dim_head(self) -> int:
        return self.hidden // self.lp_heads

    @property
    def total_tokens(self) -> int:
        return self.text_vocab + self.semantic_vocab + self.num_special

    @property
    def codebook_size(self) -> int:   # logit width, for the shared parity helpers
        return self.semantic_vocab


def make_t2s_state_dict(cfg: T2SConfig, seed: int = 0) -> dict:
    """TextToSemanticWLen.state_dict() keys (modeling_text_to_semantic.py:30-60) with deterministic values. The length head is
    centred on cfg.target_length frames so that exp(length_pred_head(.)) is a usable sequence length at random init."""
    d, sd = cfg.hidden, {}
    sd["input_embedding.weight"] = _randn("input_embedding.weight", seed, cfg.total_tokens, d)
    sd["input_embedding.weight"][0].zero_()                      # padding_idx row, as nn.Embedding initialises it
    for i in range(cfg.depth):
        _conformer_layer(sd, f"conformer.layers.{i}.", d, cfg.ff_mult, cfg.conv_expansion, cfg.conv_kernel, seed)
    sd["length_token"] = _randn("length_token", seed, 1, 1, d)
    for i in range(cfg.lp_depth):
        _conformer_layer(sd, f"length_predictor.layers.{i}.", d, cfg.ff_mult, cfg.conv_expansion, cfg.conv_kernel, seed)
    sd["pred_transform.0.weight"] = _randn("pred_transform.0.weight", seed, d, d, std=1.0 / math.sqrt(d))
    sd["pred_transform.0.bias"] = _randn("pred_transform.0.bias", seed, d, std=0.05)
    sd["pred_transform.2.weight"] = 1.0 + _randn("pred_transform.2.weight", seed, d, std=0.1)
    sd["pred_transform.2.bias"] = _randn("pred_transform.2.bias", seed, d, std=0.05)
    sd["pred_head.weight"] = _randn("pred_head.weight", seed, cfg.semantic_vocab, d, std=1.0 / math.sqrt(d))
    sd["pred_head.bias"] = _randn("pred_head.bias", seed, cfg.semantic_vocab, std=0.05)
    sd["length_pred_head.weight"] = _randn("length_pred_head.weight", seed, 1, d, std=0.2 / math.sqrt(d))
    sd["length_pred_head.bias"] = torch.tensor([math.log(cfg.target_length)], dtype=torch.float32)
    return sd


def make_t2s_noise(n_positions: int, pred_iters: int, cfg: T2SConfig, seed: int = 1234) -> dict:
    """Injected sampling noise of TextToSemanticWLen.infer: cat_gumbel [iters-1, L, V] (Categorical.sample == argmax(logits + g)) and
    remask_gumbel [iters-1, 1, L] (the Gumbel draw of random_topk_mask), L = sequence length incl. text and special tokens."""
    g = torch.Generator(device="cpu")
    g.manual_seed(seed)
    n = max(pred_iters - 1, 0)
    u = torch.rand(n, n_positions, cfg.semantic_vocab, generator=g).clamp_(1e-10, 1 - 1e-7)
    cat = -torch.log(-torch.log(u))
    u = torch.rand(n, 1, n_positions, generator=g).clamp_(1e-10, 1 - 1e-7)
    return {"cat_gumbel": cat, "remask_gumbel": -torch.log(-torch.log(u))}


def make_state_dict(cfg: OracleConfig, seed: int = 0) -> dict:
    """All parameters the hot path touches, keyed as in InjectionConformerModel.state_dict()."""
    d, sd = cfg.hidden, {}

    def linear(prefix, out_f, in_f, bias=True, gain=1.0):
        sd[prefix + ".weight"] = _randn(prefix + ".weight", seed, out_f, in_f, std=gain / math.sqrt(in_f))
        if bias:
            sd[prefix + ".bias"] = _randn(prefix + ".bias", seed, out_f, std=0.05)

    def lnorm(prefix, n):
        sd[prefix + ".weight"] = 1.0 + _randn(prefix + ".weight", seed, n, std=0.1)
        sd[prefix + ".bias"] = _randn(prefix + ".bias", seed, n, std=0.05)

    sd["mask_token"] = _randn("mask_token", seed, 1, 1, d)
    sd["semantic_embedding.weight"] = _randn("semantic_embedding.weight", seed, cfg.num_semantic, d)
    linear("acoustic_feat_proj.0", d, cfg.latent_dim)
    lnorm("acoustic_feat_proj.1", d)
    for i in range(cfg.depth):
        _conformer_layer(sd, f"encoder.layers.{i}.", d, cfg.ff_mult, cfg.conv_expansion, cfg.conv_kernel, seed)
    for k in range(len(cfg.injection_layers)):
        linear(f"encoder.project_injection.{k}.0", d, cfg.latent_dim)
        lnorm(f"encoder.project_injection.{k}.1", d)
    n_fine = cfg.n_codebooks - len(cfg.injection_layers)
    linear("encoder.fine_head.0", d * n_fine, d)
    lnorm("encoder.to_logits.0", d)
    sd["encoder.to_logits.1.weight"] = _randn("encoder.to_logits.1.weight", seed, cfg.n_codebooks, d, cfg.codebook_size, std=1 / math.sqrt(d))
    sd["encoder.to_logits.1.bias"] = _randn("encoder.to_logits.1.bias", seed, 1, 1, cfg.n_codebooks, cfg.codebook_size, std=0.05)
    sd.update(make_quantizer_state_dict(cfg, seed, prefix="acoustic_model.quantizer."))
    return sd


def make_quantizer_state_dict(cfg: OracleConfig, seed: int = 0, prefix: str = "") -> dict:
    """DAC ResidualVectorQuantize parameters (weight-normed 1x1 convs keep their original0/original1 split)."""
    sd = {}
    for i in range(cfg.n_codebooks):
        q = f"{prefix}quantizers.{i}."
        sd[q + "codebook.weight"] = _randn(q + "codebook.weight", seed, cfg.codebook_size, cfg.codebook_dim)
        v_in = _randn(q + "in_proj.v", seed, cfg.codebook_dim, cfg.latent_dim, 1, std=1 / math.sqrt(cfg.latent_dim))
        sd[q + "in_proj.parametrizations.weight.original1"] = v_in
        sd[q + "in_proj.parametrizations.weight.original0"] = v_in.flatten(1).norm(dim=1).view(-1, 1, 1) * (1.0 + _randn(q + "in_proj.g", seed, cfg.codebook_dim, 1, 1, std=0.1))
        sd[q + "in_proj.bias"] = _randn(q + "in_proj.bias", seed, cfg.codebook_dim, std=0.05)
        # later levels quantise a shrinking residual, as in a trained codec
        v_out = _randn(q + "out_proj.v", seed, cfg.latent_dim, cfg.codebook_dim, 1, std=0.35 * (0.8 ** i))
        sd[q + "out_proj.parametrizations.weight.original1"] = v_out
        sd[q + "out_proj.parametrizations.weight.original0"] = v_out.flatten(1).norm(dim=1).view(-1, 1, 1) * (1.0 + _randn(q + "out_proj.g", seed, cfg.latent_dim, 1, 1, std=0.1))
        sd[q + "out_proj.bias"] = _randn(q + "out_proj.bias", seed, cfg.latent_dim, std=0.02)
    return sd


def make_encoder_state_dict(encoder_dim: int = 64, rates=(2, 4, 5, 8), seed: int = 0, prefix: str = "") -> dict:
    """DAC Encoder parameters keyed as edm_tts/models/dac/encoder.py builds them (nn.Sequential indices): block.0 first conv,
    block.{1..n} EncoderBlocks (three ResidualUnits, Snake, strided conv), then Snake and the last conv. Weight-normed convs keep
    the original0 (g) / original1 (v) split. Gains are chosen so activations stay O(1) through the stack."""
    sd = {}

    def wnconv(key, c_out, c_in, k, gain):
        v = _randn(key + ".v", seed, c_out, c_in, k)
        sd[key + ".parametrizations.weight.original1"] = v
        sd[key + ".parametrizations.weight.original0"] = (gain * (1.0 + 0.2 * torch.rand(c_out, 1, 1, generator=_gen(key + ".g", seed)))).float()
        sd[key + ".bias"] = _randn(key + ".bias", seed, c_out, std=0.05)

    def snake(key, c):
        sd[key + ".alpha"] = (0.5 + 1.5 * torch.rand(1, c, 1, generator=_gen(key + ".alpha", seed))).float()

    d = encoder_dim
    wnconv(f"{prefix}block.0", d, 1, 7, 2.0)
    n = 1
    for stride in rates:
        d *= 2
        c = d // 2
        for u in range(3):
            ru = f"{prefix}block.{n}.block.{u}.block."
            snake(ru + "0", c)
            wnconv(ru + "1", c, c, 7, 0.6)
            snake(ru + "2", c)
            wnconv(ru + "3", c, c, 1, 0.3)
        snake(f"{prefix}block.{n}.block.3", c)
        wnconv(f"{prefix}block.{n}.block.4", d, c, 2 * stride, 0.5)
        n += 1
    snake(f"{prefix}block.{n}", d)
    wnconv(f"{prefix}block.{n + 1}", d, d, 3, 0.7)
    return sd


def make_decoder_state_dict(input_channel: int = 1024, channels: int = 1536, rates=(8, 5, 4, 2), seed: int = 0, prefix: str = "") -> dict:
    """DAC Decoder parameters keyed as edm_tts/models/dac/decoder.py builds them: model.0 first conv, model.{1..n} DecoderBlocks
    (block.0 Snake, block.1 weight-normed ConvTranspose1d [c_in, c_out, 2s], block.{2,3,4} ResidualUnits), then Snake, last conv."""
    sd = {}

    def wn(key, shape, gain):
        v = _randn(key + ".v", seed, *shape)
        sd[key + ".parametrizations.weight.original1"] = v
        sd[key + ".parametrizations.weight.original0"] = (gain * (1.0 + 0.2 * torch.rand(shape[0], 1, 1, generator=_gen(key + ".g", seed)))).float()

    def snake(key, c):
        sd[key + ".alpha"] = (0.5 + 1.5 * torch.rand(1, c, 1, generator=_gen(key + ".alpha", seed))).float()

    wn(f"{prefix}model.0", (channels, input_channel, 7), 2.0)
    sd[f"{prefix}model.0.bias"] = _randn(f"{prefix}model.0.bias", seed, channels, std=0.05)
    n = 1
    for i, stride in enumerate(rates):
        c_in, c_out = channels // 2 ** i, channels // 2 ** (i + 1)
        blk = f"{prefix}model.{n}.block."
        snake(blk + "0", c_in)
        wn(blk + "1", (c_in, c_out, 2 * stride), 0.5)        # weight_norm dim 0 of a transposed conv = the INPUT channels
        sd[blk + "1.bias"] = _randn(blk + "1.bias", seed, c_out, std=0.05)
        for u in range(3):
            ru = f"{blk}{2 + u}.block."
            snake(ru + "0", c_out)
            wn(ru + "1", (c_out, c_out, 7), 0.6)
            sd[ru + "1.bias"] = _randn(ru + "1.bias", seed, c_out, std=0.05)
            snake(ru + "2", c_out)
            wn(ru + "3", (c_out, c_out, 1), 0.3)
            sd[ru + "3.bias"] = _randn(ru + "3.bias", seed, c_out, std=0.05)
        n += 1
    c_last = channels // 2 ** len(rates)
    snake(f"{prefix}model.{n}", c_last)
    wn(f"{prefix}model.{n + 1}", (1, c_last, 7), 1.0)
    sd[f"{prefix}model.{n + 1}.bias"] = _randn(f"{prefix}model.{n + 1}.bias", seed, 1, std=0.05)
    return sd


def make_dac_state_dict(seed: int = 0) -> dict:
    """Encoder, quantizer and decoder parameters keyed as DAC.state_dict() (`encoder.`, `quantizer.`, `decoder.`) at the base config."""
    sd = make_encoder_state_dict(64, (2, 4, 5, 8), seed, prefix="encoder.")
    sd.update(make_quantizer_state_dict(OracleConfig(), seed, prefix="quantizer."))
    sd.update(make_decoder_state_dict(1024, 1536, (8, 5, 4, 2), seed, prefix="decoder."))
    return sd


def make_inputs(B: int, T: int, P: int, steps: int, cfg: OracleConfig, seed: int = 1234) -> dict:
    """Synthetic tokens + injected sampling noise (SURVEY.md section 8d), all from one CPU generator."""
    g = torch.Generator(device="cpu")
    g.manual_seed(seed)
    out = {"semantic_tokens": torch.randint(0, cfg.num_semantic, (B, T), generator=g)}
    if P > 0:
        out["acoustic_prompt_tokens"] = torch.randint(0, cfg.codebook_size, (B, cfg.n_codebooks, P), generator=g)
        out["semantic_prompt_tokens"] = torch.randint(0, cfg.num_semantic, (B, P), generator=g)
    else:
        out["acoustic_prompt_tokens"] = None
        out["semantic_prompt_tokens"] = None
    n = max(steps - 1, 0)
    u = torch.rand(n, B * T, cfg.codebook_size, generator=g).clamp_(1e-10, 1 - 1e-7)
    out["cat_gumbel"] = -torch.log(-torch.log(u))          # Gumbel(0,1): Categorical.sample == argmax(logits + g)
    u = torch.rand(n, B, T, generator=g).clamp_(1e-10, 1 - 1e-7)
    out["remask_gumbel"] = -torch.log(-torch.log(u))       # noise of random_topk_mask
    return out


def hubert_config(**overrides):
    """transformers HubertConfig of hubert-large (the semantic tokenizer's backbone): every field the kernels depend on set explicitly,
    the rest at transformers' defaults."""
    from transformers import HubertConfig

    kw = dict(hidden_size=1024, num_hidden_layers=24, num_attention_heads=16, intermediate_size=4096, feat_extract_norm="layer",
              do_stable_layer_norm=True, conv_bias=True)
    kw.update(overrides)
    return HubertConfig(**kw)


def make_hubert_state_dict(seed: int = 0, config=None) -> dict:
    """A HubertModel(config).state_dict() with transformers' own random initialisation, seeded (hubert_config() by default)."""
    from transformers import HubertModel

    cfg = config if config is not None else hubert_config()
    devnull = torch.random.fork_rng(devices=[])
    with devnull:
        torch.manual_seed(seed)
        model = HubertModel(cfg)
    return {k: v.detach().clone() for k, v in model.state_dict().items()}
