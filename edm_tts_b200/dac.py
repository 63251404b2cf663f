"""The reference's DAC module on the CUDA path: conv encoder, residual vector quantizer, conv decoder.

Mirrors edm_tts/models/dac/modeling_dac.py: DAC.preprocess (:75-93) + encode (:111-139), decode (:141-161),
encode_to_codes (:163-167), decode_from_codes (:169-171), codes_to_features / codes_to_features_unreduced (:173-182). State-dict keys
are the reference's (`encoder.block...`, `quantizer.quantizers...`, `decoder.model...`); the decoder is built only when its weights
are present.
"""
from __future__ import annotations

import json
import math
import os

import torch

from . import varlen
from .config import DACConfig
from .dac_decoder import DACDecoder
from .dac_encoder import DACEncoder, code_lengths
from .dac_rvq import ResidualVectorQuantize


class DAC:
    def __init__(self, state_dict: dict, config=None, device="cuda"):
        self.config = cfg = DACConfig.from_any(config)
        self.device = torch.device(device)
        self.sample_rate = cfg.sample_rate
        self.n_codebooks, self.codebook_size, self.codebook_dim = cfg.n_codebooks, cfg.codebook_size, cfg.codebook_dim
        self.encoder = DACEncoder(state_dict, cfg.encoder_dim, cfg.encoder_rates, prefix="encoder.", device=device)
        self.latent_dim = self.encoder.enc_dim
        self.hop_length = self.encoder.hop_length
        self.quantizer = ResidualVectorQuantize(state_dict, n_codebooks=cfg.n_codebooks, codebook_size=cfg.codebook_size,
                                                codebook_dim=cfg.codebook_dim, input_dim=self.latent_dim, prefix="quantizer.", device=device)
        self.decoder = None
        if any(k.startswith("decoder.") for k in state_dict):
            self.decoder = DACDecoder(state_dict, self.latent_dim, cfg.decoder_dim, cfg.decoder_rates, prefix="decoder.", device=device)

    @staticmethod
    def load_checkpoint(path: str):
        """HF directory written by the reference's DAC.save_pretrained (config.json + model.safetensors) -> (state_dict, DACConfig)."""
        from safetensors.torch import load_file

        with open(os.path.join(path, "config.json")) as f:
            cfg = DACConfig.from_any(json.load(f))
        return load_file(os.path.join(path, "model.safetensors")), cfg

    @classmethod
    def from_pretrained(cls, path: str, device="cuda"):
        sd, cfg = cls.load_checkpoint(path)
        return cls(sd, cfg, device=device)

    def eval(self):
        return self

    @torch.no_grad()
    def encode_to_codes(self, audio: torch.Tensor, n_quantizers=None) -> torch.Tensor:
        """audio [B, 1, L] -> codes int64 [B, n_codebooks, T] (modeling_dac.py:163-167). z stays bf16 between the encoder and the
        quantizer, as under the reference's autocast (dump_tokens.py:213)."""
        z = self.encoder(audio, out_dtype=torch.bfloat16)
        return self.quantizer.encode(z, n_quantizers)

    @torch.no_grad()
    def encode_to_codes_batch(self, audios, n_quantizers=None) -> list:
        """audios: list of mono clips [1, L_i] of different lengths -> list of int64 codes [n_codebooks, T_i], T_i =
        get_code_lengths(L_i), views of one flat buffer laid out as varlen.split_blocks (what the S2A infer_batch returns and
        decode_from_codes_batch takes). Item i equals encode_to_codes(audios[i][None], n_quantizers)[0] bit for bit. The clips of a
        chunk are encoded in one packed pass (DACEncoder.forward_batch) and quantized by one RVQ call over the packed z, whose gap
        frames are dropped."""
        T = [self.encoder.lengths(L_i)[-1] for L_i in self.encoder._check_list(audios)]
        n = self.quantizer.n_codebooks
        out = torch.empty(n * sum(T), device=self.device, dtype=torch.int64)
        cu = varlen.offsets(T)

        def gather(ch, z):
            # out[n cu_i + q T_i + t] = codes[q, a_i + t] for the chunk's clips, as one index_select over the packed codes
            codes = self.quantizer.encode(z, n_quantizers)[0]                # [n, rows], gap frames included
            meta = torch.tensor([ch.lengths[-1], ch.starts[-1]], dtype=torch.int64).to(self.device)
            sizes = n * meta[0]
            m = n * (cu[ch.stop] - cu[ch.start])
            clip = torch.repeat_interleave(torch.arange(ch.stop - ch.start, device=self.device), sizes, output_size=m)
            within = torch.arange(m, device=self.device) - (sizes.cumsum(0) - sizes)[clip]
            t_i = meta[0][clip]
            idx = (within // t_i) * codes.shape[1] + meta[1][clip] + within % t_i
            torch.index_select(codes.reshape(-1), 0, idx, out=out[n * cu[ch.start]:n * cu[ch.stop]])

        self.encoder._forward_packed(audios, torch.bfloat16, gather)
        return varlen.split_blocks(out, T, n)

    def preprocess(self, audio_data: torch.Tensor, sample_rate=None):
        """modeling_dac.py:75-93: resample to the model's rate when another one is given (torchaudio, as the reference), then right-pad
        with zeros to a multiple of the hop length. -> (padded audio, un-padded length)."""
        if sample_rate is not None and sample_rate != self.sample_rate:
            import torchaudio

            audio_data = torchaudio.functional.resample(audio_data, sample_rate, self.sample_rate)
        length = audio_data.shape[-1]
        right_pad = math.ceil(length / self.hop_length) * self.hop_length - length
        return torch.nn.functional.pad(audio_data, (0, int(right_pad))), length

    @torch.no_grad()
    def encode(self, audio_data: torch.Tensor, sample_rate=None, n_quantizers=None) -> dict:
        """modeling_dac.py:111-139: preprocess (resample + right-pad to a hop multiple), conv encoder, quantizer. encode_to_codes
        does not pad, in the reference either (:163-167)."""
        audio_data, length = self.preprocess(audio_data, sample_rate)
        z = self.encoder(audio_data, out_dtype=torch.float32)
        out = {"length": length, "z": z}
        q = self.quantizer(z, n_quantizers)
        out.update(q)
        return out

    def get_code_lengths(self, input_lengths: torch.Tensor) -> torch.Tensor:
        """Frames per utterance for padded batches (AudioTokenizer.get_code_lengths, audio_tokenizer.py:84-93)."""
        return code_lengths(input_lengths.long(), self.config.encoder_rates).int()

    def codes_to_features(self, codes):
        return self.quantizer.from_codes(codes)[0]

    def codes_to_features_unreduced(self, codes):
        return self.quantizer.from_codes_unreduced(codes)

    @torch.no_grad()
    def decode(self, z: torch.Tensor, length=None) -> dict:
        """z [B, D, T] -> {"audio": [B, 1, length]} (modeling_dac.py:141-161)."""
        if self.decoder is None:
            raise RuntimeError("this DAC was built without decoder weights")
        x = self.decoder(z)
        return {"audio": x[..., :length]}

    def decode_from_codes(self, codes: torch.Tensor, length=None) -> torch.Tensor:
        """codes [B, n, T] -> audio [B, 1, L] (modeling_dac.py:169-171; the step after the S2A decode in inference.py:49)."""
        return self.decode(self.quantizer.from_codes(codes)[0], length)["audio"]

    def _decoder_or_raise(self):
        if self.decoder is None:
            raise RuntimeError("this DAC was built without decoder weights")
        return self.decoder

    @staticmethod
    def _trim(audio: list, lengths) -> list:
        return audio if lengths is None else [a[..., :n] for a, n in zip(audio, lengths)]

    @torch.no_grad()
    def decode_batch(self, zs, lengths=None) -> list:
        """Latents of different lengths, [D, T_i] each, decoded together -> list of audio [1, L_i] (trimmed to lengths[i] when
        given). Item i equals decode(zs[i][None], lengths[i])["audio"][0] bit for bit."""
        dec = self._decoder_or_raise()
        if lengths is not None and isinstance(zs, (list, tuple)) and len(lengths) != len(zs):
            raise ValueError(f"{len(zs)} utterances but {len(lengths)} lengths")
        return self._trim(dec.forward_batch(zs), lengths)

    @torch.no_grad()
    def decode_from_codes_batch(self, codes, lengths=None) -> list:
        """codes: list of integer [n, T_i] tensors (one n for all, n <= n_codebooks), e.g. what the S2A infer_batch returns -> list of
        audio [1, L_i], views of one packed output (trimmed to lengths[i] when given). Item i equals
        decode_from_codes(codes[i][None], lengths[i])[0] bit for bit. The features of the whole list come from one codes_to_features
        pass over the concatenated codes, which works frame by frame."""
        dec = self._decoder_or_raise()
        if not isinstance(codes, (list, tuple)) or len(codes) == 0:
            raise ValueError("codes must be a non-empty list of [n, T_i] tensors")
        if any(not torch.is_tensor(c) or c.dim() != 2 for c in codes):
            raise ValueError("every codes entry must be a 2-D tensor [n, T_i]")
        if any(c.dtype.is_floating_point or c.dtype.is_complex or c.dtype == torch.bool for c in codes):
            raise ValueError("codes must be integer tensors")
        n = int(codes[0].shape[0])
        if any(int(c.shape[0]) != n for c in codes) or not 1 <= n <= self.n_codebooks:
            raise ValueError(f"every codes entry must have the same number of levels n, 1 <= n <= {self.n_codebooks}")
        T = [int(c.shape[1]) for c in codes]
        if min(T) < 1:
            raise ValueError("every utterance needs at least one frame")
        if lengths is not None and len(lengths) != len(codes):
            raise ValueError(f"{len(codes)} utterances but {len(lengths)} lengths")
        z = self.quantizer.from_codes(torch.cat([c.to(self.device, torch.int64) for c in codes], dim=1)[None])[0][0]
        return self._trim(dec._forward_packed(z.to(torch.bfloat16), T), lengths)
