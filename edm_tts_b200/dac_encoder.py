"""DAC convolutional encoder on the CUDA path, behind the reference's module API.

Mirrors edm_tts/models/dac/encoder.py:11-58 (Encoder(d_model, strides): first conv, EncoderBlocks of three dilated ResidualUnits +
Snake + strided conv, last Snake + conv) and its caller DAC.encode_to_codes (edm_tts/models/dac/modeling_dac.py:163-167:
z = encoder(audio); codes = quantizer(z)["codes"]), which utility_scripts/dump_tokens/dump_tokens.py:213-215 runs under bf16
autocast. Every conv is one launch of the implicit-GEMM kernel of csrc/dac_conv.cuh: activations are channel-last, the residual
stream is fp32, the conv operands are bf16 tensors that already hold Snake(x) and are written by the producing conv's epilogue.
"""
from __future__ import annotations

import math

import torch

from . import _lib as L
from . import varlen
from .varlen import strided_conv_length


_FUSED = (64, 128)   # channel counts whose ResidualUnits run as one launch (edm_dac_resunit); at 256 the two-launch form is as fast


def _fold(sd, key):
    """weight_norm (dim 0): w = g * v / ||v||, the norm taken over (in, k) per output channel (nn_layers.py:8-9)."""
    g = sd[key + ".parametrizations.weight.original0"].float()
    v = sd[key + ".parametrizations.weight.original1"].float()
    return v * (g / v.flatten(1).norm(dim=1).view(-1, 1, 1))


def code_lengths(input_lengths, strides=(2, 4, 5, 8)):
    """Frames produced for audio of `input_lengths` samples: what AudioTokenizer.get_code_lengths computes by walking the encoder's
    Conv1d modules (edm_tts/models/audio_tokenizer/audio_tokenizer.py:84-93)."""
    out = input_lengths
    for s in strides:
        out = strided_conv_length(out, s)
    return out


class DACEncoder:
    def __init__(self, state_dict: dict, d_model: int = 64, strides=(2, 4, 5, 8), prefix: str = "", device="cuda",
                 max_chunk_samples: int = 1 << 23, fused: bool = True):
        if not torch.cuda.is_available():
            raise L.EdmError("edm_tts_b200 needs a CUDA device (sm_100); there is no CPU fallback")
        if d_model % 64 != 0 or d_model * 2 ** len(strides) > 1024:
            raise ValueError("the conv kernels need channel counts that are multiples of 64 and at most 1024")
        self.device = torch.device(device)
        self.d_model, self.strides = d_model, tuple(strides)
        self.enc_dim = d_model * 2 ** len(strides)
        self.hop_length = math.prod(strides)
        self.max_chunk_samples = max_chunk_samples
        self.fused = fused          # False: every ResidualUnit as two conv launches (A/B timing and parity of the fused kernel)
        sd = {k: v.detach().to("cpu") for k, v in state_dict.items() if k.startswith(prefix)}
        dev = self.device

        def conv(key):
            w = _fold(sd, key)                                                   # [c_out, c_in, k]
            packed = w.permute(0, 2, 1).reshape(w.shape[0], -1)                  # K index = tap * c_in + channel
            return packed.to(dev, torch.bfloat16).contiguous(), sd[key + ".bias"].float().to(dev).contiguous()

        def alpha(key):
            return sd[key + ".alpha"].float().reshape(-1).to(dev).contiguous()

        self.w0 = _fold(sd, f"{prefix}block.0")[:, 0, :].to(dev).contiguous()   # [d_model, 7] fp32
        self.b0 = sd[f"{prefix}block.0.bias"].float().to(dev).contiguous()
        self.blocks = []
        n = 1
        for stride in self.strides:
            units = []
            for u in range(3):
                ru = f"{prefix}block.{n}.block.{u}.block."
                w7, b7 = conv(ru + "1")
                w1, b1 = conv(ru + "3")
                units.append(dict(a_in=alpha(ru + "0"), w7=w7, b7=b7, a_mid=alpha(ru + "2"), w1=w1, b1=b1))
            wd, bd = conv(f"{prefix}block.{n}.block.4")
            self.blocks.append(dict(units=units, a_down=alpha(f"{prefix}block.{n}.block.3"), wd=wd, bd=bd, stride=stride))
            n += 1
        self.a_last = alpha(f"{prefix}block.{n}")
        self.w_last, self.b_last = conv(f"{prefix}block.{n + 1}")
        self._ws = {}
        self._pws = None

    def eval(self):
        return self

    # ------------------------------------------------------------------ geometry / workspace
    def lengths(self, L_in: int):
        """Time lengths after the first conv and after each strided conv (kernel 2s, stride s, padding ceil(s/2))."""
        out = [L_in]
        for s in self.strides:
            out.append(strided_conv_length(out[-1], s))
        return out

    def _alloc(self, B: int, lens):
        """Stage buffers for B sequences of lens[k] rows at stage k."""
        dev = self.device
        ws = dict(lens=lens, y=[], sx=[], sh=[], sd=[], sm=[])
        c = self.d_model
        for k, s in enumerate(self.strides):
            Lk, Ln = lens[k], lens[k + 1]
            ws["y"].append(torch.empty(B, Lk, c, device=dev, dtype=torch.float32))
            ws["sx"].append(torch.empty(B, Lk, c, device=dev, dtype=torch.bfloat16))
            ws["sh"].append(torch.empty(B, Lk, c, device=dev, dtype=torch.bfloat16))     # sx / sh alternate as unit input / output
            # hidden activation between the two convs of a unit (two-launch form only)
            ws["sm"].append(None if self.fused and c in _FUSED else torch.empty(B, Lk, c, device=dev, dtype=torch.bfloat16))
            # operand of the strided conv: `pad` zero rows in front, (Ln + 1) * s rows in all; never-written rows stay zero
            ws["sd"].append(torch.zeros(B, (Ln + 1) * s, c, device=dev, dtype=torch.bfloat16))
            c *= 2
        ws["y"].append(None)
        ws["sx"].append(torch.empty(B, lens[-1], c, device=dev, dtype=torch.bfloat16))
        return ws

    def _workspace(self, B: int, L_in: int):
        key = (B, L_in)
        ws = self._ws.get(key)
        if ws is not None:
            return ws
        # keep two geometries (a batch that does not divide into equal chunks alternates between two chunk sizes; re-allocating
        # per chunk costs more than the kernels), drop the oldest beyond that: the buffers are large
        while len(self._ws) >= 2:
            self._ws.pop(next(iter(self._ws)))
        ws = self._alloc(B, self.lengths(L_in))
        self._ws[key] = ws
        return ws

    def _packed_workspace(self, rows0: int):
        """Grow-only workspace of the packed path, sized for rows0 packed audio rows (stage k: rows0 / r_k rows). The chunks of a list
        have different geometries; re-allocating per chunk would cost more than the kernels."""
        if self._pws is None or self._pws["lens"][0] < rows0:
            self._pws = None                                                     # release the smaller one first
            lens = [rows0]
            for s in self.strides:
                lens.append(lens[-1] // s)
            self._pws = self._alloc(1, lens)
        return self._pws

    # ------------------------------------------------------------------ forward
    def _conv(self, a, a_rows, a_cols, w, bias, taps, step, off, rows_out, B, alpha=None, x_res=None, y=None, s_out=None,
              s_row_off=0, s_rows=0, zt=None):
        c_out = w.shape[0]
        L.check(L.lib().edm_dac_conv(L.ptr(a), a_rows, a_cols, a.stride(0), B, L.ptr(w), c_out, taps, step, off, rows_out, L.ptr(bias),
                                     L.ptr(alpha), 0, L.ptr(x_res), L.ptr(y), y.stride(0) if y is not None else 0, L.ptr(s_out),
                                     s_out.stride(0) if s_out is not None else 0, s_row_off, s_rows, L.ptr(zt),
                                     int(zt is not None and zt.dtype == torch.float32), L.stream_ptr()), "dac_conv")

    def _resunit(self, src, B, rows, c, dilation, ru, a_next, y, dst, dst_off, dst_rows):
        L.check(L.lib().edm_dac_resunit(L.ptr(src), src.stride(0), B, rows, c, dilation, L.ptr(ru["w7"]), L.ptr(ru["w1"]), L.ptr(ru["b7"]),
                                        L.ptr(ru["a_mid"]), L.ptr(ru["b1"]), L.ptr(a_next), L.ptr(y), y.stride(0), L.ptr(dst),
                                        dst.stride(0), dst_off, dst_rows, L.stream_ptr()), "dac_resunit")

    @torch.no_grad()
    def forward(self, audio: torch.Tensor, out_dtype=torch.bfloat16) -> torch.Tensor:
        """audio [B, 1, L] -> z [B, enc_dim, T] (bf16 as under the reference's autocast, or fp32)."""
        if audio.dim() != 3 or audio.shape[1] != 1:
            raise ValueError("audio must be [B, 1, L]")
        if out_dtype not in (torch.bfloat16, torch.float32):
            raise ValueError("out_dtype must be bfloat16 or float32")
        audio = audio.to(self.device, torch.float32).contiguous()
        B, _, L_in = audio.shape
        T = self.lengths(L_in)[-1]
        if T <= 0:
            raise ValueError(f"audio of {L_in} samples is shorter than one frame")
        z = torch.empty(B, self.enc_dim, T, device=self.device, dtype=out_dtype)
        per = max(1, self.max_chunk_samples // L_in)
        for b0 in range(0, B, per):
            self._forward_chunk(audio[b0:b0 + per], z[b0:b0 + per])
        return z

    __call__ = forward

    def _forward_chunk(self, audio, z_out):
        B, _, L_in = audio.shape
        ws = self._workspace(B, L_in)
        return self._run(ws, B, ws["lens"], audio, z_out)

    def _run(self, ws, B, lens, audio, z_out, clear=None):
        """The encoder's launches over ws (stage k holds lens[k] rows per sequence; the buffers may be longer) from audio [B, ..., L]
        into z_out [B, enc_dim, T]. clear(k, ptr, pitch_bytes, sd), when given, runs after every launch whose bf16 operand output at
        stage k a multi-tap conv reads next; sd marks the strided conv's padded operand, whose row 0 is `pad` rows before row 0 of the
        stage."""
        c = self.d_model
        first_alpha = self.blocks[0]["units"][0]["a_in"]
        L.check(L.lib().edm_dac_conv_first(L.ptr(audio), B, lens[0], L.ptr(self.w0), L.ptr(self.b0), L.ptr(first_alpha), c, L.ptr(ws["y"][0]),
                                           L.ptr(ws["sx"][0]), L.stream_ptr()), "dac_conv_first")
        if clear:
            clear(0, ws["sx"][0].data_ptr(), c * 2, False)
        for k, blk in enumerate(self.blocks):
            s, Lk, Ln = blk["stride"], lens[k], lens[k + 1]
            y, sx, sh, sd = ws["y"][k][:, :Lk], ws["sx"][k][:, :Lk], ws["sh"][k][:, :Lk], ws["sd"][k][:, :(Ln + 1) * s]
            sm = ws["sm"][k][:, :Lk] if ws["sm"][k] is not None else None
            src = sx
            for u, ru in enumerate(blk["units"]):
                d = 3 ** u
                a_next = blk["units"][u + 1]["a_in"] if u < 2 else blk["a_down"]
                # the unit's output operand: the other 64/128-channel buffer, or the padded operand of the strided conv
                dst, dst_off, dst_rows = (sh if src is sx else sx, 0, Lk) if u < 2 else (sd, math.ceil(s / 2), (Ln + 1) * s)
                if self.fused and c in _FUSED:
                    # both convs in one launch, the hidden activation stays in shared memory (csrc/dac_conv.cuh, dac_resunit_kernel)
                    self._resunit(src, B, Lk, c, d, ru, a_next, y, dst, dst_off, dst_rows)
                else:
                    # dilated k=7 conv of Snake(x); epilogue applies the unit's second Snake
                    self._conv(src, Lk, c, ru["w7"], ru["b7"], 7, d, -3 * d, Lk, B, alpha=ru["a_mid"], s_out=sm, s_rows=Lk)
                    # 1x1 conv + residual add into the fp32 stream; epilogue applies the Snake in front of the next conv
                    self._conv(sm, Lk, c, ru["w1"], ru["b1"], 1, 1, 0, Lk, B, alpha=a_next, x_res=y, y=y, s_out=dst,
                               s_row_off=dst_off, s_rows=dst_rows)
                if clear:
                    clear(k, dst.data_ptr(), c * 2, u == 2)
                src = dst
            # strided conv on the padded operand viewed as [Ln + 1][s * c]
            nxt_alpha = self.blocks[k + 1]["units"][0]["a_in"] if k + 1 < len(self.blocks) else self.a_last
            sd_view = sd.view(B, Ln + 1, s * c)
            last = k + 1 == len(self.blocks)      # nothing reads the fp32 stream after the last strided conv
            self._conv(sd_view, Ln + 1, s * c, blk["wd"], blk["bd"], 2, 1, 0, Ln, B, alpha=nxt_alpha,
                       y=None if last else ws["y"][k + 1][:, :Ln], s_out=ws["sx"][k + 1][:, :Ln], s_rows=Ln)
            c *= 2
            if clear:
                clear(k + 1, ws["sx"][k + 1].data_ptr(), c * 2, False)
        T = lens[-1]
        self._conv(ws["sx"][-1][:, :T], T, c, self.w_last, self.b_last, 3, 1, -1, T, B, zt=z_out)
        return z_out

    # ------------------------------------------------------------------ clips of different lengths
    def _check_list(self, audios) -> list[int]:
        """Samples per clip of a list of [1, L_i] clips; ValueError for anything else or a clip shorter than one frame."""
        if not isinstance(audios, (list, tuple)) or len(audios) == 0:
            raise ValueError("audios must be a non-empty list of [1, L_i] clips")
        for a in audios:
            if not torch.is_tensor(a) or a.dim() != 2 or a.shape[0] != 1:
                raise ValueError("every clip must be a [1, L_i] tensor")
            if self.lengths(int(a.shape[1]))[-1] <= 0:
                raise ValueError(f"a clip of {int(a.shape[1])} samples is shorter than one frame")
        return [int(a.shape[1]) for a in audios]

    @torch.no_grad()
    def forward_batch(self, audios, out_dtype=torch.bfloat16) -> list:
        """List of mono clips [1, L_i] (any float dtype, converted as forward converts) -> list of z [enc_dim, T_i] (bf16 or fp32),
        T_i = lengths(L_i)[-1], views of buffers of this call. Item i equals forward(audios[i][None])[0] bit for bit."""
        out = []
        self._forward_packed(audios, out_dtype, lambda ch, z: out.extend(z[0, :, a:a + n] for a, n in zip(ch.starts[-1], ch.lengths[-1])))
        return out

    def _forward_packed(self, audios, out_dtype, consume):
        """Encodes the list chunk by chunk (varlen.enc_plan); consume(chunk, z) gets each chunk's packed z [1, enc_dim, rows[-1]], a
        fresh tensor whose gap frames hold junk."""
        if out_dtype not in (torch.bfloat16, torch.float32):
            raise ValueError("out_dtype must be bfloat16 or float32")
        lens = self._check_list(audios)
        plan = varlen.enc_plan(lens, self.strides, self.max_chunk_samples)
        K = len(self.strides)
        # one upload per call: the gap ranges of every chunk and stage ((start, end) pairs); list k <= K clears the operand of stage k,
        # list K + 1 + k the strided conv's padded operand of stage k: the same gaps `pad` rows later, the first one from row 0 (the
        # front rows) and the last one to the end of the [Ln + 1][s C] view, rows a previous larger chunk may have written
        host, at = [], []
        for ch in plan:
            at.append([])
            lists = [ch.gaps(k) for k in range(K + 1)]
            for k, s in enumerate(self.strides):
                pad = math.ceil(s / 2)
                g = [(b + pad, e + pad) for b, e in ch.gaps(k)]
                g[0], g[-1] = (0, g[0][1]), (g[-1][0], ch.rows[k] + s)
                lists.append(g)
            for g in lists:
                at[-1].append((len(host), len(g), max(e - b for b, e in g)))
                host += g
        dev_buf = torch.tensor([v for g in host for v in g], dtype=torch.int32).to(self.device)
        # the packed audio of every chunk in one copy: clips at their packed rows, zeros in between
        clips = [a.to(self.device, torch.float32).reshape(-1) for a in audios]
        zeros = torch.zeros(max(e - b for ch in plan for b, e in ch.gaps(0)), device=self.device)
        pieces = []
        for ch in plan:
            for (b, e), i in zip(ch.gaps(0), range(ch.start, ch.stop + 1)):
                pieces.append(zeros[:e - b])
                if i < ch.stop:
                    pieces.append(clips[i])
        packed = torch.cat(pieces)
        ws = self._packed_workspace(max(ch.rows[0] for ch in plan))
        o0 = 0
        for ch, at_ch in zip(plan, at):
            def clear(k, ptr, pitch, sd, at_ch=at_ch):
                first, n, widest = at_ch[K + 1 + k if sd else k]
                self._zero_rows(ptr, pitch, dev_buf.data_ptr() + 8 * first, n, widest)

            z = torch.empty(1, self.enc_dim, ch.rows[-1], device=self.device, dtype=out_dtype)
            self._run(ws, 1, ch.rows, packed[o0:o0 + ch.rows[0]], z, clear)
            o0 += ch.rows[0]
            consume(ch, z)

    def _zero_rows(self, ptr, pitch, ranges_ptr, n, widest):
        L.check(L.lib().edm_dac_zero_rows(ptr, pitch, ranges_ptr, n, widest, L.stream_ptr()), "dac_zero_rows")
