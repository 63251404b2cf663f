"""DAC convolutional decoder (vocoder side of the codec) on the CUDA path, behind the reference's module API.

Mirrors edm_tts/models/dac/decoder.py:11-62 (Decoder(input_channel, channels, rates): first conv k=7, DecoderBlocks of Snake +
weight-normed ConvTranspose1d(kernel 2s, stride s) + three dilated ResidualUnits, last Snake + conv k=7 to one channel + tanh) and
its callers DAC.decode / decode_from_codes (edm_tts/models/dac/modeling_dac.py:141-171; inference.py:49 after the S2A decode).
It reuses the encoder's kernels (csrc/dac_conv.cuh): channel-last activations, fp32 residual stream, bf16 conv operands that already
hold Snake(x). A transposed conv with kernel 2s / stride s is the 2-tap conv
    out_view[q, r * C + co] = sum_{u in {0,1}} x[q - u] . w[:, co, r + u * s],        out_view[q, r * C + co] = out[q * s + r - padding, co]
so its output "view" [L_in + 1][s * C] is just the channel-last output tensor addressed `padding` rows early; the output buffers carry
a few guard rows in front and behind for the rows of the view that fall outside [0, L_out). Channel counts that are not multiples of
64 (the last stage has 96) are zero-padded to the next multiple (weights, biases zero; Snake alpha one), which keeps the pad lanes 0.

forward_batch decodes latents of different lengths together: they are packed along time with zero gap rows between them
(varlen.dac_pack), the same launches run with B = 1 over the packed rows, and edm_dac_zero_rows clears the gap rows of every bf16
operand a multi-tap conv reads next, so each utterance sees exactly the zero padding it sees when decoded alone.
"""
from __future__ import annotations

import math

import torch

from . import _lib as L
from . import varlen
from .dac_encoder import _fold
from .varlen import conv_transpose_length

_G = 8          # guard rows in front of every stage buffer (>= the largest transposed-conv padding)
_FUSED = (128, 192)   # (padded) channel counts whose ResidualUnits run as one launch (edm_dac_resunit)


def _pad64(c):
    return (c + 63) // 64 * 64


def pack_conv_transpose(wt: torch.Tensor, stride: int, c_out_pad: int) -> torch.Tensor:
    """ConvTranspose1d weight [c_in, c_out, 2 * stride] (weight-norm folded) -> [stride * c_out_pad, 2 * c_in] fp32 for the 2-tap conv
    of the module docstring: row = phase r * c_out_pad + co, K = tap j * c_in + ci, tap 0 reads x[q - 1] (u = 1), tap 1 reads x[q]."""
    c_in, c_out, k = wt.shape
    assert k == 2 * stride
    wp = torch.zeros(stride, c_out_pad, 2, c_in, dtype=torch.float32)
    for j in range(2):
        wp[:, :c_out, j, :] = wt[:, :, (1 - j) * stride:(2 - j) * stride].permute(2, 1, 0)
    return wp.reshape(stride * c_out_pad, 2 * c_in)


class DACDecoder:
    def __init__(self, state_dict: dict, input_channel: int = 1024, channels: int = 1536, rates=(8, 5, 4, 2), prefix: str = "",
                 device="cuda", max_chunk_samples: int = 1 << 21):
        if not torch.cuda.is_available():
            raise L.EdmError("edm_tts_b200 needs a CUDA device (sm_100); there is no CPU fallback")
        if input_channel % 64 != 0 or channels % 64 != 0 or channels > 1536 or max(rates) // 2 > _G:
            raise ValueError("the conv kernels need input / first-stage channel counts that are multiples of 64 (first stage <= 1536)")
        self.device = dev = torch.device(device)
        self.input_channel, self.channels, self.rates = input_channel, channels, tuple(rates)
        self.hop_length = math.prod(rates)
        self.max_chunk_samples = max_chunk_samples
        sd = {k: v.detach().to("cpu") for k, v in state_dict.items() if k.startswith(prefix)}

        def padded(v, n, fill=0.0):
            out = torch.full((n,), fill, dtype=torch.float32)
            out[: v.numel()] = v.float().reshape(-1)
            return out.to(dev).contiguous()

        def conv(key, c_in_p, c_out_p):
            w = _fold(sd, key)                                                   # [c_out, c_in, k]
            wp = torch.zeros(c_out_p, w.shape[2], c_in_p)
            wp[: w.shape[0], :, : w.shape[1]] = w.permute(0, 2, 1)               # K index = tap * c_in_p + channel
            return wp.reshape(c_out_p, -1).to(dev, torch.bfloat16).contiguous(), padded(sd[key + ".bias"], c_out_p)

        def alpha(key, n):
            return padded(sd[key + ".alpha"], n, 1.0)

        self.w_first, self.b_first = conv(f"{prefix}model.0", input_channel, channels)
        self.blocks = []
        c_in = channels
        n = 1
        for i, s in enumerate(self.rates):
            c_out = channels // 2 ** (i + 1)
            cp = _pad64(c_out)
            blk = f"{prefix}model.{n}.block."
            wt = _fold(sd, blk + "1")                                            # [c_in, c_out, 2s], normalised per input channel
            wp = pack_conv_transpose(wt, s, cp)
            units = []
            for u in range(3):
                ru = f"{blk}{2 + u}.block."
                w7, b7 = conv(ru + "1", cp, cp)
                w1, b1 = conv(ru + "3", cp, cp)
                units.append(dict(a_in=alpha(ru + "0", cp), w7=w7, b7=b7, a_mid=alpha(ru + "2", cp), w1=w1, b1=b1))
            self.blocks.append(dict(stride=s, c_in=c_in, c=cp, a_up=alpha(blk + "0", c_in), wt=wp.to(dev, torch.bfloat16).contiguous(),
                                    bt=padded(sd[blk + "1.bias"], cp), units=units))
            c_in = cp
            n += 1
        c_last = channels // 2 ** len(self.rates)
        self.a_last = alpha(f"{prefix}model.{n}", c_in)
        w_last = _fold(sd, f"{prefix}model.{n + 1}")                             # [1, c_last, 7]
        wl = torch.zeros(7, c_in)
        wl[:, :c_last] = w_last[0].t()
        self.w_last = wl.to(dev).contiguous()
        self.b_last = float(sd[f"{prefix}model.{n + 1}.bias"].reshape(-1)[0])
        self._ws = {}
        self._pws = None

    def eval(self):
        return self

    # ------------------------------------------------------------------ geometry / workspace
    def lengths(self, T: int):
        """Time lengths after the first conv and after each transposed conv: (L - 1) s - 2 floor(s/2) + 2 s + s % 2."""
        out = [T]
        for s in self.rates:
            out.append(conv_transpose_length(out[-1], s))
        return out

    def _alloc(self, B: int, lens):
        """Stage buffers for B sequences of lens[k] rows at stage k."""
        dev = self.device
        T = lens[0]
        ws = dict(lens=lens, zin=torch.empty(B, T, self.input_channel, device=dev, dtype=torch.bfloat16),
                  s0=torch.empty(B, T, self.channels, device=dev, dtype=torch.bfloat16), y=[], sa=[], sb=[], sm=[], rows=[])
        for k, blk in enumerate(self.blocks):
            Lk, c = lens[k + 1], blk["c"]
            rows = _G + Lk + blk["stride"] + 8                                    # guard | L_k rows | tail for the view's last rows
            ws["rows"].append(rows)
            ws["y"].append(torch.empty(B, rows, c, device=dev, dtype=torch.float32))
            ws["sa"].append(torch.empty(B, rows, c, device=dev, dtype=torch.bfloat16))
            ws["sb"].append(torch.empty(B, rows, c, device=dev, dtype=torch.bfloat16))
            ws["sm"].append(None if c in _FUSED else torch.empty(B, Lk, c, device=dev, dtype=torch.bfloat16))
        ws["audio"] = torch.empty(B, lens[-1], device=dev, dtype=torch.float32)
        return ws

    def _workspace(self, B: int, T: int):
        key = (B, T)
        ws = self._ws.get(key)
        if ws is not None:
            return ws
        # keep two geometries (a batch that does not divide into equal chunks alternates between two chunk sizes; re-allocating
        # per chunk costs more than the kernels), drop the oldest beyond that: the buffers are large
        while len(self._ws) >= 2:
            self._ws.pop(next(iter(self._ws)))
        ws = self._alloc(B, self.lengths(T))
        self._ws[key] = ws
        return ws

    def _packed_workspace(self, rows0: int):
        """Grow-only workspace of the packed path, sized for rows0 packed latent rows (stage k: rows0 * r_1 ... r_k rows). The chunks
        of a list have different geometries; re-allocating per chunk would cost more than the kernels."""
        if self._pws is None or self._pws["lens"][0] < rows0:
            self._pws = None                                                     # release the smaller one first
            lens = [rows0]
            for s in self.rates:
                lens.append(lens[-1] * s)
            self._pws = self._alloc(1, lens)
        return self._pws

    # ------------------------------------------------------------------ launches (raw addresses: the stage buffers are used through
    # views that start at a guard-row offset)
    def _conv(self, a_ptr, a_rows, a_cols, a_bs, w, bias, taps, step, off, rows_out, B, alpha=None, period=0, x_res=None, y=None, y_bs=0,
              s_out=None, s_bs=0, s_rows=0):
        L.check(L.lib().edm_dac_conv(a_ptr, a_rows, a_cols, a_bs, B, L.ptr(w), w.shape[0], taps, step, off, rows_out, L.ptr(bias), L.ptr(alpha),
                                     period, x_res, y, y_bs, s_out, s_bs, 0, s_rows, None, 0, L.stream_ptr()), "dac_conv")

    def _resunit(self, a_ptr, a_bs, B, rows, c, dilation, ru, a_next, y_ptr, y_bs, s_ptr, s_bs):
        L.check(L.lib().edm_dac_resunit(a_ptr, a_bs, B, rows, c, dilation, L.ptr(ru["w7"]), L.ptr(ru["w1"]), L.ptr(ru["b7"]), L.ptr(ru["a_mid"]),
                                        L.ptr(ru["b1"]), L.ptr(a_next), y_ptr, y_bs, s_ptr, s_bs, 0, rows, L.stream_ptr()), "dac_resunit")

    @torch.no_grad()
    def forward(self, z: torch.Tensor) -> torch.Tensor:
        """z [B, input_channel, T] (fp32 / bf16) -> audio fp32 [B, 1, L]."""
        if z.dim() != 3 or z.shape[1] != self.input_channel:
            raise ValueError(f"z must be [B, {self.input_channel}, T]")
        z = z.to(self.device)
        B, _, T = z.shape
        if T < 1:
            raise ValueError("empty latent")
        L_out = self.lengths(T)[-1]
        audio = torch.empty(B, 1, L_out, device=self.device, dtype=torch.float32)
        per = max(1, self.max_chunk_samples // L_out)
        for b0 in range(0, B, per):
            audio[b0:b0 + per, 0] = self._forward_chunk(z[b0:b0 + per])
        return audio

    __call__ = forward

    def _forward_chunk(self, z):
        B, _, T = z.shape
        ws = self._workspace(B, T)
        ws["zin"].copy_(z.transpose(1, 2))                                       # channel-last bf16 operand (no Snake before the first conv)
        return self._run(ws, B, ws["lens"])

    def _run(self, ws, B, lens, clear=None, audio=None):
        """The decoder's launches over ws (stage k holds lens[k] rows per sequence) into audio (default: the workspace's).
        clear(k, ptr, pitch_bytes), when given, runs after every launch whose bf16 operand output at stage k a multi-tap conv reads
        next."""
        audio = ws["audio"] if audio is None else audio
        T = lens[0]
        first_alpha = self.blocks[0]["a_up"]
        # first conv k=7 (decoder.py:45): only the Snake'd operand of the first transposed conv is needed
        self._conv(ws["zin"].data_ptr(), T, self.input_channel, T * self.input_channel, self.w_first, self.b_first, 7, 1, -3, T, B, alpha=first_alpha,
                   s_out=ws["s0"].data_ptr(), s_bs=T * self.channels, s_rows=T)
        if clear:
            clear(0, ws["s0"].data_ptr(), self.channels * 2)
        src_ptr, src_rows, src_bs = ws["s0"].data_ptr(), T, T * self.channels
        for k, blk in enumerate(self.blocks):
            s, c, c_in, Lk, rows = blk["stride"], blk["c"], blk["c_in"], lens[k + 1], ws["rows"][k]
            y, sa, sb = ws["y"][k], ws["sa"][k], ws["sb"][k]
            bs = rows * c
            pad = s // 2
            # transposed conv as a 2-tap conv into the output view that starts `pad` rows before row 0 of the stage buffers
            self._conv(src_ptr, src_rows, c_in, src_bs, blk["wt"], blk["bt"], 2, 1, -1, src_rows + 1, B, alpha=blk["units"][0]["a_in"], period=c,
                       y=y.data_ptr() + (_G - pad) * c * 4, y_bs=bs, s_out=sa.data_ptr() + (_G - pad) * c * 2, s_bs=bs, s_rows=src_rows + 1)
            if clear:
                clear(k + 1, sa.data_ptr() + _G * c * 2, c * 2)
            y_ptr = y.data_ptr() + _G * c * 4
            cur, oth = sa, sb
            for u, ru in enumerate(blk["units"]):
                d = 3 ** u
                if u < 2:
                    a_next = blk["units"][u + 1]["a_in"]
                else:
                    a_next = self.blocks[k + 1]["a_up"] if k + 1 < len(self.blocks) else self.a_last
                cur_ptr, oth_ptr = cur.data_ptr() + _G * c * 2, oth.data_ptr() + _G * c * 2
                if c in _FUSED:
                    self._resunit(cur_ptr, bs, B, Lk, c, d, ru, a_next, y_ptr, bs, oth_ptr, bs)
                else:
                    sm = ws["sm"][k]
                    self._conv(cur_ptr, Lk, c, bs, ru["w7"], ru["b7"], 7, d, -3 * d, Lk, B, alpha=ru["a_mid"], s_out=sm.data_ptr(), s_bs=Lk * c, s_rows=Lk)
                    self._conv(sm.data_ptr(), Lk, c, Lk * c, ru["w1"], ru["b1"], 1, 1, 0, Lk, B, alpha=a_next, x_res=y_ptr, y=y_ptr, y_bs=bs,
                               s_out=oth_ptr, s_bs=bs, s_rows=Lk)
                if clear:
                    clear(k + 1, oth_ptr, c * 2)
                cur, oth = oth, cur
            src_ptr, src_rows, src_bs = cur.data_ptr() + _G * c * 2, Lk, bs
        L.check(L.lib().edm_dac_conv_last(src_ptr, src_bs, B, src_rows, self.blocks[-1]["c"], L.ptr(self.w_last), self.b_last, L.ptr(audio), 1,
                                          L.stream_ptr()), "dac_conv_last")
        return audio

    # ------------------------------------------------------------------ utterances of different lengths
    @torch.no_grad()
    def forward_batch(self, zs) -> list:
        """List of latents [input_channel, T_i] (fp32 / bf16, T_i >= 1) -> list of fp32 [1, L_i] views of one packed output,
        L_i = lengths(T_i)[-1]. Item i equals forward(zs[i][None])[0] bit for bit."""
        if not isinstance(zs, (list, tuple)) or len(zs) == 0:
            raise ValueError("zs must be a non-empty list of [input_channel, T_i] latents")
        for z in zs:
            if not torch.is_tensor(z) or z.dim() != 2 or z.shape[0] != self.input_channel:
                raise ValueError(f"every latent must be [{self.input_channel}, T_i]")
            if z.shape[1] < 1:
                raise ValueError("empty latent")
        T = [int(z.shape[1]) for z in zs]
        # fp32 -> bf16 rounds exactly as forward's copy into its bf16 operand does
        z = torch.cat([z.to(self.device, torch.bfloat16) for z in zs], dim=1)
        return self._forward_packed(z, T)

    def _forward_packed(self, z, T):
        """z [input_channel, sum(T)]: the latents of the list back to back -> list of [1, L_i] audio views."""
        plan = varlen.dac_plan(T, self.rates, self.max_chunk_samples)
        out = torch.empty(sum(ch.rows[-1] for ch in plan), device=self.device, dtype=torch.float32)
        ws = self._packed_workspace(max(ch.rows[0] for ch in plan))
        # one upload per call: the gap ranges of every chunk and stage ((start, end) pairs), then the packed row of every latent frame
        host, at = [], []
        for ch in plan:
            at.append([])
            for k in range(len(self.rates) + 1):
                g = ch.gaps(k)
                at[-1].append((len(host), len(g), max(e - b for b, e in g)))
                host += g
        n_pairs = len(host)
        host = [v for g in host for v in g] + [a + t for ch in plan for a, n in zip(ch.starts[0], ch.lengths[0]) for t in range(n)]
        dev_buf = torch.tensor(host, dtype=torch.int32).to(self.device)
        rows_of_frame = dev_buf[2 * n_pairs:].long()
        zin = ws["zin"][0]
        views, o0 = [], 0
        for ch, at_ch in zip(plan, at):
            def clear(k, ptr, pitch, at_ch=at_ch):
                first, n, widest = at_ch[k]
                self._zero_rows(ptr, pitch, dev_buf.data_ptr() + 8 * first, n, widest)

            t1 = ch.t0 + sum(ch.lengths[0])
            zin.index_copy_(0, rows_of_frame[ch.t0:t1], z[:, ch.t0:t1].t())
            clear(0, zin.data_ptr(), self.input_channel * 2)                     # latent gaps: the first conv's zero padding
            self._run(ws, 1, ch.rows, clear, audio=out[o0:o0 + ch.rows[-1]])
            views += [out[o0 + a:o0 + a + n].view(1, n) for a, n in zip(ch.starts[-1], ch.lengths[-1])]
            o0 += ch.rows[-1]
        return views

    def _zero_rows(self, ptr, pitch, ranges_ptr, n, widest):
        L.check(L.lib().edm_dac_zero_rows(ptr, pitch, ranges_ptr, n, widest, L.stream_ptr()), "dac_zero_rows")
