"""Host side shared by the DAC conv stacks (DACEncoder, DACDecoder): weight packing, the workspace caches, the edm_dac_conv /
edm_dac_resunit launches and the gap-row clears of the packed paths (varlen.dac_pack / enc_pack)."""
from __future__ import annotations

import torch

from . import _lib as L
from .weights import weight_norm_fold


def _fold(sd, key):
    """weight_norm (dim 0) of a conv, in fp32: w = g * v / ||v||, the norm taken over (in, k) per output channel (nn_layers.py:8-9)."""
    return weight_norm_fold(sd[key + ".parametrizations.weight.original0"].float(), sd[key + ".parametrizations.weight.original1"].float())


def padded(v, n: int, fill: float, device) -> torch.Tensor:
    """v flattened to fp32 and extended with `fill` to n entries, on device."""
    out = torch.full((n,), fill, dtype=torch.float32)
    out[: v.numel()] = v.float().reshape(-1)
    return out.to(device).contiguous()


def pack_conv(sd, key, c_in_pad: int, c_out_pad: int, device):
    """Weight-normed Conv1d `key` -> (bf16 [c_out_pad, k * c_in_pad] with K index = tap * c_in_pad + channel, fp32 bias [c_out_pad]);
    the pad rows, columns and bias entries are zero."""
    w = _fold(sd, key)                                                           # [c_out, c_in, k]
    wp = torch.zeros(c_out_pad, w.shape[2], c_in_pad)
    wp[: w.shape[0], :, : w.shape[1]] = w.permute(0, 2, 1)
    return wp.reshape(c_out_pad, -1).to(device, torch.bfloat16).contiguous(), padded(sd[key + ".bias"], c_out_pad, 0.0, device)


def pack_alpha(sd, key, n: int, device) -> torch.Tensor:
    """Snake alpha of `key` as fp32 [n]; pad channels get alpha one (Snake(0) = 0 keeps them zero)."""
    return padded(sd[key + ".alpha"], n, 1.0, device)


class ConvStack:
    """Base of DACEncoder and DACDecoder. A subclass supplies lengths(L) (rows of every stage for an input of L rows) and
    _alloc(B, lens) (the stage buffers for B sequences of lens[k] rows at stage k, a dict that keeps lens under "lens")."""

    def __init__(self, device, max_chunk_samples: int):
        if not torch.cuda.is_available():
            raise L.EdmError("edm_tts_b200 needs a CUDA device (sm_100); there is no CPU fallback")
        self.device = torch.device(device)
        self.max_chunk_samples = max_chunk_samples
        self._ws = {}
        self._pws = None

    def eval(self):
        return self

    # ------------------------------------------------------------------ workspaces
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

    def _packed_workspace(self, rows):
        """Grow-only workspace of the packed path, sized for the stage rows `rows` of a list's largest chunk. The chunks of a list have
        different geometries; re-allocating per chunk would cost more than the kernels."""
        if self._pws is None or self._pws["lens"][0] < rows[0]:
            self._pws = None                                                     # release the smaller one first
            self._pws = self._alloc(1, rows)
        return self._pws

    # ------------------------------------------------------------------ gap rows of the packed path
    def _upload_gaps(self, lists, extra=()):
        """One host-to-device copy of every chunk's gap ranges: lists[c][j] is list j of chunk c, (start, end) row pairs; the ints of
        `extra` follow the pairs in the same buffer. -> (int32 device buffer, per chunk a clear(j, ptr, pitch_bytes) that zeroes the
        rows of list j in the buffer at ptr)."""
        host, at = [], []
        for chunk in lists:
            at.append([])
            for g in chunk:
                at[-1].append((len(host), len(g), max(e - b for b, e in g)))
                host += g
        buf = torch.tensor([v for g in host for v in g] + list(extra), dtype=torch.int32).to(self.device)

        def clear_fn(at_ch):
            def clear(j, ptr, pitch):
                first, n, widest = at_ch[j]
                self._zero_rows(ptr, pitch, buf.data_ptr() + 8 * first, n, widest)
            return clear

        return buf, [clear_fn(at_ch) for at_ch in at]

    def _zero_rows(self, ptr, pitch, ranges_ptr, n, widest):
        L.check(L.lib().edm_dac_zero_rows(ptr, pitch, ranges_ptr, n, widest, L.stream_ptr()), "dac_zero_rows")

    # ------------------------------------------------------------------ launches (raw addresses and batch strides in elements: stage
    # buffers are used through views that start at an offset)
    def _conv(self, a, a_rows, a_cols, a_bs, w, bias, taps, step, off, rows_out, B, alpha=None, period=0, x_res=None, y=None, y_bs=0,
              s_out=None, s_bs=0, s_row_off=0, s_rows=0, zt=None, zt_f32=0):
        L.check(L.lib().edm_dac_conv(a, a_rows, a_cols, a_bs, B, L.ptr(w), w.shape[0], taps, step, off, rows_out, L.ptr(bias), L.ptr(alpha),
                                     period, x_res, y, y_bs, s_out, s_bs, s_row_off, s_rows, zt, zt_f32, L.stream_ptr()), "dac_conv")

    def _resunit(self, a, a_bs, B, rows, c, dilation, ru, a_next, y, y_bs, s_out, s_bs, s_row_off, s_rows):
        L.check(L.lib().edm_dac_resunit(a, a_bs, B, rows, c, dilation, L.ptr(ru["w7"]), L.ptr(ru["w1"]), L.ptr(ru["b7"]), L.ptr(ru["a_mid"]),
                                        L.ptr(ru["b1"]), L.ptr(a_next), y, y_bs, s_out, s_bs, s_row_off, s_rows, L.stream_ptr()), "dac_resunit")
