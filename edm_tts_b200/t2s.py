"""Host-side mirror of the reference's text-to-semantic model on the C ABI (libedm_s2a.so, edm_t2s_*).

Mirrors edm_tts/models/text_to_semantic/modeling_text_to_semantic.py:26-267 (TextToSemanticWLen): same constructor inputs (config +
state dict / HF directory), `infer(text, pred_iters, temperature, gt_length)` with the reference's argument meaning and return type
(`.speech_pred_tokens`), `embeddings_to_logits`. `infer` decodes one sequence per call, as in the reference; `infer_batch` decodes
a list of texts of different lengths together, packed back to back without padding; `infill_batch` regenerates chosen semantic
tokens of utterances given their transcripts and the other tokens (speech editing). All arithmetic runs in the CUDA kernels; the only
host round trip is the predicted length (it fixes the shape of everything after it): one read per call, or per chunk of a batch.
No CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import math
import os

import torch

from . import _lib as L
from . import varlen
from .config import TextToSemanticWLenConfig
from .s2a import MAX_CHUNK, _check_range, _on_device
from .weights import glu_interleave


class TextToSemanticWLenOutput(dict):
    """modeling_text_to_semantic.py:17-23 (a transformers ModelOutput there): attribute and key access."""

    def __init__(self, loss=None, ce_loss=None, length_loss=None, prompt_kl_loss=None, speech_pred_tokens=None):
        super().__init__(loss=loss, ce_loss=ce_loss, length_loss=length_loss, prompt_kl_loss=prompt_kl_loss, speech_pred_tokens=speech_pred_tokens)
        self.__dict__ = self


def _pad_heads(w: torch.Tensor, heads: int, axis: int) -> torch.Tensor:
    """[heads * dh] along `axis` -> [heads * 64]: dims [0, dh/2) of every head go to columns [0, dh/2), dims [dh/2, dh) to columns
    [32, 32 + dh/2), zeros elsewhere. The rotary epilogue pairs column j with column j + 32 of a 64-wide head, which then is
    exactly rotate_half's pairing (j, j + dh/2) (conformer/conformer.py:45-51); q.k and the output projection only need the same
    placement on both sides."""
    w = w.movedim(axis, 0)
    dh = w.shape[0] // heads
    half = dh // 2
    src = w.reshape(heads, dh, *w.shape[1:])
    out = torch.zeros(heads, 64, *w.shape[1:], dtype=w.dtype, device=w.device)
    out[:, :half] = src[:, :half]
    out[:, 32:32 + half] = src[:, half:]
    return out.reshape(heads * 64, *w.shape[1:]).movedim(0, axis).contiguous()


def _rope_tables(max_positions: int, dim_head: int, device):
    """RotaryEmbedding.forward (conformer/conformer.py:28-42) for dim_head <= 64, stored [pos, 32]: entries past dim_head / 2 are
    angle 0 (cos 1, sin 0) and only ever meet the zero padding columns."""
    inv_freq = 1.0 / (10000 ** (torch.arange(0, dim_head, 2, device=device).float() / dim_head))
    t = torch.arange(max_positions, device=device).type_as(inv_freq)
    freqs = torch.zeros(max_positions, 32, device=device)
    freqs[:, : dim_head // 2] = torch.einsum("i , j -> i j", t, inv_freq)
    return freqs.cos().contiguous(), freqs.sin().contiguous()


def pack_t2s_weights(sd: dict, cfg: TextToSemanticWLenConfig, device, max_positions: int) -> dict:
    """Reference state dict (TextToSemanticWLen.state_dict()) -> {abi_name: contiguous CUDA tensor}; KeyError on a missing key."""
    d = cfg.hidden_size
    f32 = lambda t: t.to(device=device, dtype=torch.float32).contiguous()
    bf16 = lambda t: t.to(device=device, dtype=torch.float32).to(torch.bfloat16).contiguous()
    out = {}

    def block(p, o, heads):
        for ff in ("ff1", "ff2"):
            out[o + ff + "_ln_w"] = f32(sd[p + ff + ".fn.norm.weight"])
            out[o + ff + "_ln_b"] = f32(sd[p + ff + ".fn.norm.bias"])
            out[o + ff + "_w1"] = bf16(sd[p + ff + ".fn.fn.net.0.weight"])
            out[o + ff + "_b1"] = f32(sd[p + ff + ".fn.fn.net.0.bias"])
            out[o + ff + "_w2"] = bf16(sd[p + ff + ".fn.fn.net.3.weight"])
            out[o + ff + "_b2"] = f32(sd[p + ff + ".fn.fn.net.3.bias"])
        out[o + "attn_ln_w"] = f32(sd[p + "attn.norm.weight"])
        out[o + "attn_ln_b"] = f32(sd[p + "attn.norm.bias"])
        wq, wkv = sd[p + "attn.fn.to_q.weight"], sd[p + "attn.fn.to_kv.weight"]
        out[o + "wqkv"] = bf16(torch.cat([_pad_heads(wq, heads, 0), _pad_heads(wkv[:d], heads, 0), _pad_heads(wkv[d:], heads, 0)], dim=0))
        out[o + "wo"] = bf16(_pad_heads(sd[p + "attn.fn.to_out.weight"], heads, 1))
        out[o + "bo"] = f32(sd[p + "attn.fn.to_out.bias"])
        out[o + "conv_ln_w"] = f32(sd[p + "conv.net.0.weight"])
        out[o + "conv_ln_b"] = f32(sd[p + "conv.net.0.bias"])
        perm = glu_interleave(sd[p + "conv.net.2.weight"].shape[0])
        out[o + "pw1_w"] = bf16(sd[p + "conv.net.2.weight"][:, :, 0][perm])
        out[o + "pw1_b"] = f32(sd[p + "conv.net.2.bias"][perm])
        out[o + "dw_w"] = f32(sd[p + "conv.net.4.conv.weight"][:, 0, :].to(torch.bfloat16).float())
        out[o + "dw_b"] = f32(sd[p + "conv.net.4.conv.bias"])
        out[o + "cln_w"] = f32(sd[p + "conv.net.6.weight"].reshape(-1))
        out[o + "pw2_w"] = bf16(sd[p + "conv.net.7.weight"][:, :, 0])
        out[o + "pw2_b"] = f32(sd[p + "conv.net.7.bias"])
        out[o + "post_ln_w"] = f32(sd[p + "post_norm.weight"])
        out[o + "post_ln_b"] = f32(sd[p + "post_norm.bias"])

    main, lp = cfg.main_encoder_args, cfg.length_predictor_args
    for i in range(int(main["depth"])):
        block(f"conformer.layers.{i}.", f"blocks.{i}.", int(main["heads"]))
    for i in range(int(lp["depth"])):
        block(f"length_predictor.layers.{i}.", f"lp_blocks.{i}.", int(lp["heads"]))
    out["emb"] = f32(sd["input_embedding.weight"])
    out["length_token"] = f32(sd["length_token"].reshape(-1))
    out["pt_w"] = bf16(sd["pred_transform.0.weight"])
    out["pt_b"] = f32(sd["pred_transform.0.bias"])
    out["pt_ln_w"] = f32(sd["pred_transform.2.weight"])
    out["pt_ln_b"] = f32(sd["pred_transform.2.bias"])
    out["head_w"] = bf16(sd["pred_head.weight"])
    out["head_b"] = f32(sd["pred_head.bias"])
    out["len_w"] = f32(sd["length_pred_head.weight"].reshape(-1))
    out["len_b"] = f32(sd["length_pred_head.bias"].reshape(-1))
    out["rope_cos"], out["rope_sin"] = _rope_tables(max_positions, d // int(main["heads"]), device)
    out["lp_rope_cos"], out["lp_rope_sin"] = _rope_tables(max_positions, d // int(lp["heads"]), device)
    return out


class TextToSemanticWLen:
    """Drop-in for the reference TextToSemanticWLen on the decode path (inference only): `infer` decodes one utterance per call as
    the reference does, `infer_batch` a list of them in one packed decode."""

    def __init__(self, config, state_dict: dict, device="cuda", max_positions: int = 2048):
        if not torch.cuda.is_available():
            raise L.EdmError("edm_tts_b200 needs a CUDA device (sm_100); there is no CPU fallback")
        self.config = cfg = TextToSemanticWLenConfig.from_any(config)
        self.device = torch.device(device)
        self.num_special_tokens = len(cfg.special_tokens)
        self.total_num_tokens = cfg.text_vocab_size + cfg.semantic_vocab_size + self.num_special_tokens
        self.pad_token_id = cfg.special_tokens["pad"]
        self.dim = cfg.hidden_size
        self.max_positions = int(max_positions)
        lib = L.lib()
        c = L.T2SConfig()
        main, lp = cfg.main_encoder_args, cfg.length_predictor_args
        c.hidden, c.heads, c.depth, c.lp_heads, c.lp_depth = cfg.hidden_size, int(main["heads"]), int(main["depth"]), int(lp["heads"]), int(lp["depth"])
        c.ff_mult, c.conv_kernel = int(main.get("ff_mult", 4)), int(main.get("conv_kernel_size", 5))
        if (int(lp.get("ff_mult", 4)), int(lp.get("conv_kernel_size", 5))) != (c.ff_mult, c.conv_kernel):
            raise ValueError("length predictor and main encoder must share ff_mult / conv_kernel_size")
        c.text_vocab, c.semantic_vocab, c.num_special, c.max_positions = cfg.text_vocab_size, cfg.semantic_vocab_size, self.num_special_tokens, self.max_positions
        self._cfg_c = c
        n = lib.edm_t2s_num_weights(C.byref(c))
        if n <= 0:
            raise ValueError("unsupported text-to-semantic configuration: " + lib.edm_last_error().decode())
        # the batch context (infer_batch / predict_length_batch) shares the weights; it is created and bound on first use
        self._bctx, self._bws, self._bcap = None, None, (0, 0)
        self.low_latency = True
        with torch.cuda.device(self.device):
            self._w = pack_t2s_weights(state_dict, cfg, self.device, self.max_positions)
            names = [lib.edm_t2s_weight_name(C.byref(c), i).decode() for i in range(n)]
            self._wptrs = (C.c_void_p * n)(*[self._w[name].data_ptr() for name in names])
            self._ctx = self._create_ctx()
            need = lib.edm_t2s_workspace_bytes(self._ctx, self.max_positions)
            self._ws = torch.empty(need, device=self.device, dtype=torch.uint8)
            L.check(lib.edm_t2s_bind(self._ctx, self._ws.data_ptr(), need, self.max_positions), "bind")
        self.training = False

    def _create_ctx(self):
        lib = L.lib()
        ctx = lib.edm_t2s_create(C.byref(self._cfg_c), self._wptrs, len(self._wptrs))
        if not ctx:
            raise L.EdmError("edm_t2s_create failed: " + lib.edm_last_error().decode())
        return ctx

    @classmethod
    def from_pretrained(cls, path: str, device="cuda", **kw):
        """HF directory (config.json + model.safetensors) as written by the reference's save_pretrained."""
        from safetensors.torch import load_file

        return cls(TextToSemanticWLenConfig.from_pretrained(path), load_file(os.path.join(path, "model.safetensors")), device=device, **kw)

    def eval(self):
        return self

    def train(self, mode: bool = True):
        if mode:
            raise NotImplementedError("edm_tts_b200.TextToSemanticWLen is inference-only; train with the reference")
        return self

    def to(self, *args, **kwargs):
        dev = kwargs.get("device", next((a for a in args if isinstance(a, (str, torch.device, int))), None))
        if dev is not None:
            dev = torch.device("cuda", dev) if isinstance(dev, int) else torch.device(dev)
            if dev.type != "cuda" or (dev.index is not None and self.device.index is not None and dev.index != self.device.index):
                raise ValueError(f"model lives on {self.device}; construct it with device={dev!s} instead of moving it (there is no CPU path)")
        return self

    def __del__(self):
        try:
            for name in ("_ctx", "_bctx"):
                if getattr(self, name, None):
                    L.lib().edm_t2s_destroy(getattr(self, name))
                    setattr(self, name, None)
        except Exception:
            pass

    # ------------------------------------------------------------------ plumbing
    def _view(self, name, shape, dtype):
        nbytes = C.c_size_t(0)
        p = L.lib().edm_t2s_buffer(self._ctx, name.encode(), C.byref(nbytes))
        if not p:
            raise L.EdmError(f"no workspace buffer {name}")
        off = p - self._ws.data_ptr()
        numel = math.prod(shape)
        esz = torch.empty(0, dtype=dtype).element_size()
        assert numel * esz <= nbytes.value, (name, shape, nbytes.value)
        return self._ws[off:off + numel * esz].view(dtype).view(*shape)

    def _bind_batch(self, rows, n_seq):
        """The batch context with a workspace for n_seq sequences of `rows` rows in all (grown, never shrunk)."""
        if self._bctx is None:
            self._bctx = self._create_ctx()
        if rows <= self._bcap[0] and n_seq <= self._bcap[1]:
            return self._bctx
        lib = L.lib()
        cap = (max(rows, self._bcap[0]), max(n_seq, MAX_CHUNK))
        need = lib.edm_t2s_workspace_bytes_batch(self._bctx, *cap)
        if need == 0:
            raise ValueError(f"invalid batch capacity {cap}")
        self._bws, self._bcap = None, (0, 0)
        self._bws = torch.empty(need, device=self.device, dtype=torch.uint8)
        L.check(lib.edm_t2s_bind_batch(self._bctx, self._bws.data_ptr(), need, *cap), "bind_batch")
        self._bcap = cap
        return self._bctx

    def set_low_latency(self, on=True):
        """on (the default): `infer` splits its long-K residual GEMMs over K, faster for one utterance (edm_t2s_set_low_latency). The
        split changes the fp32 summation order, so with it `infer` does not give the bits of the same utterance in `infer_batch`,
        which never splits; off, it does (with batch_offset = the utterance's index in the batch)."""
        L.check(L.lib().edm_t2s_set_low_latency(self._ctx, int(bool(on))), "set_low_latency")
        self.low_latency = bool(on)
        return self

    def text_tokens(self, text) -> torch.Tensor:
        """:193-194: utf-8 bytes shifted past the special tokens (int32 on the device). A LongTensor of already shifted tokens passes through."""
        if torch.is_tensor(text):
            _check_range(text, self.total_num_tokens, "text tokens")
            return text.to(self.device, torch.int32).contiguous()
        return (torch.tensor(list(text.encode("utf-8")), dtype=torch.int32) + self.num_special_tokens).to(self.device)

    # ------------------------------------------------------------------ the decode API
    @torch.no_grad()
    @_on_device
    def predict_length(self, text):
        """:198-203 -> (length, raw log-length). One device->host read of a single float."""
        tt = self.text_tokens(text)
        if tt.numel() + 1 > self.max_positions:
            raise ValueError(f"text of {tt.numel()} bytes exceeds max_positions={self.max_positions}")
        L.check(L.lib().edm_t2s_predict_length(self._ctx, L.ptr(tt) if tt.numel() else None, tt.numel(), None, L.stream_ptr()), "predict_length")
        raw = self._view("raw_len", (1,), torch.float32)
        length = int(raw.exp().ceil().long().item())
        return length, float(raw.item())

    @torch.no_grad()
    @_on_device
    def infer(self, text, pred_iters=10, temperature=1.0, gt_length=None, *, seed=0, batch_offset=0, cat_gumbel=None, remask_gumbel=None,
              forced_ids=None, forced_masks=None, **kwargs):
        """modeling_text_to_semantic.py:184-267 -> TextToSemanticWLenOutput(speech_pred_tokens=LongTensor[length]).
        seed / batch_offset drive the in-kernel Philox noise: position t draws counter batch_offset * L + t, what the utterance at
        index batch_offset of an infer_batch call draws. Keyword-only extras are for parity runs: injected noise (cat_gumbel
        [iters-1, L, 1024], remask_gumbel [iters-1, 1, L] with L = len(text bytes) + length + 4) and teacher forcing (forced_ids
        [iters, 1, L], forced_masks [iters-1, 1, L])."""
        tt = self.text_tokens(text)
        length = int(gt_length) if gt_length is not None else self.predict_length(tt)[0]
        if length < 1:
            raise ValueError(f"predicted length {length} < 1")
        n_text = tt.numel()
        Lseq = n_text + length + 4
        if Lseq > self.max_positions:
            raise ValueError(f"sequence of {Lseq} tokens exceeds max_positions={self.max_positions}")
        dev = self.device
        prep = lambda t, dt: None if (t is None or t.numel() == 0) else t.to(dev).to(dt).reshape(t.shape[0], -1).contiguous()
        cg = None if (cat_gumbel is None or cat_gumbel.numel() == 0) else cat_gumbel.to(dev).float().reshape(-1, Lseq, self.config.semantic_vocab_size).contiguous()
        rg, fi, fm = prep(remask_gumbel, torch.float32), prep(forced_ids, torch.int32), prep(forced_masks, torch.uint8)
        for name, t, rows in (("remask_gumbel", rg, pred_iters - 1), ("forced_ids", fi, pred_iters), ("forced_masks", fm, pred_iters - 1)):
            if t is not None and (t.shape[0] < rows or t.shape[1] != Lseq):
                raise ValueError(f"{name} must cover {rows} iterations x {Lseq} positions, got {tuple(t.shape)}")
        if cg is not None and cg.shape[0] < pred_iters - 1:
            raise ValueError("cat_gumbel must cover pred_iters - 1 iterations")
        out = torch.empty(length, device=dev, dtype=torch.int64)
        L.check(L.lib().edm_t2s_set_batch_offset(self._ctx, int(batch_offset)), "set_batch_offset")
        L.check(L.lib().edm_t2s_decode(self._ctx, L.ptr(tt) if n_text else None, n_text, length, int(pred_iters), float(temperature), int(seed),
                                       L.ptr(cg), L.ptr(rg), L.ptr(fi), L.ptr(fm), L.ptr(out), L.stream_ptr()), "t2s_decode")
        return TextToSemanticWLenOutput(speech_pred_tokens=out)

    @torch.no_grad()
    @_on_device
    def decode_trace(self, text, pred_iters=10, temperature=1.0, gt_length=None, *, seed=0, batch_offset=0, cat_gumbel=None, remask_gumbel=None,
                     forced_ids=None, forced_masks=None, semantic_tokens=None, regenerate=None):
        """infer run stage by stage through the entry points edm_t2s_decode composes; returns every intermediate. Parity tests only.
        With semantic_tokens / regenerate ([N] each, gt_length unused) it is the infill decode of infill_batch([text], [semantic_tokens],
        [regenerate]) instead, begun by edm_t2s_begin_masked; "tokens" then holds the regenerated positions."""
        lib, s_ = L.lib(), L.stream_ptr()
        tt = self.text_tokens(text)
        n_text = tt.numel()
        dev = self.device
        L.check(lib.edm_t2s_set_batch_offset(self._ctx, int(batch_offset)), "set_batch_offset")
        if regenerate is None:
            length = int(gt_length) if gt_length is not None else self.predict_length(tt)[0]
            n_out = length
            L.check(lib.edm_t2s_begin(self._ctx, L.ptr(tt) if n_text else None, n_text, length, s_), "begin")
        else:
            sp = varlen.t2s_infill_split([n_text], [semantic_tokens], [regenerate], self.config.semantic_vocab_size, self.max_positions)
            length, n_out = sp.N[0], sp.T[0]
            known = sp.known.to(dev, torch.int32)
            L.check(lib.edm_t2s_begin_masked(self._ctx, 1, L.ptr(tt) if n_text else None, (C.c_int * 1)(n_text), (C.c_int * 1)(length), L.ptr(known),
                                             sp.regenerate.data_ptr(), s_), "begin_masked")
        Lseq = n_text + length + 4
        tr = dict(step_logits=[], step_ids=[], step_masks=[], step_masks_raw=[], length=length,
                  input_ids=self._view("input_ids", (1, Lseq), torch.int32).clone().long(),
                  full_mask=self._view("full_mask", (1, Lseq), torch.uint8).clone().bool())
        for i in range(pred_iters):
            last = i == pred_iters - 1
            L.check(lib.edm_t2s_logits(self._ctx, None, s_), "logits")
            tr["step_logits"].append(self._view("logits", (1, Lseq, 1024), torch.float32).clone())
            cg = None if (cat_gumbel is None or last) else cat_gumbel[i].to(dev).float().reshape(Lseq, -1).contiguous()
            rg = None if (remask_gumbel is None or last) else remask_gumbel[i].to(dev).float().reshape(Lseq).contiguous()
            fi = None if forced_ids is None else forced_ids[i].to(dev).to(torch.int32).reshape(Lseq).contiguous()
            fm = None if (forced_masks is None or last) else forced_masks[i].to(dev).to(torch.uint8).reshape(Lseq).contiguous()
            L.check(lib.edm_t2s_step(self._ctx, i, int(pred_iters), float(temperature), int(seed), L.ptr(cg), L.ptr(rg), L.ptr(fi), L.ptr(fm), s_), "step")
            tr["step_ids"].append(self._view("ids_raw", (1, Lseq), torch.int32).clone().long())
            if not last:
                tr["step_masks"].append(self._view("mask", (1, Lseq), torch.uint8).clone().bool())
                tr["step_masks_raw"].append(self._view("mask_raw", (1, Lseq), torch.uint8).clone().bool())
        out = torch.empty(n_out, device=dev, dtype=torch.int64)
        L.check(lib.edm_t2s_result(self._ctx, L.ptr(out), s_), "result")
        tr["tokens"] = out
        return tr

    def _batch_tokens(self, texts):
        if not isinstance(texts, (list, tuple)) or len(texts) == 0:
            raise ValueError("texts must be a non-empty list of str or 1-D token tensors")
        for i, t in enumerate(texts):
            if torch.is_tensor(t) and t.dim() != 1:
                raise ValueError(f"texts[{i}] must be a str or a 1-D tensor of shifted tokens, got shape {tuple(t.shape)}")
        return [self.text_tokens(t) for t in texts]

    @staticmethod
    def _packed(tokens):
        """tokens of one chunk back to back (int32 on the device), or None when every text is empty"""
        n = sum(t.numel() for t in tokens)
        return torch.cat(tokens).contiguous() if n else None

    @torch.no_grad()
    @_on_device
    def predict_length_batch(self, texts):
        """predict_length for a list of texts in one pass per chunk of MAX_CHUNK -> (lengths, raw log-lengths), two lists. One
        device->host read per chunk. The raw values are the bits of predict_length(texts[i]) with set_low_latency(False)."""
        toks = self._batch_tokens(texts)
        n_text = [t.numel() for t in toks]
        for i, nt in enumerate(n_text):
            if nt + 1 > self.max_positions:
                raise ValueError(f"texts[{i}]: text of {nt} bytes exceeds max_positions={self.max_positions}")
        lib, lengths, raws = L.lib(), [], []
        for ch in varlen.plan(n_text, [0] * len(n_text), MAX_CHUNK):
            n = ch.stop - ch.start
            ctx = self._bind_batch(sum(ch.T) + n, n)
            raw = torch.empty(n, device=self.device, dtype=torch.float32)
            tt = self._packed(toks[ch.start:ch.stop])
            L.check(lib.edm_t2s_predict_length_batch(ctx, n, L.ptr(tt), (C.c_int * n)(*ch.T), L.ptr(raw), L.stream_ptr()), "predict_length_batch")
            # length as predict_length computes it (on the device), and the raw bits, in one read
            both = torch.stack([raw.exp().ceil().long(), raw.view(torch.int32).long()]).cpu()
            lengths += [int(x) for x in both[0]]
            raws += [float(x) for x in both[1].to(torch.int32).view(torch.float32)]
        return lengths, raws

    @torch.no_grad()
    @_on_device
    def infer_batch(self, texts, pred_iters=10, temperature=1.0, gt_lengths=None, *, seed=0, batch_offset=0, cat_gumbel=None, remask_gumbel=None,
                    forced_ids=None, forced_masks=None):
        """infer for a list of texts (str, or 1-D tensors of shifted tokens) of different lengths, decoded together without padding,
        in chunks of MAX_CHUNK utterances. Returns a list of LongTensor [length_i], views of one packed output. Without gt_lengths
        the lengths come from predict_length_batch. Utterance i decodes to the bits of infer(texts[i], ..., batch_offset=batch_offset
        + i) with set_low_latency(False). The keyword extras are per-utterance lists shaped as infer's extras for one utterance, with
        L_i = len(text_i bytes) + length_i + 4: cat_gumbel[i] [iters-1, L_i, 1024], remask_gumbel[i] [iters-1, 1, L_i], forced_ids[i]
        [iters, 1, L_i], forced_masks[i] [iters-1, 1, L_i]."""
        toks = self._batch_tokens(texts)
        n = len(toks)
        iters = int(pred_iters)
        if iters < 1:
            raise ValueError(f"pred_iters must be >= 1, got {pred_iters}")
        if gt_lengths is None:
            lengths = self.predict_length_batch(toks)[0]
        else:
            if len(gt_lengths) != n:
                raise ValueError(f"gt_lengths has {len(gt_lengths)} entries for {n} texts")
            lengths = [int(x) for x in gt_lengths]
        n_text = [t.numel() for t in toks]
        Lseq = [nt + ln + 4 for nt, ln in zip(n_text, lengths)]
        for i, ln in enumerate(lengths):
            if ln < 1:
                raise ValueError(f"utterance {i}: length {ln} < 1")
            if Lseq[i] > self.max_positions:
                raise ValueError(f"utterance {i}: sequence of {Lseq[i]} tokens exceeds max_positions={self.max_positions}")
        extras = self._check_extras(iters, Lseq, cat_gumbel=cat_gumbel, remask_gumbel=remask_gumbel, forced_ids=forced_ids, forced_masks=forced_masks)
        return self._decode_packed(toks, lengths, lengths, iters, temperature, seed, batch_offset, extras)

    @torch.no_grad()
    @_on_device
    def infill_batch(self, texts, semantic_tokens, regenerate, pred_iters=10, temperature=1.0, *, seed=0, batch_offset=0, cat_gumbel=None,
                     remask_gumbel=None, forced_ids=None, forced_masks=None):
        """Regenerates chosen semantic tokens of each utterance given its transcript and the rest (speech editing; with a known prefix,
        prompted continuation). texts: the transcript of the whole (edited) utterance, str or 1-D shifted-token tensors;
        semantic_tokens[i]: LongTensor [N_i], the values at regenerated positions are ignored; regenerate[i]: BoolTensor [N_i], at least
        one True. The decode is the reference's loop (:184-267) on [text] bytes [sep] [speech] s_1 .. s_N [sep] started from full_mask
        = regenerate: known positions hold their tokens and are never sampled or re-masked, and mask_len counts only the regenerated
        ones (edm_t2s_begin_masked). Returns a list of LongTensor [T_i] (T_i = regenerate[i].sum()), the regenerated tokens in time
        order, views of one packed output. With every position regenerated, utterance i decodes to the bits of infer_batch(texts,
        gt_lengths=N) at index i. Chunks of MAX_CHUNK and the parity extras are as in infer_batch, with L_i = len(text_i bytes) + N_i
        + 4. Malformed input raises ValueError naming the utterance."""
        toks = self._batch_tokens(texts)
        iters = int(pred_iters)
        if iters < 1:
            raise ValueError(f"pred_iters must be >= 1, got {pred_iters}")
        n_text = [t.numel() for t in toks]
        sp = varlen.t2s_infill_split(n_text, semantic_tokens, regenerate, self.config.semantic_vocab_size, self.max_positions)
        Lseq = [nt + n + 4 for nt, n in zip(n_text, sp.N)]
        extras = self._check_extras(iters, Lseq, cat_gumbel=cat_gumbel, remask_gumbel=remask_gumbel, forced_ids=forced_ids, forced_masks=forced_masks)
        return self._decode_packed(toks, list(sp.N), list(sp.T), iters, temperature, seed, batch_offset, extras, sp)

    def _check_extras(self, iters, Lseq, **extras):
        """the per-utterance parity extras of infer_batch / infill_batch: lists shaped as infer's extras, L_i positions each"""
        V, n = self.config.semantic_vocab_size, len(Lseq)
        shapes = dict(cat_gumbel=lambda l: (iters - 1, l, V), remask_gumbel=lambda l: (iters - 1, 1, l), forced_ids=lambda l: (iters, 1, l),
                      forced_masks=lambda l: (iters - 1, 1, l))
        for name, lst in extras.items():
            if lst is None:
                continue
            if not isinstance(lst, (list, tuple)) or len(lst) != n:
                raise ValueError(f"{name} must be a list with one entry per utterance")
            for i, x in enumerate(lst):
                if tuple(x.shape) != shapes[name](Lseq[i]):
                    raise ValueError(f"{name}[{i}] must be {shapes[name](Lseq[i])}, got {tuple(x.shape)}")
        return extras

    def _decode_packed(self, toks, lengths, out_lens, iters, temperature, seed, batch_offset, extras, infill=None):
        """The packed decode of infer_batch (infill None) or infill_batch (infill: the varlen.T2sInfill) in chunks of MAX_CHUNK:
        utterance i has toks[i] text tokens and lengths[i] speech positions, of which it returns out_lens[i]."""
        n, dev, lib = len(toks), self.device, L.lib()
        n_text = [t.numel() for t in toks]
        Lseq = [nt + ln + 4 for nt, ln in zip(n_text, lengths)]
        cu_len = varlen.offsets(lengths)
        known = None if infill is None else infill.known.to(dev, torch.int32)

        def cat(lst, sl, dim, dtype):
            if lst is None or lst[sl.start].shape[0] == 0:  # the [iters - 1, ...] extras of a 1-iteration decode are empty
                return None
            return torch.cat([x.to(dev) for x in lst[sl]], dim).to(dtype).contiguous()

        out = torch.empty(sum(out_lens), device=dev, dtype=torch.int64)
        for ch in varlen.plan(out_lens, [0] * n, MAX_CHUNK, batch_offset):
            sl, m = slice(ch.start, ch.stop), ch.stop - ch.start
            ctx = self._bind_batch(sum(Lseq[sl]), m)
            cg = cat(extras["cat_gumbel"], sl, 1, torch.float32)
            rg = cat(extras["remask_gumbel"], sl, 2, torch.float32)
            fi = cat(extras["forced_ids"], sl, 2, torch.int32)
            fm = cat(extras["forced_masks"], sl, 2, torch.uint8)
            tt = self._packed(toks[sl])
            args = (iters, float(temperature), int(seed), L.ptr(cg), L.ptr(rg), L.ptr(fi), L.ptr(fm), L.ptr(out[ch.t0:ch.t0 + sum(ch.T)]), L.stream_ptr())
            L.check(lib.edm_t2s_set_batch_offset(ctx, ch.batch_offset), "set_batch_offset")
            if infill is None:
                L.check(lib.edm_t2s_decode_batch(ctx, m, L.ptr(tt), (C.c_int * m)(*n_text[sl]), (C.c_int * m)(*lengths[sl]), *args), "t2s_decode_batch")
            else:
                a, b = cu_len[ch.start], cu_len[ch.stop]
                flags = infill.regenerate[a:b].contiguous()   # host bytes, read by the call before it returns
                L.check(lib.edm_t2s_decode_masked(ctx, m, L.ptr(tt), (C.c_int * m)(*n_text[sl]), (C.c_int * m)(*lengths[sl]), L.ptr(known[a:b]),
                                                  flags.data_ptr(), *args), "t2s_decode_masked")
        return [b[0] for b in varlen.split_blocks(out, out_lens, 1)]

    @torch.no_grad()
    @_on_device
    def embeddings_to_logits(self, embeddings, attention_mask=None, mask=None):
        """:135-152 for one un-padded sequence: embeddings [1, L, hidden] -> logits [1, L, 1024] (or [n_selected, 1024] with `mask`)."""
        if attention_mask is not None and not bool(attention_mask.all()):
            raise ValueError("padded batches are not part of the decode path (infer never passes an attention mask)")
        x = embeddings.to(self.device).float()
        if x.dim() != 3 or x.shape[0] != 1 or x.shape[2] != self.dim:
            raise ValueError(f"embeddings must be [1, L, {self.dim}]")
        Lseq = x.shape[1]
        if Lseq < 5 or Lseq > self.max_positions:
            raise ValueError(f"sequence length {Lseq} outside [5, {self.max_positions}]")
        lib, s_ = L.lib(), L.stream_ptr()
        L.check(lib.edm_t2s_begin(self._ctx, None, 0, Lseq - 4, s_), "begin")      # shapes only: the embeddings are given
        xc = x[0].contiguous()
        L.check(lib.edm_t2s_logits(self._ctx, L.ptr(xc), s_), "logits")
        logits = self._view("logits", (1, Lseq, 1024), torch.float32).clone()
        return logits[mask.to(self.device)] if mask is not None else logits

    def input_embedding(self, tokens):
        _check_range(tokens, self.total_num_tokens, "input_embedding")
        return torch.nn.functional.embedding(tokens.to(self.device), self._w["emb"])
