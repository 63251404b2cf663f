"""Host-side mirror of the reference's S2A model API on top of the C ABI (libedm_s2a.so).

Mirrors edm_tts/models/injection_conformer/modeling_injection_conformer.py:25-230 (InjectionConformerModel) and
injection_conformer_wrapper.py:9-150 (InjectionConformerWrapper): same constructor inputs (config + state dict / HF
directory), same method names and argument meaning, same error behaviour (assert on length mismatch, ValueError for
malformed prompts). Python only moves pointers; all arithmetic runs in the CUDA kernels. No CPU fallback exists.
"""
from __future__ import annotations

import ctypes as C
import functools
import os

import torch

from . import _lib as L
from . import varlen
from .config import InjectionConformerConfig
from .weights import pack_rvq_weights, pack_s2a_weights

class InjectionConformerOutput(dict):
    """modeling_injection_conformer.py:18-22 (a transformers ModelOutput there): attribute and key access."""

    def __init__(self, loss=None, output_acoustic_codes=None, target_acoustic_codes=None):
        super().__init__(loss=loss, output_acoustic_codes=output_acoustic_codes, target_acoustic_codes=target_acoustic_codes)
        self.__dict__ = self


MAX_CHUNK = 64  # sequences decoded per bound workspace (larger batches are processed in chunks; utterances are independent)


def _on_device(fn):
    """Run a public entry point with the model's device current: L.stream_ptr() and every allocation of the call then belong to the
    device that holds the weights and the workspace, whichever device the caller had selected. The context's workspace is shared by
    all calls, so a call issued on another stream than the previous one first waits for that one's recorded end (calls on one stream
    are ordered anyway); while a CUDA graph is being captured the caller owns the ordering."""
    @functools.wraps(fn)
    def wrapped(self, *a, **k):
        model = getattr(self, "_m", self)
        with torch.cuda.device(model.device):
            cur = torch.cuda.current_stream()
            capturing = torch.cuda.is_current_stream_capturing()
            last = getattr(model, "_last_use", None)
            if last is not None and not capturing and last[0] != cur.cuda_stream:
                cur.wait_event(last[1])
            try:
                return fn(self, *a, **k)
            finally:
                if not capturing:
                    ev = torch.cuda.Event()
                    ev.record(cur)
                    model._last_use = (cur.cuda_stream, ev)
    return wrapped


def _check_range(t, n, what):
    """F.embedding raises IndexError for an out-of-range index; the kernels only clamp (memory safety), so the range is checked here.
    Host tensors cost nothing; a device tensor costs one small reduction + sync, skipped while a CUDA graph is being captured."""
    if t is None or t.numel() == 0:
        return
    if t.is_cuda and torch.cuda.is_current_stream_capturing():
        return
    lo, hi = torch.aminmax(t)
    if int(lo) < 0 or int(hi) >= n:
        raise IndexError(f"{what}: index out of range [0, {n}) (min {int(lo)}, max {int(hi)})")


class _Embedding:
    """Callable embedding table (the reference's nn.Embedding attribute): table[tokens]; `.weight` is the fp32 table."""

    def __init__(self, weight):
        self.weight = weight
        self.num_embeddings, self.embedding_dim = weight.shape

    def __call__(self, tokens):
        _check_range(tokens, self.num_embeddings, "embedding")
        return torch.nn.functional.embedding(tokens.to(self.weight.device), self.weight)


class _LinearLayerNorm:
    """nn.Sequential(nn.Linear(d, d), nn.LayerNorm(d)) on the C ABI (acoustic_feat_proj / project_injection[k],
    modeling_injection_conformer.py:44-47, injection_conformer_wrapper.py:26-32): bf16 tensor-core GEMM with fp32 accumulation and
    an fp32 LayerNorm. x [..., 1024] -> fp32 [..., 1024]."""

    def __init__(self, model, w_bf16, bias, ln_w, ln_b):
        self._m, self._w, self._b, self._ln_w, self._ln_b = model, w_bf16, bias, ln_w, ln_b

    @_on_device
    def __call__(self, x):
        d = self._w.shape[1]
        lead = x.shape[:-1]
        a = x.to(self._m.device).reshape(-1, d).to(torch.bfloat16).contiguous()
        rows = a.shape[0]
        h = torch.empty(rows, d, device=a.device, dtype=torch.float32)
        L.check(L.lib().edm_gemm_bf16(L.ptr(a), d, L.ptr(self._w), d, rows, self._w.shape[0], d, L.EPI_F32, L.ptr(self._b), L.ptr(h), d, 1.0,
                                      None, None, 1, 0, L.stream_ptr()), "gemm")
        y = torch.empty_like(h)
        L.check(L.lib().edm_layernorm(L.ptr(h), 0, rows, L.ptr(self._ln_w), L.ptr(self._ln_b), None, None, L.ptr(y), None, 1, 0, 1e-5,
                                      L.stream_ptr()), "layernorm")
        return y.view(*lead, d)


class _Encoder:
    """InjectionConformerWrapper mirror: forward_first_level / forward / apply_single_to_logits."""

    def __init__(self, model: "InjectionConformerModel"):
        self._m = model

    @staticmethod
    def _layout(x, mask_time_indices):
        """-> (P, target): a common suffix [:, P:] of target rows (mask None: P = 0) runs on the uniform bind (target None); any other
        boolean mask with the same count in every row (the reference's .view(b, ...)) on the masked bind (target: the mask on the host)."""
        B, N = x.shape[:2]
        if mask_time_indices is None:
            return 0, None
        m = mask_time_indices.to("cpu", torch.bool)
        if tuple(m.shape) != (B, N):
            raise ValueError(f"mask_time_indices must be [b, n] = {(B, N)}, got {tuple(m.shape)}")
        counts = m.sum(1)
        if not bool((counts == counts[0]).all()):
            raise ValueError("mask_time_indices must select the same number of positions in every sequence")
        T = int(counts[0])
        if T == 0:
            raise ValueError("mask_time_indices selects no position")
        if bool(m[:, N - T:].all()):
            return N - T, None
        return N - T, m

    @_on_device
    def forward_first_level(self, x, mask=None, mask_time_indices=None):
        """injection_conformer_wrapper.py:65-90 -> logits [b, 1, t, codes] (fp32)."""
        assert mask is None, "the S2A decode path never passes a padding mask"
        m = self._m
        x = x.to(m.device)
        B, N, _ = x.shape
        if B > MAX_CHUNK:
            return torch.cat([self.forward_first_level(x[i:i + MAX_CHUNK], None, None if mask_time_indices is None else mask_time_indices[i:i + MAX_CHUNK])
                              for i in range(0, B, MAX_CHUNK)])
        P, target = self._layout(x, mask_time_indices)
        if target is None:
            m._bind(B, N - P, P)
        else:
            m._bind_masked([N] * B, target)
        xf = x.float().contiguous()
        L.check(L.lib().edm_s2a_first_level(m._ctx, L.ptr(xf), L.stream_ptr()), "first_level")
        return m._view("logits", (B, 1, N - P, m.num_codevectors), torch.float32).clone()

    @_on_device
    def forward(self, x, mask=None, injections=None, acoustic_model=None, mask_time_indices=None, *, prompt_codes=None,
                forced_coarse=None):
        """injection_conformer_wrapper.py:92-150 in eval mode -> logits [b, q, t, codes] (fp32).
        Prompt rows (the rows mask_time_indices leaves out: a prefix, or any rows with the same count per sequence) are injected either
        from `injections` -- the reference's argument: one feature tensor [b, n, 1024] per injection layer (cumulative DAC features of
        the prompt, zeros on the target rows), projected here with project_injection[k].0 on the tensor cores -- or from the acoustic
        prompt *codes* (prompt_codes [b, >=4, P], the prompt rows in time order) through the folded tables, which is what infer_special
        does. `acoustic_model` is accepted for signature compatibility (the model's own folded tables are used)."""
        assert mask is None, "the S2A decode path never passes a padding mask"
        m = self._m
        x = x.to(m.device)
        B, N, _ = x.shape
        if B > MAX_CHUNK:
            raise ValueError(f"encoder.forward takes at most {MAX_CHUNK} sequences per call (infer_special chunks larger batches itself)")
        P, target = self._layout(x, mask_time_indices)
        n_inj = len(m.injection_layers)
        if P > 0 and prompt_codes is None and injections is None:
            raise ValueError("prompt rows need their injections: pass injections=[features per injection layer] or prompt_codes=<acoustic prompt tokens>")
        if target is None:
            m._bind(B, N - P, P, keep_logits=True)
        else:
            m._bind_masked([N] * B, target, keep_logits=True)
        L.check(L.lib().edm_s2a_set_prompt_injections(m._ctx, None), "set_prompt_injections")
        keep = None
        if P > 0 and prompt_codes is not None:
            m._load_prompt_codes(prompt_codes, B * (N - P), B * P)
        elif P > 0:
            if len(injections) < n_inj:
                raise IndexError("one injection tensor per injection layer is required")   # reference: list index out of range
            m._load_prompt_codes(torch.zeros(B, n_inj, P, dtype=torch.int64), B * (N - P), B * P)
            # project_injection[k].0 on the prompt rows (bf16 operands as under autocast, fp32 accumulate + bias), LayerNorm in the kernel
            w = m._w
            keep = torch.empty(n_inj, B * P, 1024, device=m.device, dtype=torch.float32)
            for k in range(n_inj):
                inj = injections[k].to(m.device)
                if tuple(inj.shape) != (B, N, 1024):
                    raise ValueError(f"injections[{k}] must be [b, n, 1024], got {tuple(inj.shape)}")
                a = (inj[:, :P] if target is None else inj[~target.to(m.device)]).reshape(B * P, 1024).to(torch.bfloat16).contiguous()
                L.check(L.lib().edm_gemm_bf16(L.ptr(a), 1024, L.ptr(w["inj_w"][k]), 1024, B * P, 1024, 1024, L.EPI_F32, L.ptr(w["inj_b"][k]),
                                              L.ptr(keep[k]), 1024, 1.0, None, None, 1, 0, L.stream_ptr()), "gemm")
                del a
            L.check(L.lib().edm_s2a_set_prompt_injections(m._ctx, L.ptr(keep)), "set_prompt_injections")
        codes = torch.empty(B, m.num_quantizers, N - P, device=x.device, dtype=torch.int64)
        fc = None if forced_coarse is None else forced_coarse.to(m.device, torch.int32).contiguous()
        xf = x.float().contiguous()
        try:
            L.check(L.lib().edm_s2a_full_pass(m._ctx, L.ptr(xf), L.ptr(fc), L.ptr(codes), L.stream_ptr()), "full_pass")
        finally:
            L.check(L.lib().edm_s2a_set_prompt_injections(m._ctx, None), "set_prompt_injections")
        n_inj = len(m.injection_layers)
        coarse = m._view("coarse_logits", (4, B, N - P, m.num_codevectors), torch.float32)[:n_inj].permute(1, 0, 2, 3)
        fine = m._view("fine_logits", (B, N - P, m.num_quantizers - n_inj, m.num_codevectors), torch.float32).permute(0, 2, 1, 3)
        return torch.cat([coarse, fine], dim=1)

    __call__ = forward

    @_on_device
    def apply_single_to_logits(self, inp, idx):
        """injection_conformer_wrapper.py:56-63: LayerNorm + per-codebook head idx -> [b, 1, n, codes]."""
        m = self._m
        if not 0 <= int(idx) < m.num_quantizers:
            raise IndexError(f"head index {idx} out of range")
        inp = inp.to(m.device)
        B, n, d = inp.shape
        z = torch.empty(B * n, d, device=inp.device, dtype=torch.bfloat16)
        w = m._w
        xf = inp.float().contiguous()
        L.check(L.lib().edm_layernorm(L.ptr(xf), 0, B * n, L.ptr(w["tl_ln_w"]), L.ptr(w["tl_ln_b"]), None, None, None,
                                      L.ptr(z), 1, 0, 1e-5, L.stream_ptr()), "layernorm")
        out = torch.empty(B * n, m.num_codevectors, device=inp.device, dtype=torch.float32)
        head = w["head_w"][idx * m.num_codevectors:(idx + 1) * m.num_codevectors]
        bias = w["head_b"][idx * m.num_codevectors:(idx + 1) * m.num_codevectors]
        L.check(L.lib().edm_gemm_bf16(L.ptr(z), d, L.ptr(head), d, B * n, m.num_codevectors, d, L.EPI_F32, L.ptr(bias), L.ptr(out),
                                      m.num_codevectors, 1.0, None, None, 1, 0, L.stream_ptr()), "gemm")
        return out.view(B, 1, n, m.num_codevectors)


class _AcousticModel:
    """The slice of the DAC API the S2A path touches (dac/modeling_dac.py:173-182): code -> feature lookups."""

    def __init__(self, rvq_tables, latent_dim, n_codebooks, codebook_size, device):
        self._t = rvq_tables
        self.device = device
        self.latent_dim, self.n_codebooks, self.codebook_size = latent_dim, n_codebooks, codebook_size

    @_on_device
    def _c2f(self, codes, unreduced):
        _check_range(codes, self.codebook_size, "codes_to_features")
        codes = codes.to(self.device, torch.int64).contiguous()
        B, Lv, T = codes.shape
        if Lv > self._t["n_levels"]:
            raise ValueError(f"codes have {Lv} levels, quantizer has {self._t['n_levels']}")
        shape = (B, Lv, self.latent_dim, T) if unreduced else (B, self.latent_dim, T)
        out = torch.empty(shape, device=codes.device, dtype=torch.float32)
        L.check(L.lib().edm_codes_to_features(L.ptr(codes), L.ptr(self._t["proj"]), L.ptr(out), B, Lv, T, int(unreduced), L.stream_ptr()),
                "codes_to_features")
        return out

    def codes_to_features(self, codes):
        return self._c2f(codes, False)

    def codes_to_features_unreduced(self, codes):
        return self._c2f(codes, True)


class InjectionConformerModel:
    """Drop-in for the reference InjectionConformerModel on the decode path (inference only)."""

    def __init__(self, config, state_dict: dict, device="cuda", dac_config=None, max_positions: int = 4096):
        if not torch.cuda.is_available():
            raise L.EdmError("edm_tts_b200 needs a CUDA device (sm_100); there is no CPU fallback")
        self.config = InjectionConformerConfig.from_any(config, dac_config)
        cfg = self.config
        self.device = torch.device(device)
        self.injection_layers = list(cfg.injection_layers)
        self.num_quantizers = cfg.dac.n_codebooks
        self.num_codevectors = cfg.dac.codebook_size
        self.acoustic_size = cfg.dac.latent_dim
        self.loss_all = cfg.loss_all
        lib = L.lib()
        c = L.S2AConfig()
        c.hidden, c.heads, c.depth, c.ff_mult, c.conv_kernel = cfg.hidden_size, cfg.heads, cfg.depth, cfg.ff_mult, cfg.conv_kernel_size
        c.num_quantizers, c.num_codes, c.num_semantic = self.num_quantizers, self.num_codevectors, cfg.num_semantic_tokens
        c.n_injection = len(self.injection_layers)
        for i, l in enumerate(self.injection_layers[:4]):
            c.injection_layers[i] = l
        c.residual, c.max_positions = int(cfg.residual), max_positions
        self._cfg_c = c
        n = lib.edm_s2a_num_weights(C.byref(c))
        if n <= 0:
            raise ValueError("unsupported S2A configuration: " + lib.edm_last_error().decode())
        if not cfg.use_injection:
            raise ValueError("use_injection=False is not supported by the B200 decode path")
        with torch.cuda.device(self.device):
            self._w = pack_s2a_weights(state_dict, cfg, self.device, max_positions)
            self._rvq = pack_rvq_weights(state_dict, self.num_quantizers, "acoustic_model.quantizer.", self.device)
            names = [lib.edm_s2a_weight_name(C.byref(c), i).decode() for i in range(n)]
            ptrs = (C.c_void_p * n)(*[self._w[name].data_ptr() for name in names])
            self._ctx = lib.edm_s2a_create(C.byref(c), ptrs, n)
        if not self._ctx:
            raise L.EdmError("edm_s2a_create failed: " + lib.edm_last_error().decode())
        self._bound = None
        self._ws = None
        self.low_latency = False
        self.encoder = _Encoder(self)
        self.acoustic_model = _AcousticModel(self._rvq, self.acoustic_size, self.num_quantizers, self.num_codevectors, self.device)
        self.semantic_embedding = _Embedding(self._w["sem_emb"])
        w = self._w
        self.acoustic_feat_proj = _LinearLayerNorm(self, w["fp_w"], w["fp_b"], w["fp_ln_w"], w["fp_ln_b"])
        self.encoder.project_injection = [_LinearLayerNorm(self, w["inj_w"][k], w["inj_b"][k], w["inj_ln_w"][k], w["inj_ln_b"][k])
                                          for k in range(len(self.injection_layers))]
        self.mask_token = self._w["mask_token"].view(1, 1, -1)
        self.training = False

    # ------------------------------------------------------------------ construction helpers
    @classmethod
    def from_pretrained(cls, path: str, device="cuda", **kw):
        """HF directory (config.json + model.safetensors), as written by the reference's save_pretrained."""
        from safetensors.torch import load_file

        cfg = InjectionConformerConfig.from_pretrained(path)
        return cls(cfg, load_file(os.path.join(path, "model.safetensors")), device=device, **kw)

    # nn.Module-like surface of an inference-only model: eval() is the only mode, the weights live (packed) on the device given
    # at construction
    def eval(self):
        return self

    def train(self, mode: bool = True):
        if mode:
            raise NotImplementedError("edm_tts_b200.InjectionConformerModel is inference-only (no dropout, no autograd); train with the reference")
        return self

    def requires_grad_(self, requires_grad: bool = False):
        if requires_grad:
            raise NotImplementedError("inference-only model")
        return self

    def parameters(self):
        return iter(())

    def to(self, *args, **kwargs):
        """Accepts the device the model already lives on (and any dtype argument: precision is fixed by the kernels); moving the
        packed weights to another device is refused -- build a second model with device=... instead."""
        dev = kwargs.get("device", next((a for a in args if isinstance(a, (str, torch.device, int))), None))
        if dev is not None:
            dev = torch.device("cuda", dev) if isinstance(dev, int) else torch.device(dev)
            cur = self.device if self.device.index is not None else torch.device("cuda", torch.cuda.current_device())
            if dev.type != "cuda" or (dev.index is not None and dev.index != cur.index):
                raise ValueError(f"model lives on {cur}; construct it with device={dev!s} instead of moving it (there is no CPU path)")
        return self

    def cuda(self, device=None):
        return self.to(device if device is not None else self.device)

    def state_dict(self):
        raise NotImplementedError("the packed bf16 weights / folded tables are not the reference's parameters; keep the HF directory "
                                  "(from_pretrained) as the interchange format")

    def __del__(self):
        try:
            if getattr(self, "_ctx", None):
                L.lib().edm_s2a_destroy(self._ctx)
                self._ctx = None
        except Exception:
            pass

    # ------------------------------------------------------------------ workspace plumbing
    def _bind(self, B, T, P, keep_logits=False):
        """keep_logits: the per-level logits of the full pass are materialised (parity runs, encoder.forward, the eval-mode loss);
        infer_special leaves it off and the [b, 12, t, 1024] logits never exist (arg-max in the head GEMM's epilogue)."""
        key = (B, T, P, bool(keep_logits))
        if self._bound == key:
            return
        lib = L.lib()
        L.check(lib.edm_s2a_set_keep_logits(self._ctx, int(bool(keep_logits))), "set_keep_logits")
        need = lib.edm_s2a_workspace_bytes(self._ctx, B, T, P)
        if need == 0:
            raise ValueError(f"invalid decode shape B={B} T={T} P={P}")
        if self._ws is None or self._ws.numel() < need:
            self._ws = None
            self._ws = torch.empty(need, device=self.device, dtype=torch.uint8)
        L.check(lib.edm_s2a_bind(self._ctx, self._ws.data_ptr(), self._ws.numel(), B, T, P), "bind")
        self._bound = key

    def _bind_varlen(self, T, P):
        """Packed workspace for utterances of T[i] target / P[i] prompt frames (edm_s2a_bind_varlen); the arg-max stays in the head GEMMs."""
        key = ("varlen", tuple(T), tuple(P))
        if self._bound == key:
            return
        lib = L.lib()
        L.check(lib.edm_s2a_set_keep_logits(self._ctx, 0), "set_keep_logits")
        n = len(T)
        t_arr, p_arr = (C.c_int * n)(*T), (C.c_int * n)(*P)
        need = lib.edm_s2a_workspace_bytes_varlen(self._ctx, n, t_arr, p_arr)
        if need == 0:
            raise ValueError("invalid variable-length batch: " + lib.edm_last_error().decode("utf-8", "replace"))
        if self._ws is None or self._ws.numel() < need:
            self._ws = None
            self._ws = torch.empty(need, device=self.device, dtype=torch.uint8)
        self._bound = None
        L.check(lib.edm_s2a_bind_varlen(self._ctx, self._ws.data_ptr(), self._ws.numel(), n, t_arr, p_arr, L.stream_ptr()), "bind_varlen")
        self._bound = key

    def _bind_masked(self, N, target, keep_logits=False):
        """Packed workspace for utterances of N[i] frames whose targets are marked in `target` (host bool, all utterances
        concatenated; edm_s2a_bind_masked)."""
        tb = target.to("cpu", torch.uint8).contiguous().reshape(-1).numpy().tobytes()
        key = ("masked", tuple(N), tb, bool(keep_logits))
        if self._bound == key:
            return
        lib = L.lib()
        L.check(lib.edm_s2a_set_keep_logits(self._ctx, int(bool(keep_logits))), "set_keep_logits")
        n, cu = len(N), varlen.offsets(N)
        T = [tb[cu[i]:cu[i + 1]].count(1) for i in range(n)]
        t_arr, p_arr, n_arr = (C.c_int * n)(*T), (C.c_int * n)(*[a - b for a, b in zip(N, T)]), (C.c_int * n)(*N)
        need = lib.edm_s2a_workspace_bytes_varlen(self._ctx, n, t_arr, p_arr)
        if need == 0:
            raise ValueError("invalid infill batch: " + lib.edm_last_error().decode("utf-8", "replace"))
        if self._ws is None or self._ws.numel() < need:
            self._ws = None
            self._ws = torch.empty(need, device=self.device, dtype=torch.uint8)
        self._bound = None
        tgt = (C.c_ubyte * len(tb)).from_buffer_copy(tb)
        L.check(lib.edm_s2a_bind_masked(self._ctx, self._ws.data_ptr(), self._ws.numel(), n, n_arr, tgt, L.stream_ptr()), "bind_masked")
        self._bound = key

    def _view(self, name, shape, dtype):
        nbytes = C.c_size_t(0)
        p = L.lib().edm_s2a_buffer(self._ctx, name.encode(), C.byref(nbytes))
        if not p:
            raise L.EdmError(f"no workspace buffer {name}")
        off = p - self._ws.data_ptr()
        numel = 1
        for s in shape:
            numel *= s
        esz = torch.empty(0, dtype=dtype).element_size()
        assert numel * esz <= nbytes.value, (name, shape, nbytes.value)
        return self._ws[off:off + numel * esz].view(dtype).view(*shape)

    def _load_prompt_codes(self, prompt_codes, n_target, n_prompt):
        pc = prompt_codes.to(self.device, torch.int32).contiguous()
        dummy_sem = torch.zeros(n_target, device=self.device, dtype=torch.int32)
        dummy_sp = torch.zeros(n_prompt, device=self.device, dtype=torch.int32)
        L.check(L.lib().edm_s2a_build_input(self._ctx, L.ptr(dummy_sem), L.ptr(dummy_sp), L.ptr(pc), pc.shape[1], L.stream_ptr()), "build_input")

    def set_low_latency(self, on=True):
        """Single-utterance serving mode (the reference's own call, inference.py:43-48): decodes of <= 512 rows split their long-K
        residual GEMMs over K (edm_s2a_set_low_latency). Faster for one short utterance; the rounding noise of a row then depends on
        how many rows are decoded together, which the default mode guarantees it never does."""
        L.check(L.lib().edm_s2a_set_low_latency(self._ctx, int(bool(on))), "set_low_latency")
        self.low_latency = bool(on)
        return self

    # ------------------------------------------------------------------ the decode API
    @torch.no_grad()
    @_on_device
    def infer_special(self, semantic_tokens, acoustic_prompt_tokens=None, semantic_prompt_tokens=None, steps=1, temperature=1.0, *,
                      seed=0, batch_offset=0, cat_gumbel=None, remask_gumbel=None, forced_ids=None, forced_masks=None, forced_coarse=None):
        """modeling_injection_conformer.py:130-230. Returns LongTensor [b, num_quantizers, t].
        seed / batch_offset drive the in-kernel Philox noise: row r of the call draws from counter (batch_offset + r), so a
        batch decoded in chunks or shards gives the same tokens as in one piece. Other keyword-only extras are for parity runs: injected Gumbel noise (cat_gumbel [S-1, b*t, codes], remask_gumbel
        [S-1, b, t]) and teacher forcing (forced_ids [S, b, t], forced_masks [S-1, b, t], forced_coarse [b, 4, t])."""
        dev = self.device
        _check_range(semantic_tokens, self.config.num_semantic_tokens, "semantic_tokens")
        st = semantic_tokens.to(dev)
        B, T = st.shape
        if steps > 1 and T < 2:
            raise IndexError("re-masking needs at least 2 frames (the reference's take_along_dim is out of range for T = 1 with steps > 1)")
        _check_range(forced_ids, self.num_codevectors, "forced_ids")
        _check_range(forced_coarse, self.num_codevectors, "forced_coarse")
        has_prompt = acoustic_prompt_tokens is not None and semantic_prompt_tokens is not None
        P = 0
        if has_prompt:
            _check_range(acoustic_prompt_tokens, self.num_codevectors, "acoustic_prompt_tokens")
            _check_range(semantic_prompt_tokens, self.config.num_semantic_tokens, "semantic_prompt_tokens")
            ap, sp = acoustic_prompt_tokens.to(dev), semantic_prompt_tokens.to(dev)
            if ap.dim() != 3 or sp.dim() != 2 or ap.shape[0] != B or sp.shape[0] != B or ap.shape[-1] != sp.shape[-1]:
                raise ValueError("prompt tokens must be acoustic [b, q, p] and semantic [b, p] with matching b and p")
            if ap.shape[1] < len(self.injection_layers):
                raise IndexError("acoustic prompt needs at least one level per injection layer")  # reference: list index out of range
            P = ap.shape[-1]
        out = torch.empty(B, self.num_quantizers, T, device=dev, dtype=torch.int64)
        lib = L.lib()
        for b0 in range(0, B, MAX_CHUNK):
            b1 = min(B, b0 + MAX_CHUNK)
            nb = b1 - b0
            self._bind(nb, T, P)
            sl = slice(b0, b1)
            sem = st[sl].to(torch.int32).contiguous()
            spc = sp[sl].to(torch.int32).contiguous() if has_prompt else None
            apc = ap[sl].to(torch.int32).contiguous() if has_prompt else None
            cg = None if cat_gumbel is None else cat_gumbel.to(dev).view(-1, B, T, self.num_codevectors)[:, sl].contiguous().float()
            rg = None if remask_gumbel is None else remask_gumbel.to(dev)[:, sl].contiguous().float()
            fi = None if forced_ids is None else forced_ids.to(dev)[:, sl].to(torch.int32).contiguous()
            fm = None if forced_masks is None else forced_masks.to(dev)[:, sl].to(torch.uint8).contiguous()
            fc = None if forced_coarse is None else forced_coarse.to(dev)[sl].to(torch.int32).contiguous()
            codes = torch.empty(nb, self.num_quantizers, T, device=dev, dtype=torch.int64)
            L.check(lib.edm_s2a_set_batch_offset(self._ctx, int(batch_offset) + b0), "set_batch_offset")
            L.check(lib.edm_s2a_decode(self._ctx, L.ptr(sem), L.ptr(spc), L.ptr(apc), apc.shape[1] if has_prompt else 0, int(steps),
                                       float(temperature), int(seed), L.ptr(cg), L.ptr(rg), L.ptr(fi), L.ptr(fm), L.ptr(fc), L.ptr(codes),
                                       L.stream_ptr()), "decode")
            out[sl] = codes
        return out

    generate = infer_special

    @torch.no_grad()
    @_on_device
    def infer_batch(self, semantic_tokens, acoustic_prompt_tokens=None, semantic_prompt_tokens=None, steps=8, temperature=1.0, *,
                    seed=0, batch_offset=0, cat_gumbel=None, remask_gumbel=None, forced_ids=None, forced_masks=None, forced_coarse=None):
        """infer_special for utterances of different lengths, decoded together without padding.
        semantic_tokens: list of LongTensor [T_i]; the prompts: None, or lists of acoustic [q, P_i] (one q for all; P_i may be 0) and
        semantic [P_i] tokens. Returns a list of LongTensor [12, T_i], views of one packed output. Utterance i decodes to the bits of
        infer_special(semantic_tokens[i][None], ..., batch_offset=batch_offset + i)[0] (outside low-latency mode). The keyword extras
        are per-utterance lists shaped as infer_special's extras for one utterance: cat_gumbel[i] [S-1, T_i, codes], remask_gumbel[i]
        [S-1, 1, T_i], forced_ids[i] [S, 1, T_i], forced_masks[i] [S-1, 1, T_i], forced_coarse[i] [1, 4, T_i]."""
        if not isinstance(semantic_tokens, (list, tuple)) or len(semantic_tokens) == 0:
            raise ValueError("semantic_tokens must be a non-empty list of [T_i] tensors")
        n = len(semantic_tokens)
        if any(not torch.is_tensor(t) or t.dim() != 1 for t in semantic_tokens):
            raise ValueError("every semantic_tokens entry must be a 1-D tensor [T_i]")
        T = [int(t.shape[0]) for t in semantic_tokens]
        if min(T) < 1:
            raise ValueError("every utterance needs at least one target frame")
        if steps > 1 and min(T) < 2:
            raise IndexError("re-masking needs at least 2 frames (the reference's take_along_dim is out of range for T = 1 with steps > 1)")
        for t in semantic_tokens:
            _check_range(t, self.config.num_semantic_tokens, "semantic_tokens")
        has_prompt = acoustic_prompt_tokens is not None or semantic_prompt_tokens is not None
        P = [0] * n
        if has_prompt:
            ap, sp = acoustic_prompt_tokens, semantic_prompt_tokens
            if not isinstance(ap, (list, tuple)) or not isinstance(sp, (list, tuple)) or len(ap) != n or len(sp) != n:
                raise ValueError("acoustic_prompt_tokens and semantic_prompt_tokens must both be lists with one entry per utterance")
            if any(not torch.is_tensor(a) or a.dim() != 2 for a in ap) or any(not torch.is_tensor(x) or x.dim() != 1 for x in sp):
                raise ValueError("prompt tokens must be acoustic [q, p_i] and semantic [p_i] tensors")
            q = int(ap[0].shape[0])
            if any(int(a.shape[0]) != q for a in ap):
                raise ValueError("every acoustic prompt must have the same number of levels q")
            if any(a.shape[1] != x.shape[0] for a, x in zip(ap, sp)):
                raise ValueError("acoustic and semantic prompts of an utterance must have the same length")
            if q < len(self.injection_layers):
                raise IndexError("acoustic prompt needs at least one level per injection layer")  # reference: list index out of range
            for a, x in zip(ap, sp):
                _check_range(a, self.num_codevectors, "acoustic_prompt_tokens")
                _check_range(x, self.config.num_semantic_tokens, "semantic_prompt_tokens")
            P = [int(x.shape[0]) for x in sp]
        self._check_extras(T, int(steps), cat_gumbel=cat_gumbel, remask_gumbel=remask_gumbel, forced_ids=forced_ids, forced_masks=forced_masks,
                           forced_coarse=forced_coarse)
        q = int(acoustic_prompt_tokens[0].shape[0]) if has_prompt else 0
        return self._decode_packed(T, P, semantic_tokens, semantic_prompt_tokens if has_prompt else None,
                                   acoustic_prompt_tokens if has_prompt else None, q, None, int(steps), temperature, seed, batch_offset,
                                   cat_gumbel, remask_gumbel, forced_ids, forced_masks, forced_coarse)

    def _check_extras(self, T, S, **extras):
        """The per-utterance parity extras of infer_batch / infill_batch: shapes as infer_special's for one utterance of T[i] targets."""
        V = self.num_codevectors
        shapes = dict(cat_gumbel=lambda t: (S - 1, t, V), remask_gumbel=lambda t: (S - 1, 1, t), forced_ids=lambda t: (S, 1, t),
                      forced_masks=lambda t: (S - 1, 1, t), forced_coarse=lambda t: (1, 4, t))
        for name, lst in extras.items():
            if lst is None:
                continue
            if not isinstance(lst, (list, tuple)) or len(lst) != len(T):
                raise ValueError(f"{name} must be a list with one entry per utterance")
            for i, x in enumerate(lst):
                if tuple(x.shape) != shapes[name](T[i]):
                    raise ValueError(f"{name}[{i}] must be {shapes[name](T[i])}, got {tuple(x.shape)}")
        for name in ("forced_ids", "forced_coarse"):
            for x in extras.get(name) or ():
                _check_range(x, V, name)

    def _decode_packed(self, T, P, sem_target, sem_known, codes_known, q, target, S, temperature, seed, batch_offset, cat_gumbel,
                       remask_gumbel, forced_ids, forced_masks, forced_coarse):
        """Chunks of MAX_CHUNK utterances through one packed bind each: the varlen bind (target None: the P[i] prompt frames lead), or
        the masked bind (target: per-utterance bool masks). Per-target inputs are lists over the targets of each utterance, per-known
        inputs (sem_known [P_i], codes_known [q, P_i]) over its prompt / known frames, both in time order."""
        dev, lib = self.device, L.lib()
        Q = self.num_quantizers
        out = torch.empty(Q * sum(T), device=dev, dtype=torch.int64)

        def cat(lst, sl, dim, dtype):
            return None if lst is None else torch.cat([x.to(dev) for x in lst[sl]], dim).to(dtype).contiguous()

        for ch in varlen.plan(T, P, MAX_CHUNK, batch_offset):
            sl = slice(ch.start, ch.stop)
            if target is None:
                self._bind_varlen(ch.T, ch.P)
            else:
                self._bind_masked([t + p for t, p in zip(ch.T, ch.P)], torch.cat(target[sl]))
            known = codes_known is not None and sum(ch.P) > 0
            sem = cat(sem_target, sl, 0, torch.int32)
            spc = cat(sem_known, sl, 0, torch.int32) if known else None
            apc = torch.cat([a.to(dev).reshape(-1) for a in codes_known[sl]]).to(torch.int32).contiguous() if known else None
            cg = cat(cat_gumbel, sl, 1, torch.float32)
            rg = cat(remask_gumbel, sl, 2, torch.float32)
            fi = cat(forced_ids, sl, 2, torch.int32)
            fm = cat(forced_masks, sl, 2, torch.uint8)
            fc = None if forced_coarse is None else torch.cat([x.to(dev).reshape(-1) for x in forced_coarse[sl]]).to(torch.int32).contiguous()
            codes = out[Q * ch.t0:Q * (ch.t0 + sum(ch.T))]
            L.check(lib.edm_s2a_set_batch_offset(self._ctx, ch.batch_offset), "set_batch_offset")
            L.check(lib.edm_s2a_decode(self._ctx, L.ptr(sem), L.ptr(spc), L.ptr(apc), q if codes_known is not None else 0,
                                       S, float(temperature), int(seed), L.ptr(cg), L.ptr(rg), L.ptr(fi), L.ptr(fm), L.ptr(fc), L.ptr(codes),
                                       L.stream_ptr()), "decode")
        return varlen.split_blocks(out, T, Q)

    @torch.no_grad()
    @_on_device
    def infill_batch(self, semantic_tokens, acoustic_tokens, regenerate, steps=8, temperature=1.0, *, seed=0, batch_offset=0,
                     cat_gumbel=None, remask_gumbel=None, forced_ids=None, forced_masks=None, forced_coarse=None):
        """Speech editing: regenerate the chosen frames of each utterance given the others (the S2A model's training objective,
        modeling_injection_conformer.py:96-102, at inference). semantic_tokens: list of [N_i]; acoustic_tokens: list of [q, N_i] codes
        (one q in [1, 12]; the values at regenerated frames are ignored); regenerate: list of bool [N_i], at least one True each.
        The other frames are known and treated exactly as prompt frames (input sem + LN(Linear(feat_0)), never sampled or re-masked,
        injected with the cumulative ground-truth features of their first min(4, q) levels; q must cover every injection layer when
        any frame is known). Returns a list of LongTensor [12, T_i] (T_i = regenerate[i].sum()): the codes of the regenerated frames in
        time order, views of one packed output. With the known frames in front this is infer_batch with them as prompts, bit for bit;
        target t of utterance i draws Philox counter (batch_offset + i) T_i + t. Chunks of 64 utterances at batch offsets
        batch_offset + 64 c. The keyword extras are per-utterance lists shaped as infer_batch's for T_i targets."""
        sp = varlen.infill_split(semantic_tokens, acoustic_tokens, regenerate, self.num_codevectors, self.config.num_semantic_tokens,
                                 self.num_quantizers)
        T, P = list(sp.T), list(sp.P)
        if steps > 1 and min(T) < 2:
            raise IndexError("re-masking needs at least 2 frames to regenerate (the reference's take_along_dim is out of range for T = 1 with steps > 1)")
        q = int(acoustic_tokens[0].shape[0])
        if sum(P) > 0 and q < len(self.injection_layers):
            raise IndexError("known frames need at least one code level per injection layer")  # reference: list index out of range
        self._check_extras(T, int(steps), cat_gumbel=cat_gumbel, remask_gumbel=remask_gumbel, forced_ids=forced_ids, forced_masks=forced_masks,
                           forced_coarse=forced_coarse)
        return self._decode_packed(T, P, sp.sem_target, sp.sem_known, sp.codes_known, q, sp.target, int(steps), temperature, seed,
                                   batch_offset, cat_gumbel, remask_gumbel, forced_ids, forced_masks, forced_coarse)

    @torch.no_grad()
    @_on_device
    def decode_trace(self, semantic_tokens, acoustic_prompt_tokens=None, semantic_prompt_tokens=None, steps=1, temperature=1.0, *,
                     seed=0, cat_gumbel=None, remask_gumbel=None, forced_ids=None, forced_masks=None, forced_coarse=None):
        """infer_special run stage by stage through the same C entry points edm_s2a_decode composes, returning every
        intermediate (per-step first-level logits / own ids / masks, per-level final logits). Parity tests only."""
        dev, lib = self.device, L.lib()
        st = semantic_tokens.to(dev).to(torch.int32).contiguous()
        B, T = st.shape
        assert B <= MAX_CHUNK
        has_prompt = acoustic_prompt_tokens is not None and semantic_prompt_tokens is not None
        ap = acoustic_prompt_tokens.to(dev).to(torch.int32).contiguous() if has_prompt else None
        sp = semantic_prompt_tokens.to(dev).to(torch.int32).contiguous() if has_prompt else None
        P = ap.shape[-1] if has_prompt else 0
        self._bind(B, T, P, keep_logits=True)
        s_ = L.stream_ptr()
        L.check(lib.edm_s2a_set_batch_offset(self._ctx, 0), "set_batch_offset")
        L.check(lib.edm_s2a_build_input(self._ctx, L.ptr(st), L.ptr(sp), L.ptr(ap), ap.shape[1] if has_prompt else 0, s_), "build_input")
        tr = dict(step_logits=[], step_ids=[], step_masks=[], step_masks_raw=[], step_logp=[], x0=self._view("x_in", (B, P + T, self.config.hidden_size), torch.float32).clone())
        V = self.num_codevectors
        if steps > 1:
            for s in range(steps):
                last = s == steps - 1
                L.check(lib.edm_s2a_first_level(self._ctx, None, s_), "first_level")
                tr["step_logits"].append(self._view("logits", (B, T, V), torch.float32).clone())
                cg = None if (cat_gumbel is None or last) else cat_gumbel[s].to(dev).float().contiguous()
                rg = None if (remask_gumbel is None or last) else remask_gumbel[s].to(dev).float().contiguous()
                fi = None if forced_ids is None else forced_ids[s].to(dev).to(torch.int32).contiguous()
                fm = None if (forced_masks is None or last) else forced_masks[s].to(dev).to(torch.uint8).contiguous()
                L.check(lib.edm_s2a_step(self._ctx, s, int(steps), float(temperature), int(seed), L.ptr(cg), L.ptr(rg), L.ptr(fi), L.ptr(fm), s_), "step")
                tr["step_ids"].append(self._view("ids_raw", (B, T), torch.int32).clone().long())
                if not last:
                    tr["step_masks"].append(self._view("mask", (B, T), torch.uint8).clone().bool())
                    tr["step_masks_raw"].append(self._view("mask_raw", (B, T), torch.uint8).clone().bool())
                    tr["step_logp"].append(self._view("logp", (B, T), torch.float32).clone())
        tr["x_final"] = self._view("x_in", (B, P + T, self.config.hidden_size), torch.float32).clone()
        codes = torch.empty(B, self.num_quantizers, T, device=dev, dtype=torch.int64)
        fc = None if forced_coarse is None else forced_coarse.to(dev).to(torch.int32).contiguous()
        L.check(lib.edm_s2a_full_pass(self._ctx, None, L.ptr(fc), L.ptr(codes), s_), "full_pass")
        n_inj = len(self.injection_layers)
        coarse = self._view("coarse_logits", (4, B, T, V), torch.float32)[:n_inj].permute(1, 0, 2, 3)
        fine = self._view("fine_logits", (B, T, self.num_quantizers - n_inj, V), torch.float32).permute(0, 2, 1, 3)
        tr["all_logits"] = torch.cat([coarse, fine], dim=1).clone()
        tr["codes"] = codes
        return tr

    def cosine_schedule_mask(self, feature_length, batch_size):
        """modeling_injection_conformer.py:62-74: one masking probability cos(u), u ~ U(0, pi/2), per sequence."""
        import math

        u = torch.empty(batch_size, device=self.device).uniform_(0, math.pi / 2)
        p = torch.cos(u).unsqueeze(1).expand(batch_size, feature_length)
        return torch.bernoulli(p).bool()

    @torch.no_grad()
    @_on_device
    def forward(self, acoustic_tokens, semantic_tokens, *, mask_time_indices=None):
        """InjectionConformerModel.forward (modeling_injection_conformer.py:76-128) in eval mode: masked encoder input,
        ground-truth coarse injections, 12-level logits, mean cross-entropy over the masked positions (all positions with
        loss_all) and the arg-max codes at the same positions. No dropout, no autograd: this is the validation-loss path,
        composed from the decoder's own kernels; `mask_time_indices` replaces the cosine_schedule_mask draw (parity tests)."""
        assert acoustic_tokens.shape[-1] == semantic_tokens.shape[-1], "Acoustic and semantic tokens must have same length"
        dev, lib = self.device, L.lib()
        _check_range(acoustic_tokens, self.num_codevectors, "acoustic_tokens")
        _check_range(semantic_tokens, self.config.num_semantic_tokens, "semantic_tokens")
        ac = acoustic_tokens.to(dev)
        st = semantic_tokens.to(dev)
        B, Q, T = ac.shape
        if Q != self.num_quantizers:
            raise ValueError(f"acoustic_tokens must carry {self.num_quantizers} levels, got {Q}")
        mask = (self.cosine_schedule_mask(T, B) if mask_time_indices is None else mask_time_indices.to(dev)).bool()
        n_inj, V = len(self.injection_layers), self.num_codevectors
        logp = torch.empty(B, Q, T, device=dev, dtype=torch.float32)          # log p(target) per (b, q, t)
        out_codes = torch.empty(B, Q, T, device=dev, dtype=torch.int64)
        s_ = L.stream_ptr()
        for b0 in range(0, B, MAX_CHUNK):
            b1 = min(B, b0 + MAX_CHUNK)
            nb, sl = b1 - b0, slice(b0, b1)
            self._bind(nb, T, 0, keep_logits=True)
            sem = st[sl].to(torch.int32).contiguous()
            tgt = ac[sl].to(torch.int32).contiguous()
            L.check(lib.edm_s2a_build_input(self._ctx, L.ptr(sem), None, None, 0, s_), "build_input")
            # one schedule step with everything teacher-forced: every (still fully masked) row receives the level-0 ground-truth
            # features, then the rows of `mask` go back to the mask token = the reference's torch.where(mask, sem + mask_token, sem + feat).
            # (every temporary is bound to a name until its call is enqueued: the caching allocator may hand a freed block to
            # the next temporary, whose fill kernel would run before ours)
            tgt0, m8 = tgt[:, 0].contiguous(), mask[sl].to(torch.uint8).contiguous()
            L.check(lib.edm_s2a_step(self._ctx, 0, 2, 1.0, 0, None, None, L.ptr(tgt0), L.ptr(m8), s_), "step")
            codes = torch.empty(nb, Q, T, device=dev, dtype=torch.int64)
            tgt_c = tgt[:, :n_inj].contiguous()
            L.check(lib.edm_s2a_full_pass(self._ctx, None, L.ptr(tgt_c), L.ptr(codes), s_), "full_pass")
            out_codes[sl] = codes
            # log-softmax of the target id at every position (the sampling kernel with the targets teacher-forced)
            coarse = self._view("coarse_logits", (4, nb * T, V), torch.float32)
            keep = []
            for k in range(n_inj):
                lp = torch.empty(nb * T, device=dev, dtype=torch.float32)
                tk, ik = tgt[:, k].contiguous(), torch.empty(nb, T, device=dev, dtype=torch.int32)
                keep += [tk, ik]
                L.check(lib.edm_sample(L.ptr(coarse[k]), V, nb * T, None, 0, 0, 0, L.ptr(tk), L.ptr(ik), L.ptr(lp), T, 1, 1, 0, s_), "sample")
                logp[sl, k] = lp.view(nb, T)
            nf = Q - n_inj
            fine = self._view("fine_logits", (nb * T * nf, V), torch.float32)
            lp = torch.empty(nb * T * nf, device=dev, dtype=torch.float32)
            tf, ids_f = tgt[:, n_inj:].contiguous(), torch.empty(nb, nf, T, device=dev, dtype=torch.int32)
            L.check(lib.edm_sample(L.ptr(fine), V, nb * T * nf, None, 0, 0, 0, L.ptr(tf), L.ptr(ids_f), L.ptr(lp), T, nf, nf, 0, s_), "sample")
            logp[sl, n_inj:] = lp.view(nb, T, nf).permute(0, 2, 1)
            del keep
        sel = torch.ones_like(mask) if self.loss_all else mask
        sel3 = sel[:, None, :].expand(B, Q, T)
        loss = -(logp.masked_select(sel3).mean())
        # the reference flattens only on the masked branch (modeling_injection_conformer.py:114-120): with loss_all the arg-max codes
        # keep their [b, q, t] shape
        out_sel = out_codes if self.loss_all else out_codes.masked_select(sel3)
        return InjectionConformerOutput(loss=loss, output_acoustic_codes=out_sel, target_acoustic_codes=ac.clone())

    __call__ = forward
