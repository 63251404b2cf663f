"""HuBERT-large semantic features and tokens on the CUDA path.

Replaces the eager `transformers` HuBERT call of the reference's semantic tokenizer (semantic_tokenizer_hubert.py:74-90, run under
bf16 autocast by dump_tokens.py:213 and inference.py:33): waveform -> HubertModel(...).hidden_states[output_layer] -> k-means ids.
The model is transformers' HubertModel with feat_extract_norm="layer" and do_stable_layer_norm=True (hubert-large): a LayerNorm conv
feature extractor (7 convs, 512 channels, 320 samples per frame), a feature projection, a grouped positional conv and pre-LayerNorm
transformer layers. hidden_states[i] is the input of layer i, so features of layer `output_layer` are the residual stream after
layers 0 .. output_layer - 1, before the encoder's final LayerNorm; later layers never run. The last entry,
hidden_states[num_hidden_layers], is the exception: transformers appends it after the final LayerNorm, and so does output_layer ==
num_hidden_layers here.

Launches (csrc/hubert.cuh, include/edm_s2a.h): edm_hubert_conv0 (conv 0 + LN + GELU), edm_dac_conv + edm_hubert_ln512 per strided conv,
edm_hubert_ln512 (projection LN, gathering the valid frames) + edm_gemm_bf16, edm_hubert_pad_rows + edm_hubert_pos_conv, then per layer
edm_layernorm, the fused q|k|v GEMM, edm_attention_varlen, out_proj (residual epilogue), edm_layernorm, the GELU up-projection and the
residual down-projection. Clips of a list are packed along time (DESIGN §4b): each starts at a multiple of 320 samples, so every
conv stage runs once over the packed rows and the transformer runs on the valid frames of all clips, separated by attention's
sequence offsets.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import torch

from . import _lib as L

HOP = 320                # samples per frame: prod(conv_stride)
_KERNELS = (10, 3, 3, 3, 3, 2, 2)
_STRIDES = (5, 2, 2, 2, 2, 2, 2)
POS_PAD = 64             # zero rows around every sequence in the positional conv's operand (k = 128, padding 64)


def _cfg(config, name, default=None):
    return config.get(name, default) if isinstance(config, dict) else getattr(config, name, default)


def check_config(config, output_layer: int = 18) -> None:
    """ValueError for a configuration the kernels do not implement (they are not emulated)."""
    want = dict(hidden_size=1024, num_attention_heads=16, intermediate_size=4096, feat_extract_norm="layer", do_stable_layer_norm=True,
                conv_bias=True, num_conv_pos_embeddings=128, num_conv_pos_embedding_groups=16, feat_extract_activation="gelu",
                hidden_act="gelu", feat_proj_layer_norm=True)
    for k, v in want.items():
        got = _cfg(config, k, v)
        if got != v:
            raise ValueError(f"HuBERT config {k}={got!r} is not supported (the kernels implement {k}={v!r})")
    if tuple(_cfg(config, "conv_dim", (512,) * 7)) != (512,) * 7:
        raise ValueError("HuBERT conv_dim must be 512 x 7")
    if tuple(_cfg(config, "conv_kernel", _KERNELS)) != _KERNELS or tuple(_cfg(config, "conv_stride", _STRIDES)) != _STRIDES:
        raise ValueError(f"HuBERT conv_kernel / conv_stride must be {_KERNELS} / {_STRIDES}")
    if bool(_cfg(config, "conv_pos_batch_norm", False)):
        raise ValueError("HuBERT conv_pos_batch_norm is not supported")
    n_layers = int(_cfg(config, "num_hidden_layers", 24))
    if not isinstance(output_layer, int) or not 1 <= output_layer <= n_layers:
        raise ValueError(f"output_layer must be an int in [1, {n_layers}] (got {output_layer!r})")


def frame_count(n_samples: int) -> int:
    """Frames of a clip: HubertModel._get_feat_extract_output_lengths (floor((L - 400) / 320) + 1 for L >= 400); 0 below 400."""
    n = int(n_samples)
    for k, s in zip(_KERNELS, _STRIDES):
        n = (n - k) // s + 1
        if n <= 0:
            return 0
    return n


def fold_pos_conv_weight(g: torch.Tensor, v: torch.Tensor) -> torch.Tensor:
    """weight_norm with dim=2 (HubertPositionalConvEmbedding): w = g * v / ||v||, the norm over (out, in) per tap, in fp32."""
    g, v = g.float(), v.float()
    return v * (g / v.norm(dim=(0, 1), keepdim=True))


def pack_weights(state_dict: dict, config, output_layer: int = 18, prefix: str = "") -> dict:
    """HubertModel.state_dict() (keys under `prefix`) -> the kernels' operands on the host. Reads only what layers < output_layer use:
    masked_spec_embed, later layers and encoder.layer_norm (unless output_layer is the last layer) are ignored. KeyError names a
    missing key."""
    check_config(config, output_layer)

    def t(key):
        try:
            return state_dict[prefix + key].detach().to("cpu")
        except KeyError:
            raise KeyError(f"HuBERT state dict has no {prefix + key!r}") from None

    bf = torch.bfloat16
    fe = "feature_extractor.conv_layers."
    out = dict(
        conv0_w=t(fe + "0.conv.weight").float()[:, 0, :].t().contiguous(),          # [10][512] tap-major
        conv0_b=t(fe + "0.conv.bias").float(), conv0_ln_w=t(fe + "0.layer_norm.weight").float(), conv0_ln_b=t(fe + "0.layer_norm.bias").float(),
        convs=[],
    )
    for i in range(1, 7):
        w = t(fe + f"{i}.conv.weight").float()                                       # [512, 512, k], k = 3 or 2
        k = w.shape[2]
        # stride 2 over the [rows / 2][1024] view: view row t = input rows 2t | 2t + 1, so tap pair (0, 1) is one 1024-wide tap and
        # tap 2 (k = 3) is a second one whose upper half is zero
        taps = [torch.cat([w[:, :, 0], w[:, :, 1]], 1)]
        if k == 3:
            taps.append(torch.cat([w[:, :, 2], torch.zeros_like(w[:, :, 2])], 1))
        out["convs"].append(dict(w=torch.cat(taps, 1).to(bf).contiguous(), taps=len(taps), b=t(fe + f"{i}.conv.bias").float(),
                                 ln_w=t(fe + f"{i}.layer_norm.weight").float(), ln_b=t(fe + f"{i}.layer_norm.bias").float()))
    out.update(fp_ln_w=t("feature_projection.layer_norm.weight").float(), fp_ln_b=t("feature_projection.layer_norm.bias").float(),
               fp_w=t("feature_projection.projection.weight").to(bf).contiguous(), fp_b=t("feature_projection.projection.bias").float())
    pc = "encoder.pos_conv_embed.conv."
    if prefix + pc + "parametrizations.weight.original0" in state_dict or prefix + pc + "weight_g" not in state_dict:
        wpc = fold_pos_conv_weight(t(pc + "parametrizations.weight.original0"), t(pc + "parametrizations.weight.original1"))
    else:                                                                            # checkpoints saved with the older weight_norm hook
        wpc = fold_pos_conv_weight(t(pc + "weight_g"), t(pc + "weight_v"))
    out["pos_w_f32"] = wpc                                                           # [1024, 64, 128]
    out["pos_w"] = wpc.permute(0, 2, 1).reshape(1024, 128 * 64).to(bf).contiguous()  # column 64 j + c
    out["pos_b"] = t(pc + "bias").float()
    out["layers"] = []
    for l in range(output_layer):
        p = f"encoder.layers.{l}."
        a = p + "attention."
        out["layers"].append(dict(
            ln_w=t(p + "layer_norm.weight").float(), ln_b=t(p + "layer_norm.bias").float(),
            wqkv=torch.cat([t(a + "q_proj.weight"), t(a + "k_proj.weight"), t(a + "v_proj.weight")]).to(bf).contiguous(),
            bqkv=torch.cat([t(a + "q_proj.bias"), t(a + "k_proj.bias"), t(a + "v_proj.bias")]).float(),
            wo=t(a + "out_proj.weight").to(bf).contiguous(), bo=t(a + "out_proj.bias").float(),
            fln_w=t(p + "final_layer_norm.weight").float(), fln_b=t(p + "final_layer_norm.bias").float(),
            w1=t(p + "feed_forward.intermediate_dense.weight").to(bf).contiguous(), b1=t(p + "feed_forward.intermediate_dense.bias").float(),
            w2=t(p + "feed_forward.output_dense.weight").to(bf).contiguous(), b2=t(p + "feed_forward.output_dense.bias").float()))
    out["final_ln"] = None
    if output_layer == int(_cfg(config, "num_hidden_layers", 24)):
        out["final_ln"] = (t("encoder.layer_norm.weight").float(), t("encoder.layer_norm.bias").float())
    return out


# ---------------------------------------------------------------------------------------------------------------- packed layout
@dataclass
class Chunk:
    """Clips [start, stop) of a list, packed. Sample rows: clip i at sample_starts[i] (a multiple of HOP), n_samples rows in all;
    conv rows at stage 7 = sample rows / HOP. Compact frame rows: clip i at cu[i] .. cu[i + 1] (T_i = frames[i]). gather[r] = stage-7
    row of compact row r. Padded rows of the positional conv: clip i at pad_starts[i], POS_PAD zero rows before every clip and after
    the last; pad_map[r] = compact row of padded row r or -1."""
    start: int
    stop: int
    sample_starts: list
    n_samples: int
    frames: list
    cu: list
    gather: list = field(repr=False)
    pad_starts: list = field(repr=False)
    pad_map: list = field(repr=False)


def plan(lengths, max_chunk_samples: int) -> list:
    """Cuts clips of `lengths` samples, in order, into chunks of at most max_chunk_samples packed samples (a longer clip gets a chunk of
    its own). ValueError for a clip shorter than one frame (400 samples)."""
    lengths = [int(n) for n in lengths]
    if not lengths:
        raise ValueError("an empty list of clips")
    for n in lengths:
        if frame_count(n) <= 0:
            raise ValueError(f"a clip of {n} samples is shorter than one HuBERT frame (400 samples)")
    slots = [-(-n // HOP) * HOP for n in lengths]
    chunks, i = [], 0
    while i < len(lengths):
        j, tot = i + 1, slots[i]
        while j < len(lengths) and tot + slots[j] <= max_chunk_samples:
            tot += slots[j]
            j += 1
        starts = [sum(slots[i:k]) for k in range(i, j)]
        frames = [frame_count(n) for n in lengths[i:j]]
        cu = [0]
        for t in frames:
            cu.append(cu[-1] + t)
        gather = [s // HOP + t for s, T in zip(starts, frames) for t in range(T)]
        pad_starts, pad_map = [], [-1] * POS_PAD
        for T, c0 in zip(frames, cu):
            pad_starts.append(len(pad_map))
            pad_map += list(range(c0, c0 + T)) + [-1] * POS_PAD
        chunks.append(Chunk(i, j, starts, tot, frames, cu, gather, pad_starts, pad_map))
        i = j
    return chunks


class HubertFeatures:
    """HubertModel(config) features hidden_states[output_layer] on the CUDA path.

    forward(input_values [B, L]) -> fp32 [B, T, 1024]; forward_batch([L_i] clips) -> [fp32 [T_i, 1024]]. The model consumes
    input_values exactly as HubertModel does (no normalisation here: that is the feature extractor's job, see SemanticTokenizer).
    Item i of forward_batch equals forward(clips[i][None])[0] bit for bit."""

    def __init__(self, config, state_dict: dict, device="cuda", output_layer: int = 18, prefix: str = "", max_chunk_samples: int = 1 << 23):
        check_config(config, output_layer)
        if not torch.cuda.is_available():
            raise L.EdmError("edm_tts_b200 needs a CUDA device (sm_100); there is no CPU fallback")
        self.device = torch.device(device)
        self.output_layer = output_layer
        self.max_chunk_samples = int(max_chunk_samples)
        host = pack_weights(state_dict, config, output_layer, prefix)
        host.pop("pos_w_f32")
        dev = self.device

        def mv(x):
            if isinstance(x, torch.Tensor):
                return x.to(dev).contiguous()
            if isinstance(x, (list, tuple)):
                return type(x)(mv(v) for v in x)
            if isinstance(x, dict):
                return {k: mv(v) for k, v in x.items()}
            return x

        self.w = mv(host)

    @classmethod
    def from_pretrained(cls, path: str, device="cuda", output_layer: int = 18, **kw):
        """A transformers HubertModel directory (config.json + weights), e.g. a local copy of facebook/hubert-large-ll60k."""
        from transformers import HubertModel

        model = HubertModel.from_pretrained(path)
        return cls(model.config, model.state_dict(), device=device, output_layer=output_layer, **kw)

    def eval(self):
        return self

    # ------------------------------------------------------------------ forward
    @torch.no_grad()
    def forward(self, input_values: torch.Tensor) -> torch.Tensor:
        if input_values.dim() != 2:
            raise ValueError("input_values must be [B, L]")
        return torch.stack(self.forward_batch(list(input_values)))

    __call__ = forward

    @torch.no_grad()
    def forward_batch(self, clips) -> list:
        if not isinstance(clips, (list, tuple)) or len(clips) == 0:
            raise ValueError("clips must be a non-empty list of [L_i] tensors")
        for c in clips:
            if not torch.is_tensor(c) or c.dim() != 1:
                raise ValueError("every clip must be a 1-D [L_i] tensor")
        out = []
        for ch in plan([c.shape[0] for c in clips], self.max_chunk_samples):
            x = self._run_chunk(ch, clips[ch.start:ch.stop])
            out.extend(x[a:b] for a, b in zip(ch.cu[:-1], ch.cu[1:]))
        return out

    def _run_chunk(self, ch: Chunk, clips) -> torch.Tensor:
        c7 = self._conv_stack(ch, clips)
        idx = torch.tensor(ch.gather + ch.pad_map + ch.cu, dtype=torch.int32).to(self.device)
        N, R = ch.cu[-1], len(ch.pad_map)
        gather, pad_map, cu = idx[:N], idx[N:N + R], idx[N + R:]
        x = self._project(c7, gather)
        self._pos_conv(x, pad_map)
        bufs = self._layer_buffers(N)
        for ly in self.w["layers"]:
            self._layer(ly, x, cu, len(ch.frames), bufs)
        if self.w["final_ln"] is not None:    # hidden_states[num_hidden_layers] is taken after encoder.layer_norm
            lw, lb = self.w["final_ln"]
            L.check(L.lib().edm_layernorm(L.ptr(x), 0, N, L.ptr(lw), L.ptr(lb), None, None, L.ptr(x), None, 1, 0, 1e-5, L.stream_ptr()),
                    "layernorm (hubert)")
        return x

    # the stages, each callable on its own (the teacher-forced parity tests feed them the reference's activations)
    def _conv_stack(self, ch: Chunk, clips) -> torch.Tensor:
        """Packed audio of the chunk -> bf16 [n_samples / 320][512]: the feature extractor's output rows (valid rows: ch.gather)."""
        dev, w, st, lib = self.device, self.w, L.stream_ptr(), L.lib()
        audio = torch.zeros(ch.n_samples, device=dev, dtype=torch.float32)
        for s, c in zip(ch.sample_starts, clips):
            audio[s:s + c.shape[0]] = c.to(dev, torch.float32)
        rows = ch.n_samples // _STRIDES[0]
        c = torch.empty(rows, 512, device=dev, dtype=torch.bfloat16)
        L.check(lib.edm_hubert_conv0(L.ptr(audio), ch.n_samples, rows, L.ptr(w["conv0_w"]), L.ptr(w["conv0_b"]), L.ptr(w["conv0_ln_w"]),
                                     L.ptr(w["conv0_ln_b"]), L.ptr(c), st), "hubert_conv0")
        for cv in w["convs"]:
            # stride 2 on the [rows / 2][1024] view; rows stays even (n_samples is a multiple of 320 = 5 * 2^6)
            rows //= 2
            nxt = torch.empty(rows, 512, device=dev, dtype=torch.bfloat16)
            L.check(lib.edm_dac_conv(L.ptr(c), rows, 1024, rows * 1024, 1, L.ptr(cv["w"]), 512, cv["taps"], 1, 0, rows, L.ptr(cv["b"]), None, 0,
                                     None, None, 0, L.ptr(nxt), rows * 512, 0, rows, None, 0, st), "dac_conv (hubert)")
            L.check(lib.edm_hubert_ln512(L.ptr(nxt), None, rows, L.ptr(cv["ln_w"]), L.ptr(cv["ln_b"]), 1, L.ptr(nxt), st), "hubert_ln512")
            c = nxt
        return c

    def _project(self, c7: torch.Tensor, gather: torch.Tensor) -> torch.Tensor:
        """Feature projection of the rows `gather` of c7 -> fp32 [len(gather)][1024]."""
        N = gather.shape[0]
        f = torch.empty(N, 512, device=self.device, dtype=torch.bfloat16)
        L.check(L.lib().edm_hubert_ln512(L.ptr(c7), L.ptr(gather), N, L.ptr(self.w["fp_ln_w"]), L.ptr(self.w["fp_ln_b"]), 0, L.ptr(f),
                                         L.stream_ptr()), "hubert_ln512")
        x = torch.empty(N, 1024, device=self.device, dtype=torch.float32)
        self._gemm(f, self.w["fp_w"], L.EPI_F32, self.w["fp_b"], x)
        return x

    def _pos_conv(self, x: torch.Tensor, pad_map: torch.Tensor) -> None:
        """x += GELU(SamePad(pos_conv(x))) per sequence (pad_map: Chunk.pad_map on the device)."""
        R = pad_map.shape[0]
        xp = torch.empty(R, 1024, device=self.device, dtype=torch.bfloat16)
        L.check(L.lib().edm_hubert_pad_rows(L.ptr(x), L.ptr(pad_map), R, L.ptr(xp), L.stream_ptr()), "hubert_pad_rows")
        L.check(L.lib().edm_hubert_pos_conv(L.ptr(xp), L.ptr(pad_map), R, L.ptr(self.w["pos_w"]), L.ptr(self.w["pos_b"]), L.ptr(x),
                                            L.stream_ptr()), "hubert_pos_conv")

    def _layer_buffers(self, N: int) -> dict:
        dev, bf = self.device, torch.bfloat16
        return dict(h=torch.empty(N, 1024, device=dev, dtype=bf), qkv=torch.empty(N, 3072, device=dev, dtype=bf),
                    o=torch.empty(N, 1024, device=dev, dtype=bf), u=torch.empty(N, 4096, device=dev, dtype=bf))

    def _layer(self, ly: dict, x: torch.Tensor, cu: torch.Tensor, n_seq: int, b: dict) -> None:
        """HubertEncoderLayerStableLayerNorm on the fp32 stream x (in place); cu: int32 sequence offsets on the device."""
        self._layernorm(x, ly["ln_w"], ly["ln_b"], b["h"])
        self._gemm(b["h"], ly["wqkv"], L.EPI_BF16, ly["bqkv"], b["qkv"])
        L.check(L.lib().edm_attention_varlen(L.ptr(b["qkv"]), n_seq, L.ptr(cu), 16, L.ptr(b["o"]), L.stream_ptr()), "attention_varlen (hubert)")
        self._gemm(b["o"], ly["wo"], L.EPI_RESID_F32, ly["bo"], x)
        self._layernorm(x, ly["fln_w"], ly["fln_b"], b["h"])
        self._gemm(b["h"], ly["w1"], L.EPI_GELU_BF16, ly["b1"], b["u"])
        self._gemm(b["u"], ly["w2"], L.EPI_RESID_F32, ly["b2"], x)

    def _gemm(self, a, b, epi, bias, out):
        M, K = a.shape
        N = b.shape[0]
        L.check(L.lib().edm_gemm_bf16(L.ptr(a), K, L.ptr(b), K, M, N, K, epi, L.ptr(bias), L.ptr(out), out.shape[1], 1.0, None, None, 0, 0,
                                      L.stream_ptr()), "gemm (hubert)")

    def _layernorm(self, x, w, b, z):
        L.check(L.lib().edm_layernorm(L.ptr(x), 0, x.shape[0], L.ptr(w), L.ptr(b), None, None, None, L.ptr(z), 1, 0, 1e-5, L.stream_ptr()),
                "layernorm (hubert)")


def normalize_clip(x: torch.Tensor) -> torch.Tensor:
    """Wav2Vec2FeatureExtractor(do_normalize=True): zero mean, unit variance per clip, (x - mean) / sqrt(var + 1e-7)."""
    x = x.float()
    return (x - x.mean()) / torch.sqrt(x.var(unbiased=False) + 1e-7)


def _prep_clip(clip: torch.Tensor, device, normalize: bool) -> torch.Tensor:
    clip = clip.to(device, torch.float32)
    return normalize_clip(clip) if normalize else clip


def _check_clips(clips) -> None:
    if not isinstance(clips, (list, tuple)) or len(clips) == 0:
        raise ValueError("clips must be a non-empty list of [L_i] tensors")
    for c in clips:
        if not torch.is_tensor(c) or c.dim() != 1:
            raise ValueError("every clip must be a 1-D [L_i] tensor")


class SemanticTokenizer:
    """Semantic tokens of the reference's tokenizer (semantic_tokenizer_hubert.py encode / encode_batch): HuBERT features of
    `hubert.output_layer` followed by the nearest k-means centroid (KMeansAssigner, edm_kmeans_assign).

    normalize: per-clip zero-mean / unit-variance normalisation of the waveform before HuBERT, as Wav2Vec2FeatureExtractor does with
    do_normalize. The default True is what facebook/hubert-large-ll60k's preprocessor config specifies; it has not been checked against
    the reference's semantic_tokenizer_hubert.py, which is not available here - pass normalize=False if that file feeds raw audio."""

    def __init__(self, hubert: HubertFeatures, cluster_centers: torch.Tensor, normalize: bool = True):
        from .kmeans import KMeansAssigner

        self.hubert = hubert
        self.normalize = bool(normalize)
        self.assigner = KMeansAssigner(cluster_centers, device=hubert.device)

    @classmethod
    @torch.no_grad()
    def fit(cls, hubert: HubertFeatures, clips, n_centroids: int = 1024, normalize: bool = True, **fit_kw):
        """Fit the k-means centroids on the HuBERT features of `clips` ([L_i] at 16 kHz) and build a tokenizer on them; replaces the
        reference's offline step (utility_scripts/hubert_kmeans/: features dumped to .npy, then faiss k-means). The clips get the same
        normalisation as encode_batch; their features stay on the device and never go to disk: 4 KB of fp32 per 20 ms frame, so about
        4 GB per million frames (5.6 h of audio), held twice while they are concatenated. fit_kw go to kmeans.fit_kmeans (niter, seed,
        max_points_per_centroid, init). Returns (SemanticTokenizer, KMeansFit)."""
        from .kmeans import fit_kmeans

        _check_clips(clips)
        feats = hubert.forward_batch([_prep_clip(c, hubert.device, normalize) for c in clips])
        feats = torch.cat(feats)
        fit = fit_kmeans(feats, n_centroids=n_centroids, device=hubert.device, **fit_kw)
        return cls(hubert, fit.centroids, normalize=normalize), fit

    def _prep(self, clip):
        return _prep_clip(clip, self.hubert.device, self.normalize)

    @torch.no_grad()
    def encode(self, audio: torch.Tensor) -> torch.Tensor:
        """audio [B, L] at 16 kHz -> int64 [B, T] cluster ids."""
        if audio.dim() != 2:
            raise ValueError("audio must be [B, L]")
        feats = self.hubert.forward(torch.stack([self._prep(a) for a in audio]))
        return self.assigner.assign(feats)

    @torch.no_grad()
    def encode_batch(self, clips) -> list:
        """List of [L_i] clips at 16 kHz -> list of int64 [T_i] cluster ids (views of one buffer); item i equals encode(clips[i][None])[0]."""
        _check_clips(clips)
        feats = self.hubert.forward_batch([self._prep(c) for c in clips])
        ids = self.assigner.assign(torch.cat(feats))
        return list(torch.split(ids, [f.shape[0] for f in feats]))
