"""Nearest-centroid assignment of the semantic tokenizer (HuBERT features -> k-means cluster ids) on the CUDA path.

Mirrors the tail of SemanticModelHuBERT.encode / encode_batch
(edm_tts/models/audio_tokenizer/semantic_tokenizer_hubert/semantic_tokenizer_hubert.py:74-90):
    dists = -torch.cdist(embed, cluster_centers, p=2); clusters = dists.argmax(dim=-1)
This replaces the distance + arg-max step; the HuBERT backbone in front of it is `hubert.HubertFeatures` (`hubert.SemanticTokenizer` chains the two).
"""
from __future__ import annotations

import torch

from . import _lib as L
from .weights import tf32_round


class KMeansAssigner:
    def __init__(self, cluster_centers: torch.Tensor, device="cuda"):
        if not torch.cuda.is_available():
            raise L.EdmError("edm_tts_b200 needs a CUDA device (sm_100); there is no CPU fallback")
        c = cluster_centers.detach().to(device, torch.float32).contiguous()
        if c.dim() != 2 or c.shape[1] % 32 != 0:
            raise ValueError("cluster_centers must be [n_centroids, dim] with dim a multiple of 32")
        self.device = torch.device(device)
        self.n_centroids, self.dim = c.shape
        n_pad = (self.n_centroids + 255) // 256 * 256
        if n_pad > 4096:
            raise ValueError("at most 4096 centroids")
        norm = -0.5 * c.double().pow(2).sum(-1)
        if n_pad != self.n_centroids:  # padding centroids can never win
            c = torch.cat([c, torch.zeros(n_pad - self.n_centroids, self.dim, device=c.device)])
            norm = torch.cat([norm, torch.full((n_pad - self.n_centroids,), -3.0e38, device=c.device, dtype=torch.float64)])
        self._c_hi = tf32_round(c)
        self._c_lo = tf32_round(c - self._c_hi)
        self._norm = norm.float().contiguous()
        self._n_pad = n_pad

    @torch.no_grad()
    def assign(self, embed: torch.Tensor, return_scores: bool = False):
        """embed [..., dim] (fp32 / bf16 / fp16) -> LongTensor [...] of cluster ids."""
        if embed.shape[-1] != self.dim:
            raise ValueError(f"embed must end in dim {self.dim}")
        x = embed.to(self.device, torch.float32).reshape(-1, self.dim).contiguous()
        n = x.shape[0]
        idx = torch.empty(n, device=self.device, dtype=torch.int64)
        sc = torch.empty(n, device=self.device, dtype=torch.float32) if return_scores else None
        L.check(L.lib().edm_kmeans_assign(L.ptr(x), n, self.dim, L.ptr(self._c_hi), L.ptr(self._c_lo), L.ptr(self._norm), self._n_pad, L.ptr(idx),
                                          L.ptr(sc), L.stream_ptr()), "kmeans_assign")
        idx = idx.view(embed.shape[:-1])
        return (idx, sc.view(embed.shape[:-1])) if return_scores else idx

    __call__ = assign
