"""K-means of the semantic tokenizer (HuBERT features -> cluster ids) on the CUDA path: the assignment, and the fit of the centroids.

Assignment mirrors the tail of SemanticModelHuBERT.encode / encode_batch
(edm_tts/models/audio_tokenizer/semantic_tokenizer_hubert/semantic_tokenizer_hubert.py:74-90):
    dists = -torch.cdist(embed, cluster_centers, p=2); clusters = dists.argmax(dim=-1)
This replaces the distance + arg-max step; the HuBERT backbone in front of it is `hubert.HubertFeatures` (`hubert.SemanticTokenizer` chains the two).

The fit (`fit_kmeans`) replaces the reference's offline faiss step (utility_scripts/hubert_kmeans/): Lloyd iterations as faiss
`Clustering::train` runs them in its default configuration, with the assignment above and a deterministic centroid update
(edm_kmeans_update), so a fit gives the same bits on every run.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import torch

from . import _lib as L
from .weights import tf32_round

MAX_CENTROIDS = 4096
SPLIT_EPS = 1.0 / 1024     # faiss split_clusters: relative perturbation of a split centroid pair
SPLIT_SEED = 1234          # faiss split_clusters seeds its generator with 1234 at every call


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
        if n_pad > MAX_CENTROIDS:
            raise ValueError("at most 4096 centroids")
        # padding centroids (rows n_centroids .. n_pad) can never win: zero rows with -||c||^2 / 2 = -3e38
        self._c_hi = torch.zeros(n_pad, self.dim, device=self.device)
        self._c_lo = torch.zeros(n_pad, self.dim, device=self.device)
        self._norm = torch.full((n_pad,), -3.0e38, device=self.device)
        self._n_pad = n_pad
        self.set_centroids(c)

    @torch.no_grad()
    def set_centroids(self, cluster_centers: torch.Tensor) -> None:
        """Refill the packed operands (tf32 hi / lo split, -||c||^2 / 2) from new centroids of the same shape, in place."""
        c = cluster_centers.detach().to(self.device, torch.float32)
        if tuple(c.shape) != (self.n_centroids, self.dim):
            raise ValueError(f"cluster_centers must be [{self.n_centroids}, {self.dim}]")
        k = self.n_centroids
        hi = tf32_round(c)
        self._c_hi[:k].copy_(hi)
        self._c_lo[:k].copy_(tf32_round(c - hi))
        self._norm[:k].copy_(-0.5 * c.double().pow(2).sum(-1))

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


# ------------------------------------------------------------------------------------------------------------------ the fit
@torch.no_grad()
def kmeans_update(x: torch.Tensor, idx: torch.Tensor, centroids: torch.Tensor, sums: torch.Tensor | None = None,
                  check_ids: bool = True) -> torch.Tensor:
    """centroids[c] = mean of the rows x[r] with idx[r] == c (edm_kmeans_update: fp64 sums in a fixed order, rounded once to fp32), in
    place; clusters without rows keep their centroid. x fp32 [n, D] and centroids fp32 [k, D] contiguous on the device, idx int64 [n]
    with values in [0, k); sums (optional, fp64 [k, D]) receives the per-cluster sums. Returns the counts, int64 [k]. The rows are
    ordered cluster by cluster with a stable sort of idx (8-16 B per row against 4 B x D of features) and the offsets come from the
    sorted ids. ValueError for an id outside [0, k): the kernel would leave the rest of its segment unsummed. That check reads the
    smallest and largest sorted id back (a synchronisation); the fit passes check_ids=False for the assignment kernel's ids, which
    are in range by construction, so that nothing in its update waits for the device."""
    if x.dim() != 2 or x.dtype != torch.float32 or centroids.dtype != torch.float32 or centroids.dim() != 2 or centroids.shape[1] != x.shape[1]:
        raise ValueError("x must be fp32 [n, D] and centroids fp32 [k, D]")
    if idx.shape != (x.shape[0],) or idx.dtype != torch.int64:
        raise ValueError("idx must be int64 [n]")
    n, dim = x.shape
    k = centroids.shape[0]
    if sums is not None and (sums.shape != centroids.shape or sums.dtype != torch.float64):
        raise ValueError("sums must be fp64 [k, D]")
    srt, perm = torch.sort(idx, stable=True)
    if check_ids and n > 0:
        lo, hi = srt[[0, -1]].tolist()
        if lo < 0 or hi >= k:
            raise ValueError(f"idx must lie in [0, {k}) (got ids {lo} .. {hi})")
    offsets = torch.searchsorted(srt, torch.arange(k + 1, device=idx.device, dtype=torch.int64))
    partials = torch.empty(max(1, L.lib().edm_kmeans_update_workspace_bytes(n, dim, k) // 8), device=x.device, dtype=torch.float64)
    L.check(L.lib().edm_kmeans_update(L.ptr(x), n, dim, L.ptr(idx), L.ptr(perm), L.ptr(offsets), k, L.ptr(partials), L.ptr(centroids),
                                      L.ptr(sums), L.stream_ptr()), "kmeans_update")
    return offsets.diff()


def split_clusters(centroids: torch.Tensor, counts: list, n_used: int) -> int:
    """faiss split_clusters: every empty cluster ci (in order) takes a copy of a cluster cj picked at random with probability
    (count_cj - 1) / (n_used - k): walking cj = 0, 1, ... cyclically, with a fresh r = torch.rand(1) per candidate from a generator
    seeded with SPLIT_SEED at each call, the first cj with r < p. The pair is pushed apart, even columns of ci x (1 + EPS) and of
    cj x (1 - EPS), odd columns the other way round, and the count of cj is shared: count_ci = count_cj / 2, count_cj -= count_ci.
    centroids [k, D] (any device / float dtype) and counts (a list of k floats) are updated in place. Returns the number of splits.
    The draws are taken in blocks (torch.rand(m) of a CPU generator is the stream of m torch.rand(1) calls): a walk takes ~k of them."""
    k = len(counts)
    g = torch.Generator().manual_seed(SPLIT_SEED)
    draws, nd = [], 0
    n_split = 0
    for ci in range(k):
        if counts[ci] != 0:
            continue
        cj = 0
        while True:
            c = counts[cj] - 1.0
            p = c / (n_used - k) if n_used != k else (math.inf if c > 0 else -math.inf)
            if nd == len(draws):
                draws += torch.rand(4096, generator=g).tolist()
            nd += 1
            if draws[nd - 1] < p:
                break
            cj = (cj + 1) % k
        centroids[ci] = centroids[cj]
        centroids[ci, 0::2] *= 1 + SPLIT_EPS
        centroids[ci, 1::2] *= 1 - SPLIT_EPS
        centroids[cj, 0::2] *= 1 - SPLIT_EPS
        centroids[cj, 1::2] *= 1 + SPLIT_EPS
        counts[ci] = counts[cj] / 2
        counts[cj] -= counts[ci]
        n_split += 1
    return n_split


def subsample_indices(n: int, n_centroids: int, max_points_per_centroid, seed: int):
    """Rows the fit uses (faiss subsampling): None (all n rows) unless n > k * max_points_per_centroid, else the first
    k * max_points_per_centroid entries of torch.randperm(n) drawn from a CPU generator seeded with `seed`."""
    if max_points_per_centroid is None or n <= n_centroids * max_points_per_centroid:
        return None
    return torch.randperm(n, generator=torch.Generator().manual_seed(seed))[:n_centroids * max_points_per_centroid]


def init_indices(n_used: int, n_centroids: int, seed: int) -> torch.Tensor:
    """Rows of the (subsampled) data that start as centroids when no init is given: torch.randperm(n_used)[:k], seeded with seed + 1."""
    return torch.randperm(n_used, generator=torch.Generator().manual_seed(seed + 1))[:n_centroids]


def check_fit_args(shape, n_centroids: int, niter: int, init=None) -> None:
    """ValueError for a fit the kernels cannot run (checked before anything touches the device)."""
    if len(shape) != 2:
        raise ValueError("x must be [n, dim]")
    n, dim = shape
    if not 1 <= n_centroids <= MAX_CENTROIDS:
        raise ValueError(f"n_centroids must be in [1, {MAX_CENTROIDS}] (got {n_centroids})")
    if n < n_centroids:
        raise ValueError(f"{n} points cannot fit {n_centroids} centroids")
    if dim % 32 != 0 or dim == 0:
        raise ValueError(f"dim must be a positive multiple of 32 (got {dim})")
    if niter < 1:
        raise ValueError("niter must be >= 1")
    if init is not None and tuple(init.shape) != (n_centroids, dim):
        raise ValueError(f"init must be [{n_centroids}, {dim}] (got {tuple(init.shape)})")


@dataclass
class KMeansFit:
    centroids: torch.Tensor    # fp32 [k, D] on the device
    objective: list            # per iteration: sum over rows of min_c ||x - c||^2 (fp64), before that iteration's update
    counts: torch.Tensor       # int64 [k]: rows per cluster in the last assignment (before splits)
    n_split: list              # per iteration: empty clusters split


class Lloyd:
    """The state of one fit and its iteration in steps (fit_kmeans runs them; the benchmark times them one by one): assign
    (edm_kmeans_assign), update (edm_kmeans_update, and the objective of the assignment; it stays on the device), split (the counts
    come to the host: the one synchronisation of an iteration), repack (the assigner's operands refilled in place).

    The objective is sum_r ||x_r - c_idx(r)||^2 = sum |x|^2 - 2 sum_c c . S_c + sum_c n_c |c|^2 in fp64, with the pre-update centroids
    c and the fp64 cluster sums S_c of the update. The assignment's own scores (x.c - |c|^2 / 2, fp32 from the tensor cores) would
    give sum |x|^2 - 2 sum best, but |x|^2 and 2 best nearly cancel and their fp32 error (~1e-2 per 1024-dim row) adds up to ~2e-5 of
    sum |x|^2 over a fit."""

    def __init__(self, x: torch.Tensor, init: torch.Tensor, niter: int):
        self.x = x
        self.n, self.dim = x.shape
        self.centroids = init.to(x.device, torch.float32).contiguous().clone()
        self.k = self.centroids.shape[0]
        self.assigner = KMeansAssigner(self.centroids, device=x.device)
        # sum |x|^2 in fp64 once, in slices (a fp64 copy of x would be twice its size)
        self.sq_total = sum(x[a:a + 65536].double().pow(2).sum() for a in range(0, self.n, 65536))
        self.sums = torch.empty(self.k, self.dim, device=x.device, dtype=torch.float64)
        self.objective = torch.zeros(niter, device=x.device, dtype=torch.float64)
        self.n_split = []
        self.idx = self.counts = None

    def assign(self) -> None:
        self.idx = self.assigner.assign(self.x)

    def update(self, it: int) -> None:
        c = self.centroids.double()                                          # before the update
        self.counts = kmeans_update(self.x, self.idx, self.centroids, self.sums, check_ids=False)
        self.objective[it] = self.sq_total - 2.0 * (c * self.sums).sum() + (self.counts.double() * c.pow(2).sum(1)).sum()

    def split(self) -> None:
        self.n_split.append(split_clusters(self.centroids, [float(c) for c in self.counts.tolist()], self.n))

    def repack(self) -> None:
        self.assigner.set_centroids(self.centroids)

    def run(self, niter: int) -> KMeansFit:
        for it in range(niter):
            self.assign()
            self.update(it)
            self.split()
            self.repack()
        return KMeansFit(self.centroids, self.objective.tolist(), self.counts, self.n_split)


def prepare_fit(x: torch.Tensor, n_centroids: int = 1024, niter: int = 25, seed: int = 1234, max_points_per_centroid=256, init=None,
                device=None) -> Lloyd:
    """Checks, subsampling and initialisation of fit_kmeans; returns the Lloyd state before the first iteration."""
    check_fit_args(tuple(x.shape), n_centroids, niter, init)
    if not torch.cuda.is_available():
        raise L.EdmError("edm_tts_b200 needs a CUDA device (sm_100); there is no CPU fallback")
    dev = torch.device(device) if device is not None else (x.device if x.is_cuda else torch.device("cuda"))
    sel = subsample_indices(x.shape[0], n_centroids, max_points_per_centroid, seed)
    if sel is not None:
        x = x[sel.to(x.device)]
    x = x.detach().to(dev, torch.float32).contiguous()
    if init is None:
        init = x[init_indices(x.shape[0], n_centroids, seed).to(dev)]
    return Lloyd(x, init, niter)


@torch.no_grad()
def fit_kmeans(x: torch.Tensor, n_centroids: int = 1024, niter: int = 25, seed: int = 1234, max_points_per_centroid=256, init=None,
               device=None) -> KMeansFit:
    """K-means centroids of x [n, D] (fp32; bf16 / fp16 are converted to fp32 once) by Lloyd's algorithm, as faiss Clustering::train
    runs it by default (nredo = 1, not spherical, no point weights); faiss's random streams are not reproduced.

    If n > k * max_points_per_centroid, the fit uses the rows subsample_indices(n, k, max_points_per_centroid, seed) (None: all rows).
    The centroids start from `init` [k, D] if given, else from the rows init_indices(n_used, k, seed). Each iteration assigns every row
    to its nearest centroid (edm_kmeans_assign, 3xTF32, first maximum on ties), moves each centroid to the mean of its rows
    (edm_kmeans_update, fp64 sums in a fixed order) and records the objective of the assignment, sum ||x - c||^2 in fp64 (see Lloyd),
    splits empty clusters (split_clusters) and repacks the centroids. The same input gives the same bits on every run. Device memory:
    x in fp32 (a copy when x is given in another dtype or on the host) plus 8 B per row for the assignment and its sort."""
    return prepare_fit(x, n_centroids, niter, seed, max_points_per_centroid, init, device).run(niter)
