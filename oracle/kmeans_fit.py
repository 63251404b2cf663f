"""Restatement of the semantic tokenizer's k-means fit (test infrastructure; see oracle/__init__.py).

The reference fits its centroids offline with faiss (utility_scripts/hubert_kmeans/: Clustering::train in its default configuration).
kmeans_fit restates that loop in fp64 from the rules of faiss's Clustering.cpp: assign every row to its nearest centroid, record the
objective before the update, move each centroid to the mean of its rows, split empty clusters (split_clusters). torch's generators
stand in for faiss's. It shares no code with edm_tts_b200/kmeans.py.
"""
from __future__ import annotations

import torch


def nearest(x: torch.Tensor, c: torch.Tensor, rows: int = 8192):
    """fp64 squared distances; returns (first index of the minimum, the minimum) per row."""
    cc = (c * c).sum(1)
    ids, dmin = [], []
    for a in range(0, x.shape[0], rows):
        xa = x[a:a + rows]
        d = (xa * xa).sum(1, keepdim=True) - 2.0 * (xa @ c.T) + cc
        m, i = d.min(1)      # the first index of the minimum
        ids.append(i)
        dmin.append(m)
    return torch.cat(ids), torch.cat(dmin)


def cluster_means(x: torch.Tensor, ids: torch.Tensor, c: torch.Tensor):
    """Per-cluster fp64 mean of the rows; a cluster without rows keeps c's row. Returns (new centroids, counts int64)."""
    k = c.shape[0]
    sums = torch.zeros(k, x.shape[1], dtype=torch.float64, device=x.device).index_add_(0, ids, x.double())
    counts = torch.zeros(k, dtype=torch.int64, device=x.device).index_add_(0, ids, torch.ones_like(ids))
    return torch.where(counts[:, None] > 0, sums / counts.clamp(min=1)[:, None].double(), c), counts


def split_empty(c: torch.Tensor, hassign: list, n: int) -> int:
    """faiss split_clusters with torch.rand(1) draws of a CPU generator seeded 1234 per call: each empty ci copies the first cj
    (cyclic from 0, one draw per candidate) whose draw is below (hassign[cj] - 1) / (n - k); the pair is scaled by 1 ± 1/1024 with
    opposite signs on even and odd columns; ci takes half of cj's count. c and hassign are updated in place."""
    k, eps = c.shape[0], 1.0 / 1024
    rng = torch.Generator().manual_seed(1234)
    sign = torch.ones(c.shape[1], dtype=c.dtype, device=c.device)
    sign[1::2] = -1.0
    splits = 0
    # a split only gives a count to the empty ci being served, so the empty clusters can be listed up front
    for ci in [i for i in range(k) if hassign[i] == 0]:
        cj = -1
        while True:
            cj = (cj + 1) % k
            prob = (hassign[cj] - 1.0) / (n - k) if n > k else float("inf") * (hassign[cj] - 1.0)
            if float(torch.rand(1, generator=rng)) < prob:
                break
        base = c[cj].clone()
        c[ci] = base * (1.0 + eps * sign)
        c[cj] = base * (1.0 - eps * sign)
        hassign[ci] = hassign[cj] / 2
        hassign[cj] = hassign[cj] - hassign[ci]
        splits += 1
    return splits


def kmeans_fit(x: torch.Tensor, init: torch.Tensor, niter: int) -> dict:
    """Lloyd's algorithm in fp64 from `init` on all rows of x. Returns the centroids (fp64), objective and n_split per iteration,
    the assignment of every iteration (ids) and the counts of the last one."""
    x = x.double()
    c = init.double().clone()
    out = dict(objective=[], n_split=[], ids=[])
    for _ in range(niter):
        ids, dmin = nearest(x, c)
        out["objective"].append(dmin.sum().item())
        out["ids"].append(ids)
        c, counts = cluster_means(x, ids, c)
        out["n_split"].append(split_empty(c, [float(v) for v in counts.tolist()], x.shape[0]))
        out["counts"] = counts
    out["centroids"] = c
    return out
