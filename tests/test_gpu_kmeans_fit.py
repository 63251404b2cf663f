"""GPU checks of the k-means fit: edm_kmeans_update against fp64 per-cluster means (counts exact, centroids within one fp32 ulp, empty
clusters untouched), bit-reproducible fits, a full fit against the fp64 oracle (oracle/kmeans_fit.py) with and without an empty-cluster
split, and SemanticTokenizer.fit on synthetic HuBERT weights."""
import pytest
import torch

from oracle import kmeans_fit as O

pytestmark = pytest.mark.gpu


def _ulp(t: torch.Tensor) -> torch.Tensor:
    a = t.abs()
    return torch.nextafter(a, torch.full_like(a, float("inf"))) - a


@pytest.mark.parametrize("n,D,k,mode", [(1, 64, 1, "nearest"), (127, 64, 500, "nearest"), (50000, 1024, 1024, "nearest"),
                                        (300001, 1024, 4096, "nearest"), (300001, 64, 1024, "skew90"), (50000, 1024, 500, "skew90"),
                                        (50000, 64, 4096, "even_only"), (127, 1024, 1024, "even_only")])
def test_kmeans_update_vs_fp64_means(n, D, k, mode):
    from edm_tts_b200.kmeans import kmeans_update

    g = torch.Generator(device="cuda").manual_seed(n + D + k)
    x = torch.randn(n, D, device="cuda", generator=g) * 3 + 1
    c0 = torch.randn(k, D, device="cuda", generator=g)
    if mode == "nearest":          # the oracle's assignment to centroids drawn from the rows (k > n leaves clusters empty)
        c0[:min(n, k)] = x[:min(n, k)]
        idx = O.nearest(x.double(), c0.double())[0]
    elif mode == "skew90":         # cluster 3 holds 90 % of the rows
        idx = torch.randint(0, k, (n,), device="cuda", generator=g)
        idx[torch.rand(n, device="cuda", generator=g) < 0.9] = 3
    else:                          # odd clusters empty
        idx = torch.randint(0, (k + 1) // 2, (n,), device="cuda", generator=g) * 2
    c = c0.clone()
    counts = kmeans_update(x, idx, c)
    want_counts = torch.bincount(idx, minlength=k)
    assert torch.equal(counts, want_counts)
    ref, _ = O.cluster_means(x, idx, c0.double())
    full = want_counts > 0
    if mode == "skew90":
        assert want_counts[3].item() > 0.85 * n
    if mode == "even_only" or k > n:
        assert (~full).any()
    assert torch.equal(c[~full], c0[~full])                  # empty clusters: the same bits
    diff = (c[full].double() - ref[full]).abs()
    assert (diff <= _ulp(ref[full].float()).double()).all(), diff.max().item()
    c2, sums = c0.clone(), torch.empty(k, D, device="cuda", dtype=torch.float64)
    kmeans_update(x, idx, c2, sums)
    assert torch.equal(c, c2)                                # the same bits again, with or without the sums
    ref_sums = torch.zeros(k, D, device="cuda", dtype=torch.float64).index_add_(0, idx, x.double())
    assert torch.allclose(sums, ref_sums, rtol=1e-12, atol=1e-9) and not sums[~full].any()


def _blobs(n, n_blobs, D=1024, delta=8.0, noise=0.1, seed=0):
    """n rows, row r in blob r % n_blobs. Each blob is two tight halves at c ± delta·u with u = s ⊙ c / |c| (s = +1 on even, -1 on odd
    columns): the direction along which the ±1/1024 split perturbation separates a centroid pair, so a split blob falls apart into
    its halves with a margin of ~ 4·delta·|c| / 1024 ≈ 1 in squared distance (the fp32 scores are good to ~1e-3)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    centres = torch.randn(n_blobs, D, device="cuda", generator=g)
    s = torch.ones(D, device="cuda")
    s[1::2] = -1
    u = centres * s / centres.norm(dim=1, keepdim=True)
    lab = torch.arange(n, device="cuda") % n_blobs
    half = torch.randint(0, 2, (n,), device="cuda", generator=g).float() * 2 - 1
    return centres[lab] + delta * half[:, None] * u[lab] + noise * torch.randn(n, D, device="cuda", generator=g)


def _fit_steps(x, init, niter):
    from edm_tts_b200.kmeans import prepare_fit

    run = prepare_fit(x, n_centroids=init.shape[0], niter=niter, max_points_per_centroid=None, init=init)
    ids = []
    for it in range(niter):
        run.assign()
        ids.append(run.idx.clone())
        run.update(it)
        run.split()
        run.repack()
    return run, ids


@pytest.mark.parametrize("forced_split", [False, True])
def test_fit_vs_oracle(forced_split):
    from edm_tts_b200.kmeans import fit_kmeans

    n, k, niter = 200000, 256, 10
    n_blobs = 255 if forced_split else 256
    x = _blobs(n, n_blobs, seed=1 + forced_split)
    init = x[:k].clone()
    if forced_split:               # rows 0 .. 254 are blobs 0 .. 254; a copy of row 0 as centroid 1: the first maximum wins, so it is empty
        init = torch.cat([x[:1], x[:n_blobs]])
    run, ids = _fit_steps(x, init, niter)
    ref = O.kmeans_fit(x, init, niter)
    for it in range(niter):
        assert torch.equal(ids[it], ref["ids"][it]), (it, int((ids[it] != ref["ids"][it]).sum()))
    assert run.n_split == ref["n_split"]
    assert sum(run.n_split) == (1 if forced_split else 0)
    c, rc = run.centroids.double(), ref["centroids"]
    rel = ((c - rc).norm(dim=1) / rc.norm(dim=1)).max().item()
    assert rel < 1e-6, rel
    sq = x.double().pow(2).sum().item()
    obj = run.objective.tolist()
    assert max(abs(a - b) for a, b in zip(obj, ref["objective"])) < 1e-5 * sq
    assert torch.equal(run.counts, ref["counts"])
    fit = fit_kmeans(x, n_centroids=k, niter=niter, max_points_per_centroid=None, init=init)     # the public call: the same bits
    assert torch.equal(fit.centroids, run.centroids) and fit.objective == obj and fit.n_split == run.n_split


def test_fit_is_bit_reproducible():
    from edm_tts_b200.kmeans import fit_kmeans

    x = _blobs(120000, 300, D=256, delta=2.0, noise=1.0, seed=5)
    init = torch.cat([x[:2], x[:2], x[2:252]])            # clusters 2 and 3 start empty: splits happen
    a = fit_kmeans(x, n_centroids=254, niter=6, max_points_per_centroid=None, init=init)
    b = fit_kmeans(x, n_centroids=254, niter=6, max_points_per_centroid=None, init=init)
    assert torch.equal(a.centroids, b.centroids) and a.objective == b.objective and a.n_split == b.n_split
    assert torch.equal(a.counts, b.counts) and sum(a.n_split) >= 2
    c = fit_kmeans(x.to(torch.bfloat16), n_centroids=64, niter=3, seed=9, max_points_per_centroid=256)   # subsampled, bf16 input
    d = fit_kmeans(x.to(torch.bfloat16), n_centroids=64, niter=3, seed=9, max_points_per_centroid=256)
    assert torch.equal(c.centroids, d.centroids) and int(c.counts.sum()) == 64 * 256
    assert c.centroids.dtype == torch.float32 and c.centroids.shape == (64, 256)


def test_kmeans_update_rejects_ids_out_of_range():
    from edm_tts_b200.kmeans import kmeans_update

    x, c = torch.randn(1000, 64, device="cuda"), torch.randn(8, 64, device="cuda")
    for bad in (-1, 8):
        idx = torch.randint(0, 8, (1000,), device="cuda")
        idx[500] = bad
        c2 = c.clone()
        with pytest.raises(ValueError):
            kmeans_update(x, idx, c2)
        assert torch.equal(c2, c)


def test_set_centroids_repacks_like_a_new_assigner():
    from edm_tts_b200.kmeans import KMeansAssigner

    g = torch.Generator().manual_seed(4)
    c1, c2, x = torch.randn(500, 128, generator=g), torch.randn(500, 128, generator=g), torch.randn(3000, 128, generator=g)
    a = KMeansAssigner(c1)
    a.set_centroids(c2)
    b = KMeansAssigner(c2)
    for name in ("_c_hi", "_c_lo", "_norm"):
        assert torch.equal(getattr(a, name), getattr(b, name)), name
    assert torch.equal(a(x), b(x))


def test_semantic_tokenizer_fit():
    from edm_tts_b200 import HubertFeatures, SemanticTokenizer
    from edm_tts_b200.hubert import normalize_clip
    from edm_tts_b200.kmeans import KMeansAssigner
    from edm_tts_b200.synthetic import hubert_config, make_hubert_state_dict

    cfg = hubert_config(num_hidden_layers=2)
    hub = HubertFeatures(cfg, make_hubert_state_dict(0, cfg), device="cuda", output_layer=2)
    g = torch.Generator().manual_seed(8)
    clips = [torch.randn(n, generator=g) * 0.3 for n in (16000, 12345, 20000, 8000, 16000)]
    tok, fit = SemanticTokenizer.fit(hub, clips, n_centroids=32, niter=8)
    assert isinstance(tok, SemanticTokenizer) and fit.centroids.shape == (32, 1024) and len(fit.objective) == 8
    feats = torch.cat(hub.forward_batch([normalize_clip(c.cuda()) for c in clips]))
    assert int(fit.counts.sum()) == feats.shape[0]
    want = KMeansAssigner(fit.centroids)(feats)
    got = torch.cat(tok.encode_batch(clips))
    assert torch.equal(got, want)
