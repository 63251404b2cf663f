"""CPU checks of the k-means fit: the oracle's split rule on a hand-built case, the library's split rule against the oracle's for the
same draws, seeded subsample / init indices, argument errors, and the oracle's objective on separated blobs."""
import pytest
import torch

from edm_tts_b200 import kmeans as K
from oracle import kmeans_fit as O

EPS = 1.0 / 1024


def test_oracle_split_hand_built():
    # cluster 2 is empty; clusters 0 and 1 hold one row each (p = 0: never picked); cluster 3 holds 10 of n = 12 rows, so
    # p = (10 - 1) / (12 - 4) > 1 and it is picked at its first visit whatever the draws
    c = torch.arange(4 * 6, dtype=torch.float64).view(4, 6) + 1.0
    c0 = c.clone()
    h = [1.0, 1.0, 0.0, 10.0]
    assert O.split_empty(c, h, 12) == 1
    sign = torch.tensor([1.0, -1.0] * 3, dtype=torch.float64)
    assert torch.equal(c[2], c0[3] * (1 + EPS * sign))       # copy of cluster 3, even columns up, odd columns down
    assert torch.equal(c[3], c0[3] * (1 - EPS * sign))       # and cluster 3 the other way round
    assert torch.equal(c[:2], c0[:2])
    assert h == [1.0, 1.0, 5.0, 5.0]
    h = [1.0, 1.0, 0.0, 11.0]
    O.split_empty(c0.clone(), h, 13)
    assert h == [1.0, 1.0, 5.5, 5.5]                         # float counts, as faiss keeps them


@pytest.mark.parametrize("seed", range(4))
def test_library_split_matches_oracle(seed):
    g = torch.Generator().manual_seed(seed)
    k, d = 37, 64
    counts = torch.randint(0, 40, (k,), generator=g).tolist()
    for i in range(0, k, 5):
        counts[i] = 0                                        # cluster 0 and every fifth one empty
    n = sum(counts)
    c = torch.randn(k, d, generator=g, dtype=torch.float64)
    ca, cb = c.clone(), c.clone()
    ha, hb = [float(v) for v in counts], [float(v) for v in counts]
    na = K.split_clusters(ca, ha, n)
    nb = O.split_empty(cb, hb, n)
    assert na == nb == sum(v == 0 for v in counts)
    assert torch.equal(ca, cb)
    assert ha == hb and all(v > 0 for v in ha)


def test_split_with_n_equal_k():
    c = torch.randn(4, 32, dtype=torch.float64)
    ca, cb = c.clone(), c.clone()
    ha, hb = [2.0, 0.0, 1.0, 1.0], [2.0, 0.0, 1.0, 1.0]
    assert K.split_clusters(ca, ha, 4) == O.split_empty(cb, hb, 4) == 1
    assert torch.equal(ca, cb) and ha == hb == [1.0, 1.0, 1.0, 1.0]


def test_subsample_and_init_indices_are_seeded():
    assert K.subsample_indices(1000, 4, 256, 7) is None                 # n <= k * max_points_per_centroid: every row
    assert K.subsample_indices(10 ** 6, 4, None, 7) is None
    a = K.subsample_indices(5000, 4, 256, 7)
    assert torch.equal(a, K.subsample_indices(5000, 4, 256, 7)) and a.shape == (1024,)
    assert torch.equal(a, torch.randperm(5000, generator=torch.Generator().manual_seed(7))[:1024])
    assert not torch.equal(a, K.subsample_indices(5000, 4, 256, 8))
    assert a.unique().numel() == 1024
    b = K.init_indices(1024, 100, 7)
    assert torch.equal(b, K.init_indices(1024, 100, 7)) and b.shape == (100,) and b.unique().numel() == 100
    assert torch.equal(b, torch.randperm(1024, generator=torch.Generator().manual_seed(8))[:100])


@pytest.mark.parametrize("shape,k,init_shape", [((10, 64), 11, None), ((100, 48), 4, None), ((10000, 64), 4097, None),
                                                ((100, 64), 4, (4, 32)), ((100, 64), 4, (5, 64)), ((100,), 4, None), ((100, 64), 0, None)])
def test_fit_argument_errors(shape, k, init_shape):
    x = torch.zeros(shape)
    init = None if init_shape is None else torch.zeros(init_shape)
    with pytest.raises(ValueError):
        K.fit_kmeans(x, n_centroids=k, niter=2, init=init)


def test_fit_niter_error():
    with pytest.raises(ValueError):
        K.fit_kmeans(torch.zeros(100, 64), n_centroids=4, niter=0)


def test_oracle_objective_never_increases():
    g = torch.Generator().manual_seed(3)
    centres = torch.randn(8, 64, generator=g, dtype=torch.float64) * 3
    x = centres[torch.randint(0, 8, (2000,), generator=g)] + torch.randn(2000, 64, generator=g, dtype=torch.float64)
    init = x[K.init_indices(2000, 8, 1234)]
    r = O.kmeans_fit(x, init, 12)
    obj = r["objective"]
    assert all(b <= a * (1 + 1e-12) for a, b in zip(obj, obj[1:])), obj
    assert obj[-1] < obj[0]
    assert int(r["counts"].sum()) == 2000 and len(r["ids"]) == 12
