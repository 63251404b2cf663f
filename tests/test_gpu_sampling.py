"""The in-kernel noise of sample_kernel and remask_kernel (csrc/elementwise.cuh) against the host Philox of tests/philox_ref.py.

Every decode with a seed draws its Gumbel noise there; the parity tests inject theirs. Here the kernels' own draws are graded:
sampled ids against the float64 arg-max of logits + g_ref, the tail of the Gumbel transform, the share of draws that can reach a
column, the re-masking rule with Philox confidences, and the high words of the counter and the key through the whole decode."""
import math

import numpy as np
import pytest
import torch

from tests import philox_ref as P
from tests.philox_ref import REMASK_U1, SAMPLE_TAIL

pytestmark = pytest.mark.gpu
dev = "cuda"
V = 1024
# |g_kernel - g_ref| over every 24-bit input is at most 5.3e-5 (the fast __logf path for u <= 1 - 2^-10; about 1e-6 elsewhere),
# measured on a B200; a score is logit + g rounded to float32
G_ERR, TIE_ULPS = 6e-5, 4
# a sampled id may differ from the float64 reference only where the two scores are within the error of both Gumbel values
ID_TIE_ABS = 2 * G_ERR


@pytest.fixture(scope="module")
def L():
    from edm_tts_b200 import _lib
    _lib.lib()
    return _lib


def f32(x):
    return float(np.float32(x))


def sample(L, logits, T, Q=1, *, seed=0, step=0, philox=True, forced=None, out_q_stride=None, out_q0=0):
    """edm_sample over float32 logits [B*T*Q, 1024] (rows ordered (b, t, q)) -> ids [B, out_q_stride, T] (-1 where nothing was
    written) and logp [rows], as numpy arrays."""
    rows = logits.shape[0]
    stride = Q if out_q_stride is None else out_q_stride
    ld = torch.from_numpy(np.ascontiguousarray(logits, dtype=np.float32)).to(dev)
    ids = torch.full((rows // (T * Q), stride, T), -1, device=dev, dtype=torch.int32)
    logp = torch.full((rows,), float("nan"), device=dev)
    fi = None if forced is None else torch.from_numpy(np.ascontiguousarray(forced, dtype=np.int32)).to(dev)
    L.check(L.lib().edm_sample(L.ptr(ld), V, rows, None, int(philox), seed, step, L.ptr(fi), L.ptr(ids), L.ptr(logp), T, Q, stride, out_q0,
                               L.stream_ptr()), "sample")
    return ids.cpu().numpy(), logp.cpu().numpy()


def row_ids(ids, T, Q, out_q0=0):
    """ids [B, stride, T] -> [B*T*Q] in row order (b, t, q): row (b T + t) Q + q lands at ids[b, out_q0 + q, t]."""
    return ids[:, out_q0:out_q0 + Q, :].transpose(0, 2, 1).reshape(-1)


def log_softmax64(x):
    x = x.astype(np.float64)
    mx = x.max(-1, keepdims=True)
    return x - (mx + np.log(np.exp(x - mx).sum(-1, keepdims=True)))


def assert_ids_match(got, logits, g, what):
    """got == first arg-max of the float64 scores logits + g, except where the score of `got` is within the tie tolerance of the top."""
    score = logits.astype(np.float64) + g
    want = score.argmax(-1)
    r = np.arange(len(got))
    assert ((got >= 0) & (got < V)).all(), what
    top = score[r, want]
    margin = top - score[r, got]
    tol = ID_TIE_ABS + TIE_ULPS * np.spacing(np.abs(top).astype(np.float32)).astype(np.float64)
    bad = (got != want) & ~(margin < tol)
    assert not bad.any(), f"{what}: {int(bad.sum())} / {len(got)} rows pick another id than the reference; first row {int(np.flatnonzero(bad)[0])}"
    return int((got != want).sum())


def make_logits(rows, seed):
    """randn * 3 rows, and every fifth row of each kind: the row maximum at four columns, a third of the columns -inf, shifted by
    +1e4, shifted by -1e4. With three rows or more the last two are all -inf and all NaN."""
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal((rows, V)) * 3).astype(np.float32)
    kind = np.arange(rows) % 5
    for r in np.flatnonzero(kind == 1):
        x[r, rng.choice(V, 4, replace=False)] = x[r].max() + 0.5
    x[(kind[:, None] == 2) & (rng.random((rows, V)) < 1 / 3)] = -np.inf
    x[kind == 3] += np.float32(1e4)
    x[kind == 4] -= np.float32(1e4)
    if rows >= 3:
        x[-2] = -np.inf
        x[-1] = np.nan
    return x


# ------------------------------------------------------------------------------------------------ sampling


@pytest.mark.parametrize("seed", [0, 1, 2 ** 32 + 7, 2 ** 64 - 1])
@pytest.mark.parametrize("B,T,Q,stride,q0", [(1, 1, 1, 1, 0), (3, 77, 1, 1, 0), (2, 500, 1, 1, 0), (2, 40, 11, 12, 1)])
def test_philox_sample_matches_host_reference(L, B, T, Q, stride, q0, seed):
    rows = B * T * Q
    x = make_logits(rows, seed=rows)
    b, t, q = (a.reshape(-1) for a in np.meshgrid(np.arange(B), np.arange(T), np.arange(Q), indexing="ij"))
    ctr = P.sample_counter(b, t, q, T, Q)
    undefined = ~np.isfinite(x).any(-1)            # no finite maximum: id 0
    flips = 0
    for step in (0, 7):
        ids, logp = sample(L, x, T, Q, seed=seed, step=step, out_q_stride=stride, out_q0=q0)
        assert (ids[:, :q0] == -1).all() and (ids[:, q0 + Q:] == -1).all(), "ids written outside the levels of the call"
        got = row_ids(ids, T, Q, q0)
        assert (got[undefined] == 0).all()
        g = P.sample_gumbel(ctr, seed, step)
        flips += assert_ids_match(got[~undefined], x[~undefined], g[~undefined], f"seed {seed} step {step}")
        lp = log_softmax64(x[~undefined])[np.arange(int((~undefined).sum())), got[~undefined]]
        np.testing.assert_allclose(logp[~undefined], lp, rtol=1e-5, atol=1e-5)
    assert flips <= max(2, rows // 100)


def test_u_equal_one_draw_cannot_win(L):
    """The draw with k = 2^24 - 1 (seed 1, step 0, row 34, column 106) gives a finite Gumbel value: a column 40 below the rest of its
    row (the widest gap a finite Gumbel pair closes is 16.64 + 2.85) is never picked."""
    seed, row, col = SAMPLE_TAIL[0xFFFFFF]
    T = 64
    x = (np.random.default_rng(0).standard_normal((T, V)) * 3).astype(np.float32)
    x[row, col] = np.delete(x[row], col).min() - 40
    ids, _ = sample(L, x, T, seed=seed, step=0)
    got = row_ids(ids, T, 1)
    assert got[row] != col
    assert_ids_match(got, x, P.sample_gumbel(np.arange(T), seed, 0), "u == 1 row")


@pytest.mark.parametrize("k", sorted(k for k in SAMPLE_TAIL if k != 0xFFFFFF), ids=hex)
def test_gumbel_tail_decides_close_pairs(L, k):
    """A draw with u within 16 ulps of 1 (g_ref 13.9 .. 15.9) against one ordinary column of its row, every other column at -1e4:
    with the float64 scores 0.01 apart the pick follows the sign, so the kernel's tail value is within 0.01 of g_ref."""
    seed, row, col = SAMPLE_TAIL[k]
    T = 64
    g = P.sample_gumbel(row, seed, 0)
    other = (col + 512) % V
    for sign in (1, -1):
        x = np.full((T, V), -1e4, np.float32)
        x[row, col] = 0
        x[row, other] = g[col] - g[other] - sign * 0.01
        diff = float(x[row, col]) + g[col] - (float(x[row, other]) + g[other])
        assert abs(diff - sign * 0.01) < 1e-5
        ids, _ = sample(L, x, T, seed=seed, step=0)
        assert row_ids(ids, T, 1)[row] == (col if sign > 0 else other), (hex(k), sign, g[col])


def test_unreachable_columns_and_softmax_frequencies(L):
    """2^18 rows x 4 steps of one 1024-logit row: 512 columns 30 below all of the other 512 can never win (a finite Gumbel pair closes
    at most 19.5), and the other 512 are drawn with the softmax frequencies (chi-square at a fixed seed)."""
    from scipy.stats import chisquare

    rows, seed = 2 ** 18, 3
    rng = np.random.default_rng(1)
    high = np.sort(rng.permutation(V)[:512])
    low = np.setdiff1d(np.arange(V), high)
    base = np.zeros(V, np.float32)
    base[high] = rng.standard_normal(512) * 0.5
    base[low] = base[high].min() - 30
    logits = torch.from_numpy(base).to(dev).expand(rows, V).contiguous()   # 1 GiB, beyond the L2
    ids = torch.empty(rows, device=dev, dtype=torch.int32)
    counts = np.zeros(V, np.int64)
    for step in range(4):
        L.check(L.lib().edm_sample(L.ptr(logits), V, rows, None, 1, seed, step, None, L.ptr(ids), None, rows, 1, 1, 0, L.stream_ptr()), "sample")
        counts += torch.bincount(ids.long(), minlength=V).cpu().numpy()
    assert counts.sum() == 4 * rows
    assert counts[low].sum() == 0, f"{int(counts[low].sum())} draws on columns 30 below the rest"
    p = np.exp(log_softmax64(base[high]))
    res = chisquare(counts[high], p * counts.sum())
    assert res.pvalue > 1e-4, (res.statistic, res.pvalue)


def test_teacher_forcing_reports_the_forced_column(L):
    B, T = 2, 100
    rng = np.random.default_rng(4)
    x = (rng.standard_normal((B * T, V)) * 3).astype(np.float32)
    forced = rng.integers(0, V, (B, 1, T))
    ids, logp = sample(L, x, T, seed=5, step=1, forced=forced)
    assert np.array_equal(ids, forced)
    np.testing.assert_allclose(logp, log_softmax64(x)[np.arange(B * T), forced.reshape(-1)], rtol=1e-5, atol=1e-5)


def test_argmax_over_fine_levels(L):
    """No noise, Q = 11 levels per frame written to a [B, 11, T] block (what the fine-level decode runs): the first maximum of each
    row (four columns share the maximum in every third row) at out_offset(b, q, 11, t) = (b 11 + q) T + t."""
    B, T, Q = 3, 50, 11
    rng = np.random.default_rng(5)
    x = (rng.standard_normal((B * T * Q, V)) * 3).astype(np.float32)
    for r in range(0, B * T * Q, 3):
        x[r, rng.choice(V, 4, replace=False)] = x[r].max() + 1
    ids, logp = sample(L, x, T, Q, philox=False)
    am = torch.from_numpy(x).argmax(-1).numpy()
    want = np.full(B * Q * T, -1)
    for r in range(B * T * Q):
        b, t, q = r // Q // T, r // Q % T, r % Q
        want[(b * Q + q) * T + t] = am[r]
    assert np.array_equal(ids.reshape(-1), want)
    np.testing.assert_allclose(logp, log_softmax64(x)[np.arange(B * T * Q), am], rtol=1e-5, atol=1e-5)


def test_sample_rejects_rows_and_levels_outside_the_id_block(L):
    x = torch.zeros(12, V, device=dev)
    ids = torch.full((64,), -1, device=dev, dtype=torch.int32)

    def call(rows, T, Q, stride, q0):
        L.check(L.lib().edm_sample(L.ptr(x), V, rows, None, 1, 0, 0, None, L.ptr(ids), None, T, Q, stride, q0, L.stream_ptr()), "sample")

    for bad in ((10, 3, 1, 1, 0), (10, 2, 2, 2, 0), (8, 2, 2, 2, 1), (8, 2, 2, 3, -1), (8, 2, 2, 1, 0), (8, 0, 1, 1, 0), (-4, 2, 1, 1, 0)):
        with pytest.raises(ValueError):
            call(*bad)
    torch.cuda.synchronize()
    assert (ids == -1).all()
    call(12, 3, 2, 3, 1)   # B = 2 frames blocks of [3, 3]: levels 1 and 2 written, level 0 untouched
    got = ids[:18].view(2, 3, 3).cpu().numpy()
    assert (got[:, 0] == -1).all() and (got[:, 1:] >= 0).all() and (ids[18:] == -1).all()


# ------------------------------------------------------------------------------------------------ re-masking


def remask(L, logp, mask_old, ratio, temp_ratio, *, seed=0, step=0, gumbel=None, forced=None):
    B, T = logp.shape
    lp = torch.from_numpy(np.ascontiguousarray(logp, dtype=np.float32)).to(dev)
    mo = torch.from_numpy(mask_old.astype(np.uint8)).to(dev)
    mn = torch.full_like(mo, 7)
    g = None if gumbel is None else torch.from_numpy(np.ascontiguousarray(gumbel, dtype=np.float32)).to(dev)
    fm = None if forced is None else torch.from_numpy(forced.astype(np.uint8)).to(dev)
    L.check(L.lib().edm_remask(L.ptr(lp), L.ptr(g), L.ptr(mo), L.ptr(mn), L.ptr(fm), B, T, ratio, temp_ratio, seed, step, L.stream_ptr()), "remask")
    return mn.cpu().numpy()


def remask_ref(logp, mask_old, ratio, temp_ratio, g):
    """The kernel's rule (elementwise.cuh, re-masking) with float32 arithmetic on float32(g):
    mask_len = max(1, min(#masked - 1, floor(float32(T) * ratio))), conf = masked ? logp + temp_ratio * g : +inf,
    cut = sort(conf)[mask_len], new mask = conf < cut. Returns (new mask, conf, cut [B, 1])."""
    B, T = logp.shape
    noise = np.float32(temp_ratio) * g.astype(np.float32)
    conf = np.where(mask_old, logp.astype(np.float32) + noise, np.float32(np.inf)).astype(np.float32)
    ml = math.floor(np.float32(T) * np.float32(ratio))
    k = np.maximum(1, np.minimum(mask_old.sum(-1) - 1, ml))
    cut = np.sort(conf, -1)[np.arange(B), k][:, None]
    return conf < cut, conf, cut


def assert_masks_match(got, want, conf, cut, temp_ratio, what):
    """A re-masking decision may differ only for a confidence within the Gumbel error of the cut-off, on either side."""
    with np.errstate(invalid="ignore"):      # inf - inf where the cut-off is +inf: no tolerance there
        tol = 2 * temp_ratio * G_ERR + TIE_ULPS * np.spacing(np.abs(cut))
        bad = (got.astype(bool) != want) & ~(np.abs(conf - cut) < tol)
    assert not bad.any(), f"{what}: {int(bad.sum())} rows off the reference mask"


@pytest.mark.parametrize("T", [2, 255, 256, 257, 4096])
def test_philox_remask_matches_host_reference(L, T):
    """Every masked count from 1 to T (positions drawn at random per row), B = 3, step and ratio cycling through an 8-step schedule."""
    B, seed = 3, 2 ** 32 + 19
    rng = np.random.default_rng(T)
    logp = (-np.abs(rng.standard_normal((B, T))) * 3).astype(np.float32)
    ctr = np.arange(B * T).reshape(B, T)
    g = {s: P.remask_gumbel(ctr, seed, s) for s in range(7)}
    order = np.argsort(rng.random((B, T)), -1)
    for c in range(1, T + 1):
        mask_old = np.zeros((B, T), bool)
        np.put_along_axis(mask_old, order[:, :c], True, -1)
        step = c % 7
        ratio = f32(math.cos(math.pi / 2 * (step + 1) / 8))
        got = remask(L, logp, mask_old, ratio, ratio, seed=seed, step=step)
        want, conf, cut = remask_ref(logp, mask_old, ratio, ratio, g[step])
        assert_masks_match(got, want, conf, cut, ratio, f"T {T} count {c}")


def test_remask_exact_with_injected_noise_and_ties(L):
    """Injected noise: the confidences are the float32 operations of the reference, so the masks match exactly, with temp_ratio = 0
    and log-probabilities taking five values (ties at the cut-off), and with temp_ratio > 0."""
    B, T = 3, 257
    rng = np.random.default_rng(7)
    logp = (-rng.integers(0, 5, (B, T)) * 0.5).astype(np.float32)
    g = P.gumbel(rng.integers(0, 2 ** 32, (B, T), dtype=np.uint64).astype(np.uint32)).astype(np.float32)
    for c in (1, 2, 3, 100, 200, 256, 257):
        mask_old = np.zeros((B, T), bool)
        mask_old[:, rng.permutation(T)[:c]] = True
        for step in range(7):
            ratio = f32(math.cos(math.pi / 2 * (step + 1) / 8))
            for tr in (0.0, ratio):
                got = remask(L, logp, mask_old, ratio, tr, gumbel=g)
                want, _, _ = remask_ref(logp, mask_old, ratio, tr, g)
                assert np.array_equal(got.astype(bool), want), (c, step, tr)


def test_remask_copies_forced_mask_and_rejects_long_rows(L):
    B, T = 2, 300
    rng = np.random.default_rng(8)
    logp = rng.standard_normal((B, T)).astype(np.float32)
    forced = rng.random((B, T)) < 0.4
    got = remask(L, logp, rng.random((B, T)) < 0.8, 0.5, 0.5, seed=3, forced=forced)
    assert np.array_equal(got, forced.astype(np.uint8))
    with pytest.raises(ValueError):
        remask(L, np.zeros((1, 4097), np.float32), np.ones((1, 4097), bool), 0.5, 0.5)


def test_remask_u_equal_one_draw(L):
    """Seed 2747, step 0: row 1531 of a B = 1, T = 4096 batch draws k = 2^24 - 1. Its confidence is finite: with the lowest log p by
    100 it is re-masked, and with temp_ratio = 0 the confidences are the log-probabilities themselves (not 0 * inf)."""
    seed, step, row = REMASK_U1
    T = 4096
    rng = np.random.default_rng(9)
    logp = (-np.abs(rng.standard_normal((1, T))) * 3).astype(np.float32)
    logp[0, row] = logp.min() - 100
    mask_old = np.ones((1, T), bool)
    g = P.remask_gumbel(np.arange(T)[None], seed, step)
    for ratio in (f32(math.cos(math.pi / 2 / 8)), f32(math.cos(math.pi / 2 * 7 / 8))):
        got = remask(L, logp, mask_old, ratio, 1.0, seed=seed, step=step)
        assert got[0, row] == 1
        want, conf, cut = remask_ref(logp, mask_old, ratio, 1.0, g)
        assert_masks_match(got, want, conf, cut, 1.0, f"ratio {ratio}")
        tied = np.round(logp * 2) / 2
        got0 = remask(L, tied, mask_old, ratio, 0.0, seed=seed, step=step)
        want0, _, _ = remask_ref(tied, mask_old, ratio, 0.0, g)
        assert np.array_equal(got0.astype(bool), want0)


# ------------------------------------------------------------------------------------------------ through the decode


def test_counter_and_key_high_words_reach_the_decode():
    """B = 1, T = 64: batch offsets o and o + 2^26 give counters that differ only in their high word, seeds s and s + 2^32 keys that
    differ only in theirs; each pair must decode to different codes (and one call twice to the same codes)."""
    from oracle.weights import make_inputs
    from tests.parity_utils import full_model

    cfg, sd, model = full_model()
    sem = make_inputs(1, 64, 0, 1, cfg, seed=6)["semantic_tokens"]
    o, s = 3, 11
    a = model.infer_special(sem, steps=3, seed=s, batch_offset=o)
    assert torch.equal(a, model.infer_special(sem, steps=3, seed=s, batch_offset=o))
    assert not torch.equal(a, model.infer_special(sem, steps=3, seed=s, batch_offset=o + 2 ** 26))
    assert not torch.equal(a, model.infer_special(sem, steps=3, seed=s + 2 ** 32, batch_offset=o))
