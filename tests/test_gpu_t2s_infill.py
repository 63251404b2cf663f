"""Text-to-semantic infilling (TextToSemanticWLen.infill_batch, edm_t2s_begin_masked / edm_t2s_decode_masked): regenerate chosen
semantic tokens of an utterance given its transcript and the other tokens.

With every speech position regenerated the decode is infer_batch, bit for bit. With known positions it is graded against the infill
oracle (tests/oracle_t2s_infill.py) under teacher forcing, with the tolerances of tests/test_gpu_t2s.py. Known positions keep their
tokens through the whole decode, the batch is invariant to its composition and chunking, and the existing paths are unchanged.
"""
import pytest
import torch

from tests.test_gpu_t2s_batch import SHAPES, _gumbel, _model, _texts

pytestmark = pytest.mark.gpu

OFFSET = 5 + 256   # num_special + text_vocab


def _tokens(N, seed):
    g = torch.Generator().manual_seed(seed)
    return [torch.randint(0, 1024, (n,), generator=g) for n in N]


def _spans(n, g, k=None):
    """20-40 % of n positions in 1-3 spans (at least one position)"""
    m = torch.zeros(n, dtype=torch.bool)
    k = k or int(torch.randint(1, 4, (1,), generator=g))
    want = max(1, int(n * (0.2 + 0.2 * float(torch.rand(1, generator=g)))))
    for _ in range(k):
        ln = max(1, want // k)
        a = int(torch.randint(0, n - ln + 1, (1,), generator=g))
        m[a:a + ln] = True
    return m


@pytest.mark.parametrize("cfg_name", ["small", "base", "train"])
@pytest.mark.parametrize("iters", [1, 4, 16])
def test_all_regenerated_is_infer_batch(cfg_name, iters):
    _, _, model = _model(cfg_name)
    texts = _texts(SHAPES, seed=iters)
    N = [ln for _, ln in SHAPES]
    regen = [torch.ones(n, dtype=torch.bool) for n in N]
    got = model.infill_batch(texts, _tokens(N, iters), regen, pred_iters=iters, seed=11, batch_offset=3)
    want = model.infer_batch(texts, pred_iters=iters, gt_lengths=N, seed=11, batch_offset=3)
    assert [tuple(t.shape) for t in got] == [(n,) for n in N] and all(t.dtype == torch.int64 for t in got)
    for i in range(len(SHAPES)):
        assert torch.equal(got[i], want[i]), f"utterance {i} (n_text, N) = {SHAPES[i]}"


@pytest.mark.parametrize("cfg_name", ["small", "train"])
def test_all_regenerated_with_injected_noise_and_forcing(cfg_name):
    cfg, _, model = _model(cfg_name)
    shapes = [(11, 116), (0, 3), (40, 213), (7, 250)]
    texts = _texts(shapes, seed=21)
    N = [ln for _, ln in shapes]
    Ls = [nt + ln + 4 for nt, ln in shapes]
    S, V = 4, cfg.semantic_vocab
    g = torch.Generator().manual_seed(8)
    extras = dict(cat_gumbel=[_gumbel(g, S - 1, L, V) for L in Ls], remask_gumbel=[_gumbel(g, S - 1, 1, L) for L in Ls],
                  forced_ids=[torch.randint(0, V, (S, 1, L), generator=g) for L in Ls],
                  forced_masks=[(torch.rand(S - 1, 1, L, generator=g) < 0.5).to(torch.uint8) for L in Ls])
    regen = [torch.ones(n, dtype=torch.bool) for n in N]
    got = model.infill_batch(texts, _tokens(N, 1), regen, pred_iters=S, seed=11, batch_offset=9, **extras)
    want = model.infer_batch(texts, pred_iters=S, gt_lengths=N, seed=11, batch_offset=9, **extras)
    for i in range(len(shapes)):
        assert torch.equal(got[i], want[i]), f"utterance {i}"


def _mask(kind, n, g):
    m = torch.zeros(n, dtype=torch.bool)
    if kind == "spans":
        return _spans(n, g, k=3)
    if kind == "single":
        m[n // 2] = True
    elif kind == "prefix":      # prompted continuation: known prompt tokens, then the new speech
        m[n // 3:] = True
    elif kind == "suffix":
        m[:n // 3] = True
    return m


@pytest.mark.parametrize("kind", ["spans", "single", "prefix", "suffix"])
def test_masked_parity_vs_oracle(kind):
    """A staged, teacher-forced run of one masked sequence graded as test_unsplit_path_parity_vs_oracle grades the plain path."""
    from edm_tts_b200.synthetic import make_t2s_noise
    from oracle import t2s as ot2s
    from tests import oracle_t2s_infill as oti
    from tests.parity_utils import compare_ids, compare_logits, compare_masks
    from tests.test_gpu_t2s import MAX_TOL, MEAN_TOL, TEXTS

    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    cfg, sd, model = _model("train")
    text, iters, n = TEXTS["train"], 4, 300
    g = torch.Generator().manual_seed(len(kind))
    regen = _mask(kind, n, g)
    sem = _tokens([n], 5)[0]
    Lseq = len(text.encode("utf-8")) + n + 4
    noise = make_t2s_noise(Lseq, iters, cfg, seed=5 + Lseq)
    tr = {}
    with torch.inference_mode():
        tt = ot2s.text_tokens_of(text, cfg, "cuda")
        oti.infer_infill(sd, cfg, tt, sem.cuda(), regen.cuda(), pred_iters=iters, cat_gumbel=noise["cat_gumbel"].cuda(),
                         remask_gumbel=noise["remask_gumbel"].cuda(), trace=tr)
    forced = dict(forced_ids=torch.stack(tr["step_ids"]), forced_masks=torch.stack(tr["step_masks"]))
    ours = model.decode_trace(text, pred_iters=iters, cat_gumbel=noise["cat_gumbel"], remask_gumbel=noise["remask_gumbel"], semantic_tokens=sem,
                              regenerate=regen, **forced)
    torch.cuda.synchronize()
    assert torch.equal(ours["input_ids"], tr["input_ids"]) and torch.equal(ours["full_mask"], tr["full_mask"])
    reports = []
    for i in range(iters):
        last = i == iters - 1
        reports.append(compare_logits(ours["step_logits"][i], tr["step_logits"][i], f"logits iteration {i}"))
        scores = tr["step_logits"][i] if last else tr["step_logits"][i] + noise["cat_gumbel"][i].cuda().view(1, Lseq, -1)
        reports.append(compare_ids(ours["step_ids"][i], tr["step_ids"][i], scores, f"own sampled ids iteration {i}"))
        if not last:
            reports.append(compare_masks(ours["step_masks_raw"][i], tr["step_masks"][i], tr["step_conf"][i], tr["step_cut"][i], f"own re-masking iteration {i}"))
    for r in reports:
        if "max" in r:
            assert r["max"] < MAX_TOL and r["mean"] < MEAN_TOL, r
        assert r["n_not_near_tie"] == 0, r
    # with every decision forced, the result is the forced last-iteration ids at the regenerated positions
    assert ours["tokens"].shape == (int(regen.sum()),)
    assert torch.equal(ours["tokens"], torch.stack(tr["step_ids"])[-1][tr["full_mask"]])
    # and infill_batch (one C call on the batch context) reproduces the staged run
    one = lambda t: [t.cpu()]
    got = model.infill_batch([text], [sem], [regen], pred_iters=iters, cat_gumbel=one(noise["cat_gumbel"]), remask_gumbel=one(noise["remask_gumbel"]),
                             forced_ids=one(forced["forced_ids"]), forced_masks=one(forced["forced_masks"]))
    assert torch.equal(got[0], ours["tokens"])


@pytest.mark.parametrize("kind", ["spans", "prefix", "suffix"])
def test_known_positions_stay_fixed(kind):
    _, _, model = _model("base")
    text, n, iters = "speech editing keeps the rest of the utterance", 180, 6
    regen = _mask(kind, n, torch.Generator().manual_seed(3))
    sem = _tokens([n], 9)[0]
    tr = model.decode_trace(text, pred_iters=iters, seed=2, semantic_tokens=sem, regenerate=regen)
    start = len(text.encode("utf-8")) + 3
    Lseq = start + n + 1
    rows = start + torch.nonzero(~regen).flatten().cuda()
    tokens = model._view("tokens", (Lseq,), torch.int32).long()
    input_ids = model._view("input_ids", (Lseq,), torch.int32).long()
    known = sem[~regen].cuda() + OFFSET
    assert torch.equal(tokens[rows], known) and torch.equal(input_ids[rows], known)
    assert not model._view("full_mask", (Lseq,), torch.uint8)[rows].any()
    assert all(not m[0, rows].any() for m in tr["step_masks"])
    out = model.infill_batch([text], [sem], [regen], pred_iters=iters, seed=2)[0]
    assert torch.equal(out, tr["tokens"])
    spliced = sem.cuda().clone()
    spliced[regen.cuda()] = out
    assert spliced.min() >= 0 and spliced.max() < 1024
    assert torch.equal(spliced[~regen.cuda()], sem[~regen].cuda())


def _batch(n, seed, max_text=30, max_n=60):
    g = torch.Generator().manual_seed(seed)
    shapes = [(int(a), int(b)) for a, b in zip(torch.randint(0, max_text, (n,), generator=g), torch.randint(2, max_n, (n,), generator=g))]
    N = [ln for _, ln in shapes]
    return _texts(shapes, seed), _tokens(N, seed), [_spans(x, g) for x in N]


@pytest.mark.parametrize("n", [9, 70])
def test_batch_invariance_and_chunks(n):
    """Utterance i of a batch is that utterance alone at batch offset batch_offset + i; more than MAX_CHUNK utterances go in chunks."""
    _, _, model = _model("small")
    texts, sem, regen = _batch(n, seed=n)
    got = model.infill_batch(texts, sem, regen, pred_iters=3, seed=11, batch_offset=100)
    assert [t.shape[0] for t in got] == [int(m.sum()) for m in regen]
    for i in range(n):
        alone = model.infill_batch([texts[i]], [sem[i]], [regen[i]], pred_iters=3, seed=11, batch_offset=100 + i)[0]
        assert torch.equal(got[i], alone), f"utterance {i}"
    again = model.infill_batch(texts, sem, regen, pred_iters=3, seed=11, batch_offset=100)
    assert all(torch.equal(a, b) for a, b in zip(got, again))
    other = model.infill_batch(texts, sem, regen, pred_iters=3, seed=12, batch_offset=100)
    assert not all(torch.equal(a, b) for a, b in zip(got, other))


def test_existing_paths_unchanged():
    _, _, model = _model("train")
    assert model.low_latency is True
    text = "The quick brown fox jumps over the lazy dog, and the dog, for once, does not mind at all."
    texts = [text, "abc", "editing"]
    single = lambda: model.infer(text, pred_iters=6, gt_length=400, seed=1).speech_pred_tokens
    batch = lambda: model.infer_batch(texts, pred_iters=4, gt_lengths=[400, 20, 90], seed=1)
    a, b = single(), batch()
    sem, regen = _tokens([400], 4), [_spans(400, torch.Generator().manual_seed(1))]
    model.infill_batch([text], sem, regen, pred_iters=4)
    model.decode_trace(text, pred_iters=2, semantic_tokens=sem[0], regenerate=regen[0])   # a masked begin on the single context
    assert model.low_latency is True
    assert torch.equal(single(), a)
    assert all(torch.equal(x, y) for x, y in zip(batch(), b))


def test_errors():
    _, _, model = _model("small")
    sem, regen = _tokens([5, 4], 0), [torch.tensor([0, 1, 1, 0, 0], dtype=torch.bool), torch.tensor([1, 0, 0, 1], dtype=torch.bool)]
    model.infill_batch(["ab", "cd"], sem, regen, pred_iters=2)
    with pytest.raises(ValueError):
        model.infill_batch([], [], [])
    with pytest.raises(ValueError):
        model.infill_batch(["ab"], sem, regen)
    with pytest.raises(ValueError):
        model.infill_batch(["ab", "cd"], sem[:1], regen)
    with pytest.raises(ValueError, match="utterance 1"):
        model.infill_batch(["ab", "cd"], sem, [regen[0], regen[1][:3]])
    with pytest.raises(ValueError, match="utterance 0"):
        model.infill_batch(["ab", "cd"], sem, [torch.zeros(5, dtype=torch.bool), regen[1]])
    with pytest.raises(ValueError, match="utterance 1"):
        model.infill_batch(["ab", "cd"], [sem[0], torch.tensor([0, 1024, 0, 3])], regen)
    bad = sem[1].clone()
    bad[1] = -1
    with pytest.raises(ValueError, match="utterance 1"):
        model.infill_batch(["ab", "cd"], [sem[0], bad], regen)
    bad[1], bad[0] = 3, 5000   # out of range, but at a regenerated position: ignored
    model.infill_batch(["ab", "cd"], [sem[0], bad], regen, pred_iters=2)
    with pytest.raises(ValueError, match="utterance 1"):
        model.infill_batch(["ab", "cd"], [sem[0], torch.zeros(1019, dtype=torch.long)], [regen[0], torch.ones(1019, dtype=torch.bool)])
    with pytest.raises(ValueError):
        model.infill_batch(["ab", "cd"], sem, regen, pred_iters=0)
    with pytest.raises(ValueError, match="remask_gumbel\\[0\\]"):
        model.infill_batch(["ab", "cd"], sem, regen, pred_iters=3, remask_gumbel=[torch.zeros(2, 1, 10), torch.zeros(2, 1, 10)])
    with pytest.raises(ValueError, match="cat_gumbel"):
        model.infill_batch(["ab", "cd"], sem, regen, pred_iters=3, cat_gumbel=[torch.zeros(2, 11, 1024)])
