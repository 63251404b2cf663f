"""Batched text-to-semantic decode (TextToSemanticWLen.infer_batch / predict_length_batch, edm_t2s_*_batch).

The contract is batch invariance: utterance i of a packed decode equals infer on text i alone with split-K off
(set_low_latency(False)) and batch offset batch_offset + i, bit for bit. The sequence lengths L_i = n_text_i + length_i + 4 sit on
both sides of the 128-row GEMM tiles and the 256-row attention query pairs, with one very short sequence among long ones.
"""
import pytest
import torch

pytestmark = pytest.mark.gpu

_MODELS = {}
# (n_text, length) -> L = n_text + length + 4: 127 / 128 / 129 / 255 / 256 / 257, a 6-row sequence, an empty text, a long one
SHAPES = [(20, 103), (0, 124), (37, 88), (5, 246), (60, 192), (13, 240), (1, 1), (90, 400)]


def _model(cfg_name):
    from edm_tts_b200 import TextToSemanticWLen
    from edm_tts_b200.config import TextToSemanticWLenConfig
    from edm_tts_b200.synthetic import T2SConfig, make_t2s_state_dict
    from tests.golden.make_golden_cfg import T2S_CONFIGS

    if cfg_name not in _MODELS:
        cfg = T2SConfig(**T2S_CONFIGS[cfg_name])
        sd = make_t2s_state_dict(cfg, 0)
        hcfg = TextToSemanticWLenConfig(hidden_size=cfg.hidden, main_encoder_args=dict(depth=cfg.depth, heads=cfg.heads, ff_mult=4, conv_kernel_size=5),
                                        length_predictor_args=dict(depth=cfg.lp_depth, heads=cfg.lp_heads, ff_mult=4, conv_kernel_size=5))
        _MODELS[cfg_name] = (cfg, {k: v.cuda() for k, v in sd.items()}, TextToSemanticWLen(hcfg, sd, max_positions=1024))
    return _MODELS[cfg_name]


class _unsplit:
    """set_low_latency(False) for the block, the default (on) restored after it"""

    def __init__(self, model):
        self.model = model

    def __enter__(self):
        self.model.set_low_latency(False)
        return self.model

    def __exit__(self, *exc):
        self.model.set_low_latency(True)


def _texts(shapes, seed):
    """shifted text tokens (bytes + 5 special tokens) of the given lengths"""
    g = torch.Generator().manual_seed(seed)
    return [torch.randint(0, 256, (nt,), generator=g) + 5 for nt, _ in shapes]


def _gumbel(g, *shape):
    return -torch.log(-torch.log(torch.rand(*shape, generator=g).clamp(1e-7, 1 - 1e-7)))


def _singles(model, texts, lengths, iters, offset, **extras):
    with _unsplit(model):
        return [model.infer(t, pred_iters=iters, gt_length=ln, seed=11, batch_offset=offset + i, **{k: v[i] for k, v in extras.items()}).speech_pred_tokens
                for i, (t, ln) in enumerate(zip(texts, lengths))]


@pytest.mark.parametrize("cfg_name", ["small", "base", "train"])
@pytest.mark.parametrize("iters", [1, 4, 16])
def test_tile_edge_lengths_match_single_utterances(cfg_name, iters):
    _, _, model = _model(cfg_name)
    texts = _texts(SHAPES, seed=iters)
    lengths = [ln for _, ln in SHAPES]
    offset = 3
    got = model.infer_batch(texts, pred_iters=iters, gt_lengths=lengths, seed=11, batch_offset=offset)
    assert [tuple(t.shape) for t in got] == [(ln,) for ln in lengths] and all(t.dtype == torch.int64 for t in got)
    want = _singles(model, texts, lengths, iters, offset)
    for i in range(len(SHAPES)):
        assert torch.equal(got[i], want[i]), f"utterance {i} (n_text, length) = {SHAPES[i]}"


@pytest.mark.parametrize("cfg_name", ["small", "train"])
def test_injected_noise_and_forcing_match_single_utterances(cfg_name):
    cfg, _, model = _model(cfg_name)
    shapes = [(11, 116), (0, 3), (40, 213), (7, 250)]
    texts = _texts(shapes, seed=21)
    lengths = [ln for _, ln in shapes]
    Ls = [nt + ln + 4 for nt, ln in shapes]
    S, V = 4, cfg.semantic_vocab
    g = torch.Generator().manual_seed(8)
    noise = dict(cat_gumbel=[_gumbel(g, S - 1, L, V) for L in Ls], remask_gumbel=[_gumbel(g, S - 1, 1, L) for L in Ls])
    got = model.infer_batch(texts, pred_iters=S, gt_lengths=lengths, seed=11, **noise)
    want = _singles(model, texts, lengths, S, 0, **noise)
    for i in range(len(shapes)):
        assert torch.equal(got[i], want[i]), f"injected noise, utterance {i}"
    forced = dict(forced_ids=[torch.randint(0, V, (S, 1, L), generator=g) for L in Ls],
                  forced_masks=[(torch.rand(S - 1, 1, L, generator=g) < 0.5).to(torch.uint8) for L in Ls])
    got = model.infer_batch(texts, pred_iters=S, gt_lengths=lengths, seed=11, batch_offset=9, **noise, **forced)
    want = _singles(model, texts, lengths, S, 9, **noise, **forced)
    for i in range(len(shapes)):
        assert torch.equal(got[i], want[i]), f"teacher forcing, utterance {i}"


@pytest.mark.parametrize("cfg_name", ["small", "base"])
def test_predicted_lengths_match_single_calls(cfg_name):
    _, _, model = _model(cfg_name)
    texts = ["hello world", "", "The quick brown fox jumps over the lazy dog.", torch.tensor([72, 105, 33]) + 5, "x" * 300, "ok"]
    lengths, raws = model.predict_length_batch(texts)
    with _unsplit(model):
        single = [model.predict_length(t) for t in texts]
    assert lengths == [s[0] for s in single]
    assert raws == [s[1] for s in single]  # the same float32 bits
    # infer_batch without gt_lengths decodes at those lengths (random-init predictions: only the texts whose sequence fits)
    n_text = [len(t.encode("utf-8")) if isinstance(t, str) else t.numel() for t in texts]
    fit = [i for i in range(len(texts)) if n_text[i] + lengths[i] + 4 <= model.max_positions]
    assert len(fit) >= 2
    got = model.infer_batch([texts[i] for i in fit], pred_iters=2, seed=4)
    assert [t.shape[0] for t in got] == [lengths[i] for i in fit]


def test_unsplit_path_parity_vs_oracle():
    """The batch is bit-identical to the unsplit single path, so grading that path against the oracle grades the batch."""
    from edm_tts_b200.synthetic import make_t2s_noise
    from oracle import t2s as ot2s
    from tests.parity_utils import compare_ids, compare_logits, compare_masks
    from tests.test_gpu_t2s import MAX_TOL, MEAN_TOL, TEXTS

    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    cfg, sd, model = _model("train")
    text, iters, length = TEXTS["train"], 4, 500
    Lseq = len(text.encode("utf-8")) + length + 4
    noise = make_t2s_noise(Lseq, iters, cfg, seed=5 + Lseq)
    tr = {}
    with torch.inference_mode():
        tt = ot2s.text_tokens_of(text, cfg, "cuda")
        ot2s.infer(sd, cfg, tt, pred_iters=iters, gt_length=length, cat_gumbel=noise["cat_gumbel"].cuda(), remask_gumbel=noise["remask_gumbel"].cuda(), trace=tr)
    forced = dict(forced_ids=torch.stack(tr["step_ids"]), forced_masks=torch.stack(tr["step_masks"]))
    with _unsplit(model):
        ours = model.decode_trace(text, pred_iters=iters, gt_length=length, cat_gumbel=noise["cat_gumbel"], remask_gumbel=noise["remask_gumbel"], **forced)
    torch.cuda.synchronize()
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
    # and the batch reproduces that staged run for this utterance (forcing and noise per utterance)
    one = lambda t: [t.cpu()]
    got = model.infer_batch([text], pred_iters=iters, gt_lengths=[length], cat_gumbel=one(noise["cat_gumbel"]), remask_gumbel=one(noise["remask_gumbel"]),
                            forced_ids=one(forced["forced_ids"]), forced_masks=one(forced["forced_masks"]))
    assert torch.equal(got[0], ours["tokens"])


def test_chunked_batch():
    """More than MAX_CHUNK utterances: chunks of 64 in order, each with batch offset batch_offset + first index."""
    from edm_tts_b200.s2a import MAX_CHUNK

    _, _, model = _model("small")
    g = torch.Generator().manual_seed(1)
    n = MAX_CHUNK + 6
    shapes = [(int(a), int(b)) for a, b in zip(torch.randint(0, 30, (n,), generator=g), torch.randint(2, 60, (n,), generator=g))]
    texts = _texts(shapes, seed=2)
    lengths = [ln for _, ln in shapes]
    got = model.infer_batch(texts, pred_iters=3, gt_lengths=lengths, seed=11, batch_offset=100)
    want = _singles(model, texts, lengths, 3, 100)
    assert len(got) == n
    for i in range(n):
        assert torch.equal(got[i], want[i]), f"utterance {i}"


def test_default_mode_unchanged():
    _, _, model = _model("train")
    assert model.low_latency is True
    text = "The quick brown fox jumps over the lazy dog, and the dog, for once, does not mind at all."
    a = model.infer(text, pred_iters=6, gt_length=500, seed=1).speech_pred_tokens
    model.set_low_latency(False)
    model.infer(text, pred_iters=6, gt_length=500, seed=1)
    model.set_low_latency(True)
    b = model.infer(text, pred_iters=6, gt_length=500, seed=1).speech_pred_tokens
    assert torch.equal(a, b)
    # the batch leaves the single-utterance context alone
    model.infer_batch([text, "abc"], pred_iters=2, gt_lengths=[500, 20])
    c = model.infer(text, pred_iters=6, gt_length=500, seed=1).speech_pred_tokens
    assert torch.equal(a, c)


def test_errors():
    cfg, _, model = _model("small")
    with pytest.raises(ValueError):
        model.infer_batch([], gt_lengths=[])
    with pytest.raises(ValueError, match="utterance 1"):
        model.infer_batch(["ab", "cd"], gt_lengths=[10, 1020])
    with pytest.raises(ValueError, match="texts\\[1\\]"):
        model.predict_length_batch(["ab", "x" * 1100])
    with pytest.raises(ValueError, match="utterance 0"):
        model.infer_batch(["ab", "cd"], gt_lengths=[0, 5])
    with pytest.raises(ValueError):
        model.infer_batch(["ab", "cd"], gt_lengths=[5])
    with pytest.raises(ValueError):
        model.infer_batch(["ab"], pred_iters=0, gt_lengths=[5])
    with pytest.raises(ValueError, match="remask_gumbel\\[0\\]"):
        model.infer_batch(["ab"], pred_iters=3, gt_lengths=[5], remask_gumbel=[torch.zeros(2, 1, 10)])
    with pytest.raises(ValueError, match="cat_gumbel"):
        model.infer_batch(["ab", "c"], pred_iters=3, gt_lengths=[5, 5], cat_gumbel=[torch.zeros(2, 11, cfg.semantic_vocab)])
    with pytest.raises(ValueError):
        model.infer_batch([torch.zeros(2, 3, dtype=torch.long) + 5], gt_lengths=[5])
