"""Text-to-semantic infilling without a GPU: the infill oracle (tests/oracle_t2s_infill.py) is oracle.t2s.infer when every speech
position is regenerated and keeps the known positions fixed otherwise; the host maps of edm_t2s_begin_masked; the checks on an infill
batch (edm_tts_b200/varlen.py)."""
import math

import pytest
import torch

from edm_tts_b200 import varlen
from edm_tts_b200.synthetic import T2SConfig, make_t2s_noise, make_t2s_state_dict
from oracle import t2s as ot2s
from tests import oracle_t2s_infill as oti

CFG = T2SConfig(hidden=128, heads=4, depth=2, lp_heads=4, lp_depth=1)


@pytest.fixture(scope="module")
def sd():
    return make_t2s_state_dict(CFG, 0)


def _case(n_speech, iters, seed, text="edit me"):
    tt = ot2s.text_tokens_of(text, CFG)
    L = tt.numel() + n_speech + 4
    noise = make_t2s_noise(L, iters, CFG, seed=seed)
    sem = torch.randint(0, CFG.semantic_vocab, (n_speech,), generator=torch.Generator().manual_seed(seed))
    return tt, sem, noise


@pytest.mark.parametrize("iters", [1, 4])
def test_all_regenerated_is_infer(sd, iters):
    tt, sem, noise = _case(13, iters, seed=3 + iters)
    tr_ref, tr = {}, {}
    with torch.inference_mode():
        ref = ot2s.infer(sd, CFG, tt, pred_iters=iters, gt_length=13, trace=tr_ref, **noise)
        got = oti.infer_infill(sd, CFG, tt, sem, torch.ones(13, dtype=torch.bool), pred_iters=iters, trace=tr, **noise)
    assert torch.equal(got, ref)
    assert torch.equal(tr["input_ids"], tr_ref["input_ids"]) and torch.equal(tr["full_mask"], tr_ref["full_mask"])
    for key in ("step_logits", "step_ids", "step_masks"):
        assert len(tr[key]) == len(tr_ref[key]) and all(torch.equal(a, b) for a, b in zip(tr[key], tr_ref[key]))


@pytest.mark.parametrize("regen", [
    [0, 0, 0, 1, 1, 1, 1, 0, 0, 0, 0, 1, 0, 0],   # two spans
    [0, 0, 0, 0, 0, 0, 0, 1, 0, 0, 0, 0, 0, 0],   # a single position
    [0, 0, 0, 0, 0, 1, 1, 1, 1, 1, 1, 1, 1, 1],   # known prefix: prompted continuation
    [1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0, 0, 0],   # known suffix
])
def test_known_positions_stay_fixed(sd, regen):
    iters = 4
    regen = torch.tensor(regen, dtype=torch.bool)
    n = regen.numel()
    tt, sem, noise = _case(n, iters, seed=11)
    tr = {}
    with torch.inference_mode():
        out = oti.infer_infill(sd, CFG, tt, sem, regen, pred_iters=iters, trace=tr, **noise)
    assert out.shape == (int(regen.sum()),) and out.min() >= 0 and out.max() < CFG.semantic_vocab
    start = tt.numel() + 3
    known_rows = start + torch.nonzero(~regen).flatten()
    offset = CFG.num_special + CFG.text_vocab
    assert torch.equal(tr["full_mask"][0, start:start + n], regen) and int(tr["full_mask"].sum()) == int(regen.sum())
    assert torch.equal(tr["input_ids"][0, known_rows], sem[~regen] + offset)
    assert torch.equal(tr["input_ids"][0, start + torch.nonzero(regen).flatten()], torch.full((int(regen.sum()),), ot2s.MASK))
    for i, s in enumerate(tr["step_sampled"]):
        assert torch.equal(s[0, known_rows], sem[~regen] + offset), f"iteration {i}"
        assert torch.equal(s[0, :start], tr["input_ids"][0, :start]), f"iteration {i}"
    # re-masking never picks a known position and masks floor(T * ratio) (at least 1) of the regenerated ones
    for i, m in enumerate(tr["step_masks"]):
        assert not m[0, known_rows].any()
        ratio = math.cos(math.pi / 2 * (i + 1) / iters)
        assert int(m.sum()) == max(1, min(int(regen.sum()), int(int(regen.sum()) * ratio)))


def _maps(n_text, masks):
    return varlen.t2s_infill_maps(n_text, [torch.tensor(m, dtype=torch.bool) for m in masks])


@pytest.mark.parametrize("mask", [
    [0, 0, 1, 0, 0],         # a single regenerated position
    [1, 1, 1, 1],            # all regenerated
    [0, 0, 0, 1, 1],         # known prefix
    [1, 1, 0, 0, 0],         # known suffix
    [1, 0, 1, 0, 1, 0, 1],   # alternating
])
def test_maps_single_utterance(mask):
    n_text = 6
    slot, row = _maps([n_text], [mask])
    regen = [k for k, m in enumerate(mask) if m]
    assert row == [n_text + 3 + k for k in regen]
    assert slot == [regen.index(k) if m else -1 for k, m in enumerate(mask)]


def test_maps_packed_batch():
    # L = n_text + N + 4: 2 + 4 + 4 = 10 rows, then 0 + 1 + 4 = 5, then 3 + 3 + 4 = 10
    slot, row = _maps([2, 0, 3], [[0, 1, 1, 0], [1], [1, 0, 1]])
    assert slot == [-1, 0, 1, -1, 2, 3, -1, 4]
    assert row == [6, 7, 13, 21, 23]


def _batch(masks, seed=0):
    g = torch.Generator().manual_seed(seed)
    return [torch.randint(0, 1024, (len(m),), generator=g) for m in masks], [torch.tensor(m, dtype=torch.bool) for m in masks]


def test_split_packs_known_tokens_and_flags():
    masks = [[0, 1, 1, 0, 1], [1, 1], [1, 0, 0]]
    sem, regen = _batch(masks)
    sem[0][1] = -7                 # values at regenerated positions are ignored
    sem[2][0] = 5000
    sp = varlen.t2s_infill_split([4, 0, 9], sem, regen, 1024, 64)
    assert sp.N == (5, 2, 3) and sp.T == (3, 2, 1)
    flat = torch.cat(regen)
    assert torch.equal(sp.regenerate, flat.to(torch.uint8)) and sp.regenerate.device.type == "cpu"
    assert torch.equal(sp.known[~flat], torch.cat(sem)[~flat]) and (sp.known[flat] == 0).all()


def test_split_rejects_bad_input():
    sem, regen = _batch([[0, 1, 1], [1, 0]])
    split = lambda s, r, n_text=(3, 3), max_positions=64: varlen.t2s_infill_split(list(n_text), s, r, 1024, max_positions)
    split(sem, regen)
    with pytest.raises(ValueError):                      # lists of different lengths
        split(sem[:1], regen)
    with pytest.raises(ValueError):
        split(sem, regen, n_text=(3,))
    with pytest.raises(ValueError):
        split([], [], n_text=())
    with pytest.raises(ValueError, match="utterance 1"):  # a mask of the wrong length
        split(sem, [regen[0], torch.tensor([True, False, True])])
    with pytest.raises(ValueError, match="utterance 1"):  # nothing to regenerate
        split(sem, [regen[0], torch.zeros(2, dtype=torch.bool)])
    with pytest.raises(ValueError, match="utterance 0"):  # not a bool mask
        split(sem, [regen[0].long(), regen[1]])
    with pytest.raises(ValueError, match="utterance 1"):  # not 1-D
        split([sem[0], sem[1][None]], regen)
    with pytest.raises(ValueError, match="utterance 1"):  # a known token out of range
        split([sem[0], torch.tensor([3, 1024])], regen)
    with pytest.raises(ValueError, match="utterance 0"):
        split([torch.tensor([-1, 0, 0]), sem[1]], regen)
    with pytest.raises(ValueError, match="utterance 1"):  # L = 3 + 2 + 4 = 9 > 8
        split(sem, regen, n_text=(1, 3), max_positions=8)
    split(sem, regen, n_text=(1, 2), max_positions=8)   # L = 8 fits
