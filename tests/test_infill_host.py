"""S2A infilling without a GPU: the infill oracle (tests/oracle_infill.py) reduces to infer_special when the known frames are a prefix (or absent), the
host row maps of the masked bind, and the checks on an infill batch."""
import pytest
import torch

from edm_tts_b200 import varlen
from oracle import s2a as os2a
from oracle.weights import OracleConfig, make_inputs, make_state_dict
from tests import oracle_infill as oi

SMALL = OracleConfig(hidden=128, heads=2, depth=6, injection_layers=(1, 2, 3, 4), num_semantic=50, n_codebooks=12, codebook_size=64,
                     codebook_dim=8, latent_dim=128)


@pytest.fixture(scope="module")
def sd():
    return make_state_dict(SMALL, seed=3)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("steps", [1, 4])
def test_prefix_infill_is_infer_special(sd, mode, steps):
    B, T, P = 2, 9, 5
    inp = make_inputs(B, T, P, steps, SMALL, seed=40 + steps)
    kw = dict(steps=steps, cat_gumbel=inp["cat_gumbel"], remask_gumbel=inp["remask_gumbel"], mode=mode)
    tr_ref, tr = {}, {}
    with torch.inference_mode():
        ref = os2a.infer_special(sd, SMALL, inp["semantic_tokens"], inp["acoustic_prompt_tokens"], inp["semantic_prompt_tokens"], trace=tr_ref, **kw)
        sem = torch.cat([inp["semantic_prompt_tokens"], inp["semantic_tokens"]], 1)
        codes = torch.cat([inp["acoustic_prompt_tokens"], torch.full((B, SMALL.n_codebooks, T), 7)], 2)
        regen = (torch.arange(P + T) >= P).expand(B, P + T)
        got = oi.infer_infill(sd, SMALL, sem, codes, regen, trace=tr, **kw)
    assert torch.equal(got, ref)
    assert torch.equal(tr["all_logits"], tr_ref["all_logits"])
    for a, b in zip(tr["step_logits"], tr_ref["step_logits"]):
        assert torch.equal(a, b)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_all_target_infill_is_the_no_prompt_decode(sd, mode):
    B, T, steps = 2, 8, 4
    inp = make_inputs(B, T, 0, steps, SMALL, seed=7)
    kw = dict(steps=steps, cat_gumbel=inp["cat_gumbel"], remask_gumbel=inp["remask_gumbel"], mode=mode)
    with torch.inference_mode():
        ref = os2a.infer_special(sd, SMALL, inp["semantic_tokens"], **kw)
        got = oi.infer_infill(sd, SMALL, inp["semantic_tokens"], torch.zeros(B, 1, T, dtype=torch.long), torch.ones(B, T, dtype=torch.bool), **kw)
    assert torch.equal(got, ref)


def test_scattered_infill_keeps_known_rows_and_matches_the_training_input(sd):
    """A scattered mask: the encoder input is the training forward's where(mask, sem + mask_token, sem + feat) (oracle training_forward)
    and the known rows get the ground-truth injections."""
    N = 10
    g = torch.Generator().manual_seed(2)
    sem = torch.randint(0, SMALL.num_semantic, (1, N), generator=g)
    codes = torch.randint(0, SMALL.codebook_size, (1, SMALL.n_codebooks, N), generator=g)
    regen = torch.tensor([[1, 0, 0, 1, 1, 0, 1, 0, 0, 1]], dtype=torch.bool)
    with torch.inference_mode():
        x, sem_t, inj = oi.build_infill_input(sd, SMALL, sem, codes, regen, "fp32")
        feat = os2a.feat_proj(sd, SMALL, codes[:, 0], "fp32")
        emb = torch.nn.functional.embedding(sem, sd["semantic_embedding.weight"])
        want = torch.where(regen[..., None], emb + sd["mask_token"], emb + feat)
        torch.testing.assert_close(x, want, rtol=1e-5, atol=1e-5)
        assert torch.equal(sem_t, emb[regen].view(1, -1, SMALL.hidden))
        assert len(inj) == len(SMALL.injection_layers) and all(torch.equal(i[regen], torch.zeros_like(i[regen])) for i in inj)
        out = oi.infer_infill(sd, SMALL, sem, codes, regen, steps=2, cat_gumbel=torch.zeros(1, 5, SMALL.codebook_size),
                                remask_gumbel=torch.zeros(1, 1, 5))
    assert out.shape == (1, SMALL.n_codebooks, 5)


def _maps(masks):
    return varlen.infill_rows([torch.tensor(m, dtype=torch.bool) for m in masks])


@pytest.mark.parametrize("mask", [
    [1, 0, 0, 0, 0],        # target at the first frame
    [0, 0, 0, 0, 1],        # at the last frame
    [1, 0, 0, 0, 1],        # both
    [0, 0, 1, 0, 0],        # a single target frame
    [1, 1, 0, 1, 1],        # all frames but one
    [0, 1, 1, 0, 0, 1, 0, 1, 1, 1, 0],  # several spans
    [1, 1, 1],              # no known frame
])
def test_row_maps_single_utterance(mask):
    tgt_enc, enc_slot = _maps([mask])
    assert tgt_enc == [n for n, m in enumerate(mask) if m]
    known = [n for n, m in enumerate(mask) if not m]
    for n, m in enumerate(mask):
        assert enc_slot[n] == (tgt_enc.index(n) if m else -1 - known.index(n))


def test_row_maps_packed_batch():
    masks = [[0, 1, 1, 0], [1], [1, 0, 1], [0, 0, 1]]
    tgt_enc, enc_slot = _maps(masks)
    assert tgt_enc == [1, 2, 4, 5, 7, 10]
    assert enc_slot == [-1, 0, 1, -2, 0, 0, -1, 1, -1, -2, 0]
    # known frames in front: the closed form of a prompt prefix, target t of utterance s at row cu_n[s] + P_s + t
    tgt_enc, enc_slot = _maps([[0, 0, 1, 1, 1], [0, 1]])
    assert tgt_enc == [2, 3, 4, 6] and enc_slot == [-1, -2, 0, 1, 2, -1, 0]


def _batch(masks, q=12, seed=0):
    g = torch.Generator().manual_seed(seed)
    sem = [torch.randint(0, 50, (len(m),), generator=g) for m in masks]
    codes = [torch.randint(0, 1024, (q, len(m)), generator=g) for m in masks]
    return sem, codes, [torch.tensor(m, dtype=torch.bool) for m in masks]


def test_infill_split_orders_targets_and_known_frames():
    masks = [[0, 1, 1, 0, 1], [1, 1], [1, 0, 0]]
    sem, codes, regen = _batch(masks, q=4)
    codes[0][:, 1] = -5        # values at regenerated frames are ignored
    sp = varlen.infill_split(sem, codes, regen, 1024, 50)
    assert sp.N == (5, 2, 3) and sp.T == (3, 2, 1) and sp.P == (2, 0, 2)
    for i, m in enumerate(regen):
        assert torch.equal(sp.sem_target[i], sem[i][m]) and torch.equal(sp.sem_known[i], sem[i][~m])
        assert torch.equal(sp.codes_known[i], codes[i][:, ~m]) and sp.codes_known[i].shape == (4, sp.P[i])


def test_infill_split_rejects_bad_input():
    sem, codes, regen = _batch([[0, 1, 1], [1, 0]])
    with pytest.raises(ValueError):   # a mask of the wrong length
        varlen.infill_split(sem, codes, [regen[0], torch.tensor([True, False, True])], 1024, 50)
    with pytest.raises(ValueError):   # an utterance with no target frame
        varlen.infill_split(sem, codes, [regen[0], torch.zeros(2, dtype=torch.bool)], 1024, 50)
    with pytest.raises(ValueError):   # not a bool mask
        varlen.infill_split(sem, codes, [regen[0], regen[1].long()], 1024, 50)
    with pytest.raises(ValueError):   # lists of different lengths
        varlen.infill_split(sem, codes[:1], regen, 1024, 50)
    with pytest.raises(ValueError):   # codes of different level counts
        varlen.infill_split(sem, [codes[0], codes[1][:4]], regen, 1024, 50)
    with pytest.raises(ValueError):   # codes and tokens of different lengths
        varlen.infill_split(sem, [codes[0], codes[1][:, :1]], regen, 1024, 50)
    bad = codes[1].clone()
    bad[3, 1] = 1024                  # a known frame's code out of range
    with pytest.raises(IndexError):
        varlen.infill_split(sem, [codes[0], bad], regen, 1024, 50)
    bad = codes[1].clone()
    bad[3, 1] = -1
    with pytest.raises(IndexError):
        varlen.infill_split(sem, [codes[0], bad], regen, 1024, 50)
    with pytest.raises(IndexError):   # a semantic token out of range
        varlen.infill_split([sem[0], torch.tensor([3, 50])], codes, regen, 1024, 50)
    bad = codes[1].clone()
    bad[3, 0] = 5000                  # out of range, but at a regenerated frame: ignored
    varlen.infill_split(sem, [codes[0], bad], regen, 1024, 50)
