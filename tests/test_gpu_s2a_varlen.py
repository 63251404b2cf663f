"""Variable-length S2A decode (infer_batch / edm_s2a_bind_varlen) and the packed-layout operators.

The contract is batch invariance: utterance i of a packed decode equals infer_special on utterance i alone with batch offset
batch_offset + i, bit for bit (default mode). The lengths sit on and around the 128- and 256-row tile edges of attention, the
16-token groups of the conv module and the 5-tap conv window.
"""
import pytest
import torch

pytestmark = pytest.mark.gpu
dev = "cuda"

T_EDGES = [2, 3, 19, 20, 21, 127, 128, 129, 255, 256, 257, 500, 1500]


@pytest.fixture(scope="module")
def model():
    from tests.parity_utils import full_model

    return full_model()[2]


def _utts(model, T, P, seed):
    g = torch.Generator().manual_seed(seed)
    n_sem, V = model.config.num_semantic_tokens, model.num_codevectors
    sem = [torch.randint(0, n_sem, (t,), generator=g) for t in T]
    ap = [torch.randint(0, V, (4, p), generator=g) for p in P]
    sp = [torch.randint(0, n_sem, (p,), generator=g) for p in P]
    return sem, ap, sp


def _single(model, sem, ap, sp, i, steps, offset, prompts, **extra):
    # infer_batch's per-utterance extras are infer_special's for one utterance: cat_gumbel [S-1, 1*T, V], remask / forced [S', 1, T]
    one = {k: v[i] for k, v in extra.items()}
    if prompts and ap[i].shape[1] > 0:
        return model.infer_special(sem[i][None], ap[i][None], sp[i][None], steps=steps, batch_offset=offset + i, seed=11, **one)[0]
    return model.infer_special(sem[i][None], None, None, steps=steps, batch_offset=offset + i, seed=11, **one)[0]


@pytest.mark.parametrize("steps", [8, 1])
def test_mixed_lengths_match_single_utterances(model, steps):
    T = T_EDGES
    P = [[0, 33, 150][i % 3] for i in range(len(T))]
    sem, ap, sp = _utts(model, T, P, seed=steps)
    offset = 5
    codes = model.infer_batch(sem, ap, sp, steps=steps, seed=11, batch_offset=offset)
    assert [tuple(c.shape) for c in codes] == [(12, t) for t in T]
    for i in range(len(T)):
        assert torch.equal(codes[i], _single(model, sem, ap, sp, i, steps, offset, True)), f"utterance {i} (T={T[i]}, P={P[i]})"


def test_no_prompt_batch_matches_single_utterances(model):
    T = [129, 2, 256, 21, 500]
    sem, _, _ = _utts(model, T, [0] * len(T), seed=3)
    codes = model.infer_batch(sem, steps=4, seed=11)
    for i in range(len(T)):
        assert torch.equal(codes[i], _single(model, sem, None, None, i, 4, 0, False))


def test_injected_noise_and_forcing_match_single_utterances(model):
    T = [3, 128, 257, 20]
    P = [33, 0, 150, 0]
    S, V = 4, model.num_codevectors
    sem, ap, sp = _utts(model, T, P, seed=7)
    g = torch.Generator().manual_seed(8)
    gum = lambda *s: -torch.log(-torch.log(torch.rand(*s, generator=g).clamp(1e-7, 1 - 1e-7)))
    cat_gumbel = [gum(S - 1, t, V) for t in T]
    remask_gumbel = [gum(S - 1, 1, t) for t in T]
    forced_coarse = [torch.randint(0, V, (1, 4, t), generator=g) for t in T]
    codes = model.infer_batch(sem, ap, sp, steps=S, seed=11, cat_gumbel=cat_gumbel, remask_gumbel=remask_gumbel, forced_coarse=forced_coarse)
    for i in range(len(T)):
        ref = _single(model, sem, ap, sp, i, S, 0, True, cat_gumbel=cat_gumbel, remask_gumbel=remask_gumbel, forced_coarse=forced_coarse)
        assert torch.equal(codes[i], ref), f"utterance {i}"


def test_chunked_batch(model):
    """More than MAX_CHUNK utterances: chunks of 64 in order, each with batch offset batch_offset + first index."""
    from edm_tts_b200.s2a import MAX_CHUNK

    g = torch.Generator().manual_seed(1)
    n = MAX_CHUNK + 6
    T = [int(x) for x in torch.randint(2, 90, (n,), generator=g)]
    sem, _, _ = _utts(model, T, [0] * n, seed=2)
    codes = model.infer_batch(sem, steps=3, seed=11, batch_offset=2)
    for i in [0, 1, MAX_CHUNK - 1, MAX_CHUNK, n - 1]:
        assert torch.equal(codes[i], _single(model, sem, None, None, i, 3, 2, False)), f"utterance {i}"


def test_equal_lengths_equal_infer_special(model):
    B, T = 64, 500
    g = torch.Generator().manual_seed(5)
    sem = torch.randint(0, model.config.num_semantic_tokens, (B, T), generator=g)
    ref = model.infer_special(sem, steps=8, seed=3)
    codes = model.infer_batch(list(sem), steps=8, seed=3)
    assert torch.equal(torch.stack(codes), ref)


def test_low_latency_packed_batch_parity(model):
    """Low-latency mode on a small packed batch (<= 512 rows): deterministic, and teacher-forced parity with the oracle per utterance."""
    from oracle.weights import make_inputs
    from tests.parity_utils import NEAR_TIE_EPS, compare_ids, full_model, oracle_trace

    cfg, sd, _ = full_model()
    T, S = [150, 40, 200], 3
    refs, inps = [], []
    for i, t in enumerate(T):
        inp = make_inputs(1, t, 0, S, cfg, seed=900 + i)
        inps.append(inp)
        refs.append(oracle_trace(cfg, sd, inp, S))
    kw = dict(steps=S, cat_gumbel=[inp["cat_gumbel"].view(S - 1, t, -1) for inp, t in zip(inps, T)],
              remask_gumbel=[inp["remask_gumbel"] for inp in inps],
              forced_ids=[torch.stack(r["step_ids"]) for r in refs], forced_masks=[torch.stack(r["step_masks"]) for r in refs],
              forced_coarse=[r["all_logits"][:, :4].argmax(-1) for r in refs])
    sem = [inp["semantic_tokens"][0] for inp in inps]
    model.set_low_latency(True)
    try:
        a = model.infer_batch(sem, **kw)
        b = model.infer_batch(sem, **kw)
    finally:
        model.set_low_latency(False)
    for i in range(len(T)):
        assert torch.equal(a[i], b[i])
        r = compare_ids(a[i][None], refs[i]["codes"], refs[i]["all_logits"], f"low-latency packed utterance {i}", NEAR_TIE_EPS)
        assert r["n_not_near_tie"] == 0, r


def test_errors_match_infer_special(model):
    n_sem, V = model.config.num_semantic_tokens, model.num_codevectors
    ok = [torch.zeros(10, dtype=torch.long), torch.zeros(20, dtype=torch.long)]
    ap = [torch.zeros(4, 5, dtype=torch.long), torch.zeros(4, 6, dtype=torch.long)]
    sp = [torch.zeros(5, dtype=torch.long), torch.zeros(6, dtype=torch.long)]
    with pytest.raises(ValueError):  # mismatched list lengths
        model.infer_batch(ok, ap[:1], sp[:1])
    with pytest.raises(ValueError):  # mixed prompt q
        model.infer_batch(ok, [ap[0], torch.zeros(5, 6, dtype=torch.long)], sp)
    with pytest.raises(ValueError):  # malformed extras
        model.infer_batch(ok, steps=2, remask_gumbel=[torch.zeros(1, 1, 10)])
    with pytest.raises(IndexError):  # out-of-range tokens
        model.infer_batch([ok[0], torch.full((20,), n_sem, dtype=torch.long)])
    with pytest.raises(IndexError):
        model.infer_batch(ok, [ap[0], torch.full((4, 6), V, dtype=torch.long)], sp)
    with pytest.raises(IndexError):  # T_i < 2 with steps > 1
        model.infer_batch([ok[0], torch.zeros(1, dtype=torch.long)], steps=2)
    model.infer_batch([ok[0], torch.zeros(1, dtype=torch.long)], steps=1)
    with pytest.raises(ValueError):  # T_i > 4096
        model.infer_batch([ok[0], torch.zeros(4097, dtype=torch.long)], steps=1)
    with pytest.raises(ValueError):  # the same limit in infer_special
        model.infer_special(torch.zeros(1, 4097, dtype=torch.long), steps=1)
    t = model._cfg_c.max_positions - 5
    with pytest.raises(ValueError):  # P_i + T_i > max_positions
        model.infer_batch([ok[0], torch.zeros(t, dtype=torch.long)], [ap[0], torch.zeros(4, 6, dtype=torch.long)], sp, steps=1)
    with pytest.raises(ValueError):
        model.infer_special(torch.zeros(1, t, dtype=torch.long), torch.zeros(1, 4, 6, dtype=torch.long), torch.zeros(1, 6, dtype=torch.long), steps=1)


def test_attention_varlen_op():
    from edm_tts_b200 import _lib as L

    L.lib()
    H = 16
    lens = [1, 127, 128, 129, 300, 5, 600]
    cu = [0]
    for n in lens:
        cu.append(cu[-1] + n)
    torch.manual_seed(0)
    qkv = torch.randn(cu[-1], 3 * H * 64, device=dev).to(torch.bfloat16)
    out = torch.zeros(cu[-1], H * 64, device=dev, dtype=torch.bfloat16)
    cu_d = torch.tensor(cu, device=dev, dtype=torch.int32)
    L.check(L.lib().edm_attention_varlen(L.ptr(qkv), len(lens), L.ptr(cu_d), H, L.ptr(out), L.stream_ptr()))
    for i, n in enumerate(lens):
        x = qkv[cu[i]:cu[i + 1]]
        q, k, v = x.float().view(1, n, 3, H, 64).permute(2, 0, 3, 1, 4)
        ref = torch.nn.functional.scaled_dot_product_attention(q, k, v).permute(0, 2, 1, 3).reshape(n, H * 64)
        torch.testing.assert_close(out[cu[i]:cu[i + 1]].float(), ref, rtol=2e-2, atol=8e-3)
        one = torch.zeros(n, H * 64, device=dev, dtype=torch.bfloat16)
        L.check(L.lib().edm_attention(L.ptr(x.contiguous()), 1, n, H, L.ptr(one), L.stream_ptr()))
        assert torch.equal(one, out[cu[i]:cu[i + 1]]), f"sequence {i}"


@pytest.mark.parametrize("glu_input", [1, 0])
def test_conv_module_varlen_op(glu_input):
    from edm_tts_b200 import _lib as L
    from tests.test_gpu_ops import _conv_ref, bf, rb

    L.lib()
    lens = [1, 2, 3, 4, 5, 37, 16, 17, 150, 500]
    cu = [0]
    for n in lens:
        cu.append(cu[-1] + n)
    torch.manual_seed(1)
    torch.backends.cudnn.allow_tf32 = False
    h = bf(torch.randn(cu[-1], 4096, device=dev))
    dw_w = rb(torch.randn(2048, 5, device=dev) * 0.4)
    dw_b = torch.randn(2048, device=dev) * 0.1
    cln_w = torch.randn(2048, device=dev)
    x = h if glu_input else bf(rb(h.float()[:, :2048] * rb(torch.sigmoid(h.float()[:, 2048:]))))
    out = torch.empty(cu[-1], 2048, device=dev, dtype=torch.bfloat16)
    cu_d = torch.tensor(cu, device=dev, dtype=torch.int32)
    args = (L.ptr(dw_w), L.ptr(dw_b), L.ptr(cln_w))
    L.check(L.lib().edm_conv_module_varlen(L.ptr(x), glu_input, L.ptr(out), *args, len(lens), L.ptr(cu_d), L.stream_ptr()))
    for i, n in enumerate(lens):
        seg = out[cu[i]:cu[i + 1]]
        d = (seg.float() - _conv_ref(h[cu[i]:cu[i + 1]], dw_w, dw_b, cln_w, 1, n)).abs()
        assert d.max().item() < 0.07 and d.mean().item() < 1e-4, (i, d.max().item(), d.mean().item())
        one = torch.empty(n, 2048, device=dev, dtype=torch.bfloat16)
        L.check(L.lib().edm_conv_module(L.ptr(x[cu[i]:cu[i + 1]].contiguous()), glu_input, L.ptr(one), *args, 1, n, L.stream_ptr()))
        assert torch.equal(one, seg), f"sequence {i}"
