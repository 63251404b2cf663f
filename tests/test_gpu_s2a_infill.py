"""S2A infilling (infill_batch / edm_s2a_bind_masked): regenerate any chosen frames of an utterance given the others.

With the known frames in front, the masked bind is the prompt decode bit for bit; with scattered masks it is graded against the oracle's
infer_infill (tests/oracle_infill.py) under the teacher-forcing protocol, and it keeps the batch-invariance contract of infer_batch.
"""
import pytest
import torch

pytestmark = pytest.mark.gpu
dev = "cuda"
SEED = 11


@pytest.fixture(scope="module")
def model():
    from tests.parity_utils import full_model

    return full_model()[2]


def _utts(model, N, seed, q=12):
    g = torch.Generator().manual_seed(seed)
    sem = [torch.randint(0, model.config.num_semantic_tokens, (n,), generator=g) for n in N]
    codes = [torch.randint(0, model.num_codevectors, (q, n), generator=g) for n in N]
    return sem, codes


def _prefix(N, P):
    return [torch.arange(n) >= p for n, p in zip(N, P)]


def _spans(n, spans):
    m = torch.zeros(n, dtype=torch.bool)
    for a, b in spans:
        m[a:b] = True
    return m


def _scattered(N, seed):
    """20-40 % of each utterance in 1-3 spans."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for n in N:
        m = torch.zeros(n, dtype=torch.bool)
        k = int(torch.randint(1, 4, (1,), generator=g))
        want = max(2, int(n * (0.2 + 0.2 * float(torch.rand(1, generator=g)))))
        for j in range(k):
            ln = max(1, want // k)
            a = int(torch.randint(0, max(1, n - ln), (1,), generator=g))
            m[a:a + ln] = True
        if int(m.sum()) < 2:
            m[:2] = True
        out.append(m)
    return out


@pytest.mark.parametrize("steps", [8, 1])
def test_prefix_masks_are_the_prompt_decode(model, steps):
    N = [2, 3, 130, 257, 500, 21, 640] + ([1, 2] if steps == 1 else [])
    P = [0, 1, 30, 0, 150, 19, 511] + ([0, 1] if steps == 1 else [])
    sem, codes = _utts(model, N, seed=steps)
    regen = _prefix(N, P)
    off = 3
    got = model.infill_batch(sem, codes, regen, steps=steps, seed=SEED, batch_offset=off)
    ref = model.infer_batch([s[m] for s, m in zip(sem, regen)], [c[:, ~m] for c, m in zip(codes, regen)], [s[~m] for s, m in zip(sem, regen)],
                            steps=steps, seed=SEED, batch_offset=off)
    for i in range(len(N)):
        assert got[i].shape == (12, N[i] - P[i])
        assert torch.equal(got[i], ref[i]), f"utterance {i} (N={N[i]}, P={P[i]})"
        m = regen[i]
        if P[i] > 0:
            one = model.infer_special(sem[i][m][None], codes[i][:, ~m][None], sem[i][~m][None], steps=steps, seed=SEED, batch_offset=off + i)[0]
        else:
            one = model.infer_special(sem[i][None], steps=steps, seed=SEED, batch_offset=off + i)[0]
        assert torch.equal(got[i], one), f"utterance {i} against infer_special"


@pytest.mark.parametrize("steps", [8, 1])
def test_all_target_masks_are_the_no_prompt_decode(model, steps):
    N = [2, 129, 300, 3] + ([1] if steps == 1 else [])
    sem, codes = _utts(model, N, seed=20 + steps, q=1)
    got = model.infill_batch(sem, codes, [torch.ones(n, dtype=torch.bool) for n in N], steps=steps, seed=SEED)
    ref = model.infer_batch(sem, steps=steps, seed=SEED)
    for i in range(len(N)):
        assert torch.equal(got[i], ref[i]), f"utterance {i}"


def _oracle_infill(cfg, sd, sem, codes, regen, S, noise_seed):
    """The infill oracle (bf16 mode) of one utterance with injected noise; returns (noise, trace)."""
    from tests import oracle_infill as oi

    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    T, V = int(regen.sum()), cfg.codebook_size
    g = torch.Generator().manual_seed(noise_seed)
    gum = lambda *s: -torch.log(-torch.log(torch.rand(*s, generator=g).clamp(1e-7, 1 - 1e-7)))
    noise = dict(cat_gumbel=gum(S - 1, T, V), remask_gumbel=gum(S - 1, 1, T)) if S > 1 else {}
    tr = {}
    with torch.inference_mode():
        tr["codes"] = oi.infer_infill(sd, cfg, sem[None].to(dev), codes[None].to(dev), regen[None].to(dev), steps=S, mode="bf16", trace=tr,
                                        **{k: v.to(dev) for k, v in noise.items()})
    return noise, tr


@pytest.mark.parametrize("S,shapes", [
    (8, [(1000, [(0, 1), (400, 650)]), (37, [(36, 37), (0, 2)]), (500, [(0, 499)]), (731, [(100, 180), (300, 310), (600, 731)]),
         (64, [(0, 64)]), (2, [(1, 2), (0, 1)])]),
    (1, [(90, [(45, 46)]), (300, [(0, 1), (299, 300)]), (5, [(0, 4)])]),
])
def test_scattered_masks_match_the_oracle(S, shapes):
    from tests.parity_utils import NEAR_TIE_EPS, compare_ids, full_model, record

    cfg, sd, model = full_model()
    N = [n for n, _ in shapes]
    regen = [_spans(n, sp) for n, sp in shapes]
    sem, codes = _utts(model, N, seed=77 + S)
    refs, noises = [], []
    for i in range(len(N)):
        nz, tr = _oracle_infill(cfg, sd, sem[i], codes[i], regen[i], S, 500 + i)
        noises.append(nz)
        refs.append(tr)
    kw = dict(forced_coarse=[r["all_logits"][:, :4].argmax(-1) for r in refs])
    if S > 1:
        kw.update(cat_gumbel=[nz["cat_gumbel"] for nz in noises], remask_gumbel=[nz["remask_gumbel"] for nz in noises],
                  forced_ids=[torch.stack(r["step_ids"]) for r in refs], forced_masks=[torch.stack(r["step_masks"]) for r in refs])
    got = model.infill_batch(sem, codes, regen, steps=S, seed=SEED, **kw)
    for i in range(len(N)):
        r = compare_ids(got[i][None], refs[i]["codes"], refs[i]["all_logits"], f"infill utterance {i} N={N[i]} T={int(regen[i].sum())} S={S}",
                        NEAR_TIE_EPS)
        record("infill scattered masks", **r)
        assert r["n_not_near_tie"] == 0, r


def test_batch_invariance_and_chunks(model):
    from edm_tts_b200.s2a import MAX_CHUNK

    g = torch.Generator().manual_seed(4)
    n = MAX_CHUNK + 5
    N = [int(x) for x in torch.randint(8, 400, (n,), generator=g)]
    sem, codes = _utts(model, N, seed=5)
    regen = _scattered(N, seed=6)
    off = 9
    got = model.infill_batch(sem, codes, regen, steps=8, seed=SEED, batch_offset=off)
    for i in [0, 1, 17, MAX_CHUNK - 1, MAX_CHUNK, n - 1]:
        one = model.infill_batch([sem[i]], [codes[i]], [regen[i]], steps=8, seed=SEED, batch_offset=off + i)[0]
        assert torch.equal(got[i], one), f"utterance {i}"
    a = model.infill_batch(sem[:MAX_CHUNK], codes[:MAX_CHUNK], regen[:MAX_CHUNK], steps=8, seed=SEED, batch_offset=off)
    b = model.infill_batch(sem[MAX_CHUNK:], codes[MAX_CHUNK:], regen[MAX_CHUNK:], steps=8, seed=SEED, batch_offset=off + MAX_CHUNK)
    for i, x in enumerate(a + b):
        assert torch.equal(got[i], x), f"utterance {i} against its chunk"


def test_philox_decode_is_deterministic(model):
    N = [300, 41, 1000]
    sem, codes = _utts(model, N, seed=12)
    regen = _scattered(N, seed=13)
    a = model.infill_batch(sem, codes, regen, steps=8, seed=5)
    b = model.infill_batch(sem, codes, regen, steps=8, seed=5)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    assert [tuple(x.shape) for x in a] == [(12, int(m.sum())) for m in regen]


def test_row_maps_on_the_device(model):
    from edm_tts_b200 import varlen

    N = [7, 1, 12]
    regen = [_spans(7, [(0, 1), (5, 7)]), torch.ones(1, dtype=torch.bool), _spans(12, [(3, 9)])]
    model._bind_masked(N, torch.cat(regen))
    tgt_enc, enc_slot = varlen.infill_rows(regen)
    assert model._view("tgt_enc", (len(tgt_enc),), torch.int32).tolist() == tgt_enc
    assert model._view("enc_slot", (sum(N),), torch.int32).tolist() == enc_slot


def test_encoder_api_with_scattered_masks():
    from tests import oracle_infill as oi
    from tests.parity_utils import compare_logits, full_model, record
    from tests.test_gpu_s2a import MAX_TOL, MEAN_TOL

    cfg, sd, model = full_model()
    B, N = 2, 120
    sem, codes = _utts(model, [N] * B, seed=41)
    sem, codes = torch.stack(sem).to(dev), torch.stack(codes).to(dev)
    mti = torch.stack([_spans(N, [(0, 10), (50, 80)]), _spans(N, [(30, 60), (110, 120)])]).to(dev)
    T, P = 40, N - 40
    with torch.inference_mode():
        x, _, prompt_inj = oi.build_infill_input(sd, cfg, sem, codes, mti)
        ref_first = oi.forward_first_level(sd, cfg, x.clone(), mti)
        ref_all = oi.forward_full(sd, cfg, x.clone(), mti, prompt_inj)
    case = f"infill encoder API B={B} N={N} T={T}"
    first = model.encoder.forward_first_level(x, mask_time_indices=mti)
    assert first.shape == (B, 1, T, cfg.codebook_size)
    r = compare_logits(first[:, 0], ref_first, "encoder.forward_first_level (scattered mask)")
    record(case, **r)
    assert r["max"] < MAX_TOL and r["n_not_near_tie"] == 0, r
    forced = ref_all[:, :4].argmax(-1)
    pc = codes.transpose(1, 2)[~mti].view(B, P, -1).transpose(1, 2)           # the known rows' codes in time order [B, 12, P]
    for name, kw in (("injections", dict(injections=prompt_inj)), ("prompt_codes", dict(prompt_codes=pc))):
        logits = model.encoder(x, injections=kw.get("injections"), acoustic_model=model.acoustic_model, mask_time_indices=mti,
                               prompt_codes=kw.get("prompt_codes"), forced_coarse=forced)
        assert logits.shape == (B, cfg.n_codebooks, T, cfg.codebook_size)
        for q in range(cfg.n_codebooks):
            r = compare_logits(logits[:, q], ref_all[:, q], f"encoder.forward({name}, scattered mask) level {q}")
            record(case, **r)
            assert r["max"] < MAX_TOL and r["mean"] < MEAN_TOL and r["n_not_near_tie"] == 0, r
    uneven = mti.clone()
    uneven[0, 100] = True
    with pytest.raises(ValueError):
        model.encoder.forward_first_level(x, mask_time_indices=uneven)
    with pytest.raises(ValueError):
        model.encoder(x, injections=prompt_inj, mask_time_indices=uneven)
    with pytest.raises(ValueError):
        model.encoder(x, mask_time_indices=mti)                                  # known rows but no injections


def test_errors(model):
    sem, codes = _utts(model, [10, 6], seed=2)
    regen = [_spans(10, [(2, 5)]), _spans(6, [(0, 2)])]
    with pytest.raises(ValueError):   # no frame to regenerate
        model.infill_batch(sem, codes, [regen[0], torch.zeros(6, dtype=torch.bool)])
    with pytest.raises(ValueError):   # mask of the wrong length
        model.infill_batch(sem, codes, [regen[0], torch.ones(5, dtype=torch.bool)])
    bad = codes[1].clone()
    bad[0, 4] = model.num_codevectors
    with pytest.raises(IndexError):   # a known frame's code out of range
        model.infill_batch(sem, [codes[0], bad], regen)
    with pytest.raises(IndexError):   # fewer levels than injection layers with known frames
        model.infill_batch(sem, [c[:2] for c in codes], regen)
    with pytest.raises(IndexError):   # one target frame with steps > 1
        model.infill_batch(sem, codes, [regen[0], _spans(6, [(3, 4)])], steps=2)
    with pytest.raises(ValueError):   # malformed extras
        model.infill_batch(sem, codes, regen, steps=2, remask_gumbel=[torch.zeros(1, 1, 3), torch.zeros(1, 1, 3)])
    n = model._cfg_c.max_positions + 1
    with pytest.raises(ValueError):   # N_i above max_positions
        model.infill_batch([torch.zeros(n, dtype=torch.long)], [torch.zeros(12, n, dtype=torch.long)], [_spans(n, [(0, 2)])], steps=1)
