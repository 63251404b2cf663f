"""DAC decoder batches of different lengths on one GPU: ms per batch and decoded latent frames/s (sum of T_i) for a fixed seeded mix of
64 utterances with T_i uniform in [150, 1000] (the mix of tools/varlen_bench.py), synthetic decoder weights of the reference
architecture (decoder_dim 1536, rates 8 5 4 2):
  (a) DAC.decode_from_codes_batch on the mix; (b) decode_from_codes per utterance in a loop; (c) decode_from_codes on the mix padded
  to max T_i (wrong tails: the compute reference of "pad to the longest"); (d) the rectangular 64 x 500 batch through
  decode_from_codes and through decode_from_codes_batch; (e) the summed event time of the edm_dac_zero_rows launches inside (a), in a
  run of its own; (f) text -> waveform: T2S infer_batch (16 iterations, the batch of tools/t2s_batch_bench.py) -> S2A infer_batch
  (8 steps) -> decode_from_codes_batch, with the share of each stage.
The stage buffers (GBs) are far larger than L2. Prints one JSON line per case and writes them, with the card name and power limit
read in the same run, to the file given as the first argument."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

N_UTT, T2S_ITERS, S2A_STEPS = 64, 16, 8


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b))
    return sorted(out)[len(out) // 2], out


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    import __graft_entry__ as ge

    ge.build()
    from edm_tts_b200 import InjectionConformerModel, TextToSemanticWLen
    from edm_tts_b200.config import InjectionConformerConfig, TextToSemanticWLenConfig
    from edm_tts_b200.dac import DAC
    from edm_tts_b200.synthetic import OracleConfig, T2SConfig, make_dac_state_dict, make_state_dict, make_t2s_state_dict

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    s2a_sd = make_state_dict(OracleConfig(), 0)
    dsd = make_dac_state_dict(0)
    for k in list(dsd):      # the vocoder decodes with the quantizer the S2A model was built with
        if k.startswith("quantizer."):
            dsd[k] = s2a_sd["acoustic_model." + k].cpu()
    dac = DAC(dsd)
    dec = dac.decoder
    g = torch.Generator().manual_seed(2024)
    T = [int(x) for x in torch.randint(150, 1001, (N_UTT,), generator=g)]
    codes = [torch.randint(0, 1024, (12, t), generator=g).cuda() for t in T]
    tmax = max(T)
    codes_pad = torch.stack([torch.nn.functional.pad(c, (0, tmax - c.shape[1])) for c in codes])
    frames = sum(T)
    rows = []

    def case(name, fn, reps, n_frames=frames, **kw):
        ms, all_ms = timed(fn, reps)
        r = dict(case=name, ms_per_batch=round(ms, 3), frames=n_frames, frames_per_s=round(n_frames / ms * 1e3),
                 samples_per_s=round(n_frames * dec.hop_length / ms * 1e3), runs_ms=[round(x, 3) for x in all_ms], **kw)
        print(json.dumps(r), flush=True)
        rows.append(r)
        return r

    a = case("a_decode_from_codes_batch", lambda: dac.decode_from_codes_batch(codes), 7)
    b = case("b_decode_from_codes_loop", lambda: [dac.decode_from_codes(c[None]) for c in codes], 3)
    c = case("c_decode_from_codes_padded", lambda: dac.decode_from_codes(codes_pad), 7, padded_frames=N_UTT * tmax)
    rect = torch.randint(0, 1024, (64, 12, 500), generator=g).cuda()
    rect_l = list(rect)
    d_rect = case("d_rect_64x500/decode_from_codes", lambda: dac.decode_from_codes(rect), 7, n_frames=64 * 500)
    d_batch = case("d_rect_64x500/decode_from_codes_batch", lambda: dac.decode_from_codes_batch(rect_l), 7, n_frames=64 * 500)

    # (e) the gap clears inside (a): every edm_dac_zero_rows launch bracketed by events (a run of its own)
    ev = []
    plain = dec._zero_rows

    def bracketed(*args):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        plain(*args)
        e.record()
        ev.append((s, e))

    dec._zero_rows = bracketed
    dac.decode_from_codes_batch(codes)
    torch.cuda.synchronize()
    del dec._zero_rows
    zero_ms = sum(s.elapsed_time(e) for s, e in ev)
    e_res = dict(case="e_zero_rows_in_a", launches=len(ev), ms=round(zero_ms, 4), share_of_a=round(zero_ms / a["ms_per_batch"], 4))
    print(json.dumps(e_res), flush=True)

    # (f) text -> waveform, every stage batched (the T2S model and texts of tools/t2s_batch_bench.py, gt lengths in [150, 500])
    dims = T2SConfig(hidden=384, heads=8, depth=12, lp_heads=8, lp_depth=4)
    t2s = TextToSemanticWLen(TextToSemanticWLenConfig(hidden_size=384, main_encoder_args=dict(depth=12, heads=8), length_predictor_args=dict(depth=4, heads=8)),
                             make_t2s_state_dict(dims, 0), device="cuda", max_positions=1024)
    s2a = InjectionConformerModel(InjectionConformerConfig(), s2a_sd, device="cuda")
    gt = torch.Generator().manual_seed(2024)
    alphabet = "abcdefghijklmnopqrstuvwxyz ABCDEFGHIJKLMNOPQRSTUVWXYZ,.'"
    n_bytes = [int(x) for x in torch.randint(40, 201, (N_UTT,), generator=gt)]
    texts = ["".join(alphabet[int(i)] for i in torch.randint(0, len(alphabet), (n,), generator=gt)) for n in n_bytes]
    lengths = [int(x) for x in torch.randint(150, 501, (N_UTT,), generator=gt)]

    def pipeline():
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        evs[0].record()
        sem = t2s.infer_batch(texts, pred_iters=T2S_ITERS, gt_lengths=lengths, seed=1)
        evs[1].record()
        cb = s2a.infer_batch(sem, steps=S2A_STEPS, seed=1)
        evs[2].record()
        dac.decode_from_codes_batch(cb)
        evs[3].record()
        torch.cuda.synchronize()
        return [evs[i].elapsed_time(evs[i + 1]) for i in range(3)]

    pipeline()
    runs = [pipeline() for _ in range(5)]
    tot = sorted(runs, key=sum)[len(runs) // 2]
    f_res = dict(case="f_text_to_waveform", utterances=N_UTT, semantic_frames=sum(lengths), total_ms=round(sum(tot), 3),
                 ms_per_utterance=round(sum(tot) / N_UTT, 3), stage_ms=dict(t2s=round(tot[0], 3), s2a=round(tot[1], 3), dac=round(tot[2], 3)),
                 stage_share=dict(t2s=round(tot[0] / sum(tot), 3), s2a=round(tot[1] / sum(tot), 3), dac=round(tot[2] / sum(tot), 3)),
                 runs_ms=[[round(x, 3) for x in r] for r in runs])
    print(json.dumps(f_res), flush=True)

    summary = dict(batch_vs_loop=round(b["ms_per_batch"] / a["ms_per_batch"], 2), batch_vs_padded=round(c["ms_per_batch"] / a["ms_per_batch"], 2),
                   a_rate_over_d_rect_rate=round(a["frames_per_s"] / d_rect["frames_per_s"], 3),
                   a_rate_over_d_batch_rate=round(a["frames_per_s"] / d_batch["frames_per_s"], 3),
                   padded_row_fraction=round(1 - frames / (N_UTT * tmax), 3), zero_rows_share_of_a=e_res["share_of_a"])
    print(json.dumps(dict(case="summary", **summary)), flush=True)
    res = dict(gpu=smi, utterances=N_UTT, T_range=[150, 1000], decoder=dict(decoder_dim=1536, rates=[8, 5, 4, 2], weights="synthetic"),
               cases=rows, e_zero_rows=e_res, f_text_to_waveform=f_res, summary=summary)
    if out_path:
        with open(out_path, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
