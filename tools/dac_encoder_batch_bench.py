"""DAC encoder batches of different lengths on one GPU: ms per call, audio samples/s and frames/s (sums over the clips), synthetic DAC
weights of the reference architecture (encoder_dim 64, rates 2 4 5 8, 12 codebooks):
  (a) DAC.encode_to_codes_batch on a fixed seeded mix of 64 clips with L_i uniform in [48 000, 320 000] samples (3-20 s, the
  [150, 1000]-frame range of the other batch benches), lengths not hop-aligned; (b) encode_to_codes per clip in a loop; (c)
  encode_to_codes on the mix right-padded to the longest clip (the reference's Collator: wrong tails, the compute reference of "pad to
  the longest"); (d) the rectangular 32 x 960 160 batch (BASELINE config 4, bench.py's secondary_encode) through encode_to_codes and
  through encode_to_codes_batch; (e) the summed event time of the edm_dac_zero_rows launches inside (a), in a run of its own; (f) 256
  prompt-sized clips of 0.5-3 s: encode_to_codes_batch against the loop.
Each case is warmed up once, then timed with CUDA events; the median of the repeats is reported. The stage buffers (GBs) are far
larger than L2. Prints one JSON line per case and writes them, with the card name and power limit read in the same run, to the file
given as the first argument."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

N_CLIPS, N_PROMPTS = 64, 256


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
    from edm_tts_b200.dac import DAC
    from edm_tts_b200.dac_encoder import code_lengths
    from edm_tts_b200.synthetic import make_dac_state_dict

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    dac = DAC(make_dac_state_dict(0))
    enc = dac.encoder
    g = torch.Generator().manual_seed(2024)

    def clips(n, lo, hi):
        L = [int(x) for x in torch.randint(lo, hi + 1, (n,), generator=g)]
        return [(torch.randn(1, x, generator=g) * 0.3).clamp(-1, 1).cuda() for x in L]

    mix = clips(N_CLIPS, 48000, 320000)
    L = [a.shape[1] for a in mix]
    Lmax = max(L)
    padded = torch.stack([torch.nn.functional.pad(a, (0, Lmax - a.shape[1])) for a in mix])
    rows = []

    def case(name, fn, reps, audio):
        samples, frames = sum(x.shape[-1] for x in audio), sum(code_lengths(x.shape[-1]) for x in audio)
        ms, all_ms = timed(fn, reps)
        r = dict(case=name, ms=round(ms, 3), samples=samples, frames=frames, samples_per_s=round(samples / ms * 1e3),
                 frames_per_s=round(frames / ms * 1e3), runs_ms=[round(x, 3) for x in all_ms])
        print(json.dumps(r), flush=True)
        rows.append(r)
        return r

    a = case("a_encode_to_codes_batch", lambda: dac.encode_to_codes_batch(mix), 7, mix)
    b = case("b_encode_to_codes_loop", lambda: [dac.encode_to_codes(x[None]) for x in mix], 3, mix)
    c = case("c_encode_to_codes_padded", lambda: dac.encode_to_codes(padded), 7, mix)
    c["padded_row_fraction"] = round(1 - sum(L) / (N_CLIPS * Lmax), 3)
    del padded
    rect = (torch.randn(32, 1, 960160, device="cuda", generator=torch.Generator(device="cuda").manual_seed(5)) * 0.3).clamp(-1, 1)
    rect_l = list(rect)
    d_rect = case("d_rect_32x960160/encode_to_codes", lambda: dac.encode_to_codes(rect), 5, rect_l)
    d_batch = case("d_rect_32x960160/encode_to_codes_batch", lambda: dac.encode_to_codes_batch(rect_l), 5, rect_l)
    del rect, rect_l

    # (e) the gap clears inside (a): every edm_dac_zero_rows launch bracketed by events (a run of its own)
    ev = []
    plain = enc._zero_rows

    def bracketed(*args):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        plain(*args)
        e.record()
        ev.append((s, e))

    enc._zero_rows = bracketed
    dac.encode_to_codes_batch(mix)
    torch.cuda.synchronize()
    del enc._zero_rows
    zero_ms = sum(s.elapsed_time(e) for s, e in ev)
    e_res = dict(case="e_zero_rows_in_a", launches=len(ev), ms=round(zero_ms, 4), share_of_a=round(zero_ms / a["ms"], 4))
    print(json.dumps(e_res), flush=True)

    # (f) prompt-sized clips
    prompts = clips(N_PROMPTS, 8000, 48000)
    f_batch = case("f_prompts/encode_to_codes_batch", lambda: dac.encode_to_codes_batch(prompts), 7, prompts)
    f_loop = case("f_prompts/encode_to_codes_loop", lambda: [dac.encode_to_codes(x[None]) for x in prompts], 3, prompts)

    summary = dict(loop_over_batch=round(b["ms"] / a["ms"], 2), padded_over_batch=round(c["ms"] / a["ms"], 2),
                   padded_row_fraction=c["padded_row_fraction"], a_rate_over_d_rect_rate=round(a["samples_per_s"] / d_rect["samples_per_s"], 3),
                   d_batch_rate_over_d_rect_rate=round(d_batch["samples_per_s"] / d_rect["samples_per_s"], 3),
                   zero_rows_share_of_a=e_res["share_of_a"], prompts_loop_over_batch=round(f_loop["ms"] / f_batch["ms"], 2))
    print(json.dumps(dict(case="summary", **summary)), flush=True)
    res = dict(gpu=smi, clips=N_CLIPS, L_range=[48000, 320000], prompts=N_PROMPTS, prompt_L_range=[8000, 48000],
               dac=dict(encoder_dim=64, rates=[2, 4, 5, 8], n_codebooks=12, weights="synthetic"), cases=rows, e_zero_rows=e_res, summary=summary)
    if out_path:
        with open(out_path, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
