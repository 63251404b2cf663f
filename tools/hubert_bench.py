"""HuBERT semantic tokenizer on one GPU (HubertFeatures + SemanticTokenizer, synthetic transformers-initialised hubert-large weights,
1024 random centroids), with the card name and power limit read in the same run:
  (a) the dump_tokens batch, 32 clips x 960 160 samples (60 s) -> semantic ids through encode: ms, frames/s and algorithmic TFLOP/s
      from the per-frame count below;
  (b) the incumbent: transformers HubertModel (18 layers run, the rest unused) eager under autocast(bf16) on the same clips, the way
      the reference calls it (hidden_states[18]), followed by cdist + argmax;
  (c) 64 clips with L_i uniform in 3-20 s: encode_batch vs an encode loop vs encode on the clips right-padded to the longest;
  (d) the full dump_tokens step: DAC.encode_to_codes_batch + encode_batch on the (a) clips as a list.
Each case is warmed up once and timed with CUDA events; the median of the repeats is reported. Writes JSON to argv[1]."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

SR = 16000
# algorithmic FLOP per 20 ms frame (2 per MAC): conv feature extractor, positional conv, layers 0-17 without attention, and the
# attention score / value products per frame of a sequence of N frames
CONV_FLOP = 2 * (512 * 10 * 64 + sum(512 * 512 * k * n for k, n in ((3, 32), (3, 16), (3, 8), (3, 4), (2, 2), (2, 1))))
POS_FLOP = 2 * 1024 * 64 * 128
LAYER_FLOP = 2 * (4 * 1024 * 1024 + 2 * 1024 * 4096)
ATTN_FLOP_PER_N = 4 * 1024


def flop(frames_per_clip, layers=18):
    return sum(T * (CONV_FLOP + POS_FLOP + layers * (LAYER_FLOP + ATTN_FLOP_PER_N * T)) for T in frames_per_clip)


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
    from transformers import HubertModel

    from edm_tts_b200 import HubertFeatures, SemanticTokenizer
    from edm_tts_b200.dac import DAC
    from edm_tts_b200.hubert import frame_count
    from edm_tts_b200.synthetic import hubert_config, make_dac_state_dict, make_hubert_state_dict

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    cfg = hubert_config()
    sd = make_hubert_state_dict(0, cfg)
    hub = HubertFeatures(cfg, sd, device="cuda")
    g = torch.Generator().manual_seed(2024)
    centers = torch.randn(1024, 1024, generator=g).cuda()
    tok = SemanticTokenizer(hub, centers)
    rows = []

    def add(name, ms, frames, **kw):
        r = dict(case=name, ms=round(ms, 3), frames=frames, frames_per_s=round(frames / ms * 1e3), **kw)
        rows.append(r)
        print(json.dumps(r), flush=True)

    # (a)
    big = torch.randn(32, 960160, generator=g).clamp(-3, 3).cuda()
    T = frame_count(960160)
    ms, _ = timed(lambda: tok.encode(big), 3)
    add("a_encode_32x60s", ms, 32 * T, tflops=round(flop([T] * 32) / ms / 1e9, 1))
    # (b) incumbent: HF eager under autocast(bf16), 18 layers (hidden_states[18] needs no more)
    ref = HubertModel(hubert_config(num_hidden_layers=18)).eval()
    ref.load_state_dict({k: v for k, v in sd.items() if not any(k.startswith(f"encoder.layers.{i}.") for i in range(18, 24))})
    ref = ref.cuda()

    def hf():
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            x = (big - big.mean(-1, keepdim=True)) / torch.sqrt(big.var(-1, keepdim=True, unbiased=False) + 1e-7)
            f = ref(x, output_hidden_states=True).hidden_states[18]
            return (-torch.cdist(f.float(), centers[None].expand(32, -1, -1))).argmax(-1)

    ms_hf, _ = timed(hf, 3)
    add("b_hf_eager_autocast_32x60s", ms_hf, 32 * T, tflops=round(flop([T] * 32) / ms_hf / 1e9, 1), speedup_a=round(ms_hf / ms, 2))
    del ref
    torch.cuda.empty_cache()
    # (c)
    L = [int(x) for x in torch.randint(3 * SR, 20 * SR + 1, (64,), generator=g)]
    mix = [torch.randn(n, generator=g).cuda() for n in L]
    frames = sum(frame_count(n) for n in L)
    ms_b, _ = timed(lambda: tok.encode_batch(mix), 5)
    add("c_encode_batch_64x3-20s", ms_b, frames, tflops=round(flop([frame_count(n) for n in L]) / ms_b / 1e9, 1))
    ms_l, _ = timed(lambda: [tok.encode(a[None]) for a in mix], 3)
    add("c_encode_loop_64x3-20s", ms_l, frames, vs_batch=round(ms_l / ms_b, 2))
    Lmax = max(L)
    padded = torch.stack([torch.nn.functional.pad(a, (0, Lmax - a.shape[0])) for a in mix])
    ms_p, _ = timed(lambda: tok.encode(padded), 3)
    add("c_encode_padded_64x3-20s", ms_p, frames, vs_batch=round(ms_p / ms_b, 2), padding_frac=round(1 - sum(L) / (64 * Lmax), 3))
    del padded
    # (d)
    dac = DAC(make_dac_state_dict(0))
    clips = [a for a in big]
    step = lambda: (dac.encode_to_codes_batch([a[None] for a in clips]), tok.encode_batch(clips))
    ms_d, _ = timed(step, 3)
    ms_dac, _ = timed(lambda: dac.encode_to_codes_batch([a[None] for a in clips]), 3)
    add("d_dump_tokens_step_32x60s", ms_d, 32 * T, dac_ms=round(ms_dac, 3))
    res = dict(card=smi, note="synthetic weights; (b) runs 18 of 24 layers, all that hidden_states[18] needs", cases=rows)
    if out_path:
        os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
        with open(out_path, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
