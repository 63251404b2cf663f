"""Batched text-to-semantic decode on one GPU: ms per chunk, semantic tokens/s and ms per utterance for a fixed seeded mix of 64
texts of 40-200 bytes with gt_lengths uniform in [150, 500], 16 iterations, on the bench's T2S model (hidden 384, depth 12, lp_depth
4, 8 heads, max_positions 1024, synthetic weights; random-init predicted lengths are meaningless, so the decode uses gt_lengths):
  (a) infer_batch on the mix; (b) infer per utterance in a loop, default (low-latency) mode; (c) the same loop with split-K off;
  (d) predict_length_batch next to a predict_length loop; (e) S2A infer_batch (8 steps) on the tokens of (a), so that one report
  holds both stages from text to codes. Also the GEMM / attention share of (a) from the library's per-launch event hooks, in a run
  of its own. Prints one JSON line per case and writes them, with the card name and power limit read in the same run, to the file
  given as the first argument."""
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

ITERS, N_UTT, S2A_STEPS = 16, 64, 8


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
    from edm_tts_b200 import InjectionConformerModel, TextToSemanticWLen, _lib
    from edm_tts_b200.config import InjectionConformerConfig, TextToSemanticWLenConfig
    from edm_tts_b200.synthetic import OracleConfig, T2SConfig, make_state_dict, make_t2s_state_dict

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    dims = T2SConfig(hidden=384, heads=8, depth=12, lp_heads=8, lp_depth=4)
    t2s = TextToSemanticWLen(TextToSemanticWLenConfig(hidden_size=384, main_encoder_args=dict(depth=12, heads=8), length_predictor_args=dict(depth=4, heads=8)),
                             make_t2s_state_dict(dims, 0), device="cuda", max_positions=1024)
    g = torch.Generator().manual_seed(2024)
    alphabet = "abcdefghijklmnopqrstuvwxyz ABCDEFGHIJKLMNOPQRSTUVWXYZ,.'"
    n_bytes = [int(x) for x in torch.randint(40, 201, (N_UTT,), generator=g)]
    texts = ["".join(alphabet[int(i)] for i in torch.randint(0, len(alphabet), (n,), generator=g)) for n in n_bytes]
    lengths = [int(x) for x in torch.randint(150, 501, (N_UTT,), generator=g)]
    tokens = sum(lengths)
    rows_total = sum(n + ln + 4 for n, ln in zip(n_bytes, lengths))
    results = []

    def case(name, fn, reps, n_tokens=tokens, **kw):
        ms, all_ms = timed(fn, reps)
        r = dict(case=name, ms_per_chunk=round(ms, 3), ms_per_utterance=round(ms / N_UTT, 4), semantic_tokens=n_tokens,
                 semantic_tokens_per_s=round(n_tokens / ms * 1e3), runs_ms=[round(x, 3) for x in all_ms], **kw)
        print(json.dumps(r), flush=True)
        results.append(r)
        return r

    a = case("a_infer_batch", lambda: t2s.infer_batch(texts, pred_iters=ITERS, gt_lengths=lengths, seed=1), 5, rows=rows_total)

    def loop():
        for i in range(N_UTT):
            t2s.infer(texts[i], pred_iters=ITERS, gt_length=lengths[i], seed=1, batch_offset=i)

    b = case("b_infer_loop_default", loop, 2)
    t2s.set_low_latency(False)
    c = case("c_infer_loop_unsplit", loop, 2)
    t2s.set_low_latency(True)
    d = case("d_predict_length_batch", lambda: t2s.predict_length_batch(texts), 5, n_tokens=0, text_bytes=sum(n_bytes))
    d_loop = case("d_predict_length_loop", lambda: [t2s.predict_length(t) for t in texts], 2, n_tokens=0, text_bytes=sum(n_bytes))

    # where the time of (a) goes: GEMM / attention launches bracketed by events (a run of its own, the hooks slow the host)
    lib = _lib.lib()
    lib.edm_prof_enable(1)
    t2s.infer_batch(texts, pred_iters=ITERS, gt_lengths=lengths, seed=1)
    torch.cuda.synchronize()
    pm, pw, pc = (C.c_double * 5)(), (C.c_double * 5)(), (C.c_int * 5)()
    _lib.check(lib.edm_prof_collect(pm, pw, pc), "prof_collect")
    lib.edm_prof_enable(0)
    breakdown = {k: dict(ms=round(pm[i], 3), launches=pc[i], tflop_per_s=round(pw[i] / (pm[i] * 1e-3) / 1e12, 1) if pm[i] > 0 and i < 2 else None)
                 for i, k in enumerate(["gemm", "attention"])}
    breakdown["note"] = "event-bracketed launches of one infer_batch call; the other kernels (LayerNorm, conv, sampling, re-masking) are not bracketed"
    print(json.dumps(dict(case="a_breakdown", **breakdown)), flush=True)

    # (e) the second stage on the tokens of (a)
    s2a = InjectionConformerModel(InjectionConformerConfig(), make_state_dict(OracleConfig(), 0), device="cuda")
    sem = [t.clone() for t in t2s.infer_batch(texts, pred_iters=ITERS, gt_lengths=lengths, seed=1)]
    e = case("e_s2a_infer_batch", lambda: s2a.infer_batch(sem, steps=S2A_STEPS, seed=1), 5, s2a_steps=S2A_STEPS)

    summary = dict(batch_vs_loop_default=round(b["ms_per_chunk"] / a["ms_per_chunk"], 2), batch_vs_loop_unsplit=round(c["ms_per_chunk"] / a["ms_per_chunk"], 2),
                   predict_batch_vs_loop=round(d_loop["ms_per_chunk"] / d["ms_per_chunk"], 2),
                   text_to_codes_ms_per_utterance=round((a["ms_per_chunk"] + e["ms_per_chunk"]) / N_UTT, 3),
                   t2s_share_of_text_to_codes=round(a["ms_per_chunk"] / (a["ms_per_chunk"] + e["ms_per_chunk"]), 3))
    print(json.dumps(dict(case="summary", **summary)), flush=True)
    res = dict(gpu=smi, iters=ITERS, utterances=N_UTT, text_bytes_range=[40, 200], length_range=[150, 500], rows=rows_total,
               model=dict(hidden=384, depth=12, lp_depth=4, heads=8, max_positions=1024, weights="synthetic"), cases=results,
               a_breakdown=breakdown, summary=summary)
    if out_path:
        with open(out_path, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
