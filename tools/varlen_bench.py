"""Variable-length S2A decode on one GPU: ms per batch and decoded frames/s (sum of T_i) for
  (a) infer_batch on the packed mix, (b) infer_special per utterance in a loop, (c) infer_special on the mix padded to max T_i
  (wrong tokens: the compute reference of "pad to the longest"), for a fixed seeded mix of 64 utterances with T_i uniform in
  [150, 1000], without prompts and with P_i uniform in [50, 150]; and the rectangular bench shape 64 x 500 through infer_batch
  next to infer_special. 8 steps, synthetic weights of the reference architecture. Prints one JSON line per case and writes
  them, with the card name and power limit read in the same run, to the file given as the first argument."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

STEPS, N_UTT = 8, 64


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
    from edm_tts_b200 import InjectionConformerModel
    from edm_tts_b200.config import InjectionConformerConfig
    from edm_tts_b200.synthetic import OracleConfig, make_state_dict

    cfg = OracleConfig()
    model = InjectionConformerModel(InjectionConformerConfig(), make_state_dict(cfg, 0), device="cuda")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    g = torch.Generator().manual_seed(2024)
    T = [int(x) for x in torch.randint(150, 1001, (N_UTT,), generator=g)]
    P = [int(x) for x in torch.randint(50, 151, (N_UTT,), generator=g)]
    sem = [torch.randint(0, cfg.num_semantic, (t,), generator=g).cuda() for t in T]
    ap = [torch.randint(0, cfg.codebook_size, (4, p), generator=g).cuda() for p in P]
    sp = [torch.randint(0, cfg.num_semantic, (p,), generator=g).cuda() for p in P]
    tmax, pmax = max(T), max(P)
    sem_pad = torch.stack([torch.nn.functional.pad(s, (0, tmax - s.shape[0])) for s in sem])
    ap_pad = torch.stack([torch.nn.functional.pad(a, (0, pmax - a.shape[1])) for a in ap])
    sp_pad = torch.stack([torch.nn.functional.pad(s, (0, pmax - s.shape[0])) for s in sp])
    frames = sum(T)
    rows = []

    def case(name, fn, reps, n_frames=frames, **kw):
        ms, all_ms = timed(fn, reps)
        r = dict(case=name, ms_per_batch=round(ms, 3), frames=n_frames, frames_per_s=round(n_frames / ms * 1e3), runs_ms=[round(x, 3) for x in all_ms], **kw)
        print(json.dumps(r), flush=True)
        rows.append(r)

    for prompts in (False, True):
        tag = "prompt" if prompts else "no_prompt"
        pk = dict(sum_n=frames + (sum(P) if prompts else 0))
        a = (ap, sp) if prompts else (None, None)
        case(f"{tag}/a_infer_batch", lambda: model.infer_batch(sem, *a, steps=STEPS, seed=1), 5, **pk)
        def loop():
            for i in range(N_UTT):
                if prompts:
                    model.infer_special(sem[i][None], ap[i][None], sp[i][None], steps=STEPS, seed=1, batch_offset=i)
                else:
                    model.infer_special(sem[i][None], steps=STEPS, seed=1, batch_offset=i)
        case(f"{tag}/b_infer_special_loop", loop, 2, **pk)
        ap_ = (ap_pad, sp_pad) if prompts else (None, None)
        case(f"{tag}/c_infer_special_padded", lambda: model.infer_special(sem_pad, *ap_, steps=STEPS, seed=1), 5,
             padded_rows=N_UTT * (tmax + (pmax if prompts else 0)), **pk)
    rect = torch.randint(0, cfg.num_semantic, (64, 500), generator=g).cuda()
    rect_l = list(rect)
    case("rect_64x500/infer_batch", lambda: model.infer_batch(rect_l, steps=STEPS, seed=1), 5, n_frames=64 * 500, sum_n=64 * 500)
    case("rect_64x500/infer_special", lambda: model.infer_special(rect, steps=STEPS, seed=1), 5, n_frames=64 * 500, sum_n=64 * 500)
    res = dict(gpu=smi, steps=STEPS, utterances=N_UTT, T_range=[150, 1000], P_range=[50, 150], cases=rows)
    if out_path:
        with open(out_path, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
