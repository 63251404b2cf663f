"""S2A decode throughput on B200: decoded codec frames/s for BASELINE.json's config 2 (B=64 x 10 s = 500 frames, full
8-step first-level schedule + full pass, bf16 tensor cores) per GPU, weak-scaled over N GPUs (one process per GPU, batch-sharded
through edm_tts_b200.runner.ShardedDecoder: no collective on the decode path, the int16 codes are all-gathered once per step over
NCCL). Also in the line: the same global batch 512 split over the N GPUs (BASELINE config 3, `fixed_global_batch`), the eager-torch
bf16-autocast incumbent on the same GPU (`gpu_incumbent`), single-utterance latency, and the secondary kernels.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Prints ONE JSON line (rank 0). See DESIGN.md "Measurement" for the definition of every field. --dump-outputs DIR writes the codes the
last timed step returned to DIR/s2a_codes.npy (float32 [N*64, 12, 500]; [1, 12, 500] with --impl reference); the inputs are seeded,
so two builds run with the same arguments can be compared output for output. bench_outputs/<name> inside the tree is ignored by git.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # no __pycache__ in the tree the benchmark runs from, which may be read-only

B_PER_GPU, T_FRAMES, P_PROMPT, DECODE_STEPS = 64, 500, 0, 8
WORKLOAD = "S2A decode: batch 64 x 10 s (500 frames) per GPU, 8 first-level steps + full pass, no prompt (BASELINE config 2)"
METRIC, UNIT = "s2a_decoded_codec_frames_per_s", "frames/s"


def bench_config(world):
    """The workload both arms are quoted on (BASELINE config 2). The reference arm times a bounded sample of it (cpu_baseline.sample)."""
    return {"workload": WORKLOAD, "batch_per_gpu": B_PER_GPU, "frames": T_FRAMES, "prompt_frames": P_PROMPT, "decode_steps": DECODE_STEPS,
            "weights": "random-init, reference architecture (configs/injection_conformer/base_config)",
            "sampling_noise": "synthetic Gumbel noise: in-kernel Philox in the GPU arm, pre-generated tensors in the reference arm", "l2": "working set 3.5 GB per step >> 126 MB L2 (no flush needed)",
            "parallelism": f"batch-sharded x{world} (runner.ShardedDecoder), one all_gather of the int16 codes per step" if world > 1 else "single GPU"}


def flops_per_frame(S, T):
    """SURVEY.md section 8d: algorithmic FLOPs per target frame with no prompt."""
    return (S * (276.82e6 + 20480.0 * T) if S > 1 else 0.0) + 922.75e6 + 65536.0 * T


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons during the timed region (NVML)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.reasons, self.max_mhz = index, False, [], set(), None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {
                getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
                getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
                getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
            }
            while not self.stop_flag:
                self.sm.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(0.05)
        except Exception as e:  # NVML missing: report that instead of fabricating clocks
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    def result(self):
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return p.get("bf16_tflops_sustained", 1406.7), p.get("hbm_gbs", 6460.2), "measured"
    return 1400.0, 6650.0, "fallback"


def ncu_traffic():
    """DRAM bytes per GEMM launch from the committed ncu --set full capture of this same command (tools/gpu_ncu_bench.sh ->
    tools/ncu_traffic.py -> profiles/ncu_traffic_r02.json); None when the file is missing."""
    path = next((q for q in (os.path.join(ROOT, "profiles", f"ncu_traffic_r0{r}.json") for r in (2, 1)) if os.path.exists(q)), None)
    if path is None:
        return None, None
    with open(path) as f:
        t = json.load(f)
    e = t.get("gemm_bf16_tn_pair_kernel (all captured epilogues)")
    return (e["traffic_bytes_per_launch"], os.path.relpath(path, ROOT)) if e else (None, None)


def cpu_oracle_fps(B, T, steps, repeats, threads):
    """Times the oracle (CPU restatement of the reference, fp32) on the host cores."""
    import torch

    from oracle import s2a as os2a
    from oracle.weights import OracleConfig, make_inputs, make_state_dict

    torch.set_num_threads(threads)
    cfg = OracleConfig()
    sd = make_state_dict(cfg, 0)
    inp = make_inputs(B, T, 0, steps, cfg, seed=1234)
    times = []
    with torch.inference_mode():
        for i in range(repeats + 1):
            t0 = time.perf_counter()
            os2a.infer_special(sd, cfg, inp["semantic_tokens"], None, None, steps=steps, cat_gumbel=inp["cat_gumbel"],
                               remask_gumbel=inp["remask_gumbel"], mode="fp32")
            times.append(time.perf_counter() - t0)
    best = min(times[1:]) if repeats > 0 else times[0]
    return B * T / best, times


def gpu_incumbent_fps(dev, B, T, steps):
    """What a user gets on this GPU without this repo: the reference's algorithm as eager torch ops under autocast(bf16), fp32
    parameters (inference.py:33 runs the reference exactly so). The oracle restates that op sequence with torch library kernels
    (F.linear, F.layer_norm, SDPA, conv1d), so it serves as the incumbent here; one warm-up + one timed decode of the bench batch."""
    import torch

    from oracle import s2a as os2a
    from oracle.weights import OracleConfig, make_state_dict

    cfg = OracleConfig()
    sd = {k: v.to(dev) for k, v in make_state_dict(cfg, 0).items()}
    g = torch.Generator(device=dev).manual_seed(5)
    sem = torch.randint(0, cfg.num_semantic, (B, T), device=dev, generator=g)
    cat = -torch.log(torch.empty(steps - 1, B * T, cfg.codebook_size, device=dev).exponential_(generator=g))
    rem = -torch.log(-torch.log(torch.rand(steps - 1, B, T, device=dev, generator=g).clamp_(1e-7, 1 - 1e-7)))
    times = []
    with torch.inference_mode(), torch.autocast("cuda", dtype=torch.bfloat16):
        for _ in range(2):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            os2a.infer_special(sd, cfg, sem, None, None, steps=steps, cat_gumbel=cat, remask_gumbel=rem, mode="fp32")
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
    del sd, cat, rem
    torch.cuda.empty_cache()
    return B * T / (times[-1] * 1e-3), times


def dump_outputs(out_dir, arrays):
    """Writes each tensor of `arrays` as out_dir/<name>.npy in float32."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().to("cpu", torch.float32).numpy())


def run_reference(args):
    """--impl reference: the reference's algorithm on the host CPU (oracle port; the Python reference itself cannot
    travel to the GPU box), all host threads, one bounded sample per step: 1 utterance x 500 frames x 8 steps."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch

    from oracle import s2a as os2a
    from oracle.weights import OracleConfig, make_inputs, make_state_dict

    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    cfg = OracleConfig()
    sd = make_state_dict(cfg, 0)
    inp = make_inputs(1, T_FRAMES, 0, DECODE_STEPS, cfg, seed=1234)

    def step():
        with torch.inference_mode():
            return os2a.infer_special(sd, cfg, inp["semantic_tokens"], None, None, steps=DECODE_STEPS, cat_gumbel=inp["cat_gumbel"],
                                      remask_gumbel=inp["remask_gumbel"], mode="fp32")

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        codes = step()
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"s2a_codes": codes})
    fps = args.steps * T_FRAMES / dt
    sample = (f"bounded sample of the workload: 1 utterance x {T_FRAMES} frames x {DECODE_STEPS} steps per timed step (1/64 of the 64-utterance batch the "
              f"GPU arm decodes per step; the full batch takes ~70 s per step on these cores), oracle port of the reference in fp32 torch, {threads} threads")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": bench_config(args.gpus), "sample": sample,
        "cpu_baseline": {"value": fps, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the codes of the last timed step to DIR/s2a_codes.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    import __graft_entry__ as ge
    ge.build()
    from edm_tts_b200 import InjectionConformerModel, _lib
    from edm_tts_b200.config import InjectionConformerConfig
    from edm_tts_b200.synthetic import OracleConfig, make_state_dict

    lib = _lib.lib()
    cfg = OracleConfig()
    sd = make_state_dict(cfg, 0)          # random-init weights of the reference architecture (no checkpoints offline)
    model = InjectionConformerModel(InjectionConformerConfig(), sd, device=dev)
    del sd
    B, T = B_PER_GPU, T_FRAMES
    from edm_tts_b200.runner import ShardedDecoder, shard_bounds

    # the global batch (64 utterances per GPU) is known to every rank; ShardedDecoder decodes this rank's contiguous shard with the
    # Philox counters of the global rows and all-gathers the int16 codes, so every rank ends with the codes of all world * 64 rows
    GB = world * B
    sem_host = torch.randint(0, cfg.num_semantic, (GB, T), generator=torch.Generator().manual_seed(1234)).pin_memory()
    codes_host = torch.empty(GB, cfg.n_codebooks, T, dtype=torch.int16).pin_memory()
    sem_dev = sem_host.to(dev)
    SEED = 7
    sharded = ShardedDecoder(model.infer_special, keep_gather_dtype=True)
    lo, hi = shard_bounds(GB, rank, world)

    def step_resident():
        return sharded(sem_dev, None, None, steps=DECODE_STEPS, temperature=1.0, seed=SEED)

    def step_e2e():
        # this rank's shard of the tokens host -> device, decode, gather, all codes device -> host (pinned buffers on both sides)
        sd_ = torch.empty(GB, T, dtype=torch.int64, device=dev)
        sd_[lo:hi].copy_(sem_host[lo:hi], non_blocking=True)
        codes = sharded(sd_, None, None, steps=DECODE_STEPS, temperature=1.0, seed=SEED)
        codes_host.copy_(codes, non_blocking=True)
        return codes

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, k, profile=False):
        sync_all()
        if profile:
            lib.edm_prof_enable(1)
        l0 = lib.edm_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            out = fn()
        e1.record()
        sync_all()
        ms = e0.elapsed_time(e1)
        launches = lib.edm_launch_count() - l0
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item(), launches, out

    first = None
    for _ in range(args.warmup):
        first = step_resident()
    # N-GPU == 1-GPU: rank 0 decodes the whole global batch alone and compares with what the sharded run gathered
    sharded_ok = None
    if world > 1:
        if rank == 0:
            alone = model.infer_special(sem_dev, None, None, steps=DECODE_STEPS, temperature=1.0, seed=SEED)
            sharded_ok = bool(torch.equal(alone.to(torch.int16), first))
            assert sharded_ok, "sharded decode differs from the single-GPU decode of the same rows"
            del alone
        sync_all()
    del first
    sampler = ClockSampler(local)
    sampler.start()
    ms_total, launches, codes = timed(step_resident, args.steps)   # the headline: no per-kernel instrumentation inside
    # same K steps again with every GEMM / attention / LayerNorm / conv launch bracketed by CUDA events (roofline numbers);
    # the event records add a few % of gaps between kernels, so this pass is reported separately as instrumented_ms_per_step
    ms_prof, _, _ = timed(step_resident, args.steps, profile=True)
    sampler.stop_flag = True
    sampler.join()
    pm, pw, pc = (C.c_double * 5)(), (C.c_double * 5)(), (C.c_int * 5)()
    _lib.check(lib.edm_prof_collect(pm, pw, pc), "prof_collect")
    lib.edm_prof_enable(0)
    for _ in range(2):
        step_e2e()
    ms_e2e, _, _ = timed(step_e2e, args.steps)

    frames = world * B * T * args.steps
    value = frames / (ms_total * 1e-3)
    e2e = frames / (ms_e2e * 1e-3)

    # BASELINE config 3: a fixed global batch of 512 x 10 s split over the N GPUs (strong scaling), same sharded path
    FG = 512
    sem512 = torch.randint(0, cfg.num_semantic, (FG, T), generator=torch.Generator().manual_seed(4321)).to(dev)
    fixed_steps = 2

    def step_fixed():
        return sharded(sem512, None, None, steps=DECODE_STEPS, temperature=1.0, seed=SEED)

    step_fixed()
    ms_fixed, _, _ = timed(step_fixed, fixed_steps)
    del sem512

    # single-utterance latency (the reference's own call site, inference.py:43-48): B = 1, 150 frames, 8 steps, device time per decode
    lat_ms = None
    if rank == 0:
        tok1 = sem_dev[:1, :150].contiguous()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

        def lat_once():
            for _ in range(3):
                model.infer_special(tok1, None, None, steps=DECODE_STEPS, seed=SEED)
            torch.cuda.synchronize()
            l0 = lib.edm_launch_count()
            r0.record()
            for _ in range(10):
                model.infer_special(tok1, None, None, steps=DECODE_STEPS, seed=SEED)
            r1.record()
            torch.cuda.synchronize()
            return r0.elapsed_time(r1) / 10, (lib.edm_launch_count() - l0) // 10

        lat_default_ms, lat_launches = lat_once()   # default mode: a row's bits never depend on the batch it is decoded in
        model.set_low_latency(True)                 # single-utterance serving mode (split-K residual GEMMs below 512 rows)
        lat_ms, _ = lat_once()
        model.set_low_latency(False)
        # the same decode replayed from a CUDA graph (edm_tts_b200.serving.GraphedDecode, Philox noise with a per-request seed word)
        from edm_tts_b200.serving import GraphedDecode

        gd = GraphedDecode(model, 1, 150, steps=DECODE_STEPS, seed=SEED, fresh_noise=False)
        for _ in range(3):
            gd(tok1, clone=False)
        torch.cuda.synchronize()
        r0.record()
        for _ in range(10):
            gd(tok1, clone=False)
        r1.record()
        torch.cuda.synchronize()
        lat_graph_ms = r0.elapsed_time(r1) / 10
        del gd
    tf_peak, hbm_peak, peak_kind = peaks()
    traffic, traffic_src = ncu_traffic()
    # algorithmic bytes of the 8 GEMMs of one conformer block at M = B*T rows (operands read once, outputs written once,
    # the fp32 residual stream read + written by the three residual GEMMs): DESIGN.md section 4
    M = B * T
    blk_bytes = (M * 1024 * 2 + 4096 * 1024 * 2 + M * 4096 * 2) * 2 + (M * 4096 * 2 + 1024 * 4096 * 2 + M * 1024 * 8) * 2 \
        + (M * 1024 * 2 + 3072 * 1024 * 2 + M * 3072 * 2) + (M * 1024 * 2 + 1024 * 1024 * 2 + M * 1024 * 8) \
        + (M * 1024 * 2 + 4096 * 1024 * 2 + M * 2048 * 2) + (M * 2048 * 2 + 1024 * 2048 * 2 + M * 1024 * 8)
    gemm_tflops = pw[0] / (pm[0] * 1e-3) / 1e12 if pm[0] > 0 else 0.0
    kernels = {
        "gemm_tcgen05": {"launches": pc[0], "ms": pm[0], "tflops": gemm_tflops},
        "attention_tcgen05": {"launches": pc[1], "ms": pm[1], "tflops": pw[1] / (pm[1] * 1e-3) / 1e12 if pm[1] > 0 else 0.0},
        "layernorm": {"launches": pc[2], "ms": pm[2], "gbs": pw[2] / (pm[2] * 1e-3) / 1e9 if pm[2] > 0 else 0.0, "frac_hbm": pw[2] / (pm[2] * 1e-3) / 1e9 / hbm_peak if pm[2] > 0 else 0.0},
        "conv_module": {"launches": pc[3], "ms": pm[3], "gbs": pw[3] / (pm[3] * 1e-3) / 1e9 if pm[3] > 0 else 0.0, "frac_hbm": pw[3] / (pm[3] * 1e-3) / 1e9 / hbm_peak if pm[3] > 0 else 0.0},
    }
    # secondary kernel (BASELINE config 4): DAC RVQ encode of a dump_tokens batch, z [32, 1024, 3000] fp32 resident in HBM
    from edm_tts_b200 import ResidualVectorQuantize
    from edm_tts_b200.synthetic import make_quantizer_state_dict

    rvq = ResidualVectorQuantize(make_quantizer_state_dict(cfg, 0), device=dev)

    def time_rvq(zz):
        for _ in range(3):
            rvq.encode(zz)
        torch.cuda.synchronize()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0.record()
        for _ in range(10):
            rvq.encode(zz)
        r1.record()
        torch.cuda.synchronize()
        return r0.elapsed_time(r1) / 10

    zb = torch.randn(32, 1024, 3000, device=dev)
    rvq_ms_f32 = time_rvq(zb)
    zb = zb.to(torch.bfloat16)          # what the DAC encoder hands over under the reference's bf16 autocast (dump_tokens.py:213)
    rvq_ms = time_rvq(zb)
    del zb
    # the same dump_tokens batch from audio: DAC conv encoder + RVQ (SURVEY.md section 8f rank 1), 32 x 60 s segments resident in HBM
    from edm_tts_b200.dac import DAC
    from edm_tts_b200.synthetic import make_dac_state_dict

    dac = DAC(make_dac_state_dict(0), device=dev)
    audio = (torch.randn(32, 1, 960160, device=dev) * 0.3).clamp_(-1, 1)
    dac.encode_to_codes(audio)
    torch.cuda.synchronize()
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    r0.record()
    for _ in range(3):
        dac.encode_to_codes(audio)
    r1.record()
    torch.cuda.synchronize()
    enc_ms = r0.elapsed_time(r1) / 3
    # and the step after the S2A decode (inference.py:49): codes of the bench batch -> waveform through the DAC conv decoder
    dcodes = torch.randint(0, 1024, (B, 12, T), device=dev)
    dac.decode_from_codes(dcodes)
    torch.cuda.synchronize()
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    r0.record()
    for _ in range(3):
        wav = dac.decode_from_codes(dcodes)
    r1.record()
    torch.cuda.synchronize()
    dec_ms = r0.elapsed_time(r1) / 3
    dec_samples = wav.shape[-1]
    del audio, dac, wav, dcodes
    torch.cuda.empty_cache()
    # the step before the S2A decode (inference.py:38-41): text -> semantic tokens, TextToSemanticWLen.infer with the trained
    # configuration (train_config.yaml: hidden 384, 8 heads of 48, depth 12) and the script's pred_iters = 16, one utterance of 10 s
    from edm_tts_b200 import TextToSemanticWLen
    from edm_tts_b200.config import TextToSemanticWLenConfig
    from edm_tts_b200.synthetic import T2SConfig, make_t2s_state_dict

    t2s_dims = T2SConfig(hidden=384, heads=8, depth=12, lp_heads=8, lp_depth=4)
    t2s = TextToSemanticWLen(TextToSemanticWLenConfig(hidden_size=384, main_encoder_args=dict(depth=12, heads=8), length_predictor_args=dict(depth=4, heads=8)),
                             make_t2s_state_dict(t2s_dims, 0), device=dev, max_positions=1024)
    t2s_text = "The quick brown fox jumps over the lazy dog, and the dog, for once, does not mind at all."
    for _ in range(2):
        t2s.infer(t2s_text, pred_iters=16, gt_length=T, seed=1)
    torch.cuda.synchronize()
    l0 = lib.edm_launch_count()
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    r0.record()
    for _ in range(5):
        t2s.infer(t2s_text, pred_iters=16, gt_length=T, seed=1)
    r1.record()
    torch.cuda.synchronize()
    t2s_ms = r0.elapsed_time(r1) / 5
    t2s_launches = (lib.edm_launch_count() - l0) // 5
    t2s.predict_length(t2s_text)
    torch.cuda.synchronize()
    r0.record()
    for _ in range(5):
        t2s.predict_length(t2s_text)
    r1.record()
    torch.cuda.synchronize()
    t2s_len_ms = r0.elapsed_time(r1) / 5
    del t2s
    torch.cuda.empty_cache()
    t2s_inc_ms = None
    if rank == 0 and not args.no_cpu_baseline:
        # the incumbent for this step: the reference's op sequence as eager torch kernels under autocast(bf16) on the same GPU
        from oracle import t2s as ot2s
        from edm_tts_b200.synthetic import make_t2s_noise

        tsd = {k: v.to(dev) for k, v in make_t2s_state_dict(t2s_dims, 0).items()}
        tt = ot2s.text_tokens_of(t2s_text, t2s_dims, dev)
        tn = make_t2s_noise(len(t2s_text) + T + 4, 16, t2s_dims, seed=3)
        tcat, trem = tn["cat_gumbel"].to(dev), tn["remask_gumbel"].to(dev)
        ts = []
        with torch.inference_mode(), torch.autocast("cuda", dtype=torch.bfloat16):
            for _ in range(2):
                r0.record()
                ot2s.infer(tsd, t2s_dims, tt, pred_iters=16, gt_length=T, cat_gumbel=tcat, remask_gumbel=trem)
                r1.record()
                torch.cuda.synchronize()
                ts.append(r0.elapsed_time(r1))
        t2s_inc_ms = ts[-1]
        del tsd, tcat, trem
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": bench_config(world),
        "clocks": sampler.result(),
        "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": sem_host.numel() * 8, "d2h_bytes_per_step": codes_host.numel() * 2 * world,
                "ms_per_step": ms_e2e / args.steps,
                "note": "whole job: every rank copies its shard of the int64 tokens in and the gathered int16 codes of all rows out"},
        "gpu_launches": int(launches) * world,
        "sharded_equals_single_gpu": sharded_ok,
        "fixed_global_batch": {"global_batch": FG, "per_gpu": FG // world, "frames": T, "decode_steps": DECODE_STEPS, "steps_timed": fixed_steps,
                               "ms_per_step": ms_fixed / fixed_steps, "value": FG * T * fixed_steps / (ms_fixed * 1e-3), "unit": UNIT, "scaling": "strong",
                               "workload": "BASELINE config 3: S2A decode of 512 x 10 s utterances batch-sharded over the GPUs of the run"},
        "latency_b1_t150_s8_ms": lat_ms, "latency_b1_launches": lat_launches, "latency_b1_t150_s8_graph_replay_ms": lat_graph_ms,
        "latency_b1_t150_s8_default_mode_ms": lat_default_ms,
        "latency_note": "B=1 x 150 frames x 8 steps + full pass, device time per decode; *_ms and the graph replay in the model's low-latency mode (set_low_latency: split-K residual GEMMs, the mode for the reference's single-utterance call), *_default_mode_ms in the batch-invariant default",
        "roofline": {"bound": "tensor", "kernel": "gemm_bf16_tn_pair_kernel (tcgen05 cta_group::2; all conformer / head GEMMs of the timed region)",
                     "achieved": gemm_tflops, "peak": tf_peak, "unit": "TFLOP/s", "frac": gemm_tflops / tf_peak, "traffic": traffic,
                     "traffic_unit": "DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum, mean of the 8 GEMMs of one block)",
                     "traffic_source": traffic_src, "algorithmic_bytes_per_launch": blk_bytes / 8,
                     "peak_kind": f"{peak_kind} bf16 sustained", "gemm_share_of_step": pm[0] / ms_prof, "instrumented_ms_per_step": ms_prof / args.steps},
        "kernels": kernels,
        "secondary": {"metric": "dac_rvq_encode_frames_per_s", "value": 32 * 3000 / (rvq_ms * 1e-3), "unit": "frames/s", "ms": rvq_ms,
                      "workload": "DAC RVQ encode, z [32, 1024, 3000] bf16 (dump_tokens batch, BASELINE config 4), 12 codebooks, per GPU",
                      "hbm_gbs": 32 * 3000 * (2048 + 96) / (rvq_ms * 1e-3) / 1e9, "frac_hbm": 32 * 3000 * (2048 + 96) / (rvq_ms * 1e-3) / 1e9 / hbm_peak,
                      "fp32_z_ms": rvq_ms_f32, "fp32_z_frames_per_s": 32 * 3000 / (rvq_ms_f32 * 1e-3),
                      "note": "tcgen05 kind::tf32: 3xTF32 projection GEMM (z read once through MN-major TMA boxes) + 12-level search with the "
                              "[128 frames x 1024 codes] score tiles in TMEM; the search is bound by the latency of its level-serial pipeline (12 levels x score-tile round "
                              "trips + level boundary: 0.14 of its 0.24 ms remain without compare work, TMEM reads and 3 of 4 MMAs; DESIGN 7b), then by the "
                              "per-score compare work; the projection by the L2->SM fabric, not by HBM"},
        "secondary_encode": {"metric": "dac_encode_to_codes_frames_per_s", "value": 32 * 3000 / (enc_ms * 1e-3), "unit": "frames/s", "ms": enc_ms,
                             "workload": "DAC.encode_to_codes, audio [32, 1, 960160] fp32 (32 x 60 s at 16 kHz, dump_tokens batch) -> codes [32, 12, 3000], per GPU",
                             "algorithmic_tflops": 2 * 767.0e3 * 32 * 960160 / (enc_ms * 1e-3) / 1e12,
                             "frac_of_tensor_peak": 2 * 767.0e3 * 32 * 960160 / (enc_ms * 1e-3) / 1e12 / tf_peak,
                             # activation bytes each launch must move at least once (DESIGN.md section 4a): 8164 B per audio sample
                             "algorithmic_gbs": 8164.0 * 32 * 960160 / (enc_ms * 1e-3) / 1e9, "frac_hbm": 8164.0 * 32 * 960160 / (enc_ms * 1e-3) / 1e9 / hbm_peak,
                             "note": "conv encoder = 29 implicit-GEMM launches per chunk of 8 utterances (csrc/dac_conv.cuh, bf16 operands, fp32 stream) + the RVQ kernels above; "
                                     "767 kMAC per audio sample; the 64/128-channel stages are HBM / L2 bound, the 256..1024-channel stages run at 1.1-1.3 PFLOP/s"},
        "secondary_decode": {"metric": "dac_decode_from_codes_frames_per_s", "value": B * T / (dec_ms * 1e-3), "unit": "frames/s", "ms": dec_ms,
                             "workload": f"DAC.decode_from_codes, codes [{B}, 12, {T}] (the S2A bench batch) -> audio [{B}, 1, {dec_samples}] fp32, per GPU",
                             "algorithmic_tflops": 2 * 1.74e6 * B * dec_samples / (dec_ms * 1e-3) / 1e12,
                             "frac_of_tensor_peak": 2 * 1.74e6 * B * dec_samples / (dec_ms * 1e-3) / 1e12 / tf_peak,
                             "algorithmic_gbs": 13650.0 * B * dec_samples / (dec_ms * 1e-3) / 1e9, "frac_hbm": 13650.0 * B * dec_samples / (dec_ms * 1e-3) / 1e9 / hbm_peak,
                             "note": "conv decoder on the encoder's implicit-GEMM kernels (transposed convs as 2-tap convs into a shifted output view); 1.74 MMAC per output sample"},
        "secondary_t2s": {"metric": "t2s_semantic_tokens_per_s", "value": T / (t2s_ms * 1e-3), "unit": "tokens/s", "ms_per_utterance": t2s_ms,
                          "length_predictor_ms": t2s_len_ms, "launches_per_utterance": int(t2s_launches),
                          "gpu_incumbent_ms_per_utterance": t2s_inc_ms,
                          "workload": f"TextToSemanticWLen.infer, hidden 384 / 8 heads of 48 / depth 12 (train_config.yaml), pred_iters 16 (inference.py:38), "
                                      f"{len(t2s_text)} text bytes -> {T} semantic tokens, batch 1 (the reference's infer is batch-1), in-kernel Philox noise",
                          "note": "latency-bound: ~180 dependent launches per iteration on a 600-row sequence; device time per utterance, tokens resident"},
        "model_flops_utilisation": {"algorithmic_tflops": flops_per_frame(DECODE_STEPS, T) * B * T / (ms_total / args.steps * 1e-3) / 1e12,
                                    "frac_of_peak": flops_per_frame(DECODE_STEPS, T) * B * T / (ms_total / args.steps * 1e-3) / 1e12 / tf_peak},
    }
    if not args.no_cpu_baseline:
        del model
        torch.cuda.empty_cache()
        inc_fps, inc_ms = gpu_incumbent_fps(dev, B, T, DECODE_STEPS)
        out["gpu_incumbent"] = {"value": inc_fps, "unit": UNIT, "ms_per_step": inc_ms[-1], "runs_ms": [round(t, 1) for t in inc_ms],
                                "what": "the same decode (B=64 x 500 frames x 8 steps + full pass) as eager torch library kernels under autocast(bf16) on "
                                        "this GPU: the reference's op sequence (oracle restatement), second of two runs, CUDA events"}
        threads = os.cpu_count() or 1
        fps, times = cpu_oracle_fps(1, 150, DECODE_STEPS, repeats=3, threads=threads)
        out["cpu_baseline"] = {"value": fps, "unit": UNIT, "cores": threads, "kind": "port",
                               "sample": f"oracle (fp32 torch CPU restatement of the reference) on 1 utterance x 150 frames x {DECODE_STEPS} steps "
                                         f"(BASELINE config 1), best of 3 after 1 warm-up; runs {[round(t, 2) for t in times]} s"}
        # the same port for the DAC conv stacks on a bounded sample (10 s of audio / 500 frames of latent), best of 2
        from edm_tts_b200.synthetic import make_decoder_state_dict, make_encoder_state_dict
        from oracle.dac_decoder import decoder_forward
        from oracle.dac_encoder import encoder_forward

        def best_of(fn, n=2):
            ts = []
            for _ in range(n + 1):
                t0 = time.perf_counter()
                fn()
                ts.append(time.perf_counter() - t0)
            return min(ts[1:])
        esd, dsd = make_encoder_state_dict(64, (2, 4, 5, 8), 0), make_decoder_state_dict(1024, 1536, (8, 5, 4, 2), 0)
        a10 = torch.randn(1, 1, 160000) * 0.3
        z10 = torch.randn(1, 1024, 500) * 0.5
        with torch.inference_mode():
            t_enc = best_of(lambda: encoder_forward(esd, a10))
            t_dec = best_of(lambda: decoder_forward(dsd, z10))
        out["secondary_encode"]["cpu_baseline"] = {"value": 500 / t_enc, "unit": "frames/s", "cores": threads, "kind": "port",
                                                   "sample": "oracle conv encoder (fp32 torch CPU) on 1 x 10 s of audio, best of 2 (RVQ not included)"}
        out["secondary_decode"]["cpu_baseline"] = {"value": 500 / t_dec, "unit": "frames/s", "cores": threads, "kind": "port",
                                                   "sample": "oracle conv decoder (fp32 torch CPU) on 1 x 500 frames of latent, best of 2"}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"s2a_codes": codes})
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
