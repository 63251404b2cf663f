"""A/B CUDA-event timing of the sampling and re-masking kernels of two builds of the library, alternated in one process:
edm_sample with in-kernel Philox noise over 32 000 rows (B=64 x 500 frames of 1024 logits) and edm_remask with Philox noise at
B=64 x T=500, the shapes of one first-level decode step. The 131 MB of logits are about the size of the 126 MB L2, so back-to-back
calls may find part of them there, for both builds alike.

    python tools/ab_sampling.py path/to/base.so path/to/new.so [--reps 5] [--iters 200]

Prints one JSON line: the card's name and power limit, and per library the median over repetitions of the mean time per call."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from edm_tts_b200 import _lib as L  # noqa: E402


def load(path):
    h = C.CDLL(os.path.abspath(path))
    for name in ("edm_sample", "edm_remask", "edm_last_error"):
        res, args = L._SIGNATURES[name]
        getattr(h, name).restype, getattr(h, name).argtypes = res, args
    return h


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("libs", nargs=2)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--iters", type=int, default=200)
    a = ap.parse_args()
    libs = {p: load(p) for p in a.libs}
    B, T = 64, 500
    gen = torch.Generator(device="cuda").manual_seed(0)
    logits = torch.randn(B * T, 1024, device="cuda", generator=gen) * 3
    ids = torch.empty(B, T, device="cuda", dtype=torch.int32)
    logp = torch.randn(B, T, device="cuda", generator=gen).abs().neg()
    mo = (torch.rand(B, T, device="cuda", generator=gen) < 0.7).to(torch.uint8)
    mn = torch.empty_like(mo)
    st = L.stream_ptr()

    def check(h, rc):
        if rc != 0:
            raise RuntimeError(h.edm_last_error().decode())

    ops = {
        "sample_philox_32000_rows": lambda h, i: check(h, h.edm_sample(L.ptr(logits), 1024, B * T, None, 1, 7, i, None, L.ptr(ids), L.ptr(logp), T, 1, 1, 0, st)),
        "remask_philox_64x500": lambda h, i: check(h, h.edm_remask(L.ptr(logp), None, L.ptr(mo), L.ptr(mn), None, B, T, 0.55, 0.55, 7, i, st)),
    }
    times = {op: {k: [] for k in libs} for op in ops}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for op, fn in ops.items():
        for h in libs.values():
            for i in range(20):
                fn(h, i)
        for _ in range(a.reps):
            for k, h in libs.items():
                torch.cuda.synchronize()
                ev0.record()
                for i in range(a.iters):
                    fn(h, i)
                ev1.record()
                torch.cuda.synchronize()
                times[op][k].append(ev0.elapsed_time(ev1) * 1e3 / a.iters)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    print(json.dumps({"gpu": smi, "iters": a.iters, "reps": a.reps,
                      "us_per_call_median": {op: {k: round(statistics.median(v), 3) for k, v in t.items()} for op, t in times.items()},
                      "us_per_call_all": {op: {k: [round(x, 3) for x in v] for k, v in t.items()} for op, t in times.items()}}))


if __name__ == "__main__":
    main()
