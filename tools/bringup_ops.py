"""GPU bring-up for the stateless operators: each sub-test compares one kernel with a plain torch computation and prints
max errors (and a timing for the large shapes). Run one sub-test per process so a trap in one kernel cannot poison the
others:  for t in gemm attn ln conv sample remask rvqtc; do timeout 300 python tools/bringup_ops.py $t; done
The sweeps that poke descriptor fields (attn, rvqtc, rvqtime) need the bring-up entry points, which the product library does not
export: build gpurun_out/libedm_bringup.so with -DEDM_BRINGUP first (tools/gpu_ab.sh does); it is picked up when present.
"""
import math
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from edm_tts_b200 import _lib as L  # noqa: E402

_alt = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out", "libedm_bringup.so")
if os.path.exists(_alt):
    import ctypes as _C

    L.LIB_PATH = _alt
    _h = L.lib()
    _h.edm_attention_dbg.argtypes = [_C.c_void_p, _C.c_int, _C.c_int, _C.c_int, _C.c_void_p, _C.c_uint, _C.c_uint, _C.c_uint, _C.c_void_p]
    _h.edm_rvq_tc_debug.argtypes = [_C.c_uint, _C.c_uint, _C.c_int, _C.c_int]
    _h.edm_rvq_tc_debug.restype = None

dev = "cuda"


def bf(x):
    return x.to(torch.bfloat16)


def rb(x):
    return x.to(torch.bfloat16).float()


def timeit(fn, iters=10, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def rope_tables(npos):
    inv = 1.0 / (10000 ** (torch.arange(0, 64, 2, device=dev).float() / 64))
    t = torch.arange(npos, device=dev).float()
    f = torch.einsum("i,j->ij", t, inv)
    return f.cos().contiguous(), f.sin().contiguous()


def gemm_call(a, b, epi, bias=None, out=None, scale=1.0, cos=None, sin=None, seq_len=1, rope_cols=0):
    M, K = a.shape
    N = b.shape[0]
    L.check(L.lib().edm_gemm_bf16(L.ptr(a), K, L.ptr(b), K, M, N, K, epi, L.ptr(bias), L.ptr(out), out.shape[1], scale,
                                  L.ptr(cos), L.ptr(sin), seq_len, rope_cols, L.stream_ptr()), "gemm")


def test_gemm():
    torch.manual_seed(0)
    for (M, N, K) in [(128, 256, 64), (128, 256, 256), (300, 512, 1024), (1000, 1024, 4096)]:
        a = bf(torch.randn(M, K, device=dev))
        b = bf(torch.randn(N, K, device=dev) / math.sqrt(K))
        bias = torch.randn(N, device=dev)
        acc = a.float() @ b.float().T
        # F32
        out = torch.empty(M, N, device=dev)
        gemm_call(a, b, L.EPI_F32, bias, out)
        torch.cuda.synchronize()
        err = (out - (acc + bias)).abs().max().item()
        print(f"gemm F32   M={M} N={N} K={K} max_abs_err={err:.3e}", flush=True)
        # BF16
        outb = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
        gemm_call(a, b, L.EPI_BF16, bias, outb)
        err = (outb.float() - rb(acc + bias)).abs().max().item()
        print(f"gemm BF16  max_abs_err={err:.3e}", flush=True)
        # SWISH
        gemm_call(a, b, L.EPI_SWISH_BF16, bias, outb)
        h = rb(acc + bias)
        ref = rb(h * rb(torch.sigmoid(h)))
        err = (outb.float() - ref).abs().max().item()
        print(f"gemm SWISH max_abs_err={err:.3e}", flush=True)
        # GLU (columns interleaved 32 value | 32 gate)
        outg = torch.empty(M, N // 2, device=dev, dtype=torch.bfloat16)
        gemm_call(a, b, L.EPI_GLU_BF16, bias, outg)
        hb = rb(acc + bias).view(M, N // 64, 2, 32)
        refg = rb(hb[:, :, 0] * rb(torch.sigmoid(hb[:, :, 1]))).reshape(M, N // 2)
        err = (outg.float() - refg).abs().max().item()
        print(f"gemm GLU   max_abs_err={err:.3e}", flush=True)
        # RESID
        x0 = torch.randn(M, N, device=dev)
        x = x0.clone()
        gemm_call(a, b, L.EPI_RESID_F32, bias, x, scale=0.5)
        ref = x0 + 0.5 * rb(acc + bias)
        err = (x - ref).abs().max().item()
        print(f"gemm RESID max_abs_err={err:.3e}", flush=True)
        # ROPE (needs N multiple of 256; treat first half of the columns as rotary)
        seq = 77
        cos, sin = rope_tables(seq)
        rope_cols = N // 2 if (N // 2) % 256 == 0 else N
        gemm_call(a, b, L.EPI_QKV_ROPE, None, outb, cos=cos, sin=sin, seq_len=seq, rope_cols=rope_cols)
        t = rb(acc).view(M, N // 64, 64)
        pos = torch.arange(M, device=dev) % seq
        c = torch.cat([cos[pos], cos[pos]], -1)[:, None, :]
        s = torch.cat([sin[pos], sin[pos]], -1)[:, None, :]
        rot = torch.cat([-t[..., 32:], t[..., :32]], -1)
        r = (t * c + rot * s)
        ref = torch.where((torch.arange(N, device=dev) < rope_cols).view(1, N // 64, 64), r, t).reshape(M, N)
        err = (outb.float() - rb(ref)).abs().max().item()
        print(f"gemm ROPE  max_abs_err={err:.3e} (rope_cols={rope_cols})", flush=True)
    # timing at the bench shapes
    for (M, N, K, epi) in [(32000, 4096, 1024, L.EPI_GLU_BF16), (32000, 4096, 1024, L.EPI_SWISH_BF16), (32000, 1024, 4096, L.EPI_RESID_F32), (32000, 3072, 1024, L.EPI_BF16),
                           (32000, 1024, 1024, L.EPI_RESID_F32), (32000, 1024, 2048, L.EPI_RESID_F32), (32000, 1024, 1024, L.EPI_F32)]:
        a = bf(torch.randn(M, K, device=dev))
        b = bf(torch.randn(N, K, device=dev) / math.sqrt(K))
        bias = torch.randn(N, device=dev)
        out = torch.zeros(M, N // 2 if epi == L.EPI_GLU_BF16 else N, device=dev, dtype=torch.float32 if epi in (L.EPI_RESID_F32, L.EPI_F32) else torch.bfloat16)
        ms = timeit(lambda: gemm_call(a, b, epi, bias, out, scale=0.5))
        ms_ref = timeit(lambda: torch.matmul(a, b.T))
        print(f"gemm time M={M} N={N} K={K} epi={epi}: {ms:.3f} ms = {2 * M * N * K / ms / 1e9:.1f} TFLOP/s  (torch.matmul {ms_ref:.3f} ms = {2 * M * N * K / ms_ref / 1e9:.1f})", flush=True)


def attn_ref(qkv, B, N, H):
    q, k, v = qkv.float().view(B, N, 3, H, 64).permute(2, 0, 3, 1, 4)
    return torch.nn.functional.scaled_dot_product_attention(q, k, v).permute(0, 2, 1, 3).reshape(B * N, H * 64)


def test_attn():
    torch.manual_seed(0)
    variants = [(1024, 1024, 2048), (16, 1024, 2048), (1024, 1024, 256), (2048, 1024, 2048), (1024, 2048, 2048)]
    for (B, N, H) in [(1, 128, 1), (2, 150, 16), (2, 500, 16), (1, 1650, 16)]:
        qkv = bf(torch.randn(B * N, 3 * H * 64, device=dev))
        ref = attn_ref(qkv, B, N, H)
        for v in variants:
            out = torch.zeros(B * N, H * 64, device=dev, dtype=torch.bfloat16)
            L.check(L.lib().edm_attention_dbg(L.ptr(qkv), B, N, H, L.ptr(out), v[0], v[1], v[2], L.stream_ptr()), "attn")
            torch.cuda.synchronize()
            err = (out.float() - ref).abs().max().item()
            print(f"attn B={B} N={N} H={H} variant={v}: max_abs_err={err:.3e} nan={torch.isnan(out.float()).any().item()}", flush=True)
            if err < 2e-2:
                break
    B, N, H = 64, 500, 16
    qkv = bf(torch.randn(B * N, 3 * H * 64, device=dev))
    out = torch.zeros(B * N, H * 64, device=dev, dtype=torch.bfloat16)
    ms = timeit(lambda: L.check(L.lib().edm_attention(L.ptr(qkv), B, N, H, L.ptr(out), L.stream_ptr())))
    q, k, v = qkv.view(B, N, 3, H, 64).permute(2, 0, 3, 1, 4)
    ms_ref = timeit(lambda: torch.nn.functional.scaled_dot_product_attention(q, k, v))
    fl = 4 * B * H * N * N * 64
    print(f"attn time B={B} N={N}: {ms:.3f} ms = {fl / ms / 1e9:.1f} TFLOP/s (torch sdpa {ms_ref:.3f} ms)", flush=True)


def test_ln():
    torch.manual_seed(0)
    rows = 1003
    x = torch.randn(rows, 1024, device=dev) * 2 + 0.3
    w1, b1, w2, b2 = [torch.randn(1024, device=dev) for _ in range(4)]
    y = torch.empty_like(x)
    z = torch.empty(rows, 1024, device=dev, dtype=torch.bfloat16)
    L.check(L.lib().edm_layernorm(L.ptr(x), 0, rows, L.ptr(w1), L.ptr(b1), L.ptr(w2), L.ptr(b2), L.ptr(y), L.ptr(z), 1, 0, 1e-5, L.stream_ptr()))
    yr = torch.nn.functional.layer_norm(x, (1024,), w1, b1)
    zr = torch.nn.functional.layer_norm(yr, (1024,), w2, b2)
    print(f"ln y err={(y - yr).abs().max().item():.3e} z err={(z.float() - zr).abs().max().item():.3e} (|z| max {zr.abs().max().item():.2f})", flush=True)
    # compaction + bf16 input
    B, N, P = 3, 50, 7
    xb = bf(torch.randn(B * N, 1024, device=dev))
    zt = torch.empty(B * (N - P), 1024, device=dev, dtype=torch.bfloat16)
    L.check(L.lib().edm_layernorm(L.ptr(xb), 1, B * N, L.ptr(w1), L.ptr(b1), None, None, None, L.ptr(zt), N, P, 1e-5, L.stream_ptr()))
    ref = torch.nn.functional.layer_norm(xb.float(), (1024,), w1, b1).view(B, N, 1024)[:, P:].reshape(-1, 1024)
    print(f"ln compaction err={(zt.float() - ref).abs().max().item():.3e}", flush=True)
    rows = 32000
    x = torch.randn(rows, 1024, device=dev)
    z = torch.empty(rows, 1024, device=dev, dtype=torch.bfloat16)
    ms = timeit(lambda: L.lib().edm_layernorm(L.ptr(x), 0, rows, L.ptr(w1), L.ptr(b1), None, None, None, L.ptr(z), 1, 0, 1e-5, L.stream_ptr()))
    print(f"ln time rows={rows}: {ms * 1e3:.1f} us = {rows * 6144 / ms / 1e6:.0f} GB/s", flush=True)
    y = torch.empty(rows, 1024, device=dev)
    ms = timeit(lambda: L.lib().edm_layernorm(L.ptr(x), 0, rows, L.ptr(w1), L.ptr(b1), L.ptr(w2), L.ptr(b2), L.ptr(y), L.ptr(z), 1, 0, 1e-5, L.stream_ptr()))
    print(f"ln double (fp32 y + bf16 z) time rows={rows}: {ms * 1e3:.1f} us = {rows * 10240 / ms / 1e6:.0f} GB/s", flush=True)


def conv_ref(h, dw_w, dw_b, cln_w, B, N):
    """bf16-autocast-like restatement of GLU -> dwconv -> swish -> chanLN"""
    x = h.float().view(B, N, 4096)
    a, g = x[..., :2048], x[..., 2048:]
    glu = rb(a * rb(torch.sigmoid(g)))  # [B,N,2048]
    xp = torch.nn.functional.pad(glu.transpose(1, 2), (2, 2))
    y = torch.nn.functional.conv1d(xp, dw_w.view(2048, 1, 5), dw_b, groups=2048)  # [B,2048,N] fp32
    y = rb(y)
    s = rb(y * rb(torch.sigmoid(y)))
    var = rb(s.var(dim=1, unbiased=False, keepdim=True))
    mean = rb(s.mean(dim=1, keepdim=True))
    o = rb(rb(s - mean) * rb(var.clamp(min=1e-4).rsqrt())) * cln_w.view(1, 2048, 1)
    return rb(o).transpose(1, 2).reshape(B * N, 2048)


def test_conv():
    torch.manual_seed(0)
    for (B, N) in [(2, 37), (3, 150), (2, 500), (1, 1), (5, 3), (64, 500), (7, 1650)]:
        h = bf(torch.randn(B * N, 4096, device=dev))
        dw_w = rb(torch.randn(2048, 5, device=dev) * 0.4)
        dw_b = torch.randn(2048, device=dev) * 0.1
        cln_w = torch.randn(2048, device=dev)
        out = torch.empty(B * N, 2048, device=dev, dtype=torch.bfloat16)
        L.check(L.lib().edm_conv_module(L.ptr(h), 1, L.ptr(out), L.ptr(dw_w), L.ptr(dw_b), L.ptr(cln_w), B, N, L.stream_ptr()))
        ref = conv_ref(h, dw_w, dw_b, cln_w, B, N)
        d = (out.float() - ref).abs()
        print(f"conv B={B} N={N}: max_abs_err={d.max().item():.3e} mean={d.mean().item():.3e} frac>0.05={(d > 0.05).float().mean().item():.2e}", flush=True)
        # decoder path: GLU already applied (as the GEMM epilogue does) -> streaming kernel
        x = h.float().view(B * N, 4096)
        gated = bf(x[:, :2048] * rb(torch.sigmoid(x[:, 2048:])))
        out2 = torch.full_like(out, float("nan"))
        L.check(L.lib().edm_conv_module(L.ptr(gated), 0, L.ptr(out2), L.ptr(dw_w), L.ptr(dw_b), L.ptr(cln_w), B, N, L.stream_ptr()))
        d2 = (out2.float() - ref).abs()
        same = (out2 == out).float().mean().item()
        print(f"conv (gated, streaming) B={B} N={N}: max_abs_err={d2.max().item():.3e} mean={d2.mean().item():.3e} frac>0.05={(d2 > 0.05).float().mean().item():.2e} "
              f"bit-identical to the tiled kernel: {same:.6f} nan={torch.isnan(out2.float()).sum().item()}", flush=True)
    B, N = 64, 500
    h = bf(torch.randn(B * N, 4096, device=dev))
    out = torch.empty(B * N, 2048, device=dev, dtype=torch.bfloat16)
    ms = timeit(lambda: L.lib().edm_conv_module(L.ptr(h), 1, L.ptr(out), L.ptr(dw_w), L.ptr(dw_b), L.ptr(cln_w), B, N, L.stream_ptr()))
    print(f"conv time B={B} N={N}: {ms * 1e3:.1f} us = {B * N * 12288 / ms / 1e6:.0f} GB/s", flush=True)
    hg = bf(torch.randn(B * N, 2048, device=dev))
    ms = timeit(lambda: L.lib().edm_conv_module(L.ptr(hg), 0, L.ptr(out), L.ptr(dw_w), L.ptr(dw_b), L.ptr(cln_w), B, N, L.stream_ptr()))
    print(f"conv (pre-gated input) time B={B} N={N}: {ms * 1e3:.1f} us = {B * N * 8192 / ms / 1e6:.0f} GB/s", flush=True)


def test_sample():
    torch.manual_seed(0)
    B, T, Q = 3, 50, 1
    rows = B * T * Q
    logits = torch.randn(rows, 1024, device=dev) * 3
    g = -torch.log(-torch.log(torch.rand(rows, 1024, device=dev).clamp(1e-7, 1 - 1e-7)))
    ids = torch.empty(B, T, device=dev, dtype=torch.int32)
    logp = torch.empty(rows, device=dev)
    L.check(L.lib().edm_sample(L.ptr(logits), 1024, rows, L.ptr(g), 0, 0, 0, None, L.ptr(ids), L.ptr(logp), T, 1, 1, 0, L.stream_ptr()))
    ref_ids = (logits + g).argmax(-1)
    ref_lp = torch.log_softmax(logits, -1).gather(-1, ref_ids[:, None])[:, 0]
    print(f"sample noise: id mismatches={(ids.view(-1).long() != ref_ids).sum().item()} logp err={(logp - ref_lp).abs().max().item():.3e}", flush=True)
    L.check(L.lib().edm_sample(L.ptr(logits), 1024, rows, None, 0, 0, 0, None, L.ptr(ids), L.ptr(logp), T, 1, 1, 0, L.stream_ptr()))
    print(f"argmax: mismatches={(ids.view(-1).long() != logits.argmax(-1)).sum().item()}", flush=True)
    # multi-level layout [B*T, Q, 1024] -> ids [B, Q, T]
    Q = 8
    logits = torch.randn(B * T * Q, 1024, device=dev)
    ids = torch.empty(B, Q, T, device=dev, dtype=torch.int32)
    L.check(L.lib().edm_sample(L.ptr(logits), 1024, B * T * Q, None, 0, 0, 0, None, L.ptr(ids), None, T, Q, Q, 0, L.stream_ptr()))
    ref = logits.view(B, T, Q, 1024).argmax(-1).permute(0, 2, 1)
    print(f"argmax multi-level: mismatches={(ids.long() != ref).sum().item()}", flush=True)
    # philox statistics: empirical distribution of samples vs softmax
    rows = 4096
    base = torch.randn(1, 1024, device=dev) * 2
    logits = base.expand(rows, 1024).contiguous()
    ids = torch.empty(rows, device=dev, dtype=torch.int32)
    L.check(L.lib().edm_sample(L.ptr(logits), 1024, rows, None, 1, 1234, 0, None, L.ptr(ids), None, rows, 1, 1, 0, L.stream_ptr()))
    p = torch.softmax(base[0], -1)
    top = p.argmax().item()
    print(f"philox: empirical P(top)={(ids == top).float().mean().item():.4f} expected={p[top].item():.4f}", flush=True)


def test_remask():
    torch.manual_seed(0)
    B, T = 5, 500
    logp = -torch.rand(B, T, device=dev) * 5
    g = -torch.log(-torch.log(torch.rand(B, T, device=dev).clamp(1e-7, 1 - 1e-7)))
    mask_old = (torch.rand(B, T, device=dev) < 0.7)
    steps, step, temp = 8, 2, 1.0
    ratio = math.cos(math.pi / 2.0 * ((step + 1) / steps))
    mo = mask_old.to(torch.uint8).contiguous()
    mn = torch.empty_like(mo)
    L.check(L.lib().edm_remask(L.ptr(logp), L.ptr(g), L.ptr(mo), L.ptr(mn), None, B, T, float(torch.tensor(ratio, dtype=torch.float32)),
                               float(torch.tensor(temp * ratio, dtype=torch.float32)), 0, step, L.stream_ptr()))
    init = torch.full((B,), T, device=dev, dtype=torch.long)
    mask_len = torch.floor(init * ratio)
    mask_len = torch.maximum(torch.ones_like(mask_len), torch.minimum(mask_old.sum(-1) - 1, mask_len))
    sel = torch.where(mask_old, logp.exp(), torch.inf)
    conf = torch.log(sel) + (temp * ratio) * g
    srt, _ = torch.sort(conf, dim=-1)
    cut = torch.take_along_dim(srt, mask_len.long().unsqueeze(-1), dim=-1)
    ref = conf < cut
    print(f"remask mismatches={(mn.bool() != ref).sum().item()} masked={mn.sum(-1).tolist()} ref={ref.sum(-1).tolist()}", flush=True)


def test_rvqtc():
    """tcgen05 RVQ (csrc/rvq_tc.cuh): projection vs an fp64 einsum, teacher-forced and free-running codes vs the fp32 torch loop."""
    from edm_tts_b200.weights import tf32_round
    torch.manual_seed(0)
    Lv = 12
    w_in = torch.randn(Lv, 8, 1024, device=dev) / 32
    b_in = torch.randn(Lv, 8, device=dev) * 0.1
    cb = torch.randn(Lv, 1024, 8, device=dev)
    w_out = torch.randn(Lv, 1024, 8, device=dev) * 0.2
    b_out = torch.randn(Lv, 1024, device=dev) * 0.05
    cbn = torch.nn.functional.normalize(cb, dim=-1).contiguous()
    proj = torch.einsum("lcd,lkd->lkc", w_out, cb) + b_out[:, None, :]
    g = torch.einsum("idc,jkc->ijkd", w_in, proj).contiguous()
    w_all = w_in.view(96, 1024).contiguous()
    w_hi = tf32_round(w_all)
    w_lo = tf32_round(w_all - w_hi)
    x = -0.5 * cbn.pow(2).sum(-1)
    c_hi = tf32_round(cbn)
    c_lo = tf32_round(cbn - c_hi)
    x_hi = tf32_round(x)
    cbp = torch.zeros(Lv, 1024, 32, device=dev)
    cbp[..., 0:8], cbp[..., 8:16], cbp[..., 16:24] = c_hi, c_hi, c_lo
    cbp[..., 24], cbp[..., 25] = x_hi, tf32_round(x - x_hi)
    b_flat = b_in.view(96).contiguous()

    def run(z, forced=None, want_lat=False, e_given=None):
        B, _, T = z.shape
        codes = torch.empty(B, Lv, T, device=dev, dtype=torch.int64)
        e_ws = torch.full((B * T, 96), float("nan"), device=dev) if e_given is None else e_given.float().contiguous()
        lat = torch.empty(B, 96, T, device=dev) if want_lat else None
        L.check(L.lib().edm_rvq_encode_tc(L.ptr(z), 0, B, T, Lv, L.ptr(w_hi), L.ptr(w_lo), L.ptr(b_flat), L.ptr(cbp), L.ptr(g), L.ptr(e_ws),
                                          L.ptr(codes), L.ptr(forced), L.ptr(lat), L.stream_ptr()), "rvq_tc")
        torch.cuda.synchronize()
        return codes, e_ws, lat

    combos = [(4096, 512)] if len(sys.argv) < 4 else [(int(a), int(b)) for a, b in zip(sys.argv[2::2], sys.argv[3::2])]
    for (B, T) in [(1, 128), (2, 332), (2, 3000)]:
        z = torch.randn(B, 1024, T, device=dev)
        e_ref = (torch.einsum("nc,bct->btn", w_all.double(), z.double()) + b_flat.double()).reshape(B * T, 96)
        for lbo, sbo in combos:
            L.lib().edm_rvq_tc_debug(lbo, sbo, 0, 0)
            codes, e_ws, _ = run(z)
            err = (e_ws.double() - e_ref).abs().max().item()
            print(f"rvqtc B={B} T={T} lbo={lbo} sbo={sbo}: projection max err {err:.3e} (|e| max {e_ref.abs().max().item():.2f})", flush=True)
            if err > 1e-3 and T == 128:
                d = (e_ws.double() - e_ref).abs()
                print("   bias", b_flat[:4].tolist(), "out", e_ws[0, :4].tolist(), "ref", e_ref[0, :4].tolist())
                ones = run(torch.ones_like(z))[1]
                print("   z=1: out", ones[0, :4].tolist(), ones[77, :4].tolist(), "expected", (w_all.double().sum(1) + b_flat.double())[:4].tolist())
                print("   err by 32-frame block:", [f"{d[i * 32:(i + 1) * 32].max().item():.2e}" for i in range(4)])
                print("   err by frame (first 40):", [f"{v:.1e}" for v in d[:40].max(1)[0].tolist()])
                print("   err by output column group:", [f"{d[:, i * 8:(i + 1) * 8].max().item():.2e}" for i in range(12)])
                # which reference entry does each output equal? (permutation detection on row 0..3, col 0..3)
                for r in (0, 1, 5, 33):
                    for c in (0, 1, 9):
                        hit = ((e_ref - e_ws[r, c].double()).abs() < 1e-4).nonzero()
                        print(f"   out[{r},{c}]={e_ws[r, c].item():+.5f} matches ref at {hit[:4].tolist()}")
        # fp32 torch loop (vector_quantizer.py semantics) with margins
        res = z.clone()
        ref_codes, margins = [], []
        for i in range(Lv):
            e = torch.einsum("dc,bct->bdt", w_in[i], res) + b_in[i][None, :, None]
            enc = torch.nn.functional.normalize(e.permute(0, 2, 1).reshape(-1, 8))
            dist = enc.pow(2).sum(1, keepdim=True) - 2 * enc @ cbn[i].t() + cbn[i].pow(2).sum(1, keepdim=True).t()
            top2 = (-dist).topk(2, dim=1)[0]
            margins.append((top2[:, 0] - top2[:, 1]).view(B, T))
            idx = (-dist).max(1)[1].view(B, T)
            ref_codes.append(idx)
            res = res - (torch.einsum("cd,btd->bct", w_out[i], cb[i][idx]) + b_out[i][None, :, None])
        ref_codes, margins = torch.stack(ref_codes, 1).contiguous(), torch.stack(margins, 1)
        L.lib().edm_rvq_tc_debug(4096, 512, 1, 0)   # search kernel alone on exact latents
        forced, _, lat = run(z, ref_codes, True, e_given=e_ref)
        mism = forced != ref_codes
        print(f"  [search only, exact latents] teacher-forced mismatches per level {mism.sum((0, 2)).tolist()} of {B * T}; max oracle margin at a mismatch "
              f"{margins[mism].max().item() if mism.any() else 0.0:.2e}", flush=True)
        L.lib().edm_rvq_tc_debug(combos[-1][0], combos[-1][1], 0, 0)
        forced, _, lat = run(z, ref_codes, True)
        mism = forced != ref_codes
        print(f"  teacher-forced mismatches per level {mism.sum((0, 2)).tolist()} of {B * T}; max oracle margin at a mismatch "
              f"{margins[mism].max().item() if mism.any() else 0.0:.2e}", flush=True)
        free = run(z)[0]
        print(f"  free-running mismatches per level {(free != ref_codes).sum((0, 2)).tolist()}", flush=True)
    B, T = 32, 3000
    z = torch.randn(B, 1024, T, device=dev)
    codes = torch.empty(B, Lv, T, device=dev, dtype=torch.int64)
    e_ws = torch.empty(B * T, 96, device=dev)
    ms = timeit(lambda: L.lib().edm_rvq_encode_tc(L.ptr(z), 0, B, T, Lv, L.ptr(w_hi), L.ptr(w_lo), L.ptr(b_flat), L.ptr(cbp), L.ptr(g), L.ptr(e_ws),
                                                  L.ptr(codes), None, None, L.stream_ptr()), iters=10, warm=3)
    print(f"rvqtc time B={B} T={T}: {ms:.3f} ms = {B * T / ms / 1e3:.2f} Mframes/s, {B * T * 4192 / ms / 1e6:.0f} GB/s", flush=True)


def test_rvqtime():
    """Timing of the two tcgen05 RVQ kernels at BASELINE config 4 (z [32,1024,3000] fp32) through the public wrapper."""
    from edm_tts_b200 import ResidualVectorQuantize
    from edm_tts_b200.synthetic import OracleConfig, make_quantizer_state_dict
    q = ResidualVectorQuantize(make_quantizer_state_dict(OracleConfig(), 0))
    for (B, T) in [(32, 3000), (4, 3000), (1, 500)]:
        z = torch.randn(B, 1024, T, device=dev)
        L.lib().edm_rvq_tc_debug(4096, 512, 0, 0)
        ms = timeit(lambda: q.encode(z), iters=10, warm=3)
        L.lib().edm_rvq_tc_debug(4096, 512, 1, 0)
        ms_s = timeit(lambda: q.encode(z), iters=10, warm=3)
        L.lib().edm_rvq_tc_debug(4096, 512, 1, 1)
        ms_p = timeit(lambda: q.encode(z), iters=10, warm=3)
        L.lib().edm_rvq_tc_debug(4096, 512, 0, 0)
        print(f"rvq tcgen05 B={B} T={T}: total {ms:.3f} ms (search alone {ms_s:.3f} ms [no-compare floor {ms_p:.3f}], projection ~{ms - ms_s:.3f} ms) = {B * T / ms / 1e3:.1f} Mframes/s, "
              f"{B * T * 4192 / ms / 1e6:.0f} GB/s algorithmic", flush=True)
    zb = torch.randn(32, 1024, 3000, device=dev).to(torch.bfloat16)
    same = torch.equal(q.encode(zb), q.encode(zb.float()))
    ms_b = timeit(lambda: q.encode(zb), iters=10, warm=3)
    print(f"rvq tcgen05 bf16 z B=32 T=3000: {ms_b:.3f} ms = {32 * 3000 / ms_b / 1e3:.1f} Mframes/s, {32 * 3000 * 2144 / ms_b / 1e6:.0f} GB/s algorithmic; "
          f"codes identical to the fp32 copy of the same z: {same}", flush=True)
    for (B, T) in [(32, 3000), (375, 256), (94, 1024), (12, 8192)]:
        z = torch.randn(B, 1024, T, device=dev)
        L.lib().edm_rvq_tc_debug(4096, 512, 1, 1)
        ms_s = timeit(lambda: q.encode(z), iters=10, warm=3)
        for name, dbg in (("full", 0), ("no split math", 1), ("no MMA", 2), ("TMA stream only", 3)):
            L.lib().edm_rvq_tc_debug(4096, 512, dbg << 4, 1)
            ms_d = timeit(lambda: q.encode(z), iters=10, warm=3)
            print(f"   projection probe B={B} T={T} [{name}]: {ms_d - ms_s:.3f} ms = {B * T * 4096 / (ms_d - ms_s) / 1e6:.0f} GB/s", flush=True)
    z = torch.randn(32, 1024, 3000, device=dev)
    L.lib().edm_rvq_tc_debug(4096, 512, 0, 0)
    print(f"rvq mma.sync kernel B=32 T=3000: {ms_old:.3f} ms", flush=True)


def test_rvqmma():
    """Search kernel alone at config 4 with 4 / 2 / 1 MMAs per codebook chunk, with and without the compare work (timing only: fewer
    than 4 MMAs give wrong codes). Separates the tensor-pipe / TMEM-accumulate cost of the K = 32 packing from the scan."""
    from edm_tts_b200 import ResidualVectorQuantize
    from edm_tts_b200.synthetic import OracleConfig, make_quantizer_state_dict
    q = ResidualVectorQuantize(make_quantizer_state_dict(OracleConfig(), 0))
    z = torch.randn(32, 1024, 3000, device=dev)
    for n_mma in (4, 2, 1):
        for probe in (0, 1, 2):
            L.lib().edm_rvq_tc_debug(4096, 512, 1, probe | (n_mma << 4))
            ms = timeit(lambda: q.encode(z), iters=10, warm=3)
            print(f"rvq search alone, {n_mma} MMAs per chunk, {('full scan', 'TMEM loads only', 'no TMEM loads')[probe]}: {ms:.3f} ms", flush=True)
    # host cost of one call (no synchronisation): if it is close to the numbers above, those are launch-bound, not device time
    L.lib().edm_rvq_tc_debug(4096, 512, 1, 2 | (1 << 4))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(20):
        q.encode(z)
    host_ms = (time.perf_counter() - t0) / 20 * 1e3
    torch.cuda.synchronize()
    # the same probe replayed from a CUDA graph of 10 calls: device time without any host in the loop
    res = {}
    for probe, n_mma in ((0, 4), (1, 4), (2, 4), (2, 1), (8, 4), (10, 1)):
        L.lib().edm_rvq_tc_debug(4096, 512, 1, probe | (n_mma << 4))
        s_ = torch.cuda.Stream()
        with torch.cuda.stream(s_):
            q.encode(z)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s_):
            for _ in range(10):
                q.encode(z)
        res[(probe, n_mma)] = timeit(g.replay, iters=5, warm=2) / 10
    print(f"host time per q.encode call {host_ms:.3f} ms; graph-replayed device time per call: full scan {res[(0, 4)]:.3f} ms, TMEM loads only "
          f"{res[(1, 4)]:.3f}, no TMEM loads {res[(2, 4)]:.3f}, no loads + 1 MMA per chunk {res[(2, 1)]:.3f}; one CTA per SM: full scan "
          f"{res[(8, 4)]:.3f}, no loads + 1 MMA {res[(10, 1)]:.3f}", flush=True)
    L.lib().edm_rvq_tc_debug(4096, 512, 0, 0)


def test_gemmsus():
    """Sustained (power-capped) throughput of single GEMM shapes run back to back for ~2 s each, ours vs torch.matmul (cuBLAS),
    with the SM clock sampled through NVML: separates 'kernel efficiency per clock' from 'energy per FLOP at the 1 kW cap'."""
    import pynvml as nv
    nv.nvmlInit()
    h = nv.nvmlDeviceGetHandleByIndex(0)
    torch.manual_seed(0)
    M = 32000
    shapes = [(4096, 1024, L.EPI_SWISH_BF16), (1024, 4096, L.EPI_RESID_F32), (4096, 1024, L.EPI_GLU_BF16), (3072, 1024, L.EPI_BF16)]
    only = sys.argv[2] if len(sys.argv) > 2 else "both"
    for (N, K, epi) in shapes:
        a = bf(torch.randn(M, K, device=dev))
        b = bf(torch.randn(N, K, device=dev) / math.sqrt(K))
        bias = torch.randn(N, device=dev)
        out = torch.zeros(M, N // 2 if epi == L.EPI_GLU_BF16 else N, device=dev, dtype=torch.float32 if epi == L.EPI_RESID_F32 else torch.bfloat16)
        fns = {"ours": lambda: gemm_call(a, b, epi, bias, out, scale=0.5), "cublas": lambda: torch.matmul(a, b.T)}
        for name, fn in fns.items():
            if only not in ("both", name):
                continue
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            clocks, power = [], []
            t_end = time.time() + 2.0
            iters_done, e_mid, n_mid = 0, None, 0
            e0 = torch.cuda.Event(enable_timing=True)
            e1 = torch.cuda.Event(enable_timing=True)
            while time.time() < t_end:
                if e_mid is None and time.time() > t_end - 1.0:   # time only the second half (clocks have settled)
                    e0.record()
                    e_mid, n_mid = True, iters_done
                for _ in range(50):
                    fn()
                iters_done += 50
                torch.cuda.synchronize()
                clocks.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                power.append(nv.nvmlDeviceGetPowerUsage(h) / 1000.0)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / max(1, iters_done - n_mid)
            tail = clocks[len(clocks) // 2:]
            print(f"sustained {name:6s} N={N} K={K} epi={epi}: {2 * M * N * K / ms / 1e9:7.1f} TFLOP/s, {ms * 1e3:.1f} us, SM clock ~{sorted(tail)[len(tail) // 2]} MHz, "
                  f"power ~{sorted(power)[len(power) // 2]:.0f} W", flush=True)


def test_kmeans():
    """k-means assignment (csrc/kmeans.cuh) at the dump_tokens scale: 96 000 frames x 1024 dims vs 1024 centroids."""
    from edm_tts_b200.kmeans import KMeansAssigner
    torch.manual_seed(0)
    centers = torch.randn(1024, 1024, device=dev)
    a = KMeansAssigner(centers)
    for n in (96000, 12000, 1500):
        x = centers[torch.randint(0, 1024, (n,), device=dev)] + 0.7 * torch.randn(n, 1024, device=dev)
        ids = a(x)
        ref = (-torch.cdist(x[None], centers[None]))[0].argmax(-1)
        ms = timeit(lambda: a(x), iters=10, warm=3)
        ms_ref = timeit(lambda: (-torch.cdist(x[None], centers[None]))[0].argmax(-1), iters=5, warm=2)
        fl = 2.0 * n * 1024 * 1024
        print(f"kmeans n={n}: {ms:.3f} ms = {n / ms / 1e3:.1f} Mframes/s, {3 * fl / ms / 1e9:.0f} TFLOP/s tf32 (3xTF32), {fl / ms / 1e9:.0f} algorithmic; "
              f"torch cdist+argmax {ms_ref:.3f} ms; mismatches vs torch fp32 {(ids != ref).sum().item()}", flush=True)


def test_dacenc():
    """DAC conv encoder at the dump_tokens shape (60 s segments -> L = 960160, T = 3000): whole-encoder time, per-conv times and
    the same stack in plain torch (bf16 autocast, channels-first F.conv1d) as the GPU incumbent."""
    import math
    import torch.nn.functional as F
    from edm_tts_b200.dac_encoder import DACEncoder
    from edm_tts_b200.dac_stack import _fold
    from edm_tts_b200.synthetic import make_encoder_state_dict
    B, Ls = int(os.environ.get("DAC_B", "8")), int(os.environ.get("DAC_L", "960160"))
    sd = make_encoder_state_dict(64, (2, 4, 5, 8), 0)
    enc = DACEncoder(sd, 64)
    audio = (torch.randn(B, 1, Ls, device=dev) * 0.3).clamp(-1, 1)
    z = enc(audio)
    torch.cuda.synchronize()
    ms = timeit(lambda: enc(audio), iters=3, warm=1)
    flop = 2.0 * 767.0e3 * B * Ls
    print(f"dac encoder B={B} L={Ls}: {ms:.2f} ms = {B * z.shape[-1] / ms / 1e3:.2f} Mframes/s, {flop / ms / 1e9:.0f} TFLOP/s algorithmic", flush=True)
    # per-launch times
    times = []
    orig = enc._conv

    def timed(a, a_rows, a_cols, a_bs, w, bias, taps, step, off, rows_out, Bc, **kw):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        orig(a, a_rows, a_cols, a_bs, w, bias, taps, step, off, rows_out, Bc, **kw)
        e1.record()
        times.append((f"cin={a_cols} cout={w.shape[0]} taps={taps} step={step} rows={rows_out}", 2.0 * Bc * rows_out * w.shape[0] * w.shape[1], e0, e1))
    orig_ru = enc._resunit

    def timed_ru(a_ptr, a_bs, Bc, rows, c, dilation, *a):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        orig_ru(a_ptr, a_bs, Bc, rows, c, dilation, *a)
        e1.record()
        times.append((f"fused unit c={c} dilation={dilation} rows={rows}", 2.0 * Bc * rows * c * c * 8, e0, e1))
    enc._conv, enc._resunit = timed, timed_ru
    enc(audio)
    torch.cuda.synchronize()
    enc._conv, enc._resunit = orig, orig_ru
    tot = 0.0
    for name, fl, e0, e1 in times:
        t = e0.elapsed_time(e1)
        tot += t
        print(f"  {name:58s} {t:8.3f} ms  {fl / t / 1e9:7.0f} TFLOP/s", flush=True)
    print(f"  sum of convs {tot:.2f} ms", flush=True)

    # torch incumbent
    def fold(key):
        return _fold(sd, key).to(dev), sd[key + ".bias"].to(dev)

    def snake(x, key):
        a = sd[key + ".alpha"].to(dev)
        return x + (a + 1e-9).reciprocal() * torch.sin(a * x).pow(2)
    W = {k[: -len(".bias")]: fold(k[: -len(".bias")]) for k in sd if k.endswith(".bias")}

    def torch_enc(x):
        x = F.conv1d(x, *W["block.0"], padding=3)
        n = 1
        for s in (2, 4, 5, 8):
            for u, d in enumerate((1, 3, 9)):
                ru = f"block.{n}.block.{u}.block."
                h = F.conv1d(snake(x, ru + "0"), *W[ru + "1"], dilation=d, padding=3 * d)
                h = F.conv1d(snake(h, ru + "2"), *W[ru + "3"])
                x = x + h
            x = F.conv1d(snake(x, f"block.{n}.block.3"), *W[f"block.{n}.block.4"], stride=s, padding=math.ceil(s / 2))
            n += 1
        return F.conv1d(snake(x, f"block.{n}"), *W[f"block.{n + 1}"], padding=1)
    Bt = min(B, 4)
    with torch.inference_mode(), torch.autocast("cuda", dtype=torch.bfloat16):
        zt = torch_enc(audio[:Bt])
        torch.cuda.synchronize()
        ms_t = timeit(lambda: torch_enc(audio[:Bt]), iters=2, warm=1)
    rel = ((z[:Bt].float() - zt.float()).pow(2).sum().sqrt() / zt.float().pow(2).sum().sqrt()).item()
    print(f"torch bf16-autocast encoder B={Bt}: {ms_t:.2f} ms = {Bt * z.shape[-1] / ms_t / 1e3:.3f} Mframes/s ({ms_t / Bt * B / ms:.1f}x ours per utterance); rel L2 ours vs torch-bf16 {rel:.2e}", flush=True)


def test_dacdec():
    """DAC conv decoder at the S2A bench shape (utterances of 500 frames = 10 s): whole-decoder time, per-launch times and the same
    stack in plain torch (bf16 autocast) as the GPU incumbent."""
    import torch.nn.functional as F
    from edm_tts_b200.dac_decoder import DACDecoder
    from edm_tts_b200.dac_stack import _fold
    from edm_tts_b200.synthetic import make_decoder_state_dict
    B, T = int(os.environ.get("DAC_B", "16")), int(os.environ.get("DAC_T", "500"))
    sd = make_decoder_state_dict(1024, 1536, (8, 5, 4, 2), 0)
    dec = DACDecoder(sd, max_chunk_samples=1 << 30)
    z = torch.randn(B, 1024, T, device=dev) * 0.5
    audio = dec(z)
    torch.cuda.synchronize()
    ms = timeit(lambda: dec(z), iters=3, warm=1)
    Ls = audio.shape[-1]
    flop = 2.0 * 1.74e6 * B * Ls
    print(f"dac decoder B={B} T={T} (L={Ls}): {ms:.2f} ms = {B * T / ms / 1e3:.3f} Mframes/s, {flop / ms / 1e9:.0f} TFLOP/s algorithmic", flush=True)
    times = []
    oc, oru = dec._conv, dec._resunit

    def tc(a_ptr, a_rows, a_cols, a_bs, w, bias, taps, step, off, rows_out, Bc, **kw):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); oc(a_ptr, a_rows, a_cols, a_bs, w, bias, taps, step, off, rows_out, Bc, **kw); e1.record()
        times.append((f"cin={a_cols} cout={w.shape[0]} taps={taps} step={step} rows={rows_out}", 2.0 * Bc * rows_out * w.shape[0] * w.shape[1], e0, e1))

    def tr(a_ptr, a_bs, Bc, rows, c, dilation, *a):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); oru(a_ptr, a_bs, Bc, rows, c, dilation, *a); e1.record()
        times.append((f"fused unit c={c} dilation={dilation} rows={rows}", 2.0 * Bc * rows * c * c * 8, e0, e1))
    dec._conv, dec._resunit = tc, tr
    dec(z)
    torch.cuda.synchronize()
    dec._conv, dec._resunit = oc, oru
    tot = 0.0
    for name, fl, e0, e1 in times:
        t = e0.elapsed_time(e1)
        tot += t
        print(f"  {name:58s} {t:8.3f} ms  {fl / t / 1e9:7.0f} TFLOP/s", flush=True)
    print(f"  sum of convs {tot:.2f} ms", flush=True)

    W = {k[: -len(".bias")]: (_fold(sd, k[: -len(".bias")]).to(dev), sd[k].to(dev)) for k in sd if k.endswith(".bias")}

    def snake(x, key):
        a = sd[key + ".alpha"].to(dev)
        return x + (a + 1e-9).reciprocal() * torch.sin(a * x).pow(2)

    def torch_dec(x):
        x = F.conv1d(x, *W["model.0"], padding=3)
        n = 1
        for s in (8, 5, 4, 2):
            blk = f"model.{n}.block."
            x = F.conv_transpose1d(snake(x, blk + "0"), *W[blk + "1"], stride=s, padding=s // 2, output_padding=s % 2)
            for u, d in enumerate((1, 3, 9)):
                ru = f"{blk}{2 + u}.block."
                h = F.conv1d(snake(x, ru + "0"), *W[ru + "1"], dilation=d, padding=3 * d)
                h = F.conv1d(snake(h, ru + "2"), *W[ru + "3"])
                x = x + h
            n += 1
        return torch.tanh(F.conv1d(snake(x, f"model.{n}"), *W[f"model.{n + 1}"], padding=3))
    Bt = min(B, 8)
    with torch.inference_mode(), torch.autocast("cuda", dtype=torch.bfloat16):
        at = torch_dec(z[:Bt])
        torch.cuda.synchronize()
        ms_t = timeit(lambda: torch_dec(z[:Bt]), iters=2, warm=1)
    rel = ((audio[:Bt].float() - at.float()).pow(2).sum().sqrt() / at.float().pow(2).sum().sqrt()).item()
    print(f"torch bf16-autocast decoder B={Bt}: {ms_t:.2f} ms ({ms_t / Bt * B / ms:.1f}x ours per utterance); rel L2 ours vs torch-bf16 {rel:.2e}", flush=True)


if __name__ == "__main__":
    t0 = time.time()
    {"gemm": test_gemm, "attn": test_attn, "ln": test_ln, "conv": test_conv, "sample": test_sample, "remask": test_remask, "rvqtc": test_rvqtc, "rvqtime": test_rvqtime, "rvqmma": test_rvqmma, "gemmsus": test_gemmsus, "kmeans": test_kmeans, "dacenc": test_dacenc, "dacdec": test_dacdec}[sys.argv[1]]()
    torch.cuda.synchronize()
    print(f"[{sys.argv[1]}] done in {time.time() - t0:.1f}s", flush=True)
