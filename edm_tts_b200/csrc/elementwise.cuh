// Bandwidth-bound kernels of the S2A decode path: LayerNorm (+ fused second LayerNorm / bf16 cast / row compaction),
// the conformer conv module's GLU -> depthwise conv -> Swish -> ChanLayerNorm chain, encoder-input construction,
// code->feature injection, sampling / arg-max over 1024 logits, and confidence re-masking.
// All rows are 1024 channels wide (hidden size); one warp owns one row, each lane 8 x 128-bit (fp32) accesses.
#pragma once
#include "ptx.cuh"
#include "seq_layout.cuh"

namespace edm {

constexpr int kD = 1024;        // hidden size
constexpr int kConvC = 2048;    // conv-module inner channels
constexpr int kV = 1024;        // codebook size (logit width)

// Token / code indices come from the caller: the kernels keep them inside their tables (memory safety); range *validation* with an
// IndexError, as F.embedding raises in the reference, is done by the host mirror before the launch (the C ABI never synchronises).
__device__ __forceinline__ int clamp_index(int i, int n) { return min(max(i, 0), n - 1); }

// lane l of a warp owns columns {i*128 + 4*l .. +3 : i = 0..7}
__device__ __forceinline__ void row_load_f32(const float* row, int lane, float (&v)[32]) {
  const float4* r4 = reinterpret_cast<const float4*>(row);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    float4 t = r4[i * 32 + lane];
    v[4 * i + 0] = t.x;
    v[4 * i + 1] = t.y;
    v[4 * i + 2] = t.z;
    v[4 * i + 3] = t.w;
  }
}
__device__ __forceinline__ void row_load_f32_ldg(const float* row, int lane, float (&v)[32]) {
  const float4* r4 = reinterpret_cast<const float4*>(row);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    float4 t = __ldg(r4 + i * 32 + lane);
    v[4 * i + 0] = t.x;
    v[4 * i + 1] = t.y;
    v[4 * i + 2] = t.z;
    v[4 * i + 3] = t.w;
  }
}
__device__ __forceinline__ void row_add_f32(const float* row, int lane, float (&v)[32]) {
  const float4* r4 = reinterpret_cast<const float4*>(row);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    float4 t = r4[i * 32 + lane];
    v[4 * i + 0] += t.x;
    v[4 * i + 1] += t.y;
    v[4 * i + 2] += t.z;
    v[4 * i + 3] += t.w;
  }
}
__device__ __forceinline__ void row_add_f32_ldg(const float* row, int lane, float (&v)[32]) {
  const float4* r4 = reinterpret_cast<const float4*>(row);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    float4 t = __ldg(r4 + i * 32 + lane);
    v[4 * i + 0] += t.x;
    v[4 * i + 1] += t.y;
    v[4 * i + 2] += t.z;
    v[4 * i + 3] += t.w;
  }
}
__device__ __forceinline__ void row_load_bf16(const __nv_bfloat16* row, int lane, float (&v)[32]) {
  const uint2* r2 = reinterpret_cast<const uint2*>(row);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    uint2 t = r2[i * 32 + lane];
    __nv_bfloat162 a = *reinterpret_cast<__nv_bfloat162*>(&t.x);
    __nv_bfloat162 b = *reinterpret_cast<__nv_bfloat162*>(&t.y);
    v[4 * i + 0] = __low2float(a);
    v[4 * i + 1] = __high2float(a);
    v[4 * i + 2] = __low2float(b);
    v[4 * i + 3] = __high2float(b);
  }
}
__device__ __forceinline__ void row_store_f32(float* row, int lane, const float (&v)[32]) {
  float4* r4 = reinterpret_cast<float4*>(row);
#pragma unroll
  for (int i = 0; i < 8; ++i) r4[i * 32 + lane] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
}
__device__ __forceinline__ void row_store_bf16(__nv_bfloat16* row, int lane, const float (&v)[32]) {
  uint2* r2 = reinterpret_cast<uint2*>(row);
#pragma unroll
  for (int i = 0; i < 8; ++i) r2[i * 32 + lane] = make_uint2(pack_bf16x2(v[4 * i], v[4 * i + 1]), pack_bf16x2(v[4 * i + 2], v[4 * i + 3]));
}

// nn.LayerNorm over 1024 channels, eps 1e-5, fp32 statistics (two-pass, in registers).
__device__ __forceinline__ void row_layernorm(float (&v)[32], const float* w, const float* b, int lane, float eps) {
  // packed f32x2 arithmetic (two channels per issue slot); the operations and their roundings are those of the scalar form, only
  // the partial sums are kept per even / odd channel
  uint64_t s2 = f2_pack(0.f, 0.f);
#pragma unroll
  for (int i = 0; i < 16; ++i) s2 = f2_add(s2, f2_pack(v[2 * i], v[2 * i + 1]));
  float s0, s1;
  f2_unpack(s2, s0, s1);
  const float mean = warp_sum(s0 + s1) * (1.0f / kD);
  const uint64_t nmean2 = f2_pack(-mean, -mean);
  uint64_t q2 = f2_pack(0.f, 0.f);
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const uint64_t d2 = f2_add(f2_pack(v[2 * i], v[2 * i + 1]), nmean2);
    q2 = f2_fma(d2, d2, q2);
  }
  float q0, q1;
  f2_unpack(q2, q0, q1);
  const float rstd = rsqrtf(warp_sum(q0 + q1) * (1.0f / kD) + eps);
  const uint64_t rstd2 = f2_pack(rstd, rstd);
  const float4* w4 = reinterpret_cast<const float4*>(w);
  const float4* b4 = reinterpret_cast<const float4*>(b);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float4 ww = __ldg(w4 + i * 32 + lane), bb = __ldg(b4 + i * 32 + lane);
    const uint64_t lo = f2_fma(f2_mul(f2_add(f2_pack(v[4 * i + 0], v[4 * i + 1]), nmean2), rstd2), f2_pack(ww.x, ww.y), f2_pack(bb.x, bb.y));
    const uint64_t hi = f2_fma(f2_mul(f2_add(f2_pack(v[4 * i + 2], v[4 * i + 3]), nmean2), rstd2), f2_pack(ww.z, ww.w), f2_pack(bb.z, bb.w));
    f2_unpack(lo, v[4 * i + 0], v[4 * i + 1]);
    f2_unpack(hi, v[4 * i + 2], v[4 * i + 3]);
  }
}

// ------------------------------------------------------------------------------------------------ LayerNorm
// y = LN1(in) (skipped when w1 == nullptr); optional fp32 store of y; z = LN2(y) when w2 != nullptr else y;
// optional bf16 store of z, optionally compacted to the target rows of each sequence (drops the prompt prefix).
struct LnParams {
  const void* in;
  int in_is_bf16;
  int rows;
  const float *w1, *b1, *w2, *b2;
  float* y_out;           // nullable
  __nv_bfloat16* z_out;   // nullable
  SeqLayout lay;          // compact != 0: the bf16 store keeps only target rows, encoder row of target t of s -> target row of (s, t)
  int compact;
  float eps;
  int reverse;            // 1: rows are walked from the last to the first (L2 reuse of the producer's most recent output)
  // layernorm_splitk_kernel only: the input row is the residual stream updated by a split-K GEMM whose K ranges left raw fp32 partial
  // sums at partials + s * partial_stride (s < n_partials, [rows, 1024] each): x_io[row] += lin_scale * bf16(sum_s partial_s + lin_bias)
  const float* partials;
  int n_partials;
  long long partial_stride;
  const float* lin_bias;  // nullable
  float lin_scale;
  float* x_io;
};

// 3 CTAs / SM (80 registers): 24 warps x 4 KB of row data in flight per SM measured best (5.7 TB/s)
__global__ void __launch_bounds__(256, 3) layernorm_kernel(const LnParams p) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  KTRACE_ENTRY(kt_entry);
  pdl_trigger();
  // Few rows (single-utterance decodes): the kernel is a chain of L2 round trips (row -> statistics -> weights), so the weight lines
  // (constants) are pulled into L1 while the previous kernel is still running. With many rows L1 holds them after the first warp anyway.
  if (p.rows <= 4096) {
    const float* wb[4] = {p.w1, p.b1, p.w2, p.b2};
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (wb[j] != nullptr) prefetch_l1(wb[j] + (warp * 32 + lane) * 4);  // 8 warps x 512 B = the 4 KB vector, one 16 B touch per lane
  }
  pdl_wait();
#ifdef EDM_KTRACE
  if (threadIdx.x == 0) { KTRACE_PUT(1, kt_entry); KTRACE_PUT(2, ktrace_now()); }
#endif
  const int row = (p.reverse ? gridDim.x - 1 - blockIdx.x : blockIdx.x) * 8 + warp;
  if (row >= p.rows) return;
  float v[32];
  if (p.in_is_bf16)
    row_load_bf16(static_cast<const __nv_bfloat16*>(p.in) + static_cast<long long>(row) * kD, lane, v);
  else
    row_load_f32(static_cast<const float*>(p.in) + static_cast<long long>(row) * kD, lane, v);
  if (p.w1 != nullptr) row_layernorm(v, p.w1, p.b1, lane, p.eps);
  if (p.y_out != nullptr) row_store_f32(p.y_out + static_cast<long long>(row) * kD, lane, v);
  if (p.z_out != nullptr) {
    long long zrow = row;
    if (p.compact) {
      int s, n;
      p.lay.enc_pos(row, s, n);
      const int t = p.lay.slot(row, s, n);
      if (t < 0) return;
      zrow = p.lay.t_start(s) + t;
    }
    if (p.w2 != nullptr) row_layernorm(v, p.w2, p.b2, lane, p.eps);
    row_store_bf16(p.z_out + zrow * kD, lane, v);
  }
#ifdef EDM_KTRACE
  if (threadIdx.x == 0) KTRACE_END(1);
#endif
}

// Residual update + LayerNorm for the small-M split-K GEMMs (gemm.cuh: GemmParams::splits): the K ranges' partial sums are added in
// range order, then bias, rounding to bf16 (the Linear output of the reference under autocast), scale and the residual add - the same
// single rounded fp32 add per element the unsplit epilogue performs with red.global.add - and the LayerNorm pass of layernorm_kernel
// on the updated row. The updated row goes back to x_io unless the LayerNorm's fp32 output overwrites it anyway (post_norm in place).
__global__ void __launch_bounds__(256) layernorm_splitk_kernel(const LnParams p) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  KTRACE_ENTRY(kt_entry);
  pdl_trigger();
  {
    const float* wb[4] = {p.w1, p.b1, p.w2, p.b2};
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (wb[j] != nullptr) prefetch_l1(wb[j] + (warp * 32 + lane) * 4);
    if (p.lin_bias != nullptr) prefetch_l1(p.lin_bias + (warp * 32 + lane) * 4);
  }
  pdl_wait();
#ifdef EDM_KTRACE
  if (threadIdx.x == 0) { KTRACE_PUT(1, kt_entry); KTRACE_PUT(2, ktrace_now()); }
#endif
  const int row = blockIdx.x * 8 + warp;
  if (row >= p.rows) return;
  // every load of the row is issued before the first add (one L2 round trip instead of one per K range): 2 or 4 ranges
  float v[32], a[32];
  const float* pr = p.partials + static_cast<long long>(row) * kD;
  row_load_f32(pr, lane, a);
  if (p.n_partials == 4) {
    float b[32], c[32], d[32];
    row_load_f32(pr + p.partial_stride, lane, b);
    row_load_f32(pr + 2 * p.partial_stride, lane, c);
    row_load_f32(pr + 3 * p.partial_stride, lane, d);
    row_load_f32(p.x_io + static_cast<long long>(row) * kD, lane, v);
#pragma unroll
    for (int i = 0; i < 32; ++i) a[i] = __fadd_rn(__fadd_rn(__fadd_rn(a[i], b[i]), c[i]), d[i]);
  } else {
    float b[32];
    if (p.n_partials >= 2) row_load_f32(pr + p.partial_stride, lane, b);
    row_load_f32(p.x_io + static_cast<long long>(row) * kD, lane, v);
    if (p.n_partials >= 2) {
#pragma unroll
      for (int i = 0; i < 32; ++i) a[i] = __fadd_rn(a[i], b[i]);
    }
    for (int s = 2; s < p.n_partials; ++s) row_add_f32(pr + s * p.partial_stride, lane, a);
  }
  if (p.lin_bias != nullptr) row_add_f32_ldg(p.lin_bias, lane, a);
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __fadd_rn(v[i], __fmul_rn(p.lin_scale, bf16_round(a[i])));
  if (p.y_out != p.x_io) row_store_f32(p.x_io + static_cast<long long>(row) * kD, lane, v);
  if (p.w1 != nullptr) row_layernorm(v, p.w1, p.b1, lane, p.eps);
  if (p.y_out != nullptr) row_store_f32(p.y_out + static_cast<long long>(row) * kD, lane, v);
  if (p.z_out != nullptr) {
    long long zrow = row;
    if (p.compact) {
      int s, n;
      p.lay.enc_pos(row, s, n);
      const int t = p.lay.slot(row, s, n);
      if (t < 0) return;
      zrow = p.lay.t_start(s) + t;
    }
    if (p.w2 != nullptr) row_layernorm(v, p.w2, p.b2, lane, p.eps);
    row_store_bf16(p.z_out + zrow * kD, lane, v);
  }
#ifdef EDM_KTRACE
  if (threadIdx.x == 0) KTRACE_END(4);
#endif
}

// ------------------------------------------------------------------------------------------------ conv module core
// Reference: conformer.py:59-66 (GLU), :69-77 + :23-25 (depthwise conv, k = 5, zero pad (2,2) inside each sequence),
// :54-56 (Swish), :90-99 (ChanLayerNorm: mean / biased var over the 2048 channels of a token, scale only,
// eps = 1e-4 because the activations are bf16 under autocast). Every intermediate the reference materialises in
// bf16 is rounded to bf16 here as well.
// in  : [B*N, 4096] bf16 (pointwise-conv output: first 2048 = value, last 2048 = gate)
// out : [B*N, 2048] bf16
struct ConvModParams {
  const __nv_bfloat16* in;
  __nv_bfloat16* out;
  const float* dw_w;    // [2048, 5]
  const float* dw_b;    // [2048]
  const float* cln_w;   // [2048]
  SeqLayout lay;        // rows of sequence s: [n_start(s), n_start(s) + n_len(s))
  int max_n;            // longest sequence (grid size)
};
constexpr int kConvTT = 20;        // output tokens per CTA (4 halo rows are re-read: 20 % more loads, served by L2); 25 measured slower (wave quantisation)
constexpr int kConvThreads = 512;  // 4 channels per thread at the S2A model's 2048 inner channels
constexpr uint32_t kConvSmemBytes = kConvTT * kConvThreads * 8;  // Swish outputs of the tile (bf16 x 4 per thread and token)
constexpr uint32_t conv_smem_bytes(int channels) { return kConvTT * (channels / 4) * 8; }

// kGlu = true : in is [B*N, 4096] (value | gate), the GLU runs here.
// kGlu = false: in is [B*N, 2048], already gated by the pointwise-conv GEMM epilogue (EPI_GLU_BF16).
// Three phases per CTA (20 tokens x 2048 channels): (1) every thread streams its 4 channels through the 5-tap window and
// parks the Swish outputs in shared memory, (2) one warp per token reduces mean / variance over the 2048 channels,
// (3) every thread normalises its channels. 16 warps per CTA, two CTAs per SM.
// kC = inner channels (2048 for the S2A conformer; 1024 / 768 for the text-to-semantic model's hidden 512 / 384), kC / 4 threads.
template <bool kGlu, int kC = kConvC>
__global__ void __launch_bounds__(kC / 4, 2) conv_module_kernel(const ConvModParams p) {
  constexpr int kConvThreads = kC / 4;
  constexpr int kConvC = kC;
  static_assert(kC % 256 == 0, "one warp reduces a token's channels in 256-channel steps");
  extern __shared__ uint2 s_keep[];  // [kConvTT][kC / 4]
  __shared__ uint32_t s_mean2[kConvTT];
  __shared__ uint32_t s_rstd2[kConvTT];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int c0 = tid * 4;
  const int t0 = blockIdx.x * kConvTT;
  const int b = blockIdx.y;
  const int seq_n = p.lay.n_len(b);
  const long long row_b = p.lay.n_start(b);
  constexpr int kInW = kGlu ? 2 * kConvC : kConvC;  // input row width
  const __nv_bfloat16* base = p.in + row_b * kInW + c0;

  float wt[4][5], bias[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) {
#pragma unroll
    for (int j = 0; j < 5; ++j) wt[c][j] = __ldg(p.dw_w + (c0 + c) * 5 + j);
    bias[c] = __ldg(p.dw_b + c0 + c);
  }

  float win[5][4];
#pragma unroll
  for (int j = 0; j < 5; ++j)
#pragma unroll
    for (int c = 0; c < 4; ++c) win[j][c] = 0.f;

  pdl_sync();  // the depthwise weights above are constants; the rows below come from the previous kernel
  if (t0 >= seq_n) return;  // tile past the end of a shorter sequence of a packed batch

  // two rows of loads in flight ahead of the arithmetic
  uint2 pa[2], pg[2] = {make_uint2(0, 0), make_uint2(0, 0)};
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int t = t0 - 2 + r;
    pa[r] = make_uint2(0, 0);
    if (t >= 0 && t < seq_n) {
      pa[r] = *reinterpret_cast<const uint2*>(base + static_cast<long long>(t) * kInW);
      if constexpr (kGlu) pg[r] = *reinterpret_cast<const uint2*>(base + static_cast<long long>(t) * kInW + kConvC);
    }
  }

#pragma unroll
  for (int r = 0; r < kConvTT + 4; ++r) {
    const uint2 av = pa[r & 1], gv = pg[r & 1];
    {
      const int tn = t0 + r;  // row r + 2
      pa[r & 1] = make_uint2(0, 0);
      if (r + 2 < kConvTT + 4 && tn >= 0 && tn < seq_n) {
        pa[r & 1] = *reinterpret_cast<const uint2*>(base + static_cast<long long>(tn) * kInW);
        if constexpr (kGlu) pg[r & 1] = *reinterpret_cast<const uint2*>(base + static_cast<long long>(tn) * kInW + kConvC);
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int c = 0; c < 4; ++c) win[j][c] = win[j + 1][c];
    {
      // GLU: value * bf16(sigmoid(gate)), rounded to bf16 (zero rows stay zero: 0 * 0.5 = 0)
      const uint32_t aw[2] = {av.x, av.y}, gw[2] = {gv.x, gv.y};
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        uint32_t gl = aw[c];
        if constexpr (kGlu) {
          const uint32_t sg = pack_bf16x2(sigmoid_tanh(bf16lo(gw[c])), sigmoid_tanh(bf16hi(gw[c])));
          gl = bf16x2_mul(aw[c], sg);
        }
        win[4][2 * c + 0] = bf16lo(gl);
        win[4][2 * c + 1] = bf16hi(gl);
      }
    }
    if (r >= 4) {
      const int o = r - 4;  // output token t0 + o, window = tokens t0+o-2 .. t0+o+2
      uint32_t sp[2];
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        float acc0 = bias[2 * c], acc1 = bias[2 * c + 1];
#pragma unroll
        for (int j = 0; j < 5; ++j) {
          acc0 = fmaf(wt[2 * c][j], win[j][2 * c], acc0);
          acc1 = fmaf(wt[2 * c + 1][j], win[j][2 * c + 1], acc1);
        }
        const uint32_t y2 = pack_bf16x2(acc0, acc1);
        const uint32_t sg = pack_bf16x2(sigmoid_tanh(bf16lo(y2)), sigmoid_tanh(bf16hi(y2)));
        sp[c] = bf16x2_mul(y2, sg);
      }
      s_keep[o * kConvThreads + tid] = make_uint2(sp[0], sp[1]);
    }
  }
  __syncthreads();

  // per-token statistics over the 2048 channels (ChanLayerNorm: biased variance, bf16 mean / var / rstd)
  for (int o = warp; o < kConvTT; o += kConvThreads / 32) {
    const uint4* row = reinterpret_cast<const uint4*>(s_keep + o * kConvThreads);
    float s = 0.f, q = 0.f;
#pragma unroll
    for (int i = 0; i < kC / 256; ++i) {
      const uint4 v = row[i * 32 + lane];
      const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float lo = bf16lo(w4[k]), hi = bf16hi(w4[k]);
        s += lo + hi;
        q = fmaf(lo, lo, q);
        q = fmaf(hi, hi, q);
      }
    }
    s = warp_sum(s);
    q = warp_sum(q);
    if (lane == 0) {
      const float mean = s * (1.0f / kConvC);
      const float var = fmaxf(q * (1.0f / kConvC) - mean * mean, 0.f);
      const float rs = rsqrtf(fmaxf(bf16_round(var), 1e-4f));
      s_mean2[o] = pack_bf16x2(mean, mean);
      s_rstd2[o] = pack_bf16x2(rs, rs);
    }
  }
  __syncthreads();

  float cw[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) cw[c] = __ldg(p.cln_w + c0 + c);
#pragma unroll 4
  for (int o = 0; o < kConvTT; ++o) {
    const int t = t0 + o;
    if (t >= seq_n) break;
    const uint32_t mean2 = s_mean2[o], rstd2 = s_rstd2[o];
    const uint2 k = s_keep[o * kConvThreads + tid];
    const uint32_t n0 = bf16x2_mul(bf16x2_sub(k.x, mean2), rstd2);
    const uint32_t n1 = bf16x2_mul(bf16x2_sub(k.y, mean2), rstd2);
    *reinterpret_cast<uint2*>(p.out + (row_b + t) * kConvC + c0) =
        make_uint2(pack_bf16x2(bf16lo(n0) * cw[0], bf16hi(n0) * cw[1]), pack_bf16x2(bf16lo(n1) * cw[2], bf16hi(n1) * cw[3]));
  }
}

// ------------------------------------------------------------------------------------------------ encoder input
// Reference: modeling_injection_conformer.py:139-168. Target rows: semantic embedding + mask token. Prompt rows:
// semantic embedding + LayerNorm(Linear(level-0 DAC feature)), where Linear o codes_to_features collapses to a table
// lookup (feat_table[code] = W_fp (W_out0 codebook0[code]) , feat_const = W_fp b_out0 + b_fp), exact algebra.
struct BuildInputParams {
  float* x;                        // encoder rows [sum N_s, 1024]
  const int* sem_tokens;           // target rows [sum T_s]
  const int* sem_prompt;           // prompt rows [sum P_s] or nullptr
  const int* ac_prompt;            // sequence s: [Qp, P_s] at Qp * p_start(s) (level 0 used here) or nullptr
  int ac_prompt_levels;            // Qp
  const float* sem_emb;            // [num_semantic, 1024]
  const float* mask_token;         // [1024]
  const float* feat_table;         // [1024 codes, 1024]
  const float* feat_const;         // [1024]
  const float *fp_ln_w, *fp_ln_b;  // acoustic_feat_proj.1
  SeqLayout lay;
  int rows;                        // sum N_s
  int num_semantic;                // rows of sem_emb
  float eps;
};

__global__ void __launch_bounds__(256) build_input_kernel(const BuildInputParams p) {
  pdl_sync();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row = blockIdx.x * 8 + warp;
  if (row >= p.rows) return;
  int b, n;
  p.lay.enc_pos(row, b, n);
  const int t = p.lay.slot(row, b, n);
  float v[32];
  if (t < 0) {
    const int k = -1 - t;  // k-th known row of sequence b
    const long long pb = p.lay.p_start(b);
    const int code = clamp_index(p.ac_prompt[static_cast<long long>(p.ac_prompt_levels) * pb + k], kV);  // level 0
    row_load_f32_ldg(p.feat_table + static_cast<long long>(code) * kD, lane, v);
    row_add_f32_ldg(p.feat_const, lane, v);
    row_layernorm(v, p.fp_ln_w, p.fp_ln_b, lane, p.eps);
    row_add_f32_ldg(p.sem_emb + static_cast<long long>(clamp_index(p.sem_prompt[pb + k], p.num_semantic)) * kD, lane, v);
  } else {
    row_load_f32_ldg(p.sem_emb + static_cast<long long>(clamp_index(p.sem_tokens[p.lay.t_start(b) + t], p.num_semantic)) * kD, lane, v);
    row_add_f32_ldg(p.mask_token, lane, v);
  }
  row_store_f32(p.x + static_cast<long long>(row) * kD, lane, v);
}

// Per-step update of the target rows (modeling_injection_conformer.py:184-197, :214-218):
//   still masked after re-masking -> sem + mask_token;  masked before, kept now -> sem + LN(feat_table[id] + const);
//   already unmasked earlier -> untouched.
struct UpdateInputParams {
  float* x;
  const int* sem_tokens;   // target rows [sum T_s]
  const int* ids;          // target rows: sampled level-0 codes
  const uint8_t* mask_old; // target rows
  const uint8_t* mask_new; // target rows or nullptr (final step: nothing is re-masked)
  const float* sem_emb;
  const float* mask_token;
  const float* feat_table;
  const float* feat_const;
  const float *fp_ln_w, *fp_ln_b;
  SeqLayout lay;
  int rows;                // sum T_s
  int num_semantic;
  float eps;
};

__global__ void __launch_bounds__(256) update_input_kernel(const UpdateInputParams p) {
  pdl_sync();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r = blockIdx.x * 8 + warp;
  if (r >= p.rows) return;
  const bool was = p.mask_old[r] != 0;
  const bool now = p.mask_new != nullptr && p.mask_new[r] != 0;
  if (!was && !now) return;
  float v[32];
  if (now) {
    row_load_f32_ldg(p.mask_token, lane, v);
  } else {
    row_load_f32_ldg(p.feat_table + static_cast<long long>(clamp_index(p.ids[r], kV)) * kD, lane, v);
    row_add_f32_ldg(p.feat_const, lane, v);
    row_layernorm(v, p.fp_ln_w, p.fp_ln_b, lane, p.eps);
  }
  row_add_f32_ldg(p.sem_emb + static_cast<long long>(clamp_index(p.sem_tokens[r], p.num_semantic)) * kD, lane, v);
  int b, t;
  p.lay.tgt_pos(r, b, t);
  row_store_f32(p.x + p.lay.enc_row(b, t) * kD, lane, v);
}

// ------------------------------------------------------------------------------------------------ coarse injection
// Reference: injection_conformer_wrapper.py:107-129. At injection layer k (level k):
//   inj = LN_k(Linear_k(sum_{i<=k} W_out_i codebook_i[code_i] + b_out_i)) = LN_k(sum_i inj_table[k][i][code_i] + inj_const[k])
//   x   = block_out + inj + (k > 0 ? previous coarse block_out : 0)
// code_i comes from the arg-max of this pass for target rows and from the acoustic prompt for prompt (known) rows.
struct InjectParams {
  float* x;                 // out: encoder rows [sum N_s, 1024]
  const float* cur_out;     // block output at this injection layer (coarse_out[k])
  const float* prev_out;    // coarse_out[k-1] or nullptr
  const int* pred_codes;    // sequence s: [4, T_s] at 4 t_start(s)
  const int* ac_prompt;     // sequence s: [Qp, P_s] at Qp p_start(s), or nullptr
  int ac_prompt_levels;
  const float* prompt_proj; // prompt rows [sum P_s, 1024] or nullptr: Linear_k(prompt feature) given by the caller (feature-valued injections)
  const float* tables[4];   // inj_table[k][i] : [1024 codes, 1024]
  const float* inj_const;   // [1024]
  const float *ln_w, *ln_b; // project_injection[k].1
  int level;                // k
  SeqLayout lay;
  int rows;                 // sum N_s
  float eps;
};

__global__ void __launch_bounds__(256) inject_kernel(const InjectParams p) {
  pdl_sync();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long row = static_cast<long long>(blockIdx.x) * 8 + warp;
  if (row >= p.rows) return;
  int b, n;
  p.lay.enc_pos(static_cast<int>(row), b, n);
  const int t = p.lay.slot(static_cast<int>(row), b, n);
  float v[32];
  if (t < 0 && p.prompt_proj != nullptr) {
    row_load_f32_ldg(p.prompt_proj + (p.lay.p_start(b) + static_cast<long long>(-1 - t)) * kD, lane, v);
  } else {
    row_load_f32_ldg(p.inj_const, lane, v);
    for (int i = 0; i <= p.level; ++i) {
      int code;
      if (t < 0)
        code = p.ac_prompt[static_cast<long long>(p.ac_prompt_levels) * p.lay.p_start(b) + static_cast<long long>(i) * p.lay.p_len(b) + (-1 - t)];
      else
        code = p.pred_codes[p.lay.out_offset(b, i, 4, t)];
      row_add_f32_ldg(p.tables[i] + static_cast<long long>(clamp_index(code, kV)) * kD, lane, v);
    }
  }
  row_layernorm(v, p.ln_w, p.ln_b, lane, p.eps);
  float o[32];
  row_load_f32(p.cur_out + row * kD, lane, o);
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] += o[i];
  if (p.prev_out != nullptr) {
    row_load_f32(p.prev_out + row * kD, lane, o);
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] += o[i];
  }
  row_store_f32(p.x + row * kD, lane, v);
}

// ------------------------------------------------------------------------------------------------ sampling
// Philox4x32-10, counter = (row counter low word, column group (sampling) or 0x52454d41 (re-masking), step, row counter high word),
// key = seed (low word, high word). tests/philox_ref.py restates it on the host.
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, ctr.x), lo0 = 0xD2511F53u * ctr.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, ctr.z), lo1 = 0xCD9E8D57u * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += 0x9E3779B9u;
    key.y += 0xBB67AE85u;
  }
  return ctr;
}
// Standard Gumbel from the top 24 bits k: u = float32(k + 1/2) 2^-24, g = -log(e) with e = -log(u).
// __logf has an absolute error (about 2^-24 measured near 1, 2^-21.41 documented on [0.5, 2]) that is large against e when u is
// close to 1, where g is largest and decides the sample: for u > 1 - 2^-10, e comes from v = 1 - u (exact for u >= 1/2) as
// v + v^2/2 + v^3/3 (relative truncation below 2^-32). Below that, -__logf(u) keeps g within 5.3e-5 of -log(-log(u)) (measured
// over every k on a B200), and those draws keep the bits the fast path has always given them.
// k + 1/2 needs 25 bits, so k >= 2^23 rounds to even, and k = 2^24 - 1 rounds to u = 1: v is held at 2^-24 there, which is
// u = 1 - 2^-24, the largest float below 1, instead of e = 0 and g = +inf. So u lies in [2^-25, 1 - 2^-24] and g in [-2.85, 16.64].
__device__ __forceinline__ float gumbel_from_bits(uint32_t bits) {
  const float u = (static_cast<float>(bits >> 8) + 0.5f) * (1.0f / 16777216.0f);
  float e;
  if (u > 1.0f - 0x1p-10f) {
    const float v = fmaxf(1.0f - u, 0x1p-24f);
    e = v * (1.0f + v * (0.5f + v * (1.0f / 3.0f)));
  } else {
    e = -__logf(u);
  }
  return -__logf(e);
}

// One warp per row of 1024 logits. id = argmax(logit + gumbel) (first index wins ties); logp = log softmax(logits)[id].
// Reference: Categorical(logits).sample() (modeling_injection_conformer.py:192) == argmax(log p + Gumbel); arg-max
// decoding (:185, :228, injection_conformer_wrapper.py:121) is the same kernel with no noise.
struct SampleParams {
  const float* logits;      // [rows, 1024] with row stride ld
  long long ld;
  int rows;
  const float* noise;       // [rows, 1024] Gumbel noise (parity runs) or nullptr
  int use_philox;           // noise == nullptr && use_philox: in-kernel Gumbel noise
  unsigned long long seed;
  const unsigned long long* seed_dev;  // when set, *seed_dev is added to seed (a captured CUDA graph draws fresh noise per replay)
  unsigned int step;
  long long seq0;           // global index of sequence 0 (keeps the Philox stream independent of batch chunking / sharding)
  const int* forced_ids;    // teacher forcing (parity runs) or nullptr
  int* ids;                 // out (forced id when teacher forcing), element (row) lands at out_base(row)
  int* ids_raw;             // out, the model's own choice (nullable)
  float* logp;              // out [rows] or nullptr
  // output index mapping: row r = (target row of (b, t)) * Q + q  ->  ids[lay.out_offset(b, out_q0 + q, out_q_stride, t)], i.e.
  // (b*out_q_stride + out_q0 + q)*T + t for a uniform layout. Philox counter: lay.philox_row(seq0, b, t) * Q + q.
  SeqLayout lay;
  int Q, out_q_stride, out_q0;
};

__global__ void __launch_bounds__(256) sample_kernel(const SampleParams p) {
  pdl_sync();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long row = static_cast<long long>(blockIdx.x) * 8 + warp;
  if (row >= p.rows) return;
  int b, t;
  p.lay.tgt_pos(static_cast<int>(row / p.Q), b, t);
  const int q = static_cast<int>(row % p.Q);
  float v[32];
  row_load_f32(p.logits + row * p.ld, lane, v);
  float mx = -INFINITY;
#pragma unroll
  for (int i = 0; i < 32; ++i) mx = fmaxf(mx, v[i]);
  mx = warp_max(mx);
  float se = 0.f;
#pragma unroll
  for (int i = 0; i < 32; ++i) se += __expf(v[i] - mx);
  se = warp_sum(se);

  float best = -INFINITY;
  int best_idx = 0x7fffffff;
  if (p.noise != nullptr) {
    float g[32];
    row_load_f32(p.noise + row * kV, lane, g);
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      const float s = v[i] + g[i];
      const int idx = (i >> 2) * 128 + lane * 4 + (i & 3);
      if (s > best) {
        best = s;
        best_idx = idx;
      }
    }
  } else if (p.use_philox) {
    const unsigned long long seed = p.seed + (p.seed_dev != nullptr ? *p.seed_dev : 0ull);
    const long long ctr = p.lay.philox_row(p.seq0, b, t) * p.Q + q;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const uint4 bits = philox4x32_10(make_uint4(static_cast<uint32_t>(ctr), static_cast<uint32_t>(i * 32 + lane), p.step,
                                                  static_cast<uint32_t>(ctr >> 32)),
                                       make_uint2(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32)));
      const uint32_t bb[4] = {bits.x, bits.y, bits.z, bits.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float s = v[4 * i + j] + gumbel_from_bits(bb[j]);
        const int idx = i * 128 + lane * 4 + j;
        if (s > best) {
          best = s;
          best_idx = idx;
        }
      }
    }
  } else {
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      const int idx = (i >> 2) * 128 + lane * 4 + (i & 3);
      if (v[i] > best) {
        best = v[i];
        best_idx = idx;
      }
    }
  }
  // lane-local scan order is increasing in idx, so strict '>' keeps the first maximum; same rule across lanes
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, best_idx, o);
    if (ob > best || (ob == best && oi < best_idx)) {
      best = ob;
      best_idx = oi;
    }
  }
  // a row without any finite maximum (all NaN / all -inf) never updates best_idx: id 0, as torch.argmax gives for all -inf; ids index
  // the feature tables downstream, so they must stay inside [0, 1024)
  if (best_idx >= kV) best_idx = 0;
  const long long oidx = p.lay.out_offset(b, p.out_q0 + q, p.out_q_stride, t);
  int id = best_idx;
  if (p.forced_ids != nullptr) id = min(max(p.forced_ids[oidx], 0), kV - 1);
  if (lane == 0) {
    p.ids[oidx] = id;
    if (p.ids_raw != nullptr) p.ids_raw[oidx] = best_idx;
  }
  if (p.logp != nullptr) {
    // the owner lane of column `id` publishes its logit
    const int owner = (id & 127) >> 2;
    const int slot = ((id >> 7) << 2) | (id & 3);
    float val = 0.f;
#pragma unroll
    for (int i = 0; i < 32; ++i)
      if (i == slot) val = v[i];
    val = __shfl_sync(0xffffffffu, val, owner);
    if (lane == 0) p.logp[row] = (val - mx) - __logf(se);
  }
}

// Finishes the arg-max of the fused logits heads (gemm.cuh EPI_ARGMAX): part[row, j] = (max, first arg-max) of columns [64 j, 64 j + 64).
// Same output mapping / teacher forcing as sample_kernel with no noise; ascending j with strict '>' keeps the first maximum.
struct ArgmaxCombineParams {
  const float2* part;       // [rows, parts]
  int rows, parts;
  const int* forced_ids;
  int* ids;
  int* ids_raw;             // nullable
  SeqLayout lay;
  int Q, out_q_stride, out_q0;
};
__global__ void __launch_bounds__(256) argmax_combine_kernel(const ArgmaxCombineParams p) {
  pdl_sync();
  const long long row = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x;
  if (row >= p.rows) return;
  const float2* r = p.part + row * p.parts;
  float2 first = r[0];
  float best = first.x;
  int idx = __float_as_int(first.y);
  for (int j = 1; j < p.parts; ++j) {
    const float2 v = r[j];
    if (v.x > best) {
      best = v.x;
      idx = __float_as_int(v.y);
    }
  }
  if (!(best == best)) idx = 0;      // NaN logits: no defined maximum; stay inside the tables
  idx = clamp_index(idx, kV);
  int b, t;
  p.lay.tgt_pos(static_cast<int>(row / p.Q), b, t);
  const int q = static_cast<int>(row % p.Q);
  const long long oidx = p.lay.out_offset(b, p.out_q0 + q, p.out_q_stride, t);
  p.ids[oidx] = p.forced_ids != nullptr ? clamp_index(p.forced_ids[oidx], kV) : idx;
  if (p.ids_raw != nullptr) p.ids_raw[oidx] = idx;
}

// ------------------------------------------------------------------------------------------------ re-masking
// Reference: modeling_injection_conformer.py:199-219 + edm_tts/utils/utils.py:49-60.
//   mask_len = max(1, min(#masked - 1, floor(float32(T) * float32(ratio))))
//   conf     = masked ? logp + float32(temperature * ratio) * gumbel : +inf
//   cut      = sort(conf)[mask_len];  new_mask = conf < cut
// One CTA per sequence over its T_s target rows (mask_len from T_s); the k-th order statistic is found by rank counting in shared
// memory (T_s <= 4096). Every per-row buffer below is indexed by target row.
struct RemaskParams {
  const float* logp;
  const float* gumbel;      // or nullptr (then Philox)
  const uint8_t* mask_old;
  uint8_t* mask_new;
  uint8_t* mask_raw;        // or nullptr: the kernel's own mask (before teacher forcing), for parity runs
  const uint8_t* forced_mask;  // teacher forcing: copied to mask_new when given
  SeqLayout lay;
  int init_count;    // 0: the S2A rule mask_len = max(1, min(#masked - 1, floor(T * ratio))) (modeling_injection_conformer.py:199-202);
                     // > 0: the text-to-semantic rule max(1, min(floor(init_count * ratio), init_count)) with init_count = number of
                     // speech positions (modeling_text_to_semantic.py:237-242)
  const int* init_counts;  // nullable: init_count of sequence s is init_counts[s] (a text-to-semantic batch)
  float ratio;       // float32(cos(pi/2 (t+1)/S))
  float temp_ratio;  // float32(temperature * ratio)
  unsigned long long seed;
  const unsigned long long* seed_dev;  // see SampleParams
  unsigned int step;
  long long seq0;    // global index of sequence 0 (Philox counter lay.philox_row(seq0, s, t))
};
constexpr int kRemaskMaxT = 4096;

__global__ void __launch_bounds__(256) remask_kernel(const RemaskParams p) {
  pdl_sync();
  __shared__ float conf[kRemaskMaxT];
  __shared__ int s_count;
  __shared__ float s_cut;
  const int b = blockIdx.x, tid = threadIdx.x;
  const long long base = p.lay.t_start(b);
  const int T = p.lay.t_len(b);
  if (tid == 0) {
    s_count = 0;
    s_cut = INFINITY;  // stays when mask_len >= T (the reference's take_along_dim raises there; the host rejects T < 2 with steps > 1)
  }
  __syncthreads();
  const unsigned long long seed = p.seed + (p.seed_dev != nullptr ? *p.seed_dev : 0ull);
  int local = 0;
  for (int t = tid; t < T; t += 256) {
    const bool m = p.mask_old[base + t] != 0;
    float c = INFINITY;
    if (m) {
      float g;
      if (p.gumbel != nullptr) {
        g = p.gumbel[base + t];
      } else {
        const long long ctr = p.lay.philox_row(p.seq0, b, t);
        const uint4 bits = philox4x32_10(make_uint4(static_cast<uint32_t>(ctr), 0x52454d41u, p.step, static_cast<uint32_t>(ctr >> 32)),
                                         make_uint2(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32)));
        g = gumbel_from_bits(bits.x);
      }
      c = __fadd_rn(p.logp[base + t], __fmul_rn(p.temp_ratio, g));
      ++local;
    }
    conf[t] = c;
  }
  atomicAdd(&s_count, local);
  __syncthreads();
  if (p.forced_mask != nullptr && p.mask_raw == nullptr) {
    for (int t = tid; t < T; t += 256) p.mask_new[base + t] = p.forced_mask[base + t];
    return;
  }
  float ml;
  const int init_count = p.init_counts != nullptr ? __ldg(p.init_counts + b) : p.init_count;
  if (init_count > 0) {
    ml = fmaxf(1.0f, fminf(floorf(__fmul_rn(static_cast<float>(init_count), p.ratio)), static_cast<float>(init_count)));
  } else {
    ml = floorf(__fmul_rn(static_cast<float>(T), p.ratio));
    ml = fmaxf(1.0f, fminf(static_cast<float>(s_count - 1), ml));
  }
  const int k = static_cast<int>(ml);
  for (int t = tid; t < T; t += 256) {
    const float c = conf[t];
    int less = 0, leq = 0;
    for (int u = 0; u < T; ++u) {
      const float o = conf[u];
      less += (o < c);
      leq += (o <= c);
    }
    if (less <= k && k < leq) s_cut = c;  // every thread that qualifies writes the same value
  }
  __syncthreads();
  const float cut = s_cut;
  for (int t = tid; t < T; t += 256) {
    const uint8_t own = conf[t] < cut ? 1 : 0;
    if (p.mask_raw != nullptr) p.mask_raw[base + t] = own;
    p.mask_new[base + t] = p.forced_mask != nullptr ? p.forced_mask[base + t] : own;
  }
}

}  // namespace edm
