// Kernels of the text-to-semantic decode (TextToSemanticWLen.infer, edm_tts/models/text_to_semantic/modeling_text_to_semantic.py:184-267)
// that the S2A path does not already provide: LayerNorm for hidden sizes 384 / 512 (+ embedding gather on load, + GELU on load for
// pred_transform), the length head, and the token update of one decode iteration. GEMMs, attention, the conv module, sampling and
// re-masking are the S2A kernels (gemm.cuh small-M kernel, attention.cuh with 64-wide zero-padded heads, elementwise.cuh).
// Every kernel here takes one sequence or a batch of sequences packed back to back (T2sSeqs).
#pragma once
#include "elementwise.cuh"

namespace edm {

// A row of D = 128 * NV channels: lane l of a warp owns columns {i*128 + 4*l .. +3 : i = 0..NV-1}.
template <int NV>
__device__ __forceinline__ void rowg_load_f32(const float* row, int lane, float (&v)[4 * NV]) {
  const float4* r4 = reinterpret_cast<const float4*>(row);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const float4 t = r4[i * 32 + lane];
    v[4 * i + 0] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
  }
}
template <int NV>
__device__ __forceinline__ void rowg_load_bf16(const __nv_bfloat16* row, int lane, float (&v)[4 * NV]) {
  const uint2* r2 = reinterpret_cast<const uint2*>(row);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const uint2 t = r2[i * 32 + lane];
    v[4 * i + 0] = bf16lo(t.x); v[4 * i + 1] = bf16hi(t.x); v[4 * i + 2] = bf16lo(t.y); v[4 * i + 3] = bf16hi(t.y);
  }
}
template <int NV>
__device__ __forceinline__ void rowg_store_f32(float* row, int lane, const float (&v)[4 * NV]) {
  float4* r4 = reinterpret_cast<float4*>(row);
#pragma unroll
  for (int i = 0; i < NV; ++i) r4[i * 32 + lane] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
}
template <int NV>
__device__ __forceinline__ void rowg_store_bf16(__nv_bfloat16* row, int lane, const float (&v)[4 * NV]) {
  uint2* r2 = reinterpret_cast<uint2*>(row);
#pragma unroll
  for (int i = 0; i < NV; ++i) r2[i * 32 + lane] = make_uint2(pack_bf16x2(v[4 * i], v[4 * i + 1]), pack_bf16x2(v[4 * i + 2], v[4 * i + 3]));
}
// nn.LayerNorm over D channels, fp32 two-pass statistics in registers
template <int NV>
__device__ __forceinline__ void rowg_layernorm(float (&v)[4 * NV], const float* w, const float* b, int lane, float eps) {
  constexpr float kInvD = 1.0f / (128 * NV);
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 4 * NV; ++i) s += v[i];
  const float mean = warp_sum(s) * kInvD;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < 4 * NV; ++i) q = fmaf(v[i] - mean, v[i] - mean, q);
  const float rstd = rsqrtf(warp_sum(q) * kInvD + eps);
  const float4* w4 = reinterpret_cast<const float4*>(w);
  const float4* b4 = reinterpret_cast<const float4*>(b);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const float4 ww = __ldg(w4 + i * 32 + lane), bb = __ldg(b4 + i * 32 + lane);
    v[4 * i + 0] = fmaf((v[4 * i + 0] - mean) * rstd, ww.x, bb.x);
    v[4 * i + 1] = fmaf((v[4 * i + 1] - mean) * rstd, ww.y, bb.y);
    v[4 * i + 2] = fmaf((v[4 * i + 2] - mean) * rstd, ww.z, bb.z);
    v[4 * i + 3] = fmaf((v[4 * i + 3] - mean) * rstd, ww.w, bb.w);
  }
}

// y = LN1(f(in)) (LN1 skipped when w1 == nullptr); optional fp32 store of y; z = LN2(y) when w2 != nullptr else y; optional bf16 store.
// in row r is in[gather ? clamp(gather[r]) : r], or override_row when gather[r] < 0; f = GELU(tanh) when pre_gelu (pred_transform:
// Linear -> GELU -> LayerNorm, :56-58).
struct LnGParams {
  const void* in;
  int in_is_bf16;
  const int* gather;     // nullable: embedding lookup (nn.Embedding, :47) fused into the load
  int gather_rows;       // rows of the table
  const float* override_row;  // nullable: rows whose gather index is negative are read from here (the length token in front of every text, :199)
  int rows;
  const float *w1, *b1, *w2, *b2;
  float* y_out;
  __nv_bfloat16* z_out;
  float eps;
  int pre_gelu;
  // layernorm_g_splitk_kernel only (see LnParams in elementwise.cuh): the input row is x_io[row] += lin_scale * bf16(sum of the
  // n_partials K-range partial sums + lin_bias), written back unless y_out overwrites it
  const float* partials;
  int n_partials;
  long long partial_stride;
  const float* lin_bias;
  float lin_scale;
  float* x_io;
};

template <int NV>
__global__ void __launch_bounds__(256) layernorm_g_kernel(const LnGParams p) {
  pdl_sync();
  constexpr int D = 128 * NV;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row = blockIdx.x * 8 + warp;
  if (row >= p.rows) return;
  long long src = row;
  int gi = 0;
  if (p.gather != nullptr) {
    gi = p.gather[row];
    src = clamp_index(gi, p.gather_rows);
  }
  float v[4 * NV];
  if (p.override_row != nullptr && gi < 0)
    rowg_load_f32<NV>(p.override_row, lane, v);
  else if (p.in_is_bf16)
    rowg_load_bf16<NV>(static_cast<const __nv_bfloat16*>(p.in) + src * D, lane, v);
  else
    rowg_load_f32<NV>(static_cast<const float*>(p.in) + src * D, lane, v);
  if (p.pre_gelu) {
#pragma unroll
    for (int i = 0; i < 4 * NV; ++i) {
      const float x = v[i];
      v[i] = 0.5f * x * (1.0f + tanhf(0.7978845608028654f * (x + 0.044715f * x * x * x)));
    }
  }
  if (p.w1 != nullptr) rowg_layernorm<NV>(v, p.w1, p.b1, lane, p.eps);
  if (p.y_out != nullptr) rowg_store_f32<NV>(p.y_out + static_cast<long long>(row) * D, lane, v);
  if (p.z_out != nullptr) {
    if (p.w2 != nullptr) rowg_layernorm<NV>(v, p.w2, p.b2, lane, p.eps);
    rowg_store_bf16<NV>(p.z_out + static_cast<long long>(row) * D, lane, v);
  }
}

// Residual update + LayerNorm behind a split-K residual GEMM (gemm.cuh GemmParams::splits; the S2A form is layernorm_splitk_kernel):
// the text-to-semantic model decodes one sequence of a few hundred rows, so its long-K GEMMs (FeedForward down-projection, pointwise
// conv 2) always run as K ranges; this kernel adds their partial sums in range order, then bias, bf16 rounding, scale, residual add.
template <int NV>
__global__ void __launch_bounds__(256) layernorm_g_splitk_kernel(const LnGParams p) {
  pdl_sync();
  constexpr int D = 128 * NV;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row = blockIdx.x * 8 + warp;
  if (row >= p.rows) return;
  float v[4 * NV], a[4 * NV];
  const float* pr = p.partials + static_cast<long long>(row) * D;
  rowg_load_f32<NV>(pr, lane, a);
  if (p.n_partials == 4) {
    float b[4 * NV], c[4 * NV], d[4 * NV];
    rowg_load_f32<NV>(pr + p.partial_stride, lane, b);
    rowg_load_f32<NV>(pr + 2 * p.partial_stride, lane, c);
    rowg_load_f32<NV>(pr + 3 * p.partial_stride, lane, d);
    rowg_load_f32<NV>(p.x_io + static_cast<long long>(row) * D, lane, v);
#pragma unroll
    for (int i = 0; i < 4 * NV; ++i) a[i] = __fadd_rn(__fadd_rn(__fadd_rn(a[i], b[i]), c[i]), d[i]);
  } else {
    rowg_load_f32<NV>(p.x_io + static_cast<long long>(row) * D, lane, v);
    for (int s = 1; s < p.n_partials; ++s) {
      float b[4 * NV];
      rowg_load_f32<NV>(pr + s * p.partial_stride, lane, b);
#pragma unroll
      for (int i = 0; i < 4 * NV; ++i) a[i] = __fadd_rn(a[i], b[i]);
    }
  }
  if (p.lin_bias != nullptr) {
    float b[4 * NV];
    rowg_load_f32<NV>(p.lin_bias, lane, b);
#pragma unroll
    for (int i = 0; i < 4 * NV; ++i) a[i] = __fadd_rn(a[i], b[i]);
  }
#pragma unroll
  for (int i = 0; i < 4 * NV; ++i) v[i] = __fadd_rn(v[i], __fmul_rn(p.lin_scale, bf16_round(a[i])));
  if (p.y_out != p.x_io) rowg_store_f32<NV>(p.x_io + static_cast<long long>(row) * D, lane, v);
  if (p.w1 != nullptr) rowg_layernorm<NV>(v, p.w1, p.b1, lane, p.eps);
  if (p.y_out != nullptr) rowg_store_f32<NV>(p.y_out + static_cast<long long>(row) * D, lane, v);
  if (p.z_out != nullptr) {
    if (p.w2 != nullptr) rowg_layernorm<NV>(v, p.w2, p.b2, lane, p.eps);
    rowg_store_bf16<NV>(p.z_out + static_cast<long long>(row) * D, lane, v);
  }
}

// length head (:201-203): raw[s] = <LN_post(x[row_s, :]), w> + b on the length-token row of sequence s of the length predictor's
// output, row_s = cu_rows[s] (0 when cu_rows == nullptr: one sequence). One warp per sequence. x is the pre-post_norm residual stream;
// the post_norm of the last block is applied here.
template <int NV>
__global__ void __launch_bounds__(32) t2s_length_head_kernel(const float* x, const int* cu_rows, const float* ln_w, const float* ln_b, const float* w,
                                                             const float* b, float eps, float* raw_out) {
  pdl_sync();
  const int lane = threadIdx.x, s = blockIdx.x;
  const long long row = cu_rows != nullptr ? __ldg(cu_rows + s) : 0;
  float v[4 * NV], ww[4 * NV];
  rowg_load_f32<NV>(x + row * (128 * NV), lane, v);
  rowg_layernorm<NV>(v, ln_w, ln_b, lane, eps);
  rowg_load_f32<NV>(w, lane, ww);
  float acc = 0.f;
#pragma unroll
  for (int i = 0; i < 4 * NV; ++i) acc = fmaf(v[i], ww[i], acc);
  acc = warp_sum(acc);
  if (lane == 0) raw_out[s] = acc + b[0];
}

// The requests of a decode: sequence s is [text] bytes_s [sep] [speech] [mask] * length_s [sep] (:205-217), L_s = n_text_s + length_s + 4
// rows of `lay` starting at lay.n_start(s). Its text bytes start at cu_text[s] of the packed text, its speech tokens at cu_len[s] of the
// packed output. One sequence (cu_text == nullptr): n_text / length, both offsets 0.
struct T2sSeqs {
  SeqLayout lay;
  const int* cu_text;  // [n_seq + 1] or nullptr
  const int* cu_len;   // [n_seq + 1] or nullptr
  int n_text, length;  // the single sequence's

  __device__ __forceinline__ int text_start(int s) const { return cu_text != nullptr ? __ldg(cu_text + s) : 0; }
  __device__ __forceinline__ int n_text_of(int s) const { return cu_text != nullptr ? __ldg(cu_text + s + 1) - __ldg(cu_text + s) : n_text; }
  __device__ __forceinline__ int len_start(int s) const { return cu_len != nullptr ? __ldg(cu_len + s) : 0; }
  // the speech positions (full_mask) of sequence s are the rows [speech_start(s), speech_start(s) + length_s)
  __device__ __forceinline__ long long speech_start(int s) const { return static_cast<long long>(lay.n_start(s)) + n_text_of(s) + 3; }
};

// gather indices of the length predictor's input (:199): per sequence the length token (index -1, LnGParams::override_row), then the
// text embeddings. lay: the predictor layout, n_text_s + 1 rows per sequence.
__global__ void t2s_lp_gather_kernel(const T2sSeqs q, const int* text_tokens, int* gather) {
  pdl_sync();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= q.lay.rows) return;
  int s, n;
  q.lay.enc_pos(i, s, n);
  gather[i] = n == 0 ? -1 : text_tokens[q.text_start(s) + n - 1];
}

// token sequences of the requests (:205-222); full_mask marks the speech positions.
struct T2sBeginParams {
  T2sSeqs seqs;
  const int* text_tokens;  // packed [sum n_text_s], already shifted past the special tokens
  int tok_text, tok_sep, tok_speech, tok_mask;
  int* input_ids;          // [rows]
  int* tokens;             // [rows] the running "sampled_tokens"
  uint8_t* full_mask;      // [rows]
  uint8_t* mask;           // [rows] current mask = full_mask
};
__global__ void t2s_begin_kernel(const T2sBeginParams p) {
  pdl_sync();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.seqs.lay.rows) return;
  int s, n;
  p.seqs.lay.enc_pos(i, s, n);
  const int n_text = p.seqs.n_text_of(s), L = p.seqs.lay.n_len(s);
  int tok;
  uint8_t m = 0;
  if (n == 0) tok = p.tok_text;
  else if (n <= n_text) tok = p.text_tokens[p.seqs.text_start(s) + n - 1];
  else if (n == n_text + 1) tok = p.tok_sep;
  else if (n == n_text + 2) tok = p.tok_speech;
  else if (n < L - 1) { tok = p.tok_mask; m = 1; }
  else tok = p.tok_sep;
  p.input_ids[i] = tok;
  p.tokens[i] = tok;
  p.full_mask[i] = m;
  p.mask[i] = m;
}

// end of one iteration (:231-233 last iteration, :256-258 otherwise), row-local over the rows of every sequence:
//   last : tokens = full_mask ? id : input_ids
//   else : tokens = full_mask ? (next_mask ? [mask] : id + offset) : input_ids
struct T2sUpdateParams {
  const int* ids;            // [rows] sampled / arg-max ids (semantic vocabulary)
  const uint8_t* next_mask;  // [rows] or nullptr on the last iteration
  const uint8_t* full_mask;
  const int* input_ids;
  int* tokens;
  int rows, offset, tok_mask;
};
__global__ void t2s_update_kernel(const T2sUpdateParams p) {
  pdl_sync();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.rows) return;
  int tok = p.input_ids[i];
  if (p.full_mask[i]) {
    if (p.next_mask == nullptr) tok = p.ids[i];
    else tok = p.next_mask[i] ? p.tok_mask : p.ids[i] + p.offset;
  }
  p.tokens[i] = tok;
}

// speech_pred_tokens = sampled_tokens[full_mask] (:267) of every sequence, packed: out[len_start(s) + k] = tokens[speech_start(s) + k]
__global__ void t2s_gather_out_kernel(const T2sSeqs q, const int* tokens, int total, long long* out) {
  pdl_sync();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int s = q.cu_len != nullptr ? q.lay.search(q.cu_len, i) : 0;
  out[i] = tokens[q.speech_start(s) + (i - q.len_start(s))];
}

}  // namespace edm
