// HuBERT-large backbone of the semantic tokenizer (transformers HubertModel with feat_extract_norm="layer",
// do_stable_layer_norm=True; semantic_tokenizer_hubert.py:74-90 of the reference) - the kernels its encoder does not share with the
// S2A path. The transformer layers run on the S2A kernels unchanged (edm_layernorm, edm_gemm_bf16 with EPI_BF16 / EPI_GELU_BF16 /
// EPI_RESID_F32, edm_attention_varlen), the strided convs of the feature extractor on edm_dac_conv.
//
// Packed layout (HubertFeatures.forward_batch): clips sit back to back in one sample buffer, each starting at a multiple of the 320
// samples of one frame. The convs have no padding, so frame j of a clip at every conv stage reads only that clip's samples when
// j < T_i, and the stage-k rows of a clip start at its sample start / (5 * 2^(k-1)): every stage runs over all rows of the buffer
// and the rows past a clip's last valid frame hold finite junk that nothing valid reads. The transformer runs on the valid frames
// only, compacted to [sum T_i][1024] (cu offsets of attention); the positional conv reads them through a padded copy.
#pragma once
#include "gemm.cuh"
#include "t2s.cuh"

namespace edm {

constexpr int kHbC = 512;   // conv channels
constexpr int kHbK0 = 10, kHbS0 = 5;

// ------------------------------------------------------------------------------------------------ conv0 + LayerNorm + GELU
// Conv1d(1, 512, k 10, s 5) -> LayerNorm(512) -> GELU(erf), on CUDA cores (5120 MACs per frame; the kernel is bound by its bf16
// stores). A warp owns a frame: lane l holds channels {i * 128 + 4 l + q}, so the LayerNorm statistics are one warp reduction and
// the row leaves as coalesced 8-byte stores. Weights live in shared memory tap-major ([10][512]): every lane reads its own float4.
// Samples at index >= n_samples read as zero.
struct HbConv0Params {
  const float* audio;
  long long n_samples;
  int rows;                 // output frames
  const float* w;           // [10][512] fp32 (tap-major)
  const float* bias;        // [512]
  const float* ln_w;
  const float* ln_b;
  __nv_bfloat16* out;       // [rows][512]
};

__global__ void __launch_bounds__(256) hubert_conv0_kernel(const HbConv0Params p) {
  __shared__ float4 s_w[kHbK0 * kHbC / 4];
  __shared__ float4 s_b[kHbC / 4];
  for (int i = threadIdx.x; i < kHbK0 * kHbC / 4; i += blockDim.x) s_w[i] = __ldg(reinterpret_cast<const float4*>(p.w) + i);
  for (int i = threadIdx.x; i < kHbC / 4; i += blockDim.x) s_b[i] = __ldg(reinterpret_cast<const float4*>(p.bias) + i);
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int warps = gridDim.x * (blockDim.x >> 5);
  for (int f = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); f < p.rows; f += warps) {
    const long long s0 = static_cast<long long>(f) * kHbS0;
    const float mine = (lane < kHbK0 && s0 + lane < p.n_samples) ? __ldg(p.audio + s0 + lane) : 0.f;
    float v[16];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 b = s_b[i * 32 + lane];
      v[4 * i] = b.x; v[4 * i + 1] = b.y; v[4 * i + 2] = b.z; v[4 * i + 3] = b.w;
    }
#pragma unroll
    for (int j = 0; j < kHbK0; ++j) {
      const float x = __shfl_sync(0xffffffffu, mine, j);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float4 w = s_w[j * (kHbC / 4) + i * 32 + lane];
        v[4 * i] = fmaf(x, w.x, v[4 * i]); v[4 * i + 1] = fmaf(x, w.y, v[4 * i + 1]);
        v[4 * i + 2] = fmaf(x, w.z, v[4 * i + 2]); v[4 * i + 3] = fmaf(x, w.w, v[4 * i + 3]);
      }
    }
    rowg_layernorm<4>(v, p.ln_w, p.ln_b, lane, 1e-5f);
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = gelu_erf(v[i]);
    rowg_store_bf16<4>(p.out + static_cast<long long>(f) * kHbC, lane, v);
  }
}

// ------------------------------------------------------------------------------------------------ LayerNorm(512) [+ GELU]
// out[r] = act(LN(in[gather ? gather[r] : r])), bf16 in and out, one warp per row. With gelu != 0 it follows each strided conv of the
// feature extractor (conv -> LayerNorm -> GELU, in place on the conv's bf16 output); with gelu == 0 it is the feature projection's
// LayerNorm, gathering the valid frames of the packed conv output into the compact rows of the transformer.
struct HbLnParams {
  const __nv_bfloat16* in;
  const int* gather;   // nullable
  int rows;
  const float* w;
  const float* b;
  int gelu;
  __nv_bfloat16* out;
};

__global__ void __launch_bounds__(256) hubert_ln512_kernel(const HbLnParams p) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= p.rows) return;
  const long long src = p.gather != nullptr ? p.gather[row] : row;
  float v[16];
  rowg_load_bf16<4>(p.in + src * kHbC, lane, v);
  rowg_layernorm<4>(v, p.w, p.b, lane, 1e-5f);
  if (p.gelu) {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = gelu_erf(v[i]);
  }
  rowg_store_bf16<4>(p.out + static_cast<long long>(row) * kHbC, lane, v);
}

// ------------------------------------------------------------------------------------------------ padded operand of the pos conv
// out[r] = bf16(x[map[r]]) or zeros when map[r] < 0: the compact fp32 stream [N][1024] laid out with zero rows around every sequence
// (DESIGN §4b), so that the positional conv's zero padding is plain data and one launch covers a packed batch.
__global__ void __launch_bounds__(256) hubert_pad_rows_kernel(const float* x, const int* map, int rows, __nv_bfloat16* out) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int src = map[row];
  float v[32];
  if (src >= 0) {
    row_load_f32(x + static_cast<long long>(src) * kD, lane, v);
  } else {
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = 0.f;
  }
  row_store_bf16(out + static_cast<long long>(row) * kD, lane, v);
}

// ------------------------------------------------------------------------------------------------ positional conv (tcgen05)
// HubertPositionalConvEmbedding: Conv1d(1024, 1024, k 128, padding 64, groups 16) -> SamePad (drop the last frame) -> GELU, added to
// the residual stream (HubertEncoderStableLayerNorm.forward). Group g is an implicit GEMM of M = rows, N = 64, K = 128 taps x 64:
//     D[t, n] = sum_j sum_c  xp[t - 64 + j, 64 g + c] * W[64 g + n, 64 j + c]
// over the padded operand xp (hubert_pad_rows_kernel: every sequence has >= 64 zero rows on each side, rows before 0 are zero-filled
// by TMA). A work item is one (128-row tile, group); its K loop walks the 128 taps, each one (A box 128 rows x 64 channels shifted by a
// row, W box 64 x 64). Epilogue: x[map[t], 64 g + n] += bf16(GELU(bf16(D + bias))) for the rows with map[t] >= 0 (single writer per
// element). Warp roles as dac_conv_kernel: 0 TMA producer, 1 MMA issuer, 2-9 epilogue (two per TMEM lane quadrant, 32 columns each).
constexpr int kPcThreads = 320;
constexpr int kPcStages = 6;
constexpr int kPcTaps = 128;
constexpr uint32_t kPcABytes = 128 * 64 * 2;
constexpr uint32_t kPcBBytes = 64 * 64 * 2;
constexpr uint32_t kPcStageBytes = kPcABytes + kPcBBytes;
constexpr uint32_t kPcSmemBytes = kPcStages * kPcStageBytes + 1024 + 256;

struct HbPosConvParams {
  int rows;            // padded rows (the operand's and the map's)
  const float* bias;   // [1024]
  const int* map;      // [rows]: compact row of padded row t, or -1
  float* x;            // [N][1024] fp32 residual stream
};

__global__ void __launch_bounds__(kPcThreads, 1)
hubert_pos_conv_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_w, const HbPosConvParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kPcStages * kPcStageBytes);
  uint64_t* empty_bar = full_bar + kPcStages;
  uint64_t* tfull_bar = empty_bar + kPcStages;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_tiles = ((p.rows + 127) / 128) * 16;
  const int my_tiles = (num_tiles - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_w);
    for (int s = 0; s < kPcStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tfull_bar[b], 1);
      mbar_init(&tempty_bar[b], 256);
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc<128>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      uint32_t it = 0;
      for (int tl = 0; tl < my_tiles; ++tl) {
        const int tile = blockIdx.x + tl * gridDim.x;
        const int g = tile & 15, t0 = (tile >> 4) * 128;
        for (int j = 0; j < kPcTaps; ++j, ++it) {
          const uint32_t s = it % kPcStages;
          uint8_t* st = smem + s * kPcStageBytes;
          mbar_wait(&empty_bar[s], ((it / kPcStages) & 1) ^ 1);
          mbar_arrive_expect_tx(&full_bar[s], kPcStageBytes);
          tma_load_2d(&tma_a, &full_bar[s], st, g * 64, t0 - kPcTaps / 2 + j);
          tma_load_2d(&tma_w, &full_bar[s], st + kPcABytes, j * 64, g * 64);
        }
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = umma_idesc_bf16(128, 64, 0, 0);
    uint32_t it = 0;
    for (int tl = 0; tl < my_tiles; ++tl) {
      const uint32_t buf = tl & 1;
      mbar_wait(&tempty_bar[buf], ((tl >> 1) & 1) ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + buf * 64;
      for (int j = 0; j < kPcTaps; ++j, ++it) {
        const uint32_t s = it % kPcStages;
        mbar_wait_spin(&full_bar[s], (it / kPcStages) & 1);
        tc_fence_after();
        const uint32_t st = smem_u32(smem + s * kPcStageBytes);
        const uint64_t a_desc = umma_desc_sw128(st, 16, 1024), b_desc = umma_desc_sw128(st + kPcABytes, 16, 1024);
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_ss_warp(d_tmem, a_desc + 2 * k, b_desc + 2 * k, idesc, (j | k) != 0 ? 1u : 0u);
        umma_commit_warp(&empty_bar[s]);
      }
      umma_commit_warp(&tfull_bar[buf]);
    }
  } else {
    const int quad = warp & 3, half = (warp - 2) >> 2;
    for (int tl = 0; tl < my_tiles; ++tl) {
      const int tile = blockIdx.x + tl * gridDim.x;
      const int g = tile & 15, t = (tile >> 4) * 128 + quad * 32 + lane;
      const int col = g * 64 + half * 32;
      const uint32_t buf = tl & 1;
      const int dst = t < p.rows ? __ldg(p.map + t) : -1;
      float4 xo[8];
      float* xrow = p.x + static_cast<long long>(dst < 0 ? 0 : dst) * kD + col;
      if (dst >= 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) xo[i] = *reinterpret_cast<const float4*>(xrow + 4 * i);
      }
      mbar_wait(&tfull_bar[buf], (tl >> 1) & 1);
      tc_fence_after();
      uint32_t r[32];
      tmem_ld_32x32(tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + buf * 64 + half * 32, r);
      tmem_ld_wait_dep(r);
      tc_fence_before();
      mbar_arrive(&tempty_bar[buf]);
      if (dst < 0) continue;
      const float4* b4 = reinterpret_cast<const float4*>(p.bias + col);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float4 b = __ldg(b4 + i);
        float4 o = xo[i];
        o.x += bf16_round(gelu_erf(bf16_round(__uint_as_float(r[4 * i + 0]) + b.x)));
        o.y += bf16_round(gelu_erf(bf16_round(__uint_as_float(r[4 * i + 1]) + b.y)));
        o.z += bf16_round(gelu_erf(bf16_round(__uint_as_float(r[4 * i + 2]) + b.z)));
        o.w += bf16_round(gelu_erf(bf16_round(__uint_as_float(r[4 * i + 3]) + b.w)));
        *reinterpret_cast<float4*>(xrow + 4 * i) = o;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc<128>(tmem_base);
}

}  // namespace edm
