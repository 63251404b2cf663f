// DAC encoder convolutions as implicit GEMMs on tcgen05 (kind::f16, bf16 operands, fp32 accumulators in TMEM).
// Reference: edm_tts/models/dac/encoder.py:11-58 (Encoder / EncoderBlock), edm_tts/models/dac/nn_layers.py:8-47 (WNConv1d,
// Snake1d, ResidualUnit); the reference runs this stack under bf16 autocast (utility_scripts/dump_tokens/dump_tokens.py:213).
//
// Data layout. Activations are channel-last: [batch][time][channels]. Every conv reads a bf16 "operand" tensor that already holds
// Snake(x) (each conv of the encoder except the first is preceded by a Snake), written by the epilogue of the producing kernel, and
// the residual stream stays fp32. A conv with taps j = 0..n_taps-1 is then
//     D[t, co] = sum_j sum_ci  A[t + row_off + j * tap_step, ci] * W[co, j * Cin + ci]
// i.e. a GEMM whose K loop walks (tap, 64-channel chunk) and whose A tile of each K step is one TMA box of the operand tensor at a
// shifted time coordinate. The tensor map is 3-D (channels, time, batch): rows before 0 or past the end of a sequence are
// zero-filled by TMA, which is exactly the conv's zero padding (Snake(0) = 0), and batches never bleed into each other.
//   * dilated k=7 conv of a ResidualUnit: n_taps 7, tap_step = dilation, row_off = -3 * dilation
//   * 1x1 conv: n_taps 1
//   * strided conv (kernel 2s, stride s, padding ceil(s/2)): the producer writes the operand into a buffer with `pad` zero rows in
//     front, viewed as [time / s][s * C]: output t reads buffer rows t and t + 1 of that view -> n_taps 2, tap_step 1, Cin = s * C
//   * last conv (k=3, pad 1): n_taps 3, tap_step 1, row_off -1
// Weights are packed [Cout][n_taps * Cin] bf16 (K-major), weight-norm folded at load.
//
// Epilogue (thread <-> time row, fused, runtime-selected): v = acc + bias [+ x_res]; y = v (fp32 stream); s_out = bf16(Snake_alpha(v))
// (operand of the next conv, possibly in the padded layout of a strided conv); zt_out = v transposed to [batch][channel][time]
// (the latent z handed to the RVQ, reference layout).
//
//   warp 0     : TMA producer (A box 128 rows x 64 channels, W box NT rows x 64, NT in {64, 128, 192, 256}), 3-4 stage ring
//   warp 1     : MMA issuer (whole warp, elected lane), accumulator double-buffered in TMEM (2 x NT columns)
//   warps 2-9  : epilogue, two warps per TMEM lane quadrant, each owning half of the tile's columns. A thread owns a time row, so
//                direct global accesses would touch 32 different lines per warp instruction; instead every warp has a staging
//                box in shared memory: the residual x is fetched with fully coalesced loads (4 rows x 128 B per instruction, one
//                chunk ahead) and transposed through the box, and y (fp32) / s_out (bf16) leave as swizzled 32-row TMA store
//                boxes whose tensor maps clip the ragged last tile
#pragma once
#include "ptx.cuh"

namespace edm {

constexpr int kDcThreads = 320;
template <int NT> struct DacConvStages { static constexpr int value = NT >= 192 ? 3 : 4; };
constexpr uint32_t kDcStagingBytes = 4096 + 2048;   // per epilogue warp: y box (32 rows x 128 B, swizzle 128B) + s box (32 rows x 64 B, swizzle 64B)
constexpr int kDcBM = 128;
constexpr uint32_t kDcABytes = kDcBM * 64 * 2;  // 16 KB
constexpr int kDcMaxCout = 1536;   // capacity of the per-channel constant staging (bias / Snake alpha period)

struct DacConvParams {
  int B, rows_out, tiles_per_batch, c_out, n_tiles_n;
  int n_taps, tap_step, row_off, k_chunks;  // k_chunks = Cin / 64
  int c_mod;                                // period of bias / alpha along the output columns (c_out, or C for a transposed conv
                                            // whose columns are s phases x C channels)
  const float* bias;                        // [c_mod]
  const float* alpha;                       // [c_mod] Snake of the NEXT layer, applied to what goes to s_out; nullptr: identity
  const float* x_res;                       // fp32 [B][rows_out][c_out] residual input or nullptr (may alias y)
  float* y;                                 // fp32 stream out or nullptr
  long long y_batch_stride;                 // elements
  __nv_bfloat16* s_out;                     // bf16 operand out or nullptr: row (t + s_row_off) of batch b; the tensor map drops rows >= s_rows
  long long s_batch_stride;
  int s_row_off, s_rows;
  void* zt_out;                             // [B][c_out][rows_out] (bf16 or fp32) or nullptr
  int zt_is_f32;
};

template <int NT>
constexpr uint32_t dac_conv_smem_bytes() {
  return DacConvStages<NT>::value * (kDcABytes + NT * 128) + 8 * kDcStagingBytes + 3 * kDcMaxCout * 4 + 1024 + 256;
}

__device__ __forceinline__ float snake_act(float v, float a, float inv_a) {
  const float s = __sinf(a * v);
  return fmaf(inv_a * s, s, v);
}

template <int NT>
__global__ void __launch_bounds__(kDcThreads, 1)
dac_conv_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_w, const __grid_constant__ CUtensorMap tma_y,
                const __grid_constant__ CUtensorMap tma_s, const DacConvParams p) {
  constexpr int kDcStages = DacConvStages<NT>::value;
  constexpr uint32_t kBBytes = NT * 128;
  constexpr uint32_t kStageBytes = kDcABytes + kBBytes;
  constexpr int kTmemCols = 2 * NT <= 128 ? 128 : (2 * NT <= 256 ? 256 : 512);   // power of two >= 2 * NT
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* staging = smem + kDcStages * kStageBytes;
  float* s_bias = reinterpret_cast<float*>(staging + 8 * kDcStagingBytes);
  float* s_alpha = s_bias + kDcMaxCout;
  float* s_inva = s_alpha + kDcMaxCout;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(s_inva + kDcMaxCout);
  uint64_t* empty_bar = full_bar + kDcStages;
  uint64_t* tfull_bar = empty_bar + kDcStages;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_tiles = p.B * p.tiles_per_batch * p.n_tiles_n;
  const int my_tiles = (num_tiles - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);
  const int k_steps = p.n_taps * p.k_chunks;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_w);
    if (p.y != nullptr) tma_prefetch_desc(&tma_y);
    if (p.s_out != nullptr) tma_prefetch_desc(&tma_s);
    for (int s = 0; s < kDcStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tfull_bar[b], 1);
      mbar_init(&tempty_bar[b], 256);
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc<kTmemCols>(tmem_slot);
  for (int i = threadIdx.x; i < p.c_mod; i += kDcThreads) {
    s_bias[i] = __ldg(p.bias + i);
    const float a = p.alpha != nullptr ? __ldg(p.alpha + i) : 1.0f;
    s_alpha[i] = a;
    s_inva[i] = 1.0f / (a + 1e-9f);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // tile -> (n tile fastest, then time tile, then batch): CTAs running side by side share the A rows in L2
  auto decode = [&](int tile, int& b, int& t0, int& n0) {
    n0 = (tile % p.n_tiles_n) * NT;
    const int mt = tile / p.n_tiles_n;
    t0 = (mt % p.tiles_per_batch) * kDcBM;
    b = mt / p.tiles_per_batch;
  };

  if (warp == 0) {
    if (lane == 0) {
      uint32_t it = 0;
      for (int tl = 0; tl < my_tiles; ++tl) {
        int b, t0, n0;
        decode(blockIdx.x + tl * gridDim.x, b, t0, n0);
        for (int j = 0; j < p.n_taps; ++j) {
          const int row = t0 + p.row_off + j * p.tap_step;
          for (int c = 0; c < p.k_chunks; ++c, ++it) {
            const uint32_t s = it % kDcStages;
            uint8_t* st = smem + s * kStageBytes;
            mbar_wait(&empty_bar[s], ((it / kDcStages) & 1) ^ 1);
            mbar_arrive_expect_tx(&full_bar[s], kStageBytes);
            tma_load_3d(&tma_a, &full_bar[s], st, c * 64, row, b);
            tma_load_2d(&tma_w, &full_bar[s], st + kDcABytes, (j * p.k_chunks + c) * 64, n0);
          }
        }
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = umma_idesc_bf16(kDcBM, NT, 0, 0);
    uint32_t it = 0;
    for (int tl = 0; tl < my_tiles; ++tl) {
      const uint32_t buf = tl & 1;
      mbar_wait(&tempty_bar[buf], ((tl >> 1) & 1) ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + buf * NT;
      for (int ks = 0; ks < k_steps; ++ks, ++it) {
        const uint32_t s = it % kDcStages;
        mbar_wait_spin(&full_bar[s], (it / kDcStages) & 1);
        tc_fence_after();
        const uint32_t st = smem_u32(smem + s * kStageBytes);
        const uint64_t a_desc = umma_desc_sw128(st, 16, 1024), b_desc = umma_desc_sw128(st + kDcABytes, 16, 1024);
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_ss_warp(d_tmem, a_desc + 2 * k, b_desc + 2 * k, idesc, (ks | k) != 0 ? 1u : 0u);
        umma_commit_warp(&empty_bar[s]);
      }
      umma_commit_warp(&tfull_bar[buf]);
    }
  } else {
    const int quad = warp & 3;
    const int half = (warp - 2) >> 2;
    const int r_in = quad * 32 + lane;
    constexpr int kColsPerWarp = NT / 2;
    constexpr int kChunks = kColsPerWarp / 32;
    uint8_t* stg_y = staging + (warp - 2) * kDcStagingBytes;
    uint8_t* stg_s = stg_y + 4096;
    const uint32_t y_row = smem_u32(stg_y) + lane * 128;
    const uint32_t s_row = smem_u32(stg_s) + lane * 64;
    const int sw = lane & 7, sw64 = (lane >> 1) & 3;
    const int xr_row = lane >> 3, xr_ch = lane & 7;      // coalesced pattern: instruction k covers rows 4k .. 4k+3 of the warp's 32
    const bool has_res = p.x_res != nullptr;
    const bool has_y = p.y != nullptr, has_s = p.s_out != nullptr, has_alpha = p.alpha != nullptr;
    const int total_chunks = my_tiles * kChunks;

    // residual rows of flat chunk q (tile q / kChunks, column chunk q % kChunks), fetched one chunk ahead
    auto load_x = [&](int q, float4 (&xr)[8]) {
      int b, t0, n0;
      decode(blockIdx.x + (q / kChunks) * gridDim.x, b, t0, n0);
      const int col = n0 + half * kColsPerWarp + (q % kChunks) * 32;
      const float* base = p.x_res + static_cast<long long>(b) * p.y_batch_stride + col + xr_ch * 4;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int t = t0 + quad * 32 + k * 4 + xr_row;
        xr[k] = t < p.rows_out ? __ldg(reinterpret_cast<const float4*>(base + static_cast<long long>(t) * p.c_out)) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
    float4 xr[8];
    if (has_res && total_chunks > 0) load_x(0, xr);

    for (int tl = 0; tl < my_tiles; ++tl) {
      int b, t0, n0;
      decode(blockIdx.x + tl * gridDim.x, b, t0, n0);
      const uint32_t buf = tl & 1;
      const int t = t0 + r_in;
      mbar_wait(&tfull_bar[buf], (tl >> 1) & 1);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + buf * NT + half * kColsPerWarp;
#pragma unroll 1
      for (int cc = 0; cc < kChunks; ++cc) {
        uint32_t r[32];
        tmem_ld_32x32(taddr + cc * 32, r);
        tmem_ld_wait_dep(r);
        if (cc == kChunks - 1) {
          tc_fence_before();
          mbar_arrive(&tempty_bar[buf]);
        }
        const int col = n0 + half * kColsPerWarp + cc * 32;
        const int ccol = col % p.c_mod;      // channel of the chunk's first column (chunks never straddle a period: c_mod % 32 == 0)
        float v[32];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 b4 = lds128(smem_u32(s_bias + ccol) + 16 * i);
          v[4 * i] = __uint_as_float(r[4 * i]) + b4.x; v[4 * i + 1] = __uint_as_float(r[4 * i + 1]) + b4.y;
          v[4 * i + 2] = __uint_as_float(r[4 * i + 2]) + b4.z; v[4 * i + 3] = __uint_as_float(r[4 * i + 3]) + b4.w;
        }
        // the previous chunk's store boxes have been read out of the staging buffers
        if (lane == 0) bulk_wait_group_read0();
        __syncwarp();
        if (has_res) {
#pragma unroll
          for (int k = 0; k < 8; ++k) sts128(smem_u32(stg_y) + (k * 4 + xr_row) * 128 + ((xr_ch ^ ((k * 4 + xr_row) & 7)) << 4), xr[k]);
          __syncwarp();
          const int q = tl * kChunks + cc + 1;
          if (q < total_chunks) load_x(q, xr);     // next chunk's residual rows: in flight during this chunk's math and stores
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float4 x4 = lds128(y_row + ((i ^ sw) << 4));
            v[4 * i] += x4.x; v[4 * i + 1] += x4.y; v[4 * i + 2] += x4.z; v[4 * i + 3] += x4.w;
          }
        }
        if (has_y) {
#pragma unroll
          for (int i = 0; i < 8; ++i) sts128(y_row + ((i ^ sw) << 4), make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]));
        }
        if (p.zt_out != nullptr && t < p.rows_out) {
          const long long zo = (static_cast<long long>(b) * p.c_out + col) * p.rows_out + t;
          if (p.zt_is_f32) {
            float* z = static_cast<float*>(p.zt_out) + zo;
#pragma unroll
            for (int e = 0; e < 32; ++e) z[static_cast<long long>(e) * p.rows_out] = v[e];
          } else {
            __nv_bfloat16* z = static_cast<__nv_bfloat16*>(p.zt_out) + zo;
#pragma unroll
            for (int e = 0; e < 32; ++e) z[static_cast<long long>(e) * p.rows_out] = __float2bfloat16(v[e]);
          }
        }
        if (has_s) {
          uint32_t w[16];
          if (has_alpha) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float4 a4 = lds128(smem_u32(s_alpha + ccol) + 16 * i), ia4 = lds128(smem_u32(s_inva + ccol) + 16 * i);
              w[2 * i] = pack_bf16x2(snake_act(v[4 * i], a4.x, ia4.x), snake_act(v[4 * i + 1], a4.y, ia4.y));
              w[2 * i + 1] = pack_bf16x2(snake_act(v[4 * i + 2], a4.z, ia4.z), snake_act(v[4 * i + 3], a4.w, ia4.w));
            }
          } else {
#pragma unroll
            for (int e = 0; e < 16; ++e) w[e] = pack_bf16x2(v[2 * e], v[2 * e + 1]);
          }
#pragma unroll
          for (int i = 0; i < 4; ++i)
            sts128(s_row + ((i ^ sw64) << 4), make_float4(__uint_as_float(w[4 * i]), __uint_as_float(w[4 * i + 1]), __uint_as_float(w[4 * i + 2]),
                                                          __uint_as_float(w[4 * i + 3])));
        }
        if (has_y || has_s) {
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            if (has_y) tma_store_3d(&tma_y, stg_y, col, t0 + quad * 32, b);
            if (has_s) tma_store_3d(&tma_s, stg_s, col, t0 + quad * 32 + p.s_row_off, b);
            bulk_commit_group();
          }
        }
      }
    }
    if (lane == 0) bulk_wait_group0();   // all stores have landed before the CTA exits
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc<kTmemCols>(tmem_base);
}

// ------------------------------------------------------------------------------------------------------------------------------
// Fused ResidualUnit (nn_layers.py:33-47) for the 64- and 128-channel stages, where the two convs run one after the other on the
// same 128-row tile so that the hidden activation never goes to HBM:
//     h = Snake_mid(conv7_dilated(sx) + b7)  ->  bf16 tile in shared memory (the A operand of the second GEMM)
//     y = x + conv1x1(h) + b1 ;  s_out = bf16(Snake_next(y))
// HBM traffic per row: sx (2C) + x (4C) in, y (4C) + s_out (2C) out = 12 C bytes instead of 16 C for the two-launch form.
// Two kernels: dac_resunit_kernel<C> (general, used at 128 channels: weights streamed through a ring, phases on separate
// warpgroups) and dac_resunit64_kernel (64 channels: weights resident in shared memory). Both read the input rows once per tile with
// their halo and address the seven taps through row-shifted UMMA descriptors.
//   phase 1: acc1 -> + b7 -> Snake_mid -> bf16 -> h tile (swizzled K-major, the A operand of GEMM 2)
//   phase 2: acc2 -> + b1 + x -> y (fp32 stream) and Snake_next -> s_out (the residual epilogue of dac_conv_kernel)
struct DacResUnitParams {
  int B, rows, tiles_per_batch, dilation;
  const float* b7; const float* a_mid; const float* b1; const float* a_next;   // [C] each
  float* y; long long y_batch_stride;                                          // fp32 stream, updated in place
#ifdef EDM_DAC_TRACE
  unsigned long long* trace;   // bring-up build only (tools/gpu_dac_trace.sh): clock64 stamps of CTA 0, [tile][16 events]
#endif
};
#ifdef EDM_DAC_TRACE
#define DAC_TRACE(tl, k) do { if (blockIdx.x == 0 && p.trace != nullptr && (tl) < 64 && lane == 0) p.trace[(tl) * 16 + (k)] = clock64(); } while (0)
#else
#define DAC_TRACE(tl, k) do { } while (0)
#endif

constexpr int kRu64HaloRows = 192;                                 // >= 128 + 6 * 9
constexpr uint32_t kRu64HaloBytes = kRu64HaloRows * 128;           // 24 KB per 64-channel chunk

template <int C>
struct DacResUnitCfg {
  static constexpr int kStages = 5;                                   // weight chunks [C x 64] in flight
  static constexpr uint32_t kStageBytes = C * 128;
  static constexpr uint32_t kHaloBytes = (C / 64) * kRu64HaloBytes;   // input rows with their halo, one box per 64-channel chunk
  static constexpr uint32_t kHBytes = 128 * C * 2;
  static constexpr uint32_t kSmemBytes = kStages * kStageBytes + kHaloBytes + kHBytes + 8 * kDcStagingBytes + 6 * C * 4 + 1024 + 256;
};
constexpr int kRuThreads = 512;

// Warp roles (four warpgroups, registers redistributed with setmaxnreg): warp 0 TMA producer, warp 1 MMA issuer, warps 4-7 phase 1
// (one per TMEM lane quadrant, all C columns), warps 8-15 phase 2 (two per quadrant, half of the columns each). The epilogue phases
// are latency-bound chains (TMEM load -> math -> shared / global memory), and with both phases on the same eight warps they bounded
// the kernel (7.7 us per 128-channel tile against 4.5 us of HBM time); on separate warps phase 1 of tile i+1 runs beside phase 2 of
// tile i. Both accumulators are double-buffered (TMEM columns: acc1[0] [0,C) acc1[1] [C,2C) acc2[0] [2C,3C) acc2[1] [3C,4C)); the
// MMA warp issues GEMM 1 of tile i+1 before GEMM 2 of tile i and the producer feeds the ring in that order.
// With the phases off its back the kernel is bound by TMA latency x bytes in flight (clock64 timeline, tools/gpu_dac_trace.sh: 600
// cycles per K step with three 32 KB (A + W) stages), so the input rows are loaded once per tile with their halo (one box per
// 64-channel chunk, taps = row-shifted descriptors, see dac_resunit64_kernel) and the ring carries five 16 KB weight chunks.
// Buffer reuse: acc1[s] (GEMM 1 of tile i+2) <- the MMA warp has waited hfull of tile i; the halo tile (tile i+1) <- aempty, committed
// after GEMM 1 of tile i; h (phase 1 of tile i+1) <- the phase-1 warps wait t2full of tile i (GEMM 2 has read h); acc2[s] (GEMM 2 of
// tile i+2) <- the MMA warp waits t2empty[s] of tile i.
template <int C>
__global__ void __launch_bounds__(kRuThreads, 1)
dac_resunit_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_w7, const __grid_constant__ CUtensorMap tma_w1,
                   const __grid_constant__ CUtensorMap tma_y, const __grid_constant__ CUtensorMap tma_s, const DacResUnitParams p, const int s_row_off) {
  constexpr int kStages = DacResUnitCfg<C>::kStages;
  constexpr int kKc = C / 64;                       // 64-channel chunks
  constexpr uint32_t kStageBytes = DacResUnitCfg<C>::kStageBytes;
  constexpr uint32_t kHBytes = DacResUnitCfg<C>::kHBytes;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* s_a = smem + kStages * kStageBytes;      // kKc halo tiles of [<= 192 rows x 64 channels]
  uint8_t* s_h = s_a + DacResUnitCfg<C>::kHaloBytes;   // kKc sub-tiles of [128 rows x 64 channels] bf16, 128B-swizzled
  uint8_t* staging = s_h + kHBytes;
  float* s_b7 = reinterpret_cast<float*>(staging + 8 * kDcStagingBytes);
  float* s_am = s_b7 + C;
  float* s_iam = s_am + C;
  float* s_b1 = s_iam + C;
  float* s_an = s_b1 + C;
  float* s_ian = s_an + C;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(s_ian + C);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* t1full_bar = empty_bar + kStages;  // [2]
  uint64_t* hfull_bar = t1full_bar + 2;        // [2]
  uint64_t* t2full_bar = hfull_bar + 2;        // [2]
  uint64_t* t2empty_bar = t2full_bar + 2;      // [2]
  uint64_t* afull_bar = t2empty_bar + 2;
  uint64_t* aempty_bar = afull_bar + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(aempty_bar + 1);
  const uint32_t halo_bytes = static_cast<uint32_t>(128 + 6 * p.dilation) * 128;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_tiles = p.B * p.tiles_per_batch;
  const int my_tiles = (num_tiles - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_w7);
    tma_prefetch_desc(&tma_w1);
    tma_prefetch_desc(&tma_y);
    tma_prefetch_desc(&tma_s);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&t1full_bar[s], 1);
      mbar_init(&hfull_bar[s], 128);
      mbar_init(&t2full_bar[s], 1);
      mbar_init(&t2empty_bar[s], 256);
    }
    mbar_init(afull_bar, 1);
    mbar_init(aempty_bar, 1);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc<4 * C>(tmem_slot);
  for (int i = threadIdx.x; i < C; i += kRuThreads) {
    s_b7[i] = __ldg(p.b7 + i);
    s_b1[i] = __ldg(p.b1 + i);
    const float am = __ldg(p.a_mid + i), an = __ldg(p.a_next + i);
    s_am[i] = am; s_iam[i] = 1.0f / (am + 1e-9f);
    s_an[i] = an; s_ian[i] = 1.0f / (an + 1e-9f);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 72;");
    if (warp == 0) {
      if (lane == 0) {
        uint32_t it = 0;
        auto feed1 = [&](int tl) {      // the halo tile, then 7 * kKc W7 chunks
          const int tile = blockIdx.x + tl * gridDim.x;
          const int t0 = (tile % p.tiles_per_batch) * kDcBM, b = tile / p.tiles_per_batch;
          mbar_wait(aempty_bar, (tl & 1) ^ 1);   // GEMM 1 of the previous tile has read the halo tiles
          mbar_arrive_expect_tx(afull_bar, kKc * halo_bytes);
          for (int c = 0; c < kKc; ++c) tma_load_3d(&tma_a, afull_bar, s_a + c * kRu64HaloBytes, c * 64, t0 - 3 * p.dilation, b);
          for (int j = 0; j < 7; ++j) {
            for (int c = 0; c < kKc; ++c, ++it) {
              const uint32_t s = it % kStages;
              mbar_wait(&empty_bar[s], ((it / kStages) & 1) ^ 1);
              mbar_arrive_expect_tx(&full_bar[s], kStageBytes);
              tma_load_2d(&tma_w7, &full_bar[s], smem + s * kStageBytes, (j * kKc + c) * 64, 0);
            }
          }
        };
        auto feed2 = [&]() {            // kKc stages: W1 chunks
          for (int c = 0; c < kKc; ++c, ++it) {
            const uint32_t s = it % kStages;
            mbar_wait(&empty_bar[s], ((it / kStages) & 1) ^ 1);
            mbar_arrive_expect_tx(&full_bar[s], kStageBytes);
            tma_load_2d(&tma_w1, &full_bar[s], smem + s * kStageBytes, c * 64, 0);
          }
        };
        if (my_tiles > 0) feed1(0);
        for (int tl = 0; tl < my_tiles; ++tl) {
          if (tl + 1 < my_tiles) feed1(tl + 1);
          feed2();
        }
      }
    } else if (warp == 1) {
      constexpr uint32_t idesc = umma_idesc_bf16(kDcBM, C, 0, 0);
      uint32_t it = 0;
      auto gemm1 = [&](int tl) {
        DAC_TRACE(tl, 0);
        const uint32_t d_tmem = tmem_base + (tl & 1) * C;
        mbar_wait_spin(afull_bar, tl & 1);
        tc_fence_after();
        for (int ks = 0; ks < 7 * kKc; ++ks, ++it) {
          const uint32_t s = it % kStages;
          mbar_wait_spin(&full_bar[s], (it / kStages) & 1);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(s_a) + (ks % kKc) * kRu64HaloBytes + (ks / kKc) * p.dilation * 128;   // tap = row shift
          const uint64_t a_desc = umma_desc_sw128(a_addr, 16, 1024), b_desc = umma_desc_sw128(smem_u32(smem + s * kStageBytes), 16, 1024);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_ss_warp(d_tmem, a_desc + 2 * k, b_desc + 2 * k, idesc, (ks | k) != 0 ? 1u : 0u);
          umma_commit_warp(&empty_bar[s]);
        }
        umma_commit_warp(aempty_bar);
        umma_commit_warp(&t1full_bar[tl & 1]);
        DAC_TRACE(tl, 1);
      };
      if (my_tiles > 0) gemm1(0);
      for (int tl = 0; tl < my_tiles; ++tl) {
        if (tl + 1 < my_tiles) gemm1(tl + 1);
        mbar_wait_spin(&hfull_bar[tl & 1], (tl >> 1) & 1);
        DAC_TRACE(tl, 2);
        mbar_wait_spin(&t2empty_bar[tl & 1], ((tl >> 1) & 1) ^ 1);   // phase 2 of tile tl - 2 has drained acc2[tl & 1]
        tc_fence_after();
        DAC_TRACE(tl, 3);
        for (int c = 0; c < kKc; ++c, ++it) {
          const uint32_t s = it % kStages;
          mbar_wait_spin(&full_bar[s], (it / kStages) & 1);
          tc_fence_after();
          const uint64_t a_desc = umma_desc_sw128(smem_u32(s_h) + c * kDcABytes, 16, 1024);
          const uint64_t b_desc = umma_desc_sw128(smem_u32(smem + s * kStageBytes), 16, 1024);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_ss_warp(tmem_base + 2 * C + (tl & 1) * C, a_desc + 2 * k, b_desc + 2 * k, idesc, (c | k) != 0 ? 1u : 0u);
          umma_commit_warp(&empty_bar[s]);
        }
        umma_commit_warp(&t2full_bar[tl & 1]);
        DAC_TRACE(tl, 4);
      }
    }
  } else if (warp < 8) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 104;");
    // ---- phase 1: h = Snake_mid(acc1 + b7) -> bf16, this thread's row of the h tile
    const int quad = warp & 3;
    const int r_in = quad * 32 + lane;
    const int sw = lane & 7;
    const uint32_t tq = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
    for (int tl = 0; tl < my_tiles; ++tl) {
      const int s = tl & 1;
      if (tl >= 1) mbar_wait(&t2full_bar[s ^ 1], ((tl - 1) >> 1) & 1);   // GEMM 2 of tile tl - 1 has read h
      if (warp == 4) DAC_TRACE(tl, 5);
      mbar_wait(&t1full_bar[s], (tl >> 1) & 1);
      tc_fence_after();
      if (warp == 4) DAC_TRACE(tl, 6);
#pragma unroll 1
      for (int cc = 0; cc < C / 32; ++cc) {
        uint32_t r[32];
        tmem_ld_32x32(tq + s * C + cc * 32, r);
        tmem_ld_wait_dep(r);
        const int col = cc * 32;
        uint32_t w[16];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 b4 = lds128(smem_u32(s_b7 + col) + 16 * i), a4 = lds128(smem_u32(s_am + col) + 16 * i), ia4 = lds128(smem_u32(s_iam + col) + 16 * i);
          w[2 * i] = pack_bf16x2(snake_act(__uint_as_float(r[4 * i]) + b4.x, a4.x, ia4.x), snake_act(__uint_as_float(r[4 * i + 1]) + b4.y, a4.y, ia4.y));
          w[2 * i + 1] = pack_bf16x2(snake_act(__uint_as_float(r[4 * i + 2]) + b4.z, a4.z, ia4.z), snake_act(__uint_as_float(r[4 * i + 3]) + b4.w, a4.w, ia4.w));
        }
        const uint32_t h_row = smem_u32(s_h) + (col >> 6) * kDcABytes + r_in * 128;
        const int c0 = (col & 63) >> 3;   // first 16-byte chunk of these 32 channels inside the 128-byte row
#pragma unroll
        for (int i = 0; i < 4; ++i)
          sts128(h_row + (((c0 + i) ^ sw) << 4), make_float4(__uint_as_float(w[4 * i]), __uint_as_float(w[4 * i + 1]), __uint_as_float(w[4 * i + 2]),
                                                           __uint_as_float(w[4 * i + 3])));
      }
      fence_proxy_async_smem();
      tc_fence_before();
      mbar_arrive(&hfull_bar[s]);
      if (warp == 4) DAC_TRACE(tl, 7);
    }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 168;");
    // ---- phase 2: y = x + acc2 + b1, s_out = Snake_next(y)
    const int quad = warp & 3;
    const int half = (warp - 8) >> 2;
    constexpr int kColsPerWarp = C / 2;
    constexpr int kChunks = kColsPerWarp / 32;
    uint8_t* stg_y = staging + (warp - 8) * kDcStagingBytes;
    uint8_t* stg_s = stg_y + 4096;
    const uint32_t y_row = smem_u32(stg_y) + lane * 128;
    const uint32_t s_row = smem_u32(stg_s) + lane * 64;
    const int sw = lane & 7, sw64 = (lane >> 1) & 3;
    const int xr_row = lane >> 3, xr_ch = lane & 7;
    const int total_chunks = my_tiles * kChunks;
    const uint32_t tq = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + 2 * C + half * kColsPerWarp;

    auto load_x = [&](int q, float4 (&xr)[8]) {
      const int tile = blockIdx.x + (q / kChunks) * gridDim.x;
      const int t0 = (tile % p.tiles_per_batch) * kDcBM, b = tile / p.tiles_per_batch;
      const int col = half * kColsPerWarp + (q % kChunks) * 32;
      const float* base = p.y + static_cast<long long>(b) * p.y_batch_stride + col + xr_ch * 4;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int t = t0 + quad * 32 + k * 4 + xr_row;
        xr[k] = t < p.rows ? __ldg(reinterpret_cast<const float4*>(base + static_cast<long long>(t) * C)) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
    float4 xr[8];
    if (total_chunks > 0) load_x(0, xr);

    for (int tl = 0; tl < my_tiles; ++tl) {
      const int tile = blockIdx.x + tl * gridDim.x;
      const int t0 = (tile % p.tiles_per_batch) * kDcBM, b = tile / p.tiles_per_batch;
      if (warp == 8) DAC_TRACE(tl, 8);
      mbar_wait(&t2full_bar[tl & 1], (tl >> 1) & 1);
      tc_fence_after();
      if (warp == 8) DAC_TRACE(tl, 9);
#pragma unroll 1
      for (int cc = 0; cc < kChunks; ++cc) {
        uint32_t r[32];
        tmem_ld_32x32(tq + (tl & 1) * C + cc * 32, r);
        tmem_ld_wait_dep(r);
        if (warp == 8 && cc == 0) DAC_TRACE(tl, 10);
        if (cc == kChunks - 1) {
          tc_fence_before();
          mbar_arrive(&t2empty_bar[tl & 1]);
        }
        const int col = half * kColsPerWarp + cc * 32;
        float v[32];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 b4 = lds128(smem_u32(s_b1 + col) + 16 * i);
          v[4 * i] = __uint_as_float(r[4 * i]) + b4.x; v[4 * i + 1] = __uint_as_float(r[4 * i + 1]) + b4.y;
          v[4 * i + 2] = __uint_as_float(r[4 * i + 2]) + b4.z; v[4 * i + 3] = __uint_as_float(r[4 * i + 3]) + b4.w;
        }
        if (lane == 0) bulk_wait_group_read0();
        __syncwarp();
#pragma unroll
        for (int k = 0; k < 8; ++k) sts128(smem_u32(stg_y) + (k * 4 + xr_row) * 128 + ((xr_ch ^ ((k * 4 + xr_row) & 7)) << 4), xr[k]);
        __syncwarp();
        if (warp == 8 && cc == 0) DAC_TRACE(tl, 11);
        const int q = tl * kChunks + cc + 1;
        if (q < total_chunks) load_x(q, xr);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 x4 = lds128(y_row + ((i ^ sw) << 4));
          v[4 * i] += x4.x; v[4 * i + 1] += x4.y; v[4 * i + 2] += x4.z; v[4 * i + 3] += x4.w;
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) sts128(y_row + ((i ^ sw) << 4), make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]));
        if (warp == 8 && cc == 0) DAC_TRACE(tl, 13);
        uint32_t w[16];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 a4 = lds128(smem_u32(s_an + col) + 16 * i), ia4 = lds128(smem_u32(s_ian + col) + 16 * i);
          w[2 * i] = pack_bf16x2(snake_act(v[4 * i], a4.x, ia4.x), snake_act(v[4 * i + 1], a4.y, ia4.y));
          w[2 * i + 1] = pack_bf16x2(snake_act(v[4 * i + 2], a4.z, ia4.z), snake_act(v[4 * i + 3], a4.w, ia4.w));
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
          sts128(s_row + ((i ^ sw64) << 4), make_float4(__uint_as_float(w[4 * i]), __uint_as_float(w[4 * i + 1]), __uint_as_float(w[4 * i + 2]),
                                                        __uint_as_float(w[4 * i + 3])));
        if (warp == 8 && cc == 0) DAC_TRACE(tl, 14);
        fence_proxy_async_smem();
        __syncwarp();
        if (warp == 8 && cc == 0) DAC_TRACE(tl, 15);
        if (lane == 0) {
          tma_store_3d(&tma_y, stg_y, col, t0 + quad * 32, b);
          tma_store_3d(&tma_s, stg_s, col, t0 + quad * 32 + s_row_off, b);
          bulk_commit_group();
        }
        if (warp == 8 && cc == 0) DAC_TRACE(tl, 12);
      }
    }
    if (lane == 0) bulk_wait_group0();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc<4 * C>(tmem_base);
}

template <int C>
struct DacResUnitWideCfg {
  static constexpr int kStages = 3;                                   // (shifted A box, weight chunk [C x 64]) pairs in flight
  static constexpr uint32_t kStageBytes = kDcABytes + C * 128;
  static constexpr uint32_t kHBytes = 128 * C * 2;
  static constexpr uint32_t kSmemBytes = kStages * kStageBytes + kHBytes + 8 * kDcStagingBytes + 6 * C * 4 + 1024 + 256;
};

// Wider channel counts (192: decoder stage 3; at 256 only two ring stages fit and the two-launch form is as fast), where 4 C accumulator columns and a halo tile no longer fit: one acc1 / acc2 / h
// buffer each, the ring carries (shifted A box, W chunk) pairs as in dac_conv_kernel, same warp roles as dac_resunit_kernel. Order of
// the MMA warp: GEMM 1 (i), GEMM 2 (i), GEMM 1 (i+1) ...: GEMM 1 of the next tile runs under phase 2 of the current one.
// Buffer reuse: acc1 <- hfull of the previous tile (waited by the MMA warp before its GEMM 2); h <- the phase-1 warps wait t2full of
// the previous tile; acc2 <- t2empty (phase 2 has drained it).
template <int C>
__global__ void __launch_bounds__(kRuThreads, 1)
dac_resunit_wide_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_w7, const __grid_constant__ CUtensorMap tma_w1,
                   const __grid_constant__ CUtensorMap tma_y, const __grid_constant__ CUtensorMap tma_s, const DacResUnitParams p, const int s_row_off) {
  constexpr int kStages = DacResUnitWideCfg<C>::kStages;
  constexpr int kKc = C / 64;                       // 64-channel chunks
  constexpr uint32_t kStageBytes = DacResUnitWideCfg<C>::kStageBytes;
  constexpr uint32_t kHBytes = DacResUnitWideCfg<C>::kHBytes;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* s_h = smem + kStages * kStageBytes;      // kKc sub-tiles of [128 rows x 64 channels] bf16, 128B-swizzled
  uint8_t* staging = s_h + kHBytes;
  float* s_b7 = reinterpret_cast<float*>(staging + 8 * kDcStagingBytes);
  float* s_am = s_b7 + C;
  float* s_iam = s_am + C;
  float* s_b1 = s_iam + C;
  float* s_an = s_b1 + C;
  float* s_ian = s_an + C;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(s_ian + C);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* t1full_bar = empty_bar + kStages;
  uint64_t* hfull_bar = t1full_bar + 1;
  uint64_t* t2full_bar = hfull_bar + 1;
  uint64_t* t2empty_bar = t2full_bar + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t2empty_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_tiles = p.B * p.tiles_per_batch;
  const int my_tiles = (num_tiles - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_w7);
    tma_prefetch_desc(&tma_w1);
    tma_prefetch_desc(&tma_y);
    tma_prefetch_desc(&tma_s);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(t1full_bar, 1);
    mbar_init(hfull_bar, 128);
    mbar_init(t2full_bar, 1);
    mbar_init(t2empty_bar, 256);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc<512>(tmem_slot);
  for (int i = threadIdx.x; i < C; i += kRuThreads) {
    s_b7[i] = __ldg(p.b7 + i);
    s_b1[i] = __ldg(p.b1 + i);
    const float am = __ldg(p.a_mid + i), an = __ldg(p.a_next + i);
    s_am[i] = am; s_iam[i] = 1.0f / (am + 1e-9f);
    s_an[i] = an; s_ian[i] = 1.0f / (an + 1e-9f);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 72;");
    if (warp == 0) {
      if (lane == 0) {
        uint32_t it = 0;
        for (int tl = 0; tl < my_tiles; ++tl) {
          const int tile = blockIdx.x + tl * gridDim.x;
          const int t0 = (tile % p.tiles_per_batch) * kDcBM, b = tile / p.tiles_per_batch;
          for (int j = 0; j < 7; ++j) {
            const int row = t0 + (j - 3) * p.dilation;
            for (int c = 0; c < kKc; ++c, ++it) {
              const uint32_t s = it % kStages;
              uint8_t* st = smem + s * kStageBytes;
              mbar_wait(&empty_bar[s], ((it / kStages) & 1) ^ 1);
              mbar_arrive_expect_tx(&full_bar[s], kStageBytes);
              tma_load_3d(&tma_a, &full_bar[s], st, c * 64, row, b);
              tma_load_2d(&tma_w7, &full_bar[s], st + kDcABytes, (j * kKc + c) * 64, 0);
            }
          }
          for (int c = 0; c < kKc; ++c, ++it) {
            const uint32_t s = it % kStages;
            uint8_t* st = smem + s * kStageBytes;
            mbar_wait(&empty_bar[s], ((it / kStages) & 1) ^ 1);
            mbar_arrive_expect_tx(&full_bar[s], kStageBytes - kDcABytes);
            tma_load_2d(&tma_w1, &full_bar[s], st + kDcABytes, c * 64, 0);
          }
        }
      }
    } else if (warp == 1) {
      constexpr uint32_t idesc = umma_idesc_bf16(kDcBM, C, 0, 0);
      uint32_t it = 0;
      for (int tl = 0; tl < my_tiles; ++tl) {
        // GEMM 1 -> acc1 (free: hfull of the previous tile was waited below)
        for (int ks = 0; ks < 7 * kKc; ++ks, ++it) {
          const uint32_t s = it % kStages;
          mbar_wait_spin(&full_bar[s], (it / kStages) & 1);
          tc_fence_after();
          const uint32_t st = smem_u32(smem + s * kStageBytes);
          const uint64_t a_desc = umma_desc_sw128(st, 16, 1024), b_desc = umma_desc_sw128(st + kDcABytes, 16, 1024);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_ss_warp(tmem_base, a_desc + 2 * k, b_desc + 2 * k, idesc, (ks | k) != 0 ? 1u : 0u);
          umma_commit_warp(&empty_bar[s]);
        }
        umma_commit_warp(t1full_bar);
        mbar_wait_spin(hfull_bar, tl & 1);
        mbar_wait_spin(t2empty_bar, (tl & 1) ^ 1);   // phase 2 of the previous tile has drained acc2
        tc_fence_after();
        for (int c = 0; c < kKc; ++c, ++it) {
          const uint32_t s = it % kStages;
          mbar_wait_spin(&full_bar[s], (it / kStages) & 1);
          tc_fence_after();
          const uint64_t a_desc = umma_desc_sw128(smem_u32(s_h) + c * kDcABytes, 16, 1024);
          const uint64_t b_desc = umma_desc_sw128(smem_u32(smem + s * kStageBytes) + kDcABytes, 16, 1024);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_ss_warp(tmem_base + C, a_desc + 2 * k, b_desc + 2 * k, idesc, (c | k) != 0 ? 1u : 0u);
          umma_commit_warp(&empty_bar[s]);
        }
        umma_commit_warp(t2full_bar);
      }
    }
  } else if (warp < 8) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 104;");
    // ---- phase 1: h = Snake_mid(acc1 + b7) -> bf16, this thread's row of the h tile
    const int quad = warp & 3;
    const int r_in = quad * 32 + lane;
    const int sw = lane & 7;
    const uint32_t tq = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
    for (int tl = 0; tl < my_tiles; ++tl) {
      if (tl >= 1) mbar_wait(t2full_bar, (tl - 1) & 1);   // GEMM 2 of the previous tile has read h
      mbar_wait(t1full_bar, tl & 1);
      tc_fence_after();
#pragma unroll 1
      for (int cc = 0; cc < C / 32; ++cc) {
        uint32_t r[32];
        tmem_ld_32x32(tq + cc * 32, r);
        tmem_ld_wait_dep(r);
        const int col = cc * 32;
        uint32_t w[16];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 b4 = lds128(smem_u32(s_b7 + col) + 16 * i), a4 = lds128(smem_u32(s_am + col) + 16 * i), ia4 = lds128(smem_u32(s_iam + col) + 16 * i);
          w[2 * i] = pack_bf16x2(snake_act(__uint_as_float(r[4 * i]) + b4.x, a4.x, ia4.x), snake_act(__uint_as_float(r[4 * i + 1]) + b4.y, a4.y, ia4.y));
          w[2 * i + 1] = pack_bf16x2(snake_act(__uint_as_float(r[4 * i + 2]) + b4.z, a4.z, ia4.z), snake_act(__uint_as_float(r[4 * i + 3]) + b4.w, a4.w, ia4.w));
        }
        const uint32_t h_row = smem_u32(s_h) + (col >> 6) * kDcABytes + r_in * 128;
        const int c0 = (col & 63) >> 3;   // first 16-byte chunk of these 32 channels inside the 128-byte row
#pragma unroll
        for (int i = 0; i < 4; ++i)
          sts128(h_row + (((c0 + i) ^ sw) << 4), make_float4(__uint_as_float(w[4 * i]), __uint_as_float(w[4 * i + 1]), __uint_as_float(w[4 * i + 2]),
                                                           __uint_as_float(w[4 * i + 3])));
      }
      fence_proxy_async_smem();
      tc_fence_before();
      mbar_arrive(hfull_bar);
    }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 168;");
    // ---- phase 2: y = x + acc2 + b1, s_out = Snake_next(y)
    const int quad = warp & 3;
    const int half = (warp - 8) >> 2;
    constexpr int kColsPerWarp = C / 2;
    constexpr int kChunks = kColsPerWarp / 32;
    uint8_t* stg_y = staging + (warp - 8) * kDcStagingBytes;
    uint8_t* stg_s = stg_y + 4096;
    const uint32_t y_row = smem_u32(stg_y) + lane * 128;
    const uint32_t s_row = smem_u32(stg_s) + lane * 64;
    const int sw = lane & 7, sw64 = (lane >> 1) & 3;
    const int xr_row = lane >> 3, xr_ch = lane & 7;
    const int total_chunks = my_tiles * kChunks;
    const uint32_t tq = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + C + half * kColsPerWarp;

    auto load_x = [&](int q, float4 (&xr)[8]) {
      const int tile = blockIdx.x + (q / kChunks) * gridDim.x;
      const int t0 = (tile % p.tiles_per_batch) * kDcBM, b = tile / p.tiles_per_batch;
      const int col = half * kColsPerWarp + (q % kChunks) * 32;
      const float* base = p.y + static_cast<long long>(b) * p.y_batch_stride + col + xr_ch * 4;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int t = t0 + quad * 32 + k * 4 + xr_row;
        xr[k] = t < p.rows ? __ldg(reinterpret_cast<const float4*>(base + static_cast<long long>(t) * C)) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
    float4 xr[8];
    if (total_chunks > 0) load_x(0, xr);

    for (int tl = 0; tl < my_tiles; ++tl) {
      const int tile = blockIdx.x + tl * gridDim.x;
      const int t0 = (tile % p.tiles_per_batch) * kDcBM, b = tile / p.tiles_per_batch;
      mbar_wait(t2full_bar, tl & 1);
      tc_fence_after();
#pragma unroll 1
      for (int cc = 0; cc < kChunks; ++cc) {
        uint32_t r[32];
        tmem_ld_32x32(tq + cc * 32, r);
        tmem_ld_wait_dep(r);
        if (cc == kChunks - 1) {
          tc_fence_before();
          mbar_arrive(t2empty_bar);
        }
        const int col = half * kColsPerWarp + cc * 32;
        float v[32];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 b4 = lds128(smem_u32(s_b1 + col) + 16 * i);
          v[4 * i] = __uint_as_float(r[4 * i]) + b4.x; v[4 * i + 1] = __uint_as_float(r[4 * i + 1]) + b4.y;
          v[4 * i + 2] = __uint_as_float(r[4 * i + 2]) + b4.z; v[4 * i + 3] = __uint_as_float(r[4 * i + 3]) + b4.w;
        }
        if (lane == 0) bulk_wait_group_read0();
        __syncwarp();
#pragma unroll
        for (int k = 0; k < 8; ++k) sts128(smem_u32(stg_y) + (k * 4 + xr_row) * 128 + ((xr_ch ^ ((k * 4 + xr_row) & 7)) << 4), xr[k]);
        __syncwarp();
        const int q = tl * kChunks + cc + 1;
        if (q < total_chunks) load_x(q, xr);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 x4 = lds128(y_row + ((i ^ sw) << 4));
          v[4 * i] += x4.x; v[4 * i + 1] += x4.y; v[4 * i + 2] += x4.z; v[4 * i + 3] += x4.w;
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) sts128(y_row + ((i ^ sw) << 4), make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]));
        uint32_t w[16];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 a4 = lds128(smem_u32(s_an + col) + 16 * i), ia4 = lds128(smem_u32(s_ian + col) + 16 * i);
          w[2 * i] = pack_bf16x2(snake_act(v[4 * i], a4.x, ia4.x), snake_act(v[4 * i + 1], a4.y, ia4.y));
          w[2 * i + 1] = pack_bf16x2(snake_act(v[4 * i + 2], a4.z, ia4.z), snake_act(v[4 * i + 3], a4.w, ia4.w));
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
          sts128(s_row + ((i ^ sw64) << 4), make_float4(__uint_as_float(w[4 * i]), __uint_as_float(w[4 * i + 1]), __uint_as_float(w[4 * i + 2]),
                                                        __uint_as_float(w[4 * i + 3])));
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_3d(&tma_y, stg_y, col, t0 + quad * 32, b);
          tma_store_3d(&tma_s, stg_s, col, t0 + quad * 32 + s_row_off, b);
          bulk_commit_group();
        }
      }
    }
    if (lane == 0) bulk_wait_group0();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc<512>(tmem_base);
}

// ------------------------------------------------------------------------------------------------------------------------------
// 64-channel ResidualUnit, second form: the L2 -> SM fabric bounds dac_resunit_kernel<64> (every 128-row tile pulls seven shifted
// 16 KB copies of its input rows and 64 KB of weights). Here
//   * W7 (56 KB) and W1 (8 KB) are loaded once per CTA and stay in shared memory;
//   * the input rows are loaded once per tile with their halo ([128 + 6 d] rows x 64 channels, one TMA box), and tap j of the
//     dilated conv is the same tile read through a UMMA descriptor whose start address is advanced by j * d rows (128 B each).
//     The 128B-swizzle XOR is a function of the absolute shared-memory address bits (TMA writes and UMMA reads agree on it), so
//     a start address that is not a multiple of the 1024 B swizzle atom works as is, with the descriptor's base-offset field
//     left at zero (measured: bit-identical to the seven-box form; setting base offset = (addr >> 7) & 7 gives wrong results).
// The h tile and both accumulators are double-buffered, the MMA warp issues GEMM 1 of tile i+1 before GEMM 2 of tile i, and the two
// epilogue phases run on separate warpgroups (as in dac_resunit_kernel), so phase 1 of tile i+1 runs beside phase 2 of tile i.
constexpr uint32_t kRu64SmemBytes = 7 * 8192 + 8192 + 2 * kRu64HaloBytes + 2 * kDcABytes + 8 * kDcStagingBytes + 6 * 64 * 4 + 1024 + 256;

__global__ void __launch_bounds__(kRuThreads, 1)
dac_resunit64_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_w7, const __grid_constant__ CUtensorMap tma_w1,
                     const __grid_constant__ CUtensorMap tma_y, const __grid_constant__ CUtensorMap tma_s, const DacResUnitParams p, const int s_row_off) {
  constexpr int C = 64;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* s_w7 = smem;                              // 7 taps x [64 co x 64 ci] bf16, 128B-swizzled
  uint8_t* s_w1 = s_w7 + 7 * 8192;
  uint8_t* s_a = s_w1 + 8192;                        // 2 halo tiles
  uint8_t* s_h = s_a + 2 * kRu64HaloBytes;           // 2 x [128 x 64] bf16
  uint8_t* staging = s_h + 2 * kDcABytes;
  float* s_b7 = reinterpret_cast<float*>(staging + 8 * kDcStagingBytes);
  float* s_am = s_b7 + C;
  float* s_iam = s_am + C;
  float* s_b1 = s_iam + C;
  float* s_an = s_b1 + C;
  float* s_ian = s_an + C;
  uint64_t* w_bar = reinterpret_cast<uint64_t*>(s_ian + C);
  uint64_t* afull_bar = w_bar + 1;     // [2]
  uint64_t* aempty_bar = afull_bar + 2;  // [2]
  uint64_t* t1full_bar = aempty_bar + 2;  // [2]
  uint64_t* hfull_bar = t1full_bar + 2;   // [2]
  uint64_t* t2full_bar = hfull_bar + 2;   // [2]
  uint64_t* t2empty_bar = t2full_bar + 2; // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t2empty_bar + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_tiles = p.B * p.tiles_per_batch;
  const int my_tiles = (num_tiles - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);
  const uint32_t halo_bytes = static_cast<uint32_t>(128 + 6 * p.dilation) * 128;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_w7);
    tma_prefetch_desc(&tma_w1);
    tma_prefetch_desc(&tma_y);
    tma_prefetch_desc(&tma_s);
    mbar_init(w_bar, 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(&afull_bar[s], 1);
      mbar_init(&aempty_bar[s], 1);
      mbar_init(&t1full_bar[s], 1);
      mbar_init(&hfull_bar[s], 128);
      mbar_init(&t2full_bar[s], 1);
      mbar_init(&t2empty_bar[s], 256);
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc<256>(tmem_slot);
  for (int i = threadIdx.x; i < C; i += kRuThreads) {
    s_b7[i] = __ldg(p.b7 + i);
    s_b1[i] = __ldg(p.b1 + i);
    const float am = __ldg(p.a_mid + i), an = __ldg(p.a_next + i);
    s_am[i] = am; s_iam[i] = 1.0f / (am + 1e-9f);
    s_an[i] = an; s_ian[i] = 1.0f / (an + 1e-9f);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // warp roles as in dac_resunit_kernel: warps 0 / 1 producer / MMA, warps 4-7 phase 1, warps 8-15 phase 2 (setmaxnreg)
  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 88;");
  if (warp == 0) {
    if (lane == 0) {
      mbar_arrive_expect_tx(w_bar, 8 * 8192);
      for (int j = 0; j < 7; ++j) tma_load_2d(&tma_w7, w_bar, s_w7 + j * 8192, j * 64, 0);
      tma_load_2d(&tma_w1, w_bar, s_w1, 0, 0);
      for (int tl = 0; tl < my_tiles; ++tl) {
        const int tile = blockIdx.x + tl * gridDim.x;
        const int t0 = (tile % p.tiles_per_batch) * kDcBM, b = tile / p.tiles_per_batch;
        const int s = tl & 1;
        mbar_wait(&aempty_bar[s], ((tl >> 1) & 1) ^ 1);
        mbar_arrive_expect_tx(&afull_bar[s], halo_bytes);
        tma_load_3d(&tma_a, &afull_bar[s], s_a + s * kRu64HaloBytes, 0, t0 - 3 * p.dilation, b);
      }
    }
  } else if (warp == 1) {
    // TMEM columns: acc1[0] [0,64) acc1[1] [64,128) acc2[0] [128,192) acc2[1] [192,256). Software pipeline: GEMM 1 of tile i+1 is
    // issued before GEMM 2 of tile i, and the epilogue warps run phase 1 of tile i+1 before phase 2 of tile i, so neither side
    // waits for a hand-off round trip. Buffer reuse is ordered by the barriers already there (see the epilogue loop).
    constexpr uint32_t idesc = umma_idesc_bf16(kDcBM, C, 0, 0);
    mbar_wait_spin(w_bar, 0);
    auto gemm1 = [&](int tl) {
      const int s = tl & 1;
      mbar_wait_spin(&afull_bar[s], (tl >> 1) & 1);
      tc_fence_after();
      const uint32_t a_base = smem_u32(s_a + s * kRu64HaloBytes);
      for (int j = 0; j < 7; ++j) {
        const uint64_t a_desc = umma_desc_sw128(a_base + j * p.dilation * 128, 16, 1024);
        const uint64_t b_desc = umma_desc_sw128(smem_u32(s_w7) + j * 8192, 16, 1024);
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_ss_warp(tmem_base + s * C, a_desc + 2 * k, b_desc + 2 * k, idesc, (j | k) != 0 ? 1u : 0u);
      }
      umma_commit_warp(&aempty_bar[s]);
      umma_commit_warp(&t1full_bar[s]);
    };
    if (my_tiles > 0) gemm1(0);
    for (int tl = 0; tl < my_tiles; ++tl) {
      const int s = tl & 1;
      if (tl + 1 < my_tiles) gemm1(tl + 1);
      mbar_wait_spin(&hfull_bar[s], (tl >> 1) & 1);
      mbar_wait_spin(&t2empty_bar[s], ((tl >> 1) & 1) ^ 1);   // phase 2 of tile tl - 2 has drained acc2[s]
      tc_fence_after();
      const uint64_t a_desc = umma_desc_sw128(smem_u32(s_h) + s * kDcABytes, 16, 1024), b_desc = umma_desc_sw128(smem_u32(s_w1), 16, 1024);
#pragma unroll
      for (int k = 0; k < 4; ++k) umma_ss_warp(tmem_base + 2 * C + s * C, a_desc + 2 * k, b_desc + 2 * k, idesc, k != 0 ? 1u : 0u);
      umma_commit_warp(&t2full_bar[s]);
    }
  }
  } else if (warp < 8) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 104;");
    // ---- phase 1 (four warps, one per TMEM lane quadrant, both 32-column halves): h = Snake_mid(acc1 + b7) -> bf16
    const int quad = warp & 3;
    const int r_in = quad * 32 + lane;
    const int sw = lane & 7;
    for (int tl = 0; tl < my_tiles; ++tl) {
      if (tl >= 2) mbar_wait(&t2full_bar[tl & 1], ((tl >> 1) & 1) ^ 1);   // GEMM 2 of tile tl - 2 has read h[tl & 1]
      mbar_wait(&t1full_bar[tl & 1], (tl >> 1) & 1);
      tc_fence_after();
#pragma unroll 1
      for (int half = 0; half < 2; ++half) {
        const int col = half * 32;
        uint32_t r[32];
        tmem_ld_32x32(tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + (tl & 1) * C + col, r);
        tmem_ld_wait_dep(r);
        uint32_t w[16];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 b4 = lds128(smem_u32(s_b7 + col) + 16 * i), a4 = lds128(smem_u32(s_am + col) + 16 * i), ia4 = lds128(smem_u32(s_iam + col) + 16 * i);
          w[2 * i] = pack_bf16x2(snake_act(__uint_as_float(r[4 * i]) + b4.x, a4.x, ia4.x), snake_act(__uint_as_float(r[4 * i + 1]) + b4.y, a4.y, ia4.y));
          w[2 * i + 1] = pack_bf16x2(snake_act(__uint_as_float(r[4 * i + 2]) + b4.z, a4.z, ia4.z), snake_act(__uint_as_float(r[4 * i + 3]) + b4.w, a4.w, ia4.w));
        }
        const uint32_t h_row = smem_u32(s_h) + (tl & 1) * kDcABytes + r_in * 128;
        const int c0 = col >> 3;
#pragma unroll
        for (int i = 0; i < 4; ++i)
          sts128(h_row + (((c0 + i) ^ sw) << 4), make_float4(__uint_as_float(w[4 * i]), __uint_as_float(w[4 * i + 1]), __uint_as_float(w[4 * i + 2]),
                                                           __uint_as_float(w[4 * i + 3])));
      }
      fence_proxy_async_smem();
      tc_fence_before();
      mbar_arrive(&hfull_bar[tl & 1]);
    }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 160;");
    // ---- phase 2 (eight warps, two per quadrant, 32 columns each): y = x + acc2 + b1, s_out = Snake_next(y)
    const int quad = warp & 3;
    const int half = (warp - 8) >> 2;
    uint8_t* stg_y = staging + (warp - 8) * kDcStagingBytes;
    uint8_t* stg_s = stg_y + 4096;
    const uint32_t y_row = smem_u32(stg_y) + lane * 128;
    const uint32_t s_row = smem_u32(stg_s) + lane * 64;
    const int sw = lane & 7, sw64 = (lane >> 1) & 3;
    const int xr_row = lane >> 3, xr_ch = lane & 7;
    const uint32_t tq = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + half * 32;
    const int col = half * 32;

    auto load_x = [&](int tl, float4 (&xr)[8]) {
      const int tile = blockIdx.x + tl * gridDim.x;
      const int t0 = (tile % p.tiles_per_batch) * kDcBM, b = tile / p.tiles_per_batch;
      const float* base = p.y + static_cast<long long>(b) * p.y_batch_stride + col + xr_ch * 4;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int t = t0 + quad * 32 + k * 4 + xr_row;
        xr[k] = t < p.rows ? __ldg(reinterpret_cast<const float4*>(base + static_cast<long long>(t) * C)) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
    // residual rows are fetched two tiles ahead (two register sets, the tile loop is unrolled by two): one tile of look-ahead left
    // the loads on the critical path of the phase
    float4 xr0[8], xr1[8];
    if (my_tiles > 0) load_x(0, xr0);
    if (my_tiles > 1) load_x(1, xr1);
    auto phase2 = [&](int tl, float4 (&xr)[8]) {
      const int tile = blockIdx.x + tl * gridDim.x;
      const int t0 = (tile % p.tiles_per_batch) * kDcBM, b = tile / p.tiles_per_batch;
      // ---- phase 2
      mbar_wait(&t2full_bar[tl & 1], (tl >> 1) & 1);
      tc_fence_after();
      {
        uint32_t r[32];
        tmem_ld_32x32(tq + 2 * C + (tl & 1) * C, r);
        tmem_ld_wait_dep(r);
        tc_fence_before();
        mbar_arrive(&t2empty_bar[tl & 1]);
        float v[32];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 b4 = lds128(smem_u32(s_b1 + col) + 16 * i);
          v[4 * i] = __uint_as_float(r[4 * i]) + b4.x; v[4 * i + 1] = __uint_as_float(r[4 * i + 1]) + b4.y;
          v[4 * i + 2] = __uint_as_float(r[4 * i + 2]) + b4.z; v[4 * i + 3] = __uint_as_float(r[4 * i + 3]) + b4.w;
        }
        if (lane == 0) bulk_wait_group_read0();
        __syncwarp();
#pragma unroll
        for (int k = 0; k < 8; ++k) sts128(smem_u32(stg_y) + (k * 4 + xr_row) * 128 + ((xr_ch ^ ((k * 4 + xr_row) & 7)) << 4), xr[k]);
        __syncwarp();
        if (tl + 2 < my_tiles) load_x(tl + 2, xr);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 x4 = lds128(y_row + ((i ^ sw) << 4));
          v[4 * i] += x4.x; v[4 * i + 1] += x4.y; v[4 * i + 2] += x4.z; v[4 * i + 3] += x4.w;
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) sts128(y_row + ((i ^ sw) << 4), make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]));
        uint32_t w[16];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 a4 = lds128(smem_u32(s_an + col) + 16 * i), ia4 = lds128(smem_u32(s_ian + col) + 16 * i);
          w[2 * i] = pack_bf16x2(snake_act(v[4 * i], a4.x, ia4.x), snake_act(v[4 * i + 1], a4.y, ia4.y));
          w[2 * i + 1] = pack_bf16x2(snake_act(v[4 * i + 2], a4.z, ia4.z), snake_act(v[4 * i + 3], a4.w, ia4.w));
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
          sts128(s_row + ((i ^ sw64) << 4), make_float4(__uint_as_float(w[4 * i]), __uint_as_float(w[4 * i + 1]), __uint_as_float(w[4 * i + 2]),
                                                        __uint_as_float(w[4 * i + 3])));
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_3d(&tma_y, stg_y, col, t0 + quad * 32, b);
          tma_store_3d(&tma_s, stg_s, col, t0 + quad * 32 + s_row_off, b);
          bulk_commit_group();
        }
      }
      tc_fence_before();
    };
    for (int tl = 0; tl < my_tiles; tl += 2) {
      phase2(tl, xr0);
      if (tl + 1 < my_tiles) phase2(tl + 1, xr1);
    }
    if (lane == 0) bulk_wait_group0();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc<256>(tmem_base);
}

// First conv of the encoder: 1 -> C0 channels, k = 7, padding 3 (encoder.py:38), CUDA cores (7 MACs per output, bandwidth-bound:
// 4 B in, 6 * C0 B out per sample). A half-warp owns 64 channels (4 per lane: 28 weights, bias and Snake constants in registers)
// and walks a run of consecutive samples with the 7-tap window in registers, so a sample costs one broadcast load, and the two
// output rows of a warp instruction are whole 256 B (fp32 stream) / 128 B (bf16 operand) segments. (The first version read the
// weights from shared memory per output: 1.9 TB/s; this one is bound by the stores.)
struct DacConv0Params {
  const float* audio;   // [B][L]
  const float* w;       // [C0][7]
  const float* bias;    // [C0]
  const float* alpha;   // [C0] Snake of the first ResidualUnit
  float* y;             // [B][L][C0]
  __nv_bfloat16* s_out; // [B][L][C0]
  int B, L, C0;
};
constexpr int kDc0Run = 64;   // consecutive samples per half-warp

__global__ void __launch_bounds__(256) dac_conv0_kernel(const DacConv0Params p) {
  const int hw = threadIdx.x >> 4, cl = threadIdx.x & 15;
  const int c = blockIdx.y * 64 + cl * 4;               // this lane's 4 channels
  float w[4][7], bs[4], al[4], ia[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
#pragma unroll
    for (int j = 0; j < 7; ++j) w[q][j] = __ldg(p.w + (c + q) * 7 + j);
    bs[q] = __ldg(p.bias + c + q);
    al[q] = __ldg(p.alpha + c + q);
    ia[q] = 1.0f / (al[q] + 1e-9f);
  }
  const int runs_per_b = (p.L + kDc0Run - 1) / kDc0Run;
  const long long total = static_cast<long long>(p.B) * runs_per_b;
  for (long long run = static_cast<long long>(blockIdx.x) * 16 + hw; run < total; run += static_cast<long long>(gridDim.x) * 16) {
    const int b = static_cast<int>(run / runs_per_b);
    const int t0 = static_cast<int>(run % runs_per_b) * kDc0Run;
    const float* a = p.audio + static_cast<long long>(b) * p.L;
    const int t1 = t0 + kDc0Run < p.L ? t0 + kDc0Run : p.L;
    float x[7];
#pragma unroll
    for (int j = 0; j < 6; ++j) {
      const int tt = t0 + j - 3;
      x[j] = (tt >= 0 && tt < p.L) ? __ldg(a + tt) : 0.f;
    }
    float* yo = p.y + (static_cast<long long>(b) * p.L + t0) * p.C0 + c;
    __nv_bfloat16* so = p.s_out + (static_cast<long long>(b) * p.L + t0) * p.C0 + c;
    for (int t = t0; t < t1; ++t, yo += p.C0, so += p.C0) {
      x[6] = t + 3 < p.L ? __ldg(a + t + 3) : 0.f;
      float v[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        float acc = bs[q];
#pragma unroll
        for (int j = 0; j < 7; ++j) acc = fmaf(w[q][j], x[j], acc);
        v[q] = acc;
      }
      *reinterpret_cast<float4*>(yo) = make_float4(v[0], v[1], v[2], v[3]);
      *reinterpret_cast<uint2*>(so) = make_uint2(pack_bf16x2(snake_act(v[0], al[0], ia[0]), snake_act(v[1], al[1], ia[1])),
                                                pack_bf16x2(snake_act(v[2], al[2], ia[2]), snake_act(v[3], al[3], ia[3])));
#pragma unroll
      for (int j = 0; j < 6; ++j) x[j] = x[j + 1];
    }
  }
}

// Last conv of the decoder: C channels -> 1, k = 7, padding 3, then tanh (decoder.py:55-59), on CUDA cores. The input is the bf16
// operand Snake(x) [B][rows][c_pad] (channel-last, zero-padded channels carry zero weights). A warp produces 32 consecutive
// samples: lane <-> 8 channels (one 16 B load per row), each of the 38 rows of the window is read once and its 7 tap products go to
// the 7 outputs it touches, reduced over the lanes by shuffles at the end.
struct DacConvLastParams {
  const __nv_bfloat16* a; long long a_batch_stride; int rows, c_pad, B;
  const float* w;   // [7][c_pad] fp32 (zero for padded channels)
  float bias;
  float* out;       // [B][rows]
  int apply_tanh;
};

__global__ void __launch_bounds__(256) dac_conv_last_kernel(const DacConvLastParams p) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int lanes_used = p.c_pad / 8;                       // <= 32
  float w[7][8];
#pragma unroll
  for (int j = 0; j < 7; ++j)
#pragma unroll
    for (int e = 0; e < 8; ++e) w[j][e] = lane < lanes_used ? __ldg(p.w + j * p.c_pad + lane * 8 + e) : 0.f;
  const int runs_per_b = (p.rows + 31) / 32;
  const long long total = static_cast<long long>(p.B) * runs_per_b;
  for (long long run = static_cast<long long>(blockIdx.x) * 8 + warp; run < total; run += static_cast<long long>(gridDim.x) * 8) {
    const int b = static_cast<int>(run / runs_per_b);
    const int t0 = static_cast<int>(run % runs_per_b) * 32;
    const __nv_bfloat16* a = p.a + static_cast<long long>(b) * p.a_batch_stride + lane * 8;
    float acc[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) acc[i] = 0.f;
#pragma unroll
    for (int r = 0; r < 38; ++r) {                          // input row t0 - 3 + r contributes to outputs t0 + r - j, j = 0..6 ... (tap index = r - i)
      const int t = t0 - 3 + r;
      float x[8];
      if (t >= 0 && t < p.rows && lane < lanes_used) {
        const uint4 q = __ldg(reinterpret_cast<const uint4*>(a + static_cast<long long>(t) * p.c_pad));
        x[0] = bf16lo(q.x); x[1] = bf16hi(q.x); x[2] = bf16lo(q.y); x[3] = bf16hi(q.y);
        x[4] = bf16lo(q.z); x[5] = bf16hi(q.z); x[6] = bf16lo(q.w); x[7] = bf16hi(q.w);
      } else {
#pragma unroll
        for (int e = 0; e < 8; ++e) x[e] = 0.f;
      }
#pragma unroll
      for (int j = 0; j < 7; ++j) {
        const int i = r - j;                                // output index inside the run: out[t0 + i] += w[j] . x[t0 + i + j - 3]
        if (i >= 0 && i < 32) {
#pragma unroll
          for (int e = 0; e < 8; ++e) acc[i] = fmaf(w[j][e], x[e], acc[i]);
        }
      }
    }
    // reduce over lanes: after the butterfly lane l keeps output l
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
#pragma unroll
      for (int i = 0; i < 32; ++i) acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], off);
    }
    float mine = 0.f;
#pragma unroll
    for (int i = 0; i < 32; ++i) mine = lane == i ? acc[i] : mine;
    const int t = t0 + lane;
    if (t < p.rows) {
      const float v = mine + p.bias;
      p.out[static_cast<long long>(b) * p.rows + t] = p.apply_tanh ? tanhf(v) : v;
    }
  }
}

// Gap rows of the packed encoder and decoder batches (DACEncoder.forward_batch, DACDecoder.forward_batch, DESIGN §4a): every producer
// writes bias / Snake(bias) / junk view rows into the rows between utterances, and the next multi-tap conv must read them as its zero
// padding. A [start, end) row range of
// a channel-last buffer is one contiguous span of (end - start) * pitch bytes, so this is a memset over a list of spans: blockIdx.y
// walks the ranges, the x blocks of a range stride over its 16-byte words.
constexpr int kZeroRowsThreads = 256;

__global__ void __launch_bounds__(kZeroRowsThreads) dac_zero_rows_kernel(uint8_t* buf, long long pitch, const int2* ranges, int n_ranges) {
  for (int r = blockIdx.y; r < n_ranges; r += gridDim.y) {
    const int2 rg = __ldg(ranges + r);
    uint4* span = reinterpret_cast<uint4*>(buf + static_cast<long long>(rg.x) * pitch);
    const long long words = static_cast<long long>(rg.y - rg.x) * pitch / 16;
    for (long long w = static_cast<long long>(blockIdx.x) * kZeroRowsThreads + threadIdx.x; w < words;
         w += static_cast<long long>(gridDim.x) * kZeroRowsThreads)
      span[w] = make_uint4(0u, 0u, 0u, 0u);
  }
}

}  // namespace edm
