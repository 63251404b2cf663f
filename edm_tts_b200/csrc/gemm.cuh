// Persistent warp-specialised bf16 GEMMs for sm_100a: C[M,N] = A[M,K] * B[N,K]^T (both operands K-major, which is
// how activations [tokens, channels] and nn.Linear weights [out, in] already sit in HBM). Two kernels: CTA pairs on 256 x 256 tiles
// (tcgen05.mma.cta_group::2) for large M, 128 x 64 tiles for small M / N that is not a multiple of 256. Roles in both:
//
//   warp 0       : TMA producer  (cp.async.bulk.tensor, 128B swizzle, mbarrier ring)
//   warp 1       : TMEM allocator + tcgen05.mma issue (whole warp runs the descriptor arithmetic, one elected lane issues; fp32 accum in TMEM)
//   warps 2..17  : epilogue. Warp w owns TMEM lane quadrant w % 4 and 64 of the tile's 256 columns: it pulls its
//                  128 x 64 slice into registers with two tcgen05.ld, releases the accumulator buffer at once
//                  (so the MMA warp never waits for epilogue arithmetic), then applies the fused op and stores.
//                  Two TMEM accumulator buffers (2 x 256 columns = all 512) overlap epilogue and next mainloop.
//   The bias vector is staged in shared memory once per CTA (broadcast LDS instead of a dependent global load).
//
// Fused epilogues cover every GEMM of the conformer block (reference: edm_tts/models/conformer/conformer.py:149-181,
// 113-146) and the logits heads (injection_conformer_wrapper.py:38-63); rounding points follow bf16 autocast:
// Linear/Conv outputs are rounded to bf16 before the activation / residual add, the residual stream stays fp32.
#pragma once
#include "ptx.cuh"
#include "seq_layout.cuh"

namespace edm {

enum EpiKind : int {
  EPI_BF16 = 0,        // out_bf16 = bf16(acc + bias)
  EPI_SWISH_BF16 = 1,  // h = bf16(acc + bias); out_bf16 = bf16(h * bf16(sigmoid(h)))          (FeedForward up-proj)
  EPI_QKV_ROPE = 2,    // cols < rope_cols: rotary embedding on bf16(acc) per 64-wide head; others bf16(acc)
  EPI_RESID_F32 = 3,   // x_f32[r, c] += scale * bf16(acc + bias)                                (residual branches)
  EPI_F32 = 4,         // out_f32 = acc + bias                                                   (logits heads)
  EPI_GLU_BF16 = 5,    // per 64 columns: first 32 = value, last 32 = gate (weights interleaved at pack time);
                       // out_bf16[., N/2] = bf16(bf16(value) * bf16(sigmoid(bf16(gate))))       (conv module pointwise-1 + GLU)
  EPI_ARGMAX = 10,     // logits heads whose only consumer is an arg-max (injection_conformer_wrapper.py:119-121, modeling :228): the
                       // logits acc + bias never leave the SM; every epilogue thread writes (max, first arg-max) of its 64 columns
                       // of one row to out_part[row * ldo + col / 64] (float2: value, index bits); argmax_combine_kernel finishes the row
  EPI_F32_TMA = 9,     // EPI_F32 with TMA store boxes (logits heads)
  EPI_ROPE_TMA = 8,    // EPI_QKV_ROPE with TMA store boxes
  EPI_SWISH_TMA = 7,   // EPI_SWISH_BF16 with the tile leaving as TMA store boxes (pair kernel only; launcher's choice)
  EPI_RESID_TMA = 6,   // EPI_RESID_F32 with the add carried out as TMA reduce-add boxes (pair kernel only; chosen by the
                       // launcher, not part of the ABI): 128 B rows reach L2 as whole lines instead of 16 B reductions
  EPI_GELU_BF16 = 11,  // h = bf16(acc + bias); out_bf16 = bf16(GELU_erf(h))                       (HuBERT FeedForward up-proj)
  EPI_GELU_TMA = 12,   // EPI_GELU_BF16 with TMA store boxes (pair kernel only; launcher's choice)
};

// exact (erf) GELU, nn.GELU() / ACT2FN["gelu"]
__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.7071067811865476f)); }

struct GemmParams {
  int M, N, K;
  int a_k_offset;    // starting column inside A's tensor map (grouped per-codebook heads share one activation map)
  int b_row_offset;  // starting row inside B's tensor map (stacked per-codebook weights)
  const float* bias;  // [N] (already offset for the group) or nullptr
  void* out;          // bf16 / fp32, row-major with leading dimension ldo (elements); already offset for the group
  long long ldo;
  float scale;
  const float* rope_cos;  // [max_pos, 32] fp32
  const float* rope_sin;
  int reverse;    // 1: walk the output tiles from the last to the first (see edm_s2a_ctx::flip: each kernel of the decoder starts
                  // where its producer finished, so the most recently written ~100 MB of its input are still in L2)
  SeqLayout rope_lay;  // rotary position of a row = its position inside its sequence
  int rope_cols;  // columns [0, rope_cols) get rotary (q and k parts of the fused QKV projection)
  // small-M kernel, EPI_F32 only: K is cut into `splits` equal ranges, one work item per (tile, range); range s writes its raw fp32
  // partial sums (no bias) to out + s * split_stride. The consumer adds them in range order (layernorm_kernel with LnParams::partials).
  int splits;
  long long split_stride;
};

__device__ __forceinline__ int rope_pos(const GemmParams& p, int row) {
  int s, n;
  p.rope_lay.enc_pos(row, s, n);
  return n;
}

constexpr int kGemmBM = 128;
constexpr int kGemmBN = 256;
constexpr int kGemmBK = 64;
constexpr int kGemmEpiWarps = 16;  // four per TMEM lane quadrant, each owning 64 of the tile's 256 columns
constexpr int kGemmThreads = 64 + 32 * kGemmEpiWarps;
constexpr int kGemmMaxN = 8192;    // bias staging capacity
constexpr uint32_t kGemmABytes = kGemmBM * kGemmBK * 2;

// 32 consecutive columns of one row. v: accumulators (+ bias already added by the caller).
template <int EPI>
__device__ __forceinline__ void gemm_store_32(const GemmParams& p, int row, int col, float (&v)[32]) {
  if constexpr (EPI == EPI_F32) {
    float4* o = reinterpret_cast<float4*>(static_cast<float*>(p.out) + static_cast<long long>(row) * p.ldo + col);
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
  } else if constexpr (EPI == EPI_RESID_F32) {
    // x += scale * bf16(v): fire-and-forget vector reductions resolved in L2. Every element has exactly one writer per
    // GEMM, so the result is the same single rounded add a load/add/store would give, without pulling x through the SM.
    float* o = static_cast<float*>(p.out) + static_cast<long long>(row) * p.ldo + col;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(o + 4 * i), "f"(p.scale * bf16_round(v[4 * i + 0])),
                   "f"(p.scale * bf16_round(v[4 * i + 1])), "f"(p.scale * bf16_round(v[4 * i + 2])),
                   "f"(p.scale * bf16_round(v[4 * i + 3]))
                   : "memory");
    }
  } else {
    uint32_t w[16];
    if constexpr (EPI == EPI_SWISH_BF16) {
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const uint32_t h2 = pack_bf16x2(v[2 * i], v[2 * i + 1]);
        const uint32_t s2 = pack_bf16x2(sigmoid_tanh(bf16lo(h2)), sigmoid_tanh(bf16hi(h2)));
        w[i] = bf16x2_mul(h2, s2);
      }
    } else if constexpr (EPI == EPI_GELU_BF16) {
#pragma unroll
      for (int i = 0; i < 16; ++i) w[i] = pack_bf16x2(gelu_erf(bf16_round(v[2 * i])), gelu_erf(bf16_round(v[2 * i + 1])));
    } else {
#pragma unroll
      for (int i = 0; i < 16; ++i) w[i] = pack_bf16x2(v[2 * i], v[2 * i + 1]);
    }
    uint4* o = reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(p.out) + static_cast<long long>(row) * p.ldo + col);
#pragma unroll
    for (int i = 0; i < 4; ++i) o[i] = make_uint4(w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]);
  }
}

// EPI_ARGMAX: v = the 64 logits (acc + bias) of columns [col, col + 64) of one row, as two 32-column halves. Strict '>' in ascending
// column order keeps the first maximum, as torch.argmax does; a row of NaNs keeps index col (the combine step clamps).
__device__ __forceinline__ void gemm_store_argmax(const GemmParams& p, int row, int col, const float (&a)[32], const float (&b)[32]) {
  float best = a[0];
  int idx = 0;
#pragma unroll
  for (int i = 1; i < 32; ++i)
    if (a[i] > best) {
      best = a[i];
      idx = i;
    }
#pragma unroll
  for (int i = 0; i < 32; ++i)
    if (b[i] > best) {
      best = b[i];
      idx = 32 + i;
    }
  float2* o = reinterpret_cast<float2*>(p.out) + static_cast<long long>(row) * p.ldo + (col >> 6);
  *o = make_float2(best, __int_as_float(col + idx));
}

// One 64-wide head: lo = columns [col, col+32), hi = [col+32, col+64). Reference: conformer.py:45-51 (rotate_half),
// applied to the bf16 projection output in fp32 and rounded to bf16 when SDPA consumes it.
// GLU over one 64-column group: a = 32 value accumulators (+bias), g = their 32 gates (+bias). Reference: Conv1d output is
// bf16, GLU = out * gate.sigmoid() in bf16 (conformer/conformer.py:59-66,170-171). Writes 32 bf16 at column col_out.
__device__ __forceinline__ void gemm_store_glu(const GemmParams& p, int row, int col_out, const float (&a)[32], const float (&g)[32]) {
  uint32_t w[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const uint32_t a2 = pack_bf16x2(a[2 * i], a[2 * i + 1]);
    const uint32_t g2 = pack_bf16x2(g[2 * i], g[2 * i + 1]);
    const uint32_t s2 = pack_bf16x2(sigmoid_tanh(bf16lo(g2)), sigmoid_tanh(bf16hi(g2)));
    w[i] = bf16x2_mul(a2, s2);
  }
  uint4* o = reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(p.out) + static_cast<long long>(row) * p.ldo + col_out);
#pragma unroll
  for (int i = 0; i < 4; ++i) o[i] = make_uint4(w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]);
}

// tab_row: shared-space address of this row's cos|sin (16 float4, chunk index XOR-swizzled by swz), or 0 to read the
// global tables directly.
// stg_row != 0: the 8 output chunks go to this row of a 128B-swizzled shared-memory staging box (chunk c at (c ^ swz) * 16)
// instead of global memory.
__device__ __forceinline__ void gemm_epilogue_rope64(const GemmParams& p, int row, int col, const uint32_t (&lo)[32],
                                                     const uint32_t (&hi)[32], uint32_t tab_row = 0, int swz = 0, uint32_t stg_row = 0) {
  uint4* o = reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(p.out) + static_cast<long long>(row) * p.ldo + col);
  auto put = [&](int c, uint4 v) {
    if (stg_row != 0)
      sts128(stg_row + ((c ^ swz) << 4), make_float4(__uint_as_float(v.x), __uint_as_float(v.y), __uint_as_float(v.z), __uint_as_float(v.w)));
    else
      o[c] = v;
  };
  // the projection output is bf16 in the reference: round first (also halves the live registers)
  uint32_t l2[16], h2[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    l2[i] = pack_bf16x2(__uint_as_float(lo[2 * i]), __uint_as_float(lo[2 * i + 1]));
    h2[i] = pack_bf16x2(__uint_as_float(hi[2 * i]), __uint_as_float(hi[2 * i + 1]));
  }
  if (col < p.rope_cols) {
    const int pos = rope_pos(p, row);
    const float4* c4 = reinterpret_cast<const float4*>(p.rope_cos + static_cast<long long>(pos) * 32);
    const float4* s4 = reinterpret_cast<const float4*>(p.rope_sin + static_cast<long long>(pos) * 32);
#pragma unroll
    for (int g = 0; g < 4; ++g) {  // 8 columns of each half per group: cos/sin chunks 2g, 2g+1
      float4 cs[2], sn[2];
      if (tab_row != 0) {
        cs[0] = lds128(tab_row + 16 * ((2 * g) ^ swz));
        cs[1] = lds128(tab_row + 16 * ((2 * g + 1) ^ swz));
        sn[0] = lds128(tab_row + 16 * (8 + ((2 * g) ^ swz)));
        sn[1] = lds128(tab_row + 16 * (8 + ((2 * g + 1) ^ swz)));
      } else {
        cs[0] = __ldg(c4 + 2 * g);
        cs[1] = __ldg(c4 + 2 * g + 1);
        sn[0] = __ldg(s4 + 2 * g);
        sn[1] = __ldg(s4 + 2 * g + 1);
      }
      uint32_t ol[4], oh[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int i = 4 * g + q;  // packed pair index: columns 2i, 2i+1
        const float4 c = cs[q >> 1], s = sn[q >> 1];
        const float c0 = (q & 1) ? c.z : c.x, c1 = (q & 1) ? c.w : c.y;
        const float s0 = (q & 1) ? s.z : s.x, s1 = (q & 1) ? s.w : s.y;
        const float x1a = bf16lo(l2[i]), x1b = bf16hi(l2[i]), x2a = bf16lo(h2[i]), x2b = bf16hi(h2[i]);
        ol[q] = pack_bf16x2(__fadd_rn(__fmul_rn(x1a, c0), __fmul_rn(-x2a, s0)), __fadd_rn(__fmul_rn(x1b, c1), __fmul_rn(-x2b, s1)));
        oh[q] = pack_bf16x2(__fadd_rn(__fmul_rn(x2a, c0), __fmul_rn(x1a, s0)), __fadd_rn(__fmul_rn(x2b, c1), __fmul_rn(x1b, s1)));
      }
      put(g, make_uint4(ol[0], ol[1], ol[2], ol[3]));
      put(4 + g, make_uint4(oh[0], oh[1], oh[2], oh[3]));
    }
  } else {
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      put(g, make_uint4(l2[4 * g], l2[4 * g + 1], l2[4 * g + 2], l2[4 * g + 3]));
      put(4 + g, make_uint4(h2[4 * g], h2[4 * g + 1], h2[4 * g + 2], h2[4 * g + 3]));
    }
  }
}

// ------------------------------------------------------------------------------------------------ small-M variant
// At M <= a few hundred rows (single-utterance decodes) the 256 x 256 CTA-pair tiles leave 4-32 CTAs, each streaming 128 weight rows
// x K from HBM, while the other SMs idle: the GEMM is a weight-streaming problem, not a tensor-pipe one. This variant uses
// 128 x 64 tiles (N / 64 CTAs per 128 rows: 16-128 CTAs pull the weights concurrently) and an 8-stage ring of 24 KB stages so each
// CTA keeps 190 KB of loads in flight. Epilogues store from registers ( a 64-column tile is one epilogue
// sub-tile: GLU pairs and rotary heads never straddle it). The weight tensor map has 64-row boxes (WMap::small in abi.cu).
// Round 2 (tools/ktrace.py timeline: 2.2 us per kernel boundary, 0.75 us to the first A tile, 250 ns per k-step = the ring's ~2 us
// round trip / 8 stages): (1) under programmatic dependent launch the producer requests the first ring-full of WEIGHT tiles before
// griddepcontrol.wait - they are constants - and only the A tiles after it; (2) the epilogue loads its bias / touches its rotary rows
// before it waits for the accumulator; (3) a work item may be one of `splits` K ranges of a tile (EPI_F32 raw partial sums, reduced in
// range order by layernorm_splitk_kernel): the long-K residual GEMMs of single-utterance decodes then use 128 instead of 32 CTAs.
constexpr int kSmBN = 64;
constexpr int kSmStages = 8;
constexpr int kSmThreads = 64 + 32 * 4;
constexpr uint32_t kSmBBytes = kSmBN * kGemmBK * 2;
constexpr uint32_t kSmStageBytes = kGemmABytes + kSmBBytes;
constexpr uint32_t kSmSmemBytes = kSmStages * kSmStageBytes + 1024 + 256;

template <int EPI>
__global__ void __launch_bounds__(kSmThreads, 1)
gemm_bf16_tn_small_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b, const GemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kSmStages * kSmStageBytes);
  uint64_t* empty_bar = full_bar + kSmStages;
  uint64_t* tmem_full_bar = empty_bar + kSmStages;
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;
  uint32_t* tmem_base_slot = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_m = (p.M + kGemmBM - 1) / kGemmBM;
  const int num_n = p.N / kSmBN;
  const int splits = (EPI == EPI_F32 && p.splits > 1) ? p.splits : 1;
  const int num_tiles = num_m * num_n * splits;  // work items: (tile, K range), the ranges of a tile adjacent
  const int num_kb = p.K / kGemmBK / splits;      // k-blocks per work item

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_b);
    for (int s = 0; s < kSmStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tmem_full_bar[b], 1);
      mbar_init(&tmem_empty_bar[b], 4);  // one elected lane per epilogue warp
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc<128>(tmem_base_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_base_slot;
  // Prologue done (barriers, TMEM). Everything the previous kernel of the stream wrote (the activations: A operand, residual stream)
  // may be touched only after pdl_wait; the weights are constants, so the producer requests the first ring-full of weight tiles
  // before it waits: their DRAM latency (the whole cost of a single-utterance GEMM) overlaps the previous kernel's tail.
  KTRACE_ENTRY(kt_entry);
  pdl_trigger();
  if (warp == 0) {
    if (lane == 0) {
      const int t0 = blockIdx.x;
      const int pre = t0 < num_tiles ? (num_kb < kSmStages ? num_kb : kSmStages) : 0;
      for (int kb = 0; kb < pre; ++kb) {
        mbar_arrive_expect_tx(&full_bar[kb], kSmStageBytes);
        tma_load_2d(&tma_b, &full_bar[kb], smem + kb * kSmStageBytes + kGemmABytes, ((t0 % splits) * num_kb + kb) * kGemmBK,
                    p.b_row_offset + ((t0 / splits) % num_n) * kSmBN);
      }
      pdl_wait();
      KTRACE_PUT(1, kt_entry);
      KTRACE_PUT(2, ktrace_now());
      uint32_t it = 0;
      for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
        const int m_blk = (t / splits) / num_n, n_blk = (t / splits) % num_n, kb0 = (t % splits) * num_kb;
        for (int kb = 0; kb < num_kb; ++kb, ++it) {
          const uint32_t stage = it % kSmStages;
          uint8_t* sa = smem + stage * kSmStageBytes;
          if (it >= static_cast<uint32_t>(pre)) {
            // polling wait: the ring is latency-bound at small M (8 stages = 192 KB in flight per SM against a ~2 us load + hand-back
            // round trip), and the hardware-suspended try_wait adds its 0.4-0.7 us wake-up to every round
            mbar_wait_spin(&empty_bar[stage], ((it / kSmStages) & 1) ^ 1);
            mbar_arrive_expect_tx(&full_bar[stage], kSmStageBytes);
            tma_load_2d(&tma_b, &full_bar[stage], sa + kGemmABytes, (kb0 + kb) * kGemmBK, p.b_row_offset + n_blk * kSmBN);
          }
          tma_load_2d(&tma_a, &full_bar[stage], sa, p.a_k_offset + (kb0 + kb) * kGemmBK, m_blk * kGemmBM);
        }
      }
    }
  } else if (warp == 1) {
    pdl_wait();
    constexpr uint32_t idesc = umma_idesc_bf16(kGemmBM, kSmBN, 0, 0);
    uint32_t it = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
      mbar_wait_spin(&tmem_empty_bar[acc], acc_phase ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * kSmBN;
      for (int kb = 0; kb < num_kb; ++kb, ++it) {
        const uint32_t stage = it % kSmStages;
        mbar_wait_spin(&full_bar[stage], (it / kSmStages) & 1);
        tc_fence_after();
#ifdef EDM_KTRACE
        if (it == 0 && lane == 0) KTRACE_PUT(3, ktrace_now());
#endif
        const uint32_t sa = smem_u32(smem + stage * kSmStageBytes);
        const uint64_t adesc = umma_desc_sw128(sa, 16, 1024);
        const uint64_t bdesc = umma_desc_sw128(sa + kGemmABytes, 16, 1024);
#pragma unroll
        for (int k = 0; k < kGemmBK / 16; ++k) umma_ss_warp(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
        umma_commit_warp(&empty_bar[stage]);
      }
      umma_commit_warp(&tmem_full_bar[acc]);
#ifdef EDM_KTRACE
      if (lane == 0) KTRACE_PUT(4, ktrace_now());
#endif
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  } else {
    pdl_wait();
    const int quad = warp & 3;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
      const int m_blk = (t / splits) / num_n, n_blk = (t / splits) % num_n;
      const int row = m_blk * kGemmBM + quad * 32 + lane;
      const int col0 = n_blk * kSmBN;
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + acc * kSmBN;
      // the tile's 64 bias values are requested before the wait for the accumulator: an L2 round trip off the critical path
      float4 bias_v[16];
      if constexpr (EPI == EPI_QKV_ROPE) {
        if (col0 < p.rope_cols && row < p.M) {  // this row's cos | sin lines (constants): in L1 by the time the accumulator is ready
          prefetch_l1(p.rope_cos + static_cast<long long>(rope_pos(p, row)) * 32);
          prefetch_l1(p.rope_sin + static_cast<long long>(rope_pos(p, row)) * 32);
        }
      }
      if constexpr (EPI != EPI_QKV_ROPE) {
        const float4* bg = reinterpret_cast<const float4*>(p.bias != nullptr ? p.bias + col0 : nullptr);
#pragma unroll
        for (int i = 0; i < 16; ++i) bias_v[i] = bg != nullptr ? __ldg(bg + i) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      mbar_wait(&tmem_full_bar[acc], acc_phase);
      tc_fence_after();
      uint32_t r0[32], r1[32];
      tmem_ld_32x32(taddr, r0);
      tmem_ld_32x32(taddr + 32, r1);
      tmem_ld_wait_dep(r0);
      tmem_ld_wait_dep(r1);
      tc_fence_before();
      __syncwarp();
#ifdef EDM_KTRACE
      if (warp == 2 && lane == 0) KTRACE_PUT(5, ktrace_now());
#endif
      if (lane == 0) mbar_arrive(&tmem_empty_bar[acc]);
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
      if (row >= p.M) continue;
      if constexpr (EPI == EPI_QKV_ROPE) {
        gemm_epilogue_rope64(p, row, col0, r0, r1);
      } else {
        auto bias4 = [&](int i) { return bias_v[i]; };
        float v[32];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 b = bias4(i);
          v[4 * i + 0] = __uint_as_float(r0[4 * i + 0]) + b.x;
          v[4 * i + 1] = __uint_as_float(r0[4 * i + 1]) + b.y;
          v[4 * i + 2] = __uint_as_float(r0[4 * i + 2]) + b.z;
          v[4 * i + 3] = __uint_as_float(r0[4 * i + 3]) + b.w;
        }
        if constexpr (EPI == EPI_GLU_BF16 || EPI == EPI_ARGMAX) {
          float g[32];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float4 b = bias4(8 + i);
            g[4 * i + 0] = __uint_as_float(r1[4 * i + 0]) + b.x;
            g[4 * i + 1] = __uint_as_float(r1[4 * i + 1]) + b.y;
            g[4 * i + 2] = __uint_as_float(r1[4 * i + 2]) + b.z;
            g[4 * i + 3] = __uint_as_float(r1[4 * i + 3]) + b.w;
          }
          if constexpr (EPI == EPI_GLU_BF16)
            gemm_store_glu(p, row, col0 >> 1, v, g);
          else
            gemm_store_argmax(p, row, col0, v, g);
        } else {
          GemmParams q = p;
          if constexpr (EPI == EPI_F32) q.out = static_cast<float*>(p.out) + (t % splits) * p.split_stride;  // this K range's partial sums
          gemm_store_32<EPI>(q, row, col0, v);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float4 b = bias4(8 + i);
            v[4 * i + 0] = __uint_as_float(r1[4 * i + 0]) + b.x;
            v[4 * i + 1] = __uint_as_float(r1[4 * i + 1]) + b.y;
            v[4 * i + 2] = __uint_as_float(r1[4 * i + 2]) + b.z;
            v[4 * i + 3] = __uint_as_float(r1[4 * i + 3]) + b.w;
          }
          gemm_store_32<EPI>(q, row, col0 + 32, v);
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
#ifdef EDM_KTRACE
  if (threadIdx.x == 64) KTRACE_END(100 + EPI);
#endif
  if (warp == 1) tmem_dealloc<128>(tmem_base);
}

// ------------------------------------------------------------------------------------------------ CTA-pair variant
// Same roles, but two CTAs of a cluster (two SMs of one TPC) share each 256 x 256 output tile through
// tcgen05.mma.cta_group::2: CTA r loads rows r*128.. of A and rows r*128.. of the B tile (half the B bytes per SM, a third
// less L2->SM operand traffic per FLOP than 128 x 256 tiles), CTA 0's MMA thread issues M = 256 instructions that read
// both CTAs' shared memory and write each CTA's own TMEM half, completion is multicast to both CTAs' barriers.
// 32 KB per stage instead of 48 KB -> a 6-deep ring in the same shared memory.
// Shared memory of one CTA: a ring of 32 KB stages, then (TMA-output epilogues) a 4 KB staging box per epilogue warp, then (rotary
// epilogues) the 32 KB cos|sin table of the tile's rows, barriers at a fixed offset. The bias is read through the read-only path by
// the epilogue threads (64 floats each, L1-resident), not staged: that leaves room for 7 / 5 ring stages instead of 6 / 4.
constexpr uint32_t kPairStageBytes = 2 * kGemmABytes;  // A (128 x 64) + half of B (128 x 64)
constexpr uint32_t kPairStagingBytes = 32 * 32 * 4;    // 32 rows x 32 fp32 columns (or 32 rows x 64 bf16)
constexpr uint32_t kPairRopeTabBytes = 128 * 16 * 16;  // 128 rows x (8 cos + 8 sin float4 chunks)
constexpr uint32_t kPairBarOffset = 7 * kPairStageBytes;
constexpr uint32_t kPairSmemBytes = kPairBarOffset + 256 + 1024;
__host__ __device__ constexpr int pair_stages(bool tma_out, bool rope) { return rope ? (tma_out ? 4 : 6) : (tma_out ? 5 : 7); }
constexpr int kPairMaxStages = 7;

template <int EPI>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kGemmThreads, 1)
gemm_bf16_tn_pair_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
                         const __grid_constant__ CUtensorMap tma_c, const GemmParams p) {
  constexpr bool kTmaOut = EPI == EPI_RESID_TMA || EPI == EPI_SWISH_TMA || EPI == EPI_GELU_TMA || EPI == EPI_ROPE_TMA || EPI == EPI_F32_TMA;
  constexpr bool kRope = EPI == EPI_QKV_ROPE || EPI == EPI_ROPE_TMA;
  constexpr int kSt = pair_stages(kTmaOut, kRope);
  constexpr uint32_t kStagingOffset = kSt * kPairStageBytes;
  constexpr uint32_t kRopeTabOffset = kStagingOffset + (kTmaOut ? kGemmEpiWarps * kPairStagingBytes : 0);
  static_assert(kRopeTabOffset + (kRope ? kPairRopeTabBytes : 0) <= kPairBarOffset, "smem budget");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  float* s_rope = reinterpret_cast<float*>(smem + kRopeTabOffset);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kPairBarOffset);
  uint64_t* empty_bar = full_bar + kPairMaxStages;
  uint64_t* tmem_full_bar = empty_bar + kPairMaxStages;
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;
  uint32_t* tmem_base_slot = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;

  const int num_m = (p.M + 2 * kGemmBM - 1) / (2 * kGemmBM);
  const int num_n = p.N / kGemmBN;
  const int num_tiles = num_m * num_n;
  const int num_kb = p.K / kGemmBK;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_b);
    for (int s = 0; s < kSt; ++s) {
      mbar_init(&full_bar[s], 1);   // CTA 0's expect_tx arrive; the bytes of both CTAs land here
      mbar_init(&empty_bar[s], 1);  // one multicast commit per use
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tmem_full_bar[b], 1);
      mbar_init(&tmem_empty_bar[b], 2 * kGemmEpiWarps);  // one lane per epilogue warp of both CTAs arrives on CTA 0's barrier
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc_pair<512>(tmem_base_slot);
  tc_fence_before();
  cluster_sync_all();  // both CTAs' barriers initialised and TMEM allocated before any cross-CTA signal
  tc_fence_after();
  const uint32_t tmem_base = *tmem_base_slot;
  pdl_sync();  // prologue done (barriers, TMEM): the previous kernel's activations are read from here on

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int t = pair; t < num_tiles; t += num_pairs) {
        const int tt = p.reverse ? num_tiles - 1 - t : t;
        const int m_blk = tt / num_n, n_blk = tt % num_n;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem + stage * kPairStageBytes;
          uint8_t* sb = sa + kGemmABytes;
          if (rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * kPairStageBytes);
          tma_load_2d_pair(&tma_a, &full_bar[stage], sa, p.a_k_offset + kb * kGemmBK, m_blk * 2 * kGemmBM + rank * kGemmBM);
          tma_load_2d_pair(&tma_b, &full_bar[stage], sb, kb * kGemmBK, p.b_row_offset + n_blk * kGemmBN + rank * (kGemmBN / 2));
          if (++stage == kSt) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    if (rank == 0) {  // whole warp of CTA 0, warp-uniform control flow; one elected lane issues (umma_*_pair_warp, see ptx.cuh)
      constexpr uint32_t idesc = umma_idesc_bf16(2 * kGemmBM, kGemmBN, 0, 0);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int t = pair; t < num_tiles; t += num_pairs) {
        mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * kGemmBN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * kPairStageBytes);
          const uint64_t adesc = umma_desc_sw128(sa, 16, 1024);
          const uint64_t bdesc = umma_desc_sw128(sa + kGemmABytes, 16, 1024);
#pragma unroll
          for (int k = 0; k < kGemmBK / 16; ++k) umma_ss_pair_warp(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
          umma_commit_pair_warp(&empty_bar[stage]);
          if (++stage == kSt) {
            stage = 0;
            phase ^= 1;
          }
        }
        umma_commit_pair_warp(&tmem_full_bar[acc]);
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    }
  } else {
    const int quad = warp & 3;
    const int sub = (warp - 2) >> 2;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int t = pair; t < num_tiles; t += num_pairs) {
      const int tt = p.reverse ? num_tiles - 1 - t : t;
      const int m_blk = tt / num_n, n_blk = tt % num_n;
      const int row = m_blk * 2 * kGemmBM + static_cast<int>(rank) * kGemmBM + quad * 32 + lane;
      const int col0 = n_blk * kGemmBN + sub * 64;
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + acc * kGemmBN + sub * 64;
      // this thread's 64 bias values as 16 float4 chunks: the same addresses in every lane (one broadcast transaction each), L1-resident
      const float4* bias_g = reinterpret_cast<const float4*>(p.bias != nullptr ? p.bias + col0 : nullptr);
      auto bias4 = [&](int k) { return bias_g != nullptr ? __ldg(bias_g + k) : make_float4(0.f, 0.f, 0.f, 0.f); };
      bool rope_tile = false;
      if constexpr (kRope) {
        // The rotary cos|sin rows of this CTA's 128 token rows go to shared memory
        // while the tile's mainloop is still running: one coalesced 32 KB read per tile instead of 4 x 128 rows x 256 B
        // of dependent 16-byte loads. Chunk index is XOR-swizzled with (row & 7) so row-per-lane reads are conflict-free.
        rope_tile = n_blk * kGemmBN < p.rope_cols;
        if (rope_tile) {
          float4* tab = reinterpret_cast<float4*>(s_rope);
          const int et = threadIdx.x - 64;
          asm volatile("bar.sync 1, 512;" ::: "memory");  // previous tile's readers are done
#pragma unroll
          for (int i = et; i < 128 * 16; i += 32 * kGemmEpiWarps) {
            const int r = i >> 4, c = i & 15;
            const int grow = m_blk * 2 * kGemmBM + static_cast<int>(rank) * kGemmBM + r;
            const int pos = rope_pos(p, grow < p.M ? grow : 0);
            const float* src = (c < 8 ? p.rope_cos : p.rope_sin) + static_cast<long long>(pos) * 32 + (c & 7) * 4;
            tab[r * 16 + (c ^ (r & 7))] = __ldg(reinterpret_cast<const float4*>(src));
          }
          asm volatile("bar.sync 1, 512;" ::: "memory");
        }
      }
      mbar_wait(&tmem_full_bar[acc], acc_phase);
      tc_fence_after();
      uint32_t r0[32], r1[32];
      tmem_ld_32x32(taddr, r0);
      tmem_ld_32x32(taddr + 32, r1);
      tmem_ld_wait_dep(r0);
      tmem_ld_wait_dep(r1);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(&tmem_empty_bar[acc], 0);
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
      if constexpr (EPI == EPI_ROPE_TMA) {
        uint8_t* stg = smem + kStagingOffset + (warp - 2) * kPairStagingBytes;
        const int tr = quad * 32 + lane;
        if (lane == 0) bulk_wait_group_read0();
        __syncwarp();
        gemm_epilogue_rope64(p, row, col0, r0, r1, rope_tile ? smem_u32(s_rope) + tr * 256 : 0u, tr & 7, smem_u32(stg) + lane * 128);
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_2d(&tma_c, stg, col0, m_blk * 2 * kGemmBM + static_cast<int>(rank) * kGemmBM + quad * 32);
          bulk_commit_group();
        }
        continue;
      }
      if constexpr (EPI == EPI_GELU_TMA) {
        // as EPI_SWISH_TMA below, but each 16-byte chunk goes to the staging box as soon as it is computed (erf is long: fewer live
        // registers than converting the whole slice first)
        uint8_t* stg = smem + kStagingOffset + (warp - 2) * kPairStagingBytes;
        const uint32_t stg_row = smem_u32(stg) + lane * 128;
        const int sw = lane & 7;
        if (lane == 0) bulk_wait_group_read0();
        __syncwarp();
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const uint32_t* r = c < 4 ? r0 : r1;
          const int q = (c & 3) * 8;
          uint32_t w[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float4 b = bias4((q + 2 * e) / 4 + 8 * (c >> 2));
            const float b0 = (e & 1) ? b.z : b.x, b1 = (e & 1) ? b.w : b.y;
            w[e] = pack_bf16x2(gelu_erf(bf16_round(__uint_as_float(r[q + 2 * e]) + b0)), gelu_erf(bf16_round(__uint_as_float(r[q + 2 * e + 1]) + b1)));
          }
          sts128(stg_row + ((c ^ sw) << 4), make_float4(__uint_as_float(w[0]), __uint_as_float(w[1]), __uint_as_float(w[2]), __uint_as_float(w[3])));
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_2d(&tma_c, stg, col0, m_blk * 2 * kGemmBM + static_cast<int>(rank) * kGemmBM + quad * 32);
          bulk_commit_group();
        }
        continue;
      }
      if constexpr (EPI == EPI_SWISH_TMA) {
        // bf16 output: the warp's 32 x 64 slice is one 32-row x 128-byte box in its staging buffer (128B-swizzled rows), stored
        // by TMA as whole lines instead of 32 x 8 scattered 16-byte stores; rows beyond M are clipped by the tensor map
        uint8_t* stg = smem + kStagingOffset + (warp - 2) * kPairStagingBytes;
        const uint32_t stg_row = smem_u32(stg) + lane * 128;
        const int sw = lane & 7;
        const int row0 = m_blk * 2 * kGemmBM + static_cast<int>(rank) * kGemmBM + quad * 32;
        uint32_t w[32];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const uint32_t* r = h == 0 ? r0 : r1;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float4 b = bias4(8 * h + i);
            const uint32_t h01 = pack_bf16x2(__uint_as_float(r[4 * i + 0]) + b.x, __uint_as_float(r[4 * i + 1]) + b.y);
            const uint32_t h23 = pack_bf16x2(__uint_as_float(r[4 * i + 2]) + b.z, __uint_as_float(r[4 * i + 3]) + b.w);
            w[16 * h + 2 * i] = bf16x2_mul(h01, pack_bf16x2(sigmoid_tanh(bf16lo(h01)), sigmoid_tanh(bf16hi(h01))));
            w[16 * h + 2 * i + 1] = bf16x2_mul(h23, pack_bf16x2(sigmoid_tanh(bf16lo(h23)), sigmoid_tanh(bf16hi(h23))));
          }
        }
        if (lane == 0) bulk_wait_group_read0();  // the previous tile's box has been read out of the staging buffer
        __syncwarp();
#pragma unroll
        for (int c = 0; c < 8; ++c)
          sts128(stg_row + ((c ^ sw) << 4), make_float4(__uint_as_float(w[4 * c]), __uint_as_float(w[4 * c + 1]), __uint_as_float(w[4 * c + 2]),
                                                       __uint_as_float(w[4 * c + 3])));
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_2d(&tma_c, stg, col0, row0);
          bulk_commit_group();
        }
        continue;
      }
      if constexpr (EPI == EPI_RESID_TMA || EPI == EPI_F32_TMA) {
        // RESID: x[rows, cols] += scale * bf16(acc + bias) (TMA reduce-add); F32: out = acc + bias (TMA store).
        // The warp's 32 x 64 slice leaves as two 32 x 32 fp32 boxes through its
        // 4 KB staging buffer (128B-swizzled rows); rows beyond M are clipped by the tensor map
        uint8_t* stg = smem + kStagingOffset + (warp - 2) * kPairStagingBytes;
        const uint32_t stg_row = smem_u32(stg) + lane * 128;
        const int sw = lane & 7;
        const int row0 = m_blk * 2 * kGemmBM + static_cast<int>(rank) * kGemmBM + quad * 32;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          if (lane == 0) bulk_wait_group_read0();  // the previous box has been read out of the staging buffer
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float4 b = bias4(8 * h + i);
            const uint32_t* r = h == 0 ? r0 : r1;
            if constexpr (EPI == EPI_RESID_TMA)
              sts128(stg_row + ((i ^ sw) << 4),
                     make_float4(p.scale * bf16_round(__uint_as_float(r[4 * i + 0]) + b.x), p.scale * bf16_round(__uint_as_float(r[4 * i + 1]) + b.y),
                                 p.scale * bf16_round(__uint_as_float(r[4 * i + 2]) + b.z), p.scale * bf16_round(__uint_as_float(r[4 * i + 3]) + b.w)));
            else
              sts128(stg_row + ((i ^ sw) << 4), make_float4(__uint_as_float(r[4 * i + 0]) + b.x, __uint_as_float(r[4 * i + 1]) + b.y,
                                                            __uint_as_float(r[4 * i + 2]) + b.z, __uint_as_float(r[4 * i + 3]) + b.w));
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            if constexpr (EPI == EPI_RESID_TMA)
              tma_reduce_add_2d(&tma_c, stg, col0 + 32 * h, row0);
            else
              tma_store_2d(&tma_c, stg, col0 + 32 * h, row0);
            bulk_commit_group();
          }
        }
        continue;
      }
      if (row >= p.M) continue;
      if constexpr (EPI == EPI_QKV_ROPE) {
        const int tr = quad * 32 + lane;
        gemm_epilogue_rope64(p, row, col0, r0, r1, rope_tile ? smem_u32(s_rope) + tr * 256 : 0u, tr & 7);
      } else {
        float v[32];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 b = bias4(i);
          v[4 * i + 0] = __uint_as_float(r0[4 * i + 0]) + b.x;
          v[4 * i + 1] = __uint_as_float(r0[4 * i + 1]) + b.y;
          v[4 * i + 2] = __uint_as_float(r0[4 * i + 2]) + b.z;
          v[4 * i + 3] = __uint_as_float(r0[4 * i + 3]) + b.w;
        }
        if constexpr (EPI == EPI_GLU_BF16 || EPI == EPI_ARGMAX) {
          float g[32];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float4 b = bias4(8 + i);
            g[4 * i + 0] = __uint_as_float(r1[4 * i + 0]) + b.x;
            g[4 * i + 1] = __uint_as_float(r1[4 * i + 1]) + b.y;
            g[4 * i + 2] = __uint_as_float(r1[4 * i + 2]) + b.z;
            g[4 * i + 3] = __uint_as_float(r1[4 * i + 3]) + b.w;
          }
          if constexpr (EPI == EPI_GLU_BF16)
            gemm_store_glu(p, row, col0 >> 1, v, g);
          else
            gemm_store_argmax(p, row, col0, v, g);
        } else {
          gemm_store_32<EPI>(p, row, col0, v);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float4 b = bias4(8 + i);
            v[4 * i + 0] = __uint_as_float(r1[4 * i + 0]) + b.x;
            v[4 * i + 1] = __uint_as_float(r1[4 * i + 1]) + b.y;
            v[4 * i + 2] = __uint_as_float(r1[4 * i + 2]) + b.z;
            v[4 * i + 3] = __uint_as_float(r1[4 * i + 3]) + b.w;
          }
          gemm_store_32<EPI>(p, row, col0 + 32, v);
        }
      }
    }
  }

  if constexpr (kTmaOut) {
    if (warp >= 2 && lane == 0) bulk_wait_group0();  // staging buffers must outlive the reductions that read them
  }
  tc_fence_before();
  cluster_sync_all();  // the peer may still be reading our shared memory / signalling our barriers
  if (warp == 1) tmem_dealloc_pair<512>(tmem_base);
}

}  // namespace edm
