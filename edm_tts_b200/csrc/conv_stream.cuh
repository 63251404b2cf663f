// Conformer conv-module core on an already gated input, streaming version.
// Reference: conformer.py:69-77 + :23-25 (depthwise conv k = 5, zero pad (2,2) inside each sequence), :54-56 (Swish),
// :90-99 (ChanLayerNorm: mean / biased var over the 2048 channels of a token, scale only, eps = 1e-4 under bf16 autocast).
// Arithmetic and rounding points are those of conv_module_kernel<false> (elementwise.cuh); what changes is the data movement
// and the instruction count:
//   * persistent CTAs (one per SM) walk "runs" of consecutive tokens of one sequence with the 5-tap window carried in
//     registers, so only 4 halo rows per run are read twice (7 % at the bench shape instead of 20 %);
//   * token rows (4 KB, contiguous in memory within a run) are pulled into a 32-row shared-memory ring by cp.async.bulk, 8 rows
//     (32 KB) per copy and per mbarrier: 64 KB of loads stay in flight per SM while all 16 warps compute;
//   * the fp32 conv / Swish / statistics arithmetic works on channel pairs with the packed f32x2 instructions of sm_100
//     (fma.rn.f32x2 and friends), which halves the FMA-pipe instruction count;
//   * per-token statistics: every thread contributes one (sum, sum of squares) pair per token through shared memory, one warp
//     per token reduces them; the Swish outputs themselves never leave registers.
// in : [rows, 2048] bf16 (GLU already applied by the pointwise-conv GEMM epilogue)     out : [rows, 2048] bf16
// Sequences are placed by a SeqLayout; a run never crosses the end of its sequence, so the zero padding is per sequence.
#pragma once
#include <type_traits>

#include "elementwise.cuh"

namespace edm {

constexpr int kCsThreads = 512;   // 4 channels per thread
constexpr int kCsGroup = 16;      // tokens per statistics group = one per warp
constexpr int kCsRing = 32;       // ring slots (token rows of 4 KB)
constexpr int kCsChunk = 8;       // rows per mbarrier: the ring is 4 chunks of 8 rows, each filled by one or two bulk copies
constexpr uint32_t kCsRowBytes = kConvC * 2;
constexpr uint32_t kCsSmemBytes = kCsRing * kCsRowBytes + kCsGroup * kCsThreads * 8 + kCsGroup * 8 + (kCsRing / kCsChunk) * 8 + 128;

struct ConvStreamParams {
  const __nv_bfloat16* in;
  __nv_bfloat16* out;
  const float* dw_w;    // [2048, 5]
  const float* dw_b;    // [2048]
  const float* cln_w;   // [2048]
  SeqLayout lay;
  int run_len;          // tokens per run
  int runs_per_seq;     // uniform layout: runs of every sequence
  const int* cu_runs;   // packed layout: [n_seq + 1] first run of each sequence (nullptr: uniform)
  int num_units;        // runs in all
  int reverse;          // 1: the runs are walked from the last to the first
};

__device__ __forceinline__ void bulk_load_row(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src),
               "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// mbarrier wait without the printf watchdog of mbar_wait (it sits in a fully unrolled 16-token loop and must stay two
// instructions on the fast path); a wedged pipeline still traps instead of hanging the GPU
__device__ __forceinline__ void cs_wait(uint32_t bar_addr, uint32_t parity) {
  uint32_t ok, spins = 0;
  do {
    asm volatile(
        "{\n\t"
        ".reg .pred P;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, P;\n\t"
        "}\n"
        : "=r"(ok)
        : "r"(bar_addr), "r"(parity)
        : "memory");
    if (!ok && ++spins > (1u << 28)) __trap();
  } while (!ok);
}

struct CsRun {
  long long row0;                     // first row of the run's sequence
  int t_begin, t_end, t_lo, t_hi;     // output tokens [t_begin, t_end), rows that exist in memory [t_lo, t_hi)
};
__device__ __forceinline__ CsRun cs_run(const ConvStreamParams& p, int unit) {
  CsRun r;
  if (p.reverse) unit = p.num_units - 1 - unit;
  int b, k;
  if (p.cu_runs != nullptr) {
    b = p.lay.search(p.cu_runs, unit);
    k = unit - __ldg(p.cu_runs + b);
  } else {
    b = unit / p.runs_per_seq;
    k = unit % p.runs_per_seq;
  }
  const int n = p.lay.n_len(b);
  r.row0 = p.lay.n_start(b);
  r.t_begin = k * p.run_len;
  r.t_end = min(n, r.t_begin + p.run_len);
  r.t_lo = max(0, r.t_begin - 2);
  r.t_hi = min(n, r.t_end + 2);
  return r;
}

__global__ void __launch_bounds__(kCsThreads, 1) conv_stream_kernel(const ConvStreamParams p) {
  extern __shared__ __align__(128) uint8_t cs_smem[];
  uint8_t* s_ring = cs_smem;                                                          // [32][4096]
  float2* s_part = reinterpret_cast<float2*>(s_ring + kCsRing * kCsRowBytes);         // [16][512] (sum, sum of squares)
  uint2* s_stat = reinterpret_cast<uint2*>(s_part + kCsGroup * kCsThreads);           // [16] (mean, mean | rstd, rstd) bf16x2
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_stat + kCsGroup);                   // [4] one per ring chunk

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int c0 = tid * 4;
  const int num_units = p.num_units;

  if (tid == 0) {
    for (int s = 0; s < kCsRing / kCsChunk; ++s) mbar_init(&s_bar[s], 1);
    fence_mbar_init();
  }
  __syncthreads();
  KTRACE_ENTRY(kt_entry);
  pdl_sync();
#ifdef EDM_KTRACE
  if (tid == 0) { KTRACE_PUT(1, kt_entry); KTRACE_PUT(2, ktrace_now()); }
#endif

  // producer state (thread 0 only): next row to request, as (unit, row inside the unit's [t_lo, t_hi))
  int pu = blockIdx.x, pr = 0;
  uint32_t q_issued = 0;
  CsRun prun = cs_run(p, pu < num_units ? pu : 0);
  // fills whole chunks (8 ring rows) while their slots are free: rows with sequence number < limit may be requested
  auto producer_fill = [&](uint32_t limit) {
    while (pu < num_units && q_issued + kCsChunk <= limit) {
      uint64_t* bar = &s_bar[(q_issued / kCsChunk) % (kCsRing / kCsChunk)];
      int room = kCsChunk;
      while (room > 0 && pu < num_units) {  // a chunk spans at most the tail of one run and the head of the next ones
        const int n = min(room, prun.t_hi - prun.t_lo - pr);
        asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(n * kCsRowBytes) : "memory");
        bulk_load_row(s_ring + (q_issued % kCsRing) * kCsRowBytes, p.in + (prun.row0 + prun.t_lo + pr) * kConvC,
                      n * kCsRowBytes, bar);
        q_issued += n;
        room -= n;
        pr += n;
        if (pr == prun.t_hi - prun.t_lo) {
          pr = 0;
          pu += gridDim.x;
          if (pu < num_units) prun = cs_run(p, pu);
        }
      }
      q_issued += room;  // end of this CTA's stream: the last chunk stays partly empty
      mbar_arrive(bar);
    }
  };
  if (tid == 0) producer_fill(kCsRing);

  // per-thread constants: 4 channels = 2 pairs
  uint64_t wt[2][5], bias2[2], gam2[2];
#pragma unroll
  for (int c = 0; c < 2; ++c) {
#pragma unroll
    for (int j = 0; j < 5; ++j) wt[c][j] = f2_pack(__ldg(p.dw_w + (c0 + 2 * c) * 5 + j), __ldg(p.dw_w + (c0 + 2 * c + 1) * 5 + j));
    bias2[c] = f2_pack(__ldg(p.dw_b + c0 + 2 * c), __ldg(p.dw_b + c0 + 2 * c + 1));
    gam2[c] = f2_pack(__ldg(p.cln_w + c0 + 2 * c), __ldg(p.cln_w + c0 + 2 * c + 1));
  }
  const uint64_t half2 = f2_pack(0.5f, 0.5f);

  uint32_t q = 0;  // rows consumed so far by this CTA (ring sequence number)
  const uint32_t bar0 = smem_u32(s_bar), row0 = smem_u32(s_ring) + tid * 8;
  for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
    const CsRun run = cs_run(p, unit);
    uint64_t win[5][2];
#pragma unroll
    for (int j = 0; j < 5; ++j) win[j][0] = win[j][1] = 0ull;

    auto chunk_wait = [&](uint32_t chunk) { cs_wait(bar0 + (chunk % (kCsRing / kCsChunk)) * 8, (chunk / (kCsRing / kCsChunk)) & 1); };
    // one input row: token tr (zero outside the sequence) -> window slot 4. checked = false: the row exists and its chunk
    // has already been waited for (full groups wait for their 16 rows up front, which keeps their unrolled body branch-free)
    auto pull_row = [&](int tr, auto checked) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        win[j][0] = win[j + 1][0];
        win[j][1] = win[j + 1][1];
      }
      if (!decltype(checked)::value || (tr >= run.t_lo && tr < run.t_hi)) {
        if (decltype(checked)::value && (q & (kCsChunk - 1)) == 0) chunk_wait(q / kCsChunk);
        uint2 v;
        asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(row0 + (q % kCsRing) * kCsRowBytes));
        win[4][0] = f2_from_bf16x2(v.x);
        win[4][1] = f2_from_bf16x2(v.y);
        ++q;
      } else {
        win[4][0] = win[4][1] = 0ull;
      }
    };
    // window prologue: tokens t_begin-2 .. t_begin+1
#pragma unroll
    for (int r = 0; r < 4; ++r) pull_row(run.t_begin - 2 + r, std::true_type{});

    // one statistics group of up to 16 tokens; full = all 16 tokens exist and none of their window rows is padding, so the
    // unrolled body carries no per-token branches (the window then rotates by register renaming)
    auto group = [&](int tg, auto full) {
      constexpr bool kFull = decltype(full)::value;
      uint32_t u[kCsGroup][2];
      if (kFull) {  // rows q .. q+15 were requested a group ago: in steady state these waits fall through
        for (uint32_t c = q / kCsChunk; c <= (q + kCsGroup - 1) / kCsChunk; ++c) chunk_wait(c);
      }
      // ---- phase 1: conv + Swish; park (sum, sumsq) of this thread's 4 channels per token
#pragma unroll
      for (int o = 0; o < kCsGroup; ++o) {
        const int t = tg + o;
        if (kFull || t < run.t_end) {
          pull_row(t + 2, std::integral_constant<bool, !kFull>{});
          uint64_t s2 = 0ull, q2 = 0ull;
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            uint64_t acc = bias2[c];
#pragma unroll
            for (int j = 0; j < 5; ++j) acc = f2_fma(wt[c][j], win[j][c], acc);
            const uint32_t y2 = f2_to_bf16x2(acc);                       // depthwise conv output is bf16
            const uint64_t h = f2_mul(f2_from_bf16x2(y2), half2);
            float h0, h1, t0, t1;
            f2_unpack(h, h0, h1);
            asm("tanh.approx.f32 %0, %1;" : "=f"(t0) : "f"(h0));
            asm("tanh.approx.f32 %0, %1;" : "=f"(t1) : "f"(h1));
            const uint32_t sg = f2_to_bf16x2(f2_fma(f2_pack(t0, t1), half2, half2));  // bf16(sigmoid(y))
            const uint32_t uu = bf16x2_mul(y2, sg);                                    // Swish output, bf16
            u[o][c] = uu;
            const uint64_t uf = f2_from_bf16x2(uu);
            s2 = c == 0 ? uf : f2_add(s2, uf);
            q2 = c == 0 ? f2_mul(uf, uf) : f2_fma(uf, uf, q2);
          }
          float sa, sb, qa, qb;
          f2_unpack(s2, sa, sb);
          f2_unpack(q2, qa, qb);
          s_part[o * kCsThreads + tid] = make_float2(sa + sb, qa + qb);
        } else {
          u[o][0] = u[o][1] = 0u;
        }
      }
      __syncthreads();
      // the rows consumed so far are free: top the ring up while the statistics and the normalisation run
      if (tid == 0) producer_fill((q & ~static_cast<uint32_t>(kCsChunk - 1)) + kCsRing);

      // ---- phase 2: one warp per token reduces the 512 partial pairs (ChanLayerNorm: biased variance, bf16 mean / var / rstd)
      if (kFull || tg + warp < run.t_end) {
        const float2* row = s_part + warp * kCsThreads;
        float s = 0.f, qq = 0.f;
#pragma unroll
        for (int i = 0; i < kCsThreads / 32; ++i) {
          const float2 v = row[i * 32 + lane];
          s += v.x;
          qq += v.y;
        }
        s = warp_sum(s);
        qq = warp_sum(qq);
        if (lane == 0) {
          const float mean = s * (1.0f / kConvC);
          const float var = fmaxf(qq * (1.0f / kConvC) - mean * mean, 0.f);
          const float rs = rsqrtf(fmaxf(bf16_round(var), 1e-4f));
          s_stat[warp] = make_uint2(pack_bf16x2(mean, mean), pack_bf16x2(rs, rs));
        }
      }
      __syncthreads();

      // ---- phase 3: normalise from registers and store
      __nv_bfloat16* orow = p.out + (run.row0 + tg) * kConvC + c0;
#pragma unroll
      for (int o = 0; o < kCsGroup; ++o) {
        if (kFull || tg + o < run.t_end) {
          const uint2 st = s_stat[o];
          uint32_t w[2];
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            const uint32_t n = bf16x2_mul(bf16x2_sub(u[o][c], st.x), st.y);
            w[c] = f2_to_bf16x2(f2_mul(f2_from_bf16x2(n), gam2[c]));
          }
          *reinterpret_cast<uint2*>(orow + static_cast<long long>(o) * kConvC) = make_uint2(w[0], w[1]);
        }
      }
    };

    for (int tg = run.t_begin; tg < run.t_end; tg += kCsGroup) {
      if (tg + kCsGroup <= run.t_end && tg + kCsGroup + 2 <= run.t_hi)
        group(tg, std::true_type{});
      else
        group(tg, std::false_type{});
    }
    // rows t_end+2.. never requested: the run's last window rows were pulled by the loop above (t + 2 <= t_end + 1)
  }
#ifdef EDM_KTRACE
  __syncthreads();
  if (tid == 0) KTRACE_END(3);
#endif
}

}  // namespace edm
