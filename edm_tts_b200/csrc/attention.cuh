// Non-causal multi-head attention for the conformer block (reference: edm_tts/models/conformer/attend.py:63-115 via
// conformer.py:128-146): softmax(q k^T / sqrt(64)) v, H heads of 64, no mask, one sequence = one batch element.
// Sequences are placed by a SeqLayout (packed back to back, possibly of different lengths). qkv is read through a 2-D tensor map
// over all rows: a key tile starts at the sequence's first row + 128 j, and the columns at or past the sequence's end (rows of the
// next sequence, or TMA's zero fill after the last row) get -inf scores, so they add exact zeros to every sum; query rows past the
// end are computed and not stored. Each query row is one lane with its own running max and rescale factor, so a row's result
// does not depend on its neighbours.
//
// Persistent CTAs (one per SM) loop over work items; one item = 256 query rows (two 128-row tiles, "ping" and "pong")
// of one (sequence, head). A packed layout lists its (sequence, query pair) items longest sequence first (built at bind), so the
// static round-robin hands out the long items first. The TMA producer runs one item ahead (Q is double-buffered, the K/V ring is continuous across
// items), so the next item's first scores are issued while the current item's last tile is in its exp2 phase. Both contractions run on
// tcgen05 with fp32 accumulators in TMEM (all 512 columns: S0 | S1 | O0 | O1):
//   S_w = Q_w K^T : A = Q_w [128 x 64] K-major smem,  B = K tile [128 x 64] K-major smem        -> 128 TMEM columns
//   O_w += P_w V  : A = P_w [128 x 128] K-major smem (bf16, written by the softmax warps),
//                   B = V tile [128 kv x 64]: TMA delivers it with the head dim contiguous = MN-major B  -> 64 columns
//   warps 0..3 / 4..7 : softmax warpgroup of tile 0 / 1, one query row per thread (TMEM lane == row, no shuffles).
//                       The whole S row (128 fp32) is pulled into registers once; P goes to 128B-swizzled smem.
//                       O stays in TMEM and is rescaled there only when the running max moves by more than 2^8
//                       (warp-uniform decision), so after the first tile the rescale path is practically never taken.
//   warp 8            : TMA producer (both Q tiles once, then a 3-deep K/V ring shared by the two query tiles)
//   warp 9            : TMEM allocator + MMA issuer (whole warp in warp-uniform code, one elected lane issues). S_w(j+1) is issued as soon as the warpgroup has pulled
//                       S_w(j) into registers (s_free), i.e. before P_w(j) V(j), so the next scores are ready when the
//                       exp2 phase of the current tile ends.
//                       (One issuer per query tile, warp 10 taking tile 1, was measured slower: 0.171 vs 0.154 ms at B=64,
//                       N=500. The single in-order issuer keeps the two warpgroups half a tile apart, so one is in its MUFU
//                       phase while the other's MMAs run.)
//   Tried and dropped (round 2, tools/gpu_attn_variants.sh): taking 25 / 50 % of the exp2 from the FMA pipe (Cody-Waite split + degree-3
//   minimax polynomial in packed f32x2, exponent merged with one integer multiply-add), as FlashAttention-4 does. 122.8 us -> 124.7 /
//   137.0 us at B=64, N=500: with the ping-pong hand-over only one warp per SM sub-partition is in its exp2 phase at a time, and that
//   phase is bound by its own instruction stream (scale, exp2, sum, bf16 pack, swizzled store: ~6 issue slots per column pair), not by
//   MUFU throughput; every polynomial pair adds ~10 slots to it.
//   warps 10..11      : idle; they exist so the producer/MMA warpgroup can hand its registers to the softmax warpgroups
//                       (setmaxnreg 88 / 208): a 128-wide fp32 score row per thread does not fit in 168 registers.
#pragma once
#include "ptx.cuh"
#include "seq_layout.cuh"

namespace edm {

struct AttnParams {
  SeqLayout lay;          // where the sequences are
  int H;                  // heads (head dim fixed at 64)
  const int* pairs;       // packed layout: [n_pairs] (sequence << 16 | 256-row query pair), longest sequence first; nullptr: uniform
  int n_items;            // work items = query pairs x heads
  int q_col0, k_col0, v_col0;  // first column of q / k / v inside the fused projection buffer
  __nv_bfloat16* out;     // [B*N, H*64]
  long long ldo;
  float scale_log2e;      // softmax scale * log2(e)
  // MN-major V descriptor knobs (bytes); defaults 1024 / 1024 / 2048, exposed so a bring-up run can sweep them.
  uint32_t v_lbo, v_sbo, v_kstep;
  int reverse;            // 1: work items are walked from the last to the first
#ifdef EDM_ATTN_TRACE
  unsigned long long* trace;  // bring-up build only (tools/gpu_attn_trace.sh): clock64 stamps of CTA 0, [kv iteration][32 events]
#endif
};
#ifdef EDM_ATTN_TRACE
#define ATTN_TRACE(g, k) do { if (blockIdx.x == 0 && p.trace != nullptr && (g) < 96) p.trace[(g) * 32 + (k)] = clock64(); } while (0)
#else
#define ATTN_TRACE(g, k) do { } while (0)
#endif

constexpr int kAttnThreads = 384;
constexpr int kAttnKvStages = 3;
constexpr uint32_t kAttnTile = 128 * 64 * 2;  // 16 KB: one [128 x 64] bf16 tile
constexpr uint32_t kAttnSmemBytes = 4 * kAttnTile /*Q0,Q1 x 2 slots*/ + 2 * kAttnKvStages * kAttnTile /*K,V ring*/ + 4 * kAttnTile /*P0,P1*/ + 256;
constexpr float kAttnRescaleThreshold = 8.0f;  // log2 units

__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0],"
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16,"
      " %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};\n" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
      "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]),
      "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]),
      "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// work item -> (sequence, query-tile pair, head)
__device__ __forceinline__ void attn_item(const AttnParams& p, int it, int& b, int& qt2, int& h) {
  if (p.pairs != nullptr) {
    const int pr = __ldg(p.pairs + it / p.H);
    b = pr >> 16;
    qt2 = pr & 0xffff;
    h = it % p.H;
  } else {
    const int n_q2 = (p.lay.N + 255) / 256;
    qt2 = it % n_q2;
    h = (it / n_q2) % p.H;
    b = it / (n_q2 * p.H);
  }
}

__global__ void __launch_bounds__(kAttnThreads, 1)
attention_fwd_kernel(const __grid_constant__ CUtensorMap tma_qkv, const AttnParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sQ = smem;                                   // 2 slots x 2 tiles
  uint8_t* sK = sQ + 4 * kAttnTile;                     // kAttnKvStages tiles
  uint8_t* sV = sK + kAttnKvStages * kAttnTile;         // kAttnKvStages tiles
  uint8_t* sP = sV + kAttnKvStages * kAttnTile;         // 2 x (2 half tiles)
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP + 4 * kAttnTile);
  uint64_t* q_full = bars + 0;                          // [2]
  uint64_t* q_empty = bars + 2;                         // [2]
  uint64_t* kv_full = bars + 4;                         // [3]
  uint64_t* kv_empty = kv_full + kAttnKvStages;         // [3]
  uint64_t* s_full = kv_empty + kAttnKvStages;          // [2]
  uint64_t* p_full = s_full + 2;                        // [2]
  uint64_t* o_full = p_full + 2;                        // [2]
  uint64_t* s_free = o_full + 2;                        // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(s_free + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int total_items = p.n_items;
  // persistent: this CTA handles work items blockIdx.x, blockIdx.x + gridDim.x, ... ; item -> (query-tile pair, head, sequence).
  // The kv iterations of this CTA are numbered g = 0, 1, ... across its items (n_kv of them per item, set by the item's sequence);
  // ring stages and barrier phases follow g.
  const int my_items = (total_items - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);
  auto item_of = [&](int i) {
    return p.reverse ? total_items - 1 - (static_cast<int>(blockIdx.x) + i * static_cast<int>(gridDim.x)) : static_cast<int>(blockIdx.x) + i * static_cast<int>(gridDim.x);
  };
  auto item_nkv = [&](int i) {
    int b, qt2, h;
    attn_item(p, item_of(i), b, qt2, h);
    return (p.lay.n_len(b) + 127) >> 7;
  };

  if (threadIdx.x == 0) {
    if ((smem_u32(smem) & 1023u) != 0) {
      printf("edm: attention smem base not 1024-aligned\n");
      __trap();
    }
    tma_prefetch_desc(&tma_qkv);
    for (int s = 0; s < 2; ++s) {
      mbar_init(&q_full[s], 1);
      mbar_init(&q_empty[s], 1);
    }
    for (int s = 0; s < kAttnKvStages; ++s) {
      mbar_init(&kv_full[s], 1);
      mbar_init(&kv_empty[s], 1);
    }
    for (int w = 0; w < 2; ++w) {
      mbar_init(&s_full[w], 1);
      mbar_init(&p_full[w], 128);
      mbar_init(&o_full[w], 1);
      mbar_init(&s_free[w], 128);
    }
    fence_mbar_init();
  }
  if (warp == 9) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  KTRACE_ENTRY(kt_entry);
  pdl_sync();
#ifdef EDM_KTRACE
  if (threadIdx.x == 0) { KTRACE_PUT(1, kt_entry); KTRACE_PUT(2, ktrace_now()); }
#endif

  if (warp >= 8) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 88;");
    if (warp == 8) {
      if (lane == 0) {
        int g = 0;
        for (int i = 0; i < my_items; ++i) {
          int b, qt2, h;
          attn_item(p, item_of(i), b, qt2, h);
          const int row0 = p.lay.n_start(b), n_kv = (p.lay.n_len(b) + 127) >> 7;
          const int qs = i & 1;
          mbar_wait(&q_empty[qs], ((i >> 1) & 1) ^ 1);
          mbar_arrive_expect_tx(&q_full[qs], 2 * kAttnTile);
          tma_load_2d(&tma_qkv, &q_full[qs], sQ + qs * 2 * kAttnTile, p.q_col0 + h * 64, row0 + qt2 * 256);
          tma_load_2d(&tma_qkv, &q_full[qs], sQ + qs * 2 * kAttnTile + kAttnTile, p.q_col0 + h * 64, row0 + qt2 * 256 + 128);
          for (int j = 0; j < n_kv; ++j, ++g) {
            const int s = g % kAttnKvStages;
            mbar_wait(&kv_empty[s], ((g / kAttnKvStages) & 1) ^ 1);
            mbar_arrive_expect_tx(&kv_full[s], 2 * kAttnTile);
            tma_load_2d(&tma_qkv, &kv_full[s], sK + s * kAttnTile, p.k_col0 + h * 64, row0 + j * 128);
            tma_load_2d(&tma_qkv, &kv_full[s], sV + s * kAttnTile, p.v_col0 + h * 64, row0 + j * 128);
          }
        }
      }
    } else if (warp == 9) {
      int total_g = 0;
      for (int i = 0; i < my_items; ++i) total_g += item_nkv(i);
      if (total_g > 0) {  // whole warp, warp-uniform control flow; one elected lane issues (umma_*_warp)
        constexpr uint32_t idesc_s = umma_idesc_bf16(128, 128, 0, 0);
        constexpr uint32_t idesc_o = umma_idesc_bf16(128, 64, 0, 1);  // B (= V) is MN-major
        // scores of kv iteration g for tile w (both tiles are issued back to back by the callers)
        // scores of kv iteration g (of item i) for tile w
        auto issue_s = [&](int w, int g, int i) {
          const uint64_t qdesc = umma_desc_sw128(smem_u32(sQ + (i & 1) * 2 * kAttnTile + w * kAttnTile), 16, 1024);
          const uint64_t kdesc = umma_desc_sw128(smem_u32(sK + (g % kAttnKvStages) * kAttnTile), 16, 1024);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_ss_warp(tmem_base + w * 128, qdesc + 2 * k, kdesc + 2 * k, idesc_s, k != 0);
          umma_commit_warp(&s_full[w]);
        };
        // descriptor fields that do not change (layout, LBO / SBO) are built once; per tile only the 14-bit start address moves
        const uint64_t vdesc_fixed = umma_desc_sw128(0, p.v_lbo, p.v_sbo);
        const uint32_t v_kstep16 = p.v_kstep >> 4;
        auto issue_pv = [&](int w, int g, bool first) {  // first: the item's first kv tile overwrites O
          const uint32_t p_addr = smem_u32(sP + w * 2 * kAttnTile);
          const uint64_t pdesc0 = umma_desc_sw128(p_addr, 16, 1024);
          const uint64_t pdesc1 = pdesc0 + (kAttnTile >> 4);
          const uint64_t vdesc = vdesc_fixed + (smem_u32(sV + (g % kAttnKvStages) * kAttnTile) >> 4);
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            const uint64_t adesc = (k < 4 ? pdesc0 : pdesc1) + 2 * (k & 3);
            umma_ss_warp(tmem_base + 256 + w * 64, adesc, vdesc + k * v_kstep16, idesc_o, (!first || k != 0) ? 1u : 0u);
          }
          umma_commit_warp(&o_full[w]);
        };
        mbar_wait_spin(&q_full[0], 0);
        mbar_wait_spin(&kv_full[0], 0);
        tc_fence_after();
        // (item, kv tile, tiles of the item) of iteration g (P V) and of iteration g + 1 (scores)
        int j = 0, n_kv = item_nkv(0), i1 = 0, j1 = 0, n_kv1 = n_kv;
        issue_s(0, 0, 0);
        issue_s(1, 0, 0);
        if (n_kv == 1) umma_commit_warp(&q_empty[0]);
        for (int g = 0; g < total_g; ++g) {
          if (g + 1 < total_g) {
            // next scores as soon as each warpgroup has drained S_w(g) into registers
            const int g1 = g + 1;
            if (++j1 == n_kv1) {
              j1 = 0;
              n_kv1 = item_nkv(++i1);
            }
            if (j1 == 0) mbar_wait_spin(&q_full[i1 & 1], (i1 >> 1) & 1);
            mbar_wait_spin(&kv_full[g1 % kAttnKvStages], (g1 / kAttnKvStages) & 1);
            mbar_wait_spin(&s_free[0], g & 1);
            tc_fence_after();
            ATTN_TRACE(g1, 18);
            issue_s(0, g1, i1);
            ATTN_TRACE(g1, 8);
            mbar_wait_spin(&s_free[1], g & 1);
            tc_fence_after();
            issue_s(1, g1, i1);
            ATTN_TRACE(g1, 9);
            if (j1 == n_kv1 - 1) umma_commit_warp(&q_empty[i1 & 1]);  // Q slot reusable once the item's last scores are done
          }
          // P_w(g) is in smem (and O_w rescaled if needed)
          mbar_wait_spin(&p_full[0], g & 1);
          tc_fence_after();
          ATTN_TRACE(g, 16);
          issue_pv(0, g, j == 0);
          ATTN_TRACE(g, 10);
          mbar_wait_spin(&p_full[1], g & 1);
          tc_fence_after();
          ATTN_TRACE(g, 17);
          issue_pv(1, g, j == 0);
          ATTN_TRACE(g, 11);
          umma_commit_warp(&kv_empty[g % kAttnKvStages]);  // K / V stage free once everything issued so far has completed
          if (++j == n_kv) {  // iteration g + 1 opened the next item (the scores cursor is already there)
            j = 0;
            n_kv = n_kv1;
          }
        }
      }
    }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 208;");
    // ---- softmax warpgroups: w = 0 (warps 0..3) / 1 (warps 4..7); thread <-> query row
    const int w = warp >> 2;
    const int row_in_tile = (warp & 3) * 32 + lane;
    const uint32_t lane_off = static_cast<uint32_t>((warp & 3) * 32) << 16;
    const uint32_t tmem_S = tmem_base + w * 128 + lane_off;
    const uint32_t tmem_O = tmem_base + 256 + w * 64 + lane_off;
    const float sl2 = p.scale_log2e;
    uint8_t* p_row = sP + w * 2 * kAttnTile + row_in_tile * 128;
    const int sw = row_in_tile & 7;

    if (w == 1) asm volatile("bar.arrive 2, 256;" ::: "memory");  // warpgroup 0 takes the first softmax phase
    int g0 = 0;  // first kv iteration of the current item
    for (int i = 0; i < my_items; ++i) {
      int b, qt2, h;
      attn_item(p, item_of(i), b, qt2, h);
      const int row_b = p.lay.n_start(b), seq_n = p.lay.n_len(b), n_kv = (seq_n + 127) >> 7;
      float m_ref = -INFINITY;  // reference max in scaled log2 units
      float l_run = 0.f;

      for (int j = 0; j < n_kv; ++j) {
        const int g = g0 + j;
        mbar_wait(&s_full[w], g & 1);
        tc_fence_after();
        if ((warp & 3) == 0 && lane == 0) ATTN_TRACE(g, 4 * w + 0);
        uint32_t s0[32], s1[32], s2[32], s3[32];
        tmem_ld_32x32(tmem_S, s0);
        tmem_ld_32x32(tmem_S + 32, s1);
        tmem_ld_32x32(tmem_S + 64, s2);
        tmem_ld_32x32(tmem_S + 96, s3);
        tmem_ld_wait_dep(s0);
        tmem_ld_wait_dep(s1);
        tmem_ld_wait_dep(s2);
        tmem_ld_wait_dep(s3);
        tc_fence_before();
        mbar_arrive(&s_free[w]);  // S_w may be overwritten by the next Q K^T
        if ((warp & 3) == 0 && lane == 0) ATTN_TRACE(g, 4 * w + 1);
        const int kv_valid = seq_n - j * 128;
        if (kv_valid < 128) {  // only the last tile of a ragged sequence: key columns past its end -> -inf
#pragma unroll
          for (int c = 0; c < 32; ++c) {
            if (c >= kv_valid) s0[c] = 0xff800000u;
            if (32 + c >= kv_valid) s1[c] = 0xff800000u;
            if (64 + c >= kv_valid) s2[c] = 0xff800000u;
            if (96 + c >= kv_valid) s3[c] = 0xff800000u;
          }
        }
        float mx0 = -INFINITY, mx1 = -INFINITY, mx2 = -INFINITY, mx3 = -INFINITY;
#pragma unroll
        for (int c = 0; c < 32; ++c) {
          mx0 = fmaxf(mx0, __uint_as_float(s0[c]));
          mx1 = fmaxf(mx1, __uint_as_float(s1[c]));
          mx2 = fmaxf(mx2, __uint_as_float(s2[c]));
          mx3 = fmaxf(mx3, __uint_as_float(s3[c]));
        }
        const float m_new = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3)) * sl2;
        // lazy rescale: keep the old reference unless the max moved by more than 2^8 (p stays <= 256, exact enough in fp32/bf16)
        const bool need = m_new - m_ref > kAttnRescaleThreshold;  // true at j == 0 (m_ref = -inf)
        float alpha = 1.0f;
        if (need) {
          alpha = ex2_approx(m_ref - m_new);  // 0 at j == 0
          m_ref = m_new;
        }
        if (j > 0) {
          // P_w V(g-1) must have completed before P_w is overwritten or O_w rescaled (it normally has, long ago)
          mbar_wait(&o_full[w], (g - 1) & 1);
          tc_fence_after();
        }
        if ((warp & 3) == 0 && lane == 0) ATTN_TRACE(g, 4 * w + 2);
        if (j > 0 && __any_sync(0xffffffffu, need)) {
          // O_w *= alpha in TMEM; PV(g) is not issued before our p_full arrive
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            uint32_t o[32];
            tmem_ld_32x32(tmem_O + c * 32, o);
            tmem_ld_wait_dep(o);
#pragma unroll
            for (int e = 0; e < 32; ++e) o[e] = __float_as_uint(__uint_as_float(o[e]) * alpha);
            tmem_st_32x32(tmem_O + c * 32, o);
          }
          tmem_st_wait();
        }
        l_run *= alpha;
        // packed f32x2 arithmetic around the exp2: the scale / subtract and the row sums take one issue slot per column pair
        // (same roundings as the scalar fma / add: the two halves are independent)
        uint64_t ls2 = f2_pack(0.f, 0.f);
        const uint64_t sl2_2 = f2_pack(sl2, sl2), nm2 = f2_pack(-m_ref, -m_ref);
        auto emit = [&](uint32_t (&s)[32], int c) {
          uint32_t wv[16];
#pragma unroll
          for (int e = 0; e < 16; ++e) {
            float x0, x1;
            f2_unpack(f2_fma(f2_pack(__uint_as_float(s[2 * e]), __uint_as_float(s[2 * e + 1])), sl2_2, nm2), x0, x1);
            const float p0 = ex2_approx(x0), p1 = ex2_approx(x1);
            ls2 = f2_add(ls2, f2_pack(p0, p1));
            wv[e] = pack_bf16x2(p0, p1);
          }
          // 32 kv columns = 64 B = four 16 B chunks of this row; 128B swizzle: chunk index ^= (row & 7)
          uint8_t* half = p_row + (c >> 1) * kAttnTile;
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int chunk = ((c & 1) * 4 + q) ^ sw;
            *reinterpret_cast<uint4*>(half + chunk * 16) = make_uint4(wv[4 * q], wv[4 * q + 1], wv[4 * q + 2], wv[4 * q + 3]);
          }
        };
        // Ping-pong the softmax phases of the two warpgroups (named barriers 2 + w, 256 threads: 128 waiting + 128 arriving): the
        // phase is MUFU-bound (128 ex2 per thread), so two warpgroups inside it at once just take twice as long, while strict
        // alternation lets one warpgroup's TMEM drain / row max / barrier waits run under the other's exp2 phase. Left alone the
        // two drift into lock-step (measured: 3.6 k cycles per kv iteration, 2.5 k of them in a contended exp2 phase; 3.2 k
        // with the hand-over). Narrower critical sections (ex2 only, or ex2 + sums) were measured slower.
        if (w == 0) asm volatile("bar.sync 2, 256;" ::: "memory"); else asm volatile("bar.sync 3, 256;" ::: "memory");
        emit(s0, 0);
        emit(s1, 1);
        emit(s2, 2);
        emit(s3, 3);
        if (w == 0) asm volatile("bar.arrive 3, 256;" ::: "memory"); else asm volatile("bar.arrive 2, 256;" ::: "memory");
        float ls0, ls1;
        f2_unpack(ls2, ls0, ls1);
        l_run += ls0 + ls1;
        tc_fence_before();
        fence_proxy_async_smem();
        mbar_arrive(&p_full[w]);
        if ((warp & 3) == 0 && lane == 0) ATTN_TRACE(g, 4 * w + 3);
        if ((warp & 3) == 3 && lane == 0) ATTN_TRACE(g, 22 + w);
      }
      // item epilogue: O_w / l
      const int g_last = g0 + n_kv - 1;
      g0 += n_kv;
      mbar_wait(&o_full[w], g_last & 1);
      tc_fence_after();
      if ((warp & 3) == 0 && lane == 0) ATTN_TRACE(g_last, 12 + 2 * w);
      const float inv_l = 1.0f / l_run;
      uint32_t o0[32], o1[32];
      tmem_ld_32x32(tmem_O, o0);
      tmem_ld_32x32(tmem_O + 32, o1);
      tmem_ld_wait_dep(o0);
      tmem_ld_wait_dep(o1);
      if ((warp & 3) == 0 && lane == 0) ATTN_TRACE(g_last, 20 + w);
      // Each thread holds one 128 B output row. Storing it directly costs 32 L1 wavefronts per STG (32 rows 2 KB apart per warp
      // instruction; measured 1.9 k cycles per item); instead the warp parks its 32 rows in its own slice of the (now idle) P_w
      // buffer and writes them back four full rows per instruction. Only this warp touches these smem rows: __syncwarp suffices.
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        *reinterpret_cast<uint4*>(p_row + ((e ^ sw) * 16)) =
            make_uint4(pack_bf16x2(__uint_as_float(o0[8 * e + 0]) * inv_l, __uint_as_float(o0[8 * e + 1]) * inv_l),
                       pack_bf16x2(__uint_as_float(o0[8 * e + 2]) * inv_l, __uint_as_float(o0[8 * e + 3]) * inv_l),
                       pack_bf16x2(__uint_as_float(o0[8 * e + 4]) * inv_l, __uint_as_float(o0[8 * e + 5]) * inv_l),
                       pack_bf16x2(__uint_as_float(o0[8 * e + 6]) * inv_l, __uint_as_float(o0[8 * e + 7]) * inv_l));
        *reinterpret_cast<uint4*>(p_row + (((4 + e) ^ sw) * 16)) =
            make_uint4(pack_bf16x2(__uint_as_float(o1[8 * e + 0]) * inv_l, __uint_as_float(o1[8 * e + 1]) * inv_l),
                       pack_bf16x2(__uint_as_float(o1[8 * e + 2]) * inv_l, __uint_as_float(o1[8 * e + 3]) * inv_l),
                       pack_bf16x2(__uint_as_float(o1[8 * e + 4]) * inv_l, __uint_as_float(o1[8 * e + 5]) * inv_l),
                       pack_bf16x2(__uint_as_float(o1[8 * e + 6]) * inv_l, __uint_as_float(o1[8 * e + 7]) * inv_l));
      }
      __syncwarp();
      {
        const int r_sub = lane >> 3, ch = lane & 7;
        const int row0 = (warp & 3) * 32;                                    // this warp's first row in the tile
        const uint8_t* src = sP + w * 2 * kAttnTile;
        __nv_bfloat16* dst = p.out + static_cast<long long>(row_b) * p.ldo + h * 64 + ch * 8;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const int r = row0 + k * 4 + r_sub;
          const int qr = qt2 * 256 + w * 128 + r;
          const uint4 v = *reinterpret_cast<const uint4*>(src + r * 128 + ((ch ^ (r & 7)) * 16));
          if (qr < seq_n) *reinterpret_cast<uint4*>(dst + static_cast<long long>(qr) * p.ldo) = v;
        }
      }
      __syncwarp();   // the rows are overwritten by the next item's first P
      if ((warp & 3) == 0 && lane == 0) ATTN_TRACE(g_last, 13 + 2 * w);
    }
  }

  tc_fence_before();
  __syncthreads();
#ifdef EDM_KTRACE
  if (threadIdx.x == 0) KTRACE_END(2);
#endif
  if (warp == 9) tmem_dealloc<512>(tmem_base);
}

}  // namespace edm
