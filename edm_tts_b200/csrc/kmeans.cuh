// Nearest-centroid assignment of HuBERT features (the semantic tokenizer's k-means step) on tcgen05 kind::tf32.
// Reference: edm_tts/models/audio_tokenizer/semantic_tokenizer_hubert/semantic_tokenizer_hubert.py:74-90
//     dists = -torch.cdist(embed, cluster_centers, p=2);  clusters = dists.argmax(dim=-1)
// argmin ||x - c||^2 = argmax (x . c - ||c||^2 / 2): a [frames, D] x [D, C] distance GEMM with a fused first-arg-max, the same
// shape of work as the RVQ search (rvq_tc.cuh) with K = D instead of 8. fp32-level accuracy comes from the 3xTF32 split:
// x is split into hi / lo by four "split" warps on the staged tile, the centroids are split at pack time.
//
//   warp 0     : TMA producer. Stage = x chunk [128 frames x 32 channels] + centroid chunk [256 codes x 32 channels] hi and lo.
//   warp 1     : MMA issuer: per 8 channels  D[128 x 256] += x_lo c_hi + x_hi c_lo + x_hi c_hi  (M = 128, N = 256, K = 8).
//   warps 2-5  : split warps (x -> hi in place, lo beside it).
//   warps 6-9  : scan: thread <-> frame; after the K loop of a 256-code chunk the scores are pulled from TMEM, -||c||^2 / 2 is
//                added from shared memory and the running first maximum is updated; the next chunk's MMAs run meanwhile
//                (two 256-column accumulators).
#pragma once
#include "ptx.cuh"

namespace edm {

constexpr int kKmFrames = 128;
constexpr int kKmCodes = 256;                                   // codes per accumulator chunk (UMMA N)
constexpr int kKmKc = 32;                                       // channels per stage (one 128 B swizzle row of fp32)
constexpr int kKmStages = 2;
constexpr uint32_t kKmABytes = kKmFrames * kKmKc * 4;           // 16 KB
constexpr uint32_t kKmBBytes = kKmCodes * kKmKc * 4;            // 32 KB
constexpr uint32_t kKmStageBytes = 2 * kKmABytes + 2 * kKmBBytes;   // x_hi | x_lo | c_hi | c_lo = 96 KB
constexpr int kKmMaxCentroids = 4096;
constexpr uint32_t kKmSmemBytes = kKmStages * kKmStageBytes + kKmMaxCentroids * 4 + 1024 + 256;
constexpr int kKmThreads = 320;

struct KmeansParams {
  int n_frames, dim, n_centroids;   // dim % 32 == 0, n_centroids % 256 == 0 and <= 4096
  const float* half_neg_norm;       // [n_centroids]  -||c||^2 / 2
  long long* idx_out;               // [n_frames]
  float* score_out;                 // [n_frames] best score (x.c - ||c||^2/2) or nullptr
};

__global__ void __launch_bounds__(kKmThreads, 1)
kmeans_assign_kernel(const __grid_constant__ CUtensorMap tma_x, const __grid_constant__ CUtensorMap tma_chi,
                     const __grid_constant__ CUtensorMap tma_clo, const KmeansParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  float* s_norm = reinterpret_cast<float*>(smem + kKmStages * kKmStageBytes);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(s_norm + kKmMaxCentroids);
  uint64_t* split_bar = full_bar + kKmStages;
  uint64_t* empty_bar = split_bar + kKmStages;
  uint64_t* tfull_bar = empty_bar + kKmStages;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_tiles = (p.n_frames + kKmFrames - 1) / kKmFrames;
  const int n_kc = p.dim / kKmKc, n_nc = p.n_centroids / kKmCodes;
  const int my_tiles = (num_tiles - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);
  const uint32_t steps_per_tile = static_cast<uint32_t>(n_nc) * n_kc;
  const uint32_t total_steps = static_cast<uint32_t>(my_tiles) * steps_per_tile;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_x);
    tma_prefetch_desc(&tma_chi);
    tma_prefetch_desc(&tma_clo);
    for (int s = 0; s < kKmStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&split_bar[s], 128);
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tfull_bar[b], 1);
      mbar_init(&tempty_bar[b], 128);
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc<512>(tmem_slot);
  for (int i = threadIdx.x; i < p.n_centroids; i += kKmThreads) s_norm[i] = __ldg(p.half_neg_norm + i);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      for (uint32_t it = 0; it < total_steps; ++it) {
        const int tile = blockIdx.x + (it / steps_per_tile) * gridDim.x;
        const int nc = (it % steps_per_tile) / n_kc, kc = it % n_kc;
        const uint32_t s = it % kKmStages;
        uint8_t* st = smem + s * kKmStageBytes;
        mbar_wait(&empty_bar[s], ((it / kKmStages) & 1) ^ 1);
        mbar_arrive_expect_tx(&full_bar[s], kKmABytes + 2 * kKmBBytes);
        tma_load_2d(&tma_x, &full_bar[s], st, kc * kKmKc, tile * kKmFrames);                 // rows past n_frames: zero fill
        tma_load_2d(&tma_chi, &full_bar[s], st + 2 * kKmABytes, kc * kKmKc, nc * kKmCodes);
        tma_load_2d(&tma_clo, &full_bar[s], st + 2 * kKmABytes + kKmBBytes, kc * kKmKc, nc * kKmCodes);
      }
    }
  } else if (warp == 1) {
    {  // whole warp, warp-uniform control flow; one elected lane issues (umma_*_warp, see ptx.cuh)
      constexpr uint32_t idesc = umma_idesc_tf32(kKmFrames, kKmCodes, 0, 0);
      for (uint32_t it = 0; it < total_steps; ++it) {
        const uint32_t chunk = it / n_kc;              // (tile, code chunk) counter of this CTA
        const int kc = it % n_kc;
        const uint32_t s = it % kKmStages, buf = chunk & 1;
        if (kc == 0) {
          mbar_wait(&tempty_bar[buf], ((chunk >> 1) & 1) ^ 1);
          tc_fence_after();
        }
        mbar_wait(&full_bar[s], (it / kKmStages) & 1);
        mbar_wait(&split_bar[s], (it / kKmStages) & 1);
        tc_fence_after();
        const uint32_t st = smem_u32(smem + s * kKmStageBytes);
        const uint64_t a_hi = umma_desc_sw128(st, 16, 1024), a_lo = umma_desc_sw128(st + kKmABytes, 16, 1024);
        const uint64_t b_hi = umma_desc_sw128(st + 2 * kKmABytes, 16, 1024), b_lo = umma_desc_sw128(st + 2 * kKmABytes + kKmBBytes, 16, 1024);
        const uint32_t d_tmem = tmem_base + buf * kKmCodes;
#pragma unroll
        for (int k = 0; k < kKmKc / 8; ++k) {
          umma_ss_tf32_warp(d_tmem, a_lo + 2 * k, b_hi + 2 * k, idesc, (kc | k) != 0 ? 1u : 0u);
          umma_ss_tf32_warp(d_tmem, a_hi + 2 * k, b_lo + 2 * k, idesc, 1u);
          umma_ss_tf32_warp(d_tmem, a_hi + 2 * k, b_hi + 2 * k, idesc, 1u);
        }
        umma_commit_warp(&empty_bar[s]);
        if (kc == n_kc - 1) umma_commit_warp(&tfull_bar[buf]);
      }
    }
  } else if (warp < 6) {
    const int st_tid = threadIdx.x - 64;
    for (uint32_t it = 0; it < total_steps; ++it) {
      const uint32_t s = it % kKmStages;
      mbar_wait(&full_bar[s], (it / kKmStages) & 1);
      const uint32_t xh = smem_u32(smem + s * kKmStageBytes) + st_tid * 16;
#pragma unroll
      for (int i = 0; i < static_cast<int>(kKmABytes) / (128 * 16); ++i) {
        const float4 v = lds128(xh + i * 2048);
        float4 h, l;
        h.x = tf32_rna(v.x); h.y = tf32_rna(v.y); h.z = tf32_rna(v.z); h.w = tf32_rna(v.w);
        l.x = tf32_rna(v.x - h.x); l.y = tf32_rna(v.y - h.y); l.z = tf32_rna(v.z - h.z); l.w = tf32_rna(v.w - h.w);
        sts128(xh + i * 2048, h);
        sts128(xh + kKmABytes + i * 2048, l);
      }
      fence_proxy_async_smem();
      mbar_arrive(&split_bar[s]);
    }
  } else {
    const int quad = warp & 3;
    const int f = quad * 32 + lane;
    uint32_t chunk = 0;
    for (int tl = 0; tl < my_tiles; ++tl) {
      const int tile = blockIdx.x + tl * gridDim.x;
      const long long frame = static_cast<long long>(tile) * kKmFrames + f;
      float best = -INFINITY;
      int bidx = 0;
      for (int nc = 0; nc < n_nc; ++nc, ++chunk) {
        const uint32_t buf = chunk & 1;
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + buf * kKmCodes;
        mbar_wait(&tfull_bar[buf], (chunk >> 1) & 1);
        tc_fence_after();
#pragma unroll 1
        for (int c = 0; c < kKmCodes / 32; ++c) {
          uint32_t r[32];
          tmem_ld_32x32(taddr + c * 32, r);
          tmem_ld_wait_dep(r);
          if (c == kKmCodes / 32 - 1) {
            tc_fence_before();
            mbar_arrive(&tempty_bar[buf]);
          }
          const int code0 = nc * kKmCodes + c * 32;
          const uint32_t nb = smem_u32(s_norm + code0);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float4 hn = lds128(nb + 16 * i);   // broadcast read: every lane takes the same four constants
            const float v0 = __uint_as_float(r[4 * i]) + hn.x, v1 = __uint_as_float(r[4 * i + 1]) + hn.y,
                        v2 = __uint_as_float(r[4 * i + 2]) + hn.z, v3 = __uint_as_float(r[4 * i + 3]) + hn.w;
            // strict '>' in increasing code order: the first maximum wins (torch argmax)
            if (v0 > best) { best = v0; bidx = code0 + 4 * i; }
            if (v1 > best) { best = v1; bidx = code0 + 4 * i + 1; }
            if (v2 > best) { best = v2; bidx = code0 + 4 * i + 2; }
            if (v3 > best) { best = v3; bidx = code0 + 4 * i + 3; }
          }
        }
      }
      if (frame < p.n_frames) {
        p.idx_out[frame] = bidx;
        if (p.score_out != nullptr) p.score_out[frame] = best;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc<512>(tmem_base);
}

// ---------------------------------------------------------------------------------------------- centroid update (one Lloyd step)
// centroid[c] = (sum of the rows assigned to c) / count_c, accumulated in fp64 and rounded once to fp32; empty clusters are left as
// they are. The rows are read through perm, which lists them cluster by cluster (offsets[c] .. offsets[c + 1] are c's positions).
//   pass 1 (kmeans_update_partial_kernel): item = (segment j of kKmUpdRows consecutive perm positions, column slice). The item walks
//          its positions one cluster run at a time and writes one fp64 partial sum per (cluster c, segment j) to slot c + j. Along
//          perm, c + j strictly increases from one run to the next (the next non-empty cluster c' > c starts in the segment where c
//          ends or later), so slots never collide: at most n_centroids + ceil(n / kKmUpdRows) of them.
//   pass 2 (kmeans_update_finalize_kernel): item = (cluster, column slice): the cluster's partials in segment order, / count; the
//          fp64 sums themselves on request (the fit takes the objective of the assignment from them).
// Segments are fixed by kKmUpdRows and n alone, never by the grid, so every launch on every device adds the same numbers in the same
// order: the centroids are the same bits from run to run. A cluster holding most rows spreads over many pass-1 items.
constexpr int kKmUpdRows = 256;        // perm positions per pass-1 segment
constexpr int kKmUpdThreads = 128;
// Rows per unrolled group. ptxas interleaves a group's adds with its loads (2-3 rows in flight per thread). At 32 registers an SM
// holds 2048 threads, so that is ~80 KB of loads in flight per SM, about twice HBM latency x bandwidth / 148 SMs.
constexpr int kKmUpdUnroll = 8;

struct KmeansUpdateParams {
  const float* x;                      // [n, dim]
  const long long* idx;                // [n] cluster of each row
  const long long* perm;               // [n] rows cluster by cluster
  const long long* offsets;            // [n_centroids + 1] first perm position of each cluster, offsets[n_centroids] = n
  double* partials;                    // [n_centroids + ceil(n / kKmUpdRows)][dim]
  float* centroids;                    // [n_centroids, dim], rewritten for non-empty clusters
  double* sums;                        // [n_centroids, dim] the fp64 sums of the clusters (0 for empty ones), or nullptr
  long long n;
  int dim, n_centroids;
};

__device__ __forceinline__ void acc4(double (&a)[4], const float4 v) {
  a[0] += v.x; a[1] += v.y; a[2] += v.z; a[3] += v.w;
}

// grid (ceil(n / kKmUpdRows), ceil(dim / 4 / blockDim.x)); thread <-> 4 consecutive columns
__global__ void __launch_bounds__(kKmUpdThreads) kmeans_update_partial_kernel(const KmeansUpdateParams p) {
  __shared__ long long s_row[kKmUpdRows];
  const long long seg = blockIdx.x;
  const long long pos0 = seg * kKmUpdRows;
  const int rows = static_cast<int>(min(static_cast<long long>(kKmUpdRows), p.n - pos0));
  for (int i = threadIdx.x; i < rows; i += blockDim.x) s_row[i] = __ldg(p.perm + pos0 + i);
  __syncthreads();
  const int d4 = p.dim / 4;
  const int q = blockIdx.y * blockDim.x + threadIdx.x;
  const bool active = q < d4;
  const float4* x4 = reinterpret_cast<const float4*>(p.x) + q;
  int i = 0;
  while (i < rows) {   // block-uniform: one cluster run of the segment per trip
    const long long c = __ldg(p.idx + s_row[i]);
    if (c < 0 || c >= p.n_centroids) break;                          // inconsistent idx / offsets: stop rather than run away
    const int end = static_cast<int>(min(static_cast<long long>(rows), __ldg(p.offsets + c + 1) - pos0));
    if (end <= i) break;
    if (active) {
      double a[4] = {0.0, 0.0, 0.0, 0.0};
      int r = i;
      for (; r + kKmUpdUnroll <= end; r += kKmUpdUnroll) {
        float4 v[kKmUpdUnroll];
#pragma unroll
        for (int u = 0; u < kKmUpdUnroll; ++u) v[u] = __ldg(x4 + s_row[r + u] * d4);
#pragma unroll
        for (int u = 0; u < kKmUpdUnroll; ++u) acc4(a, v[u]);
      }
      for (; r < end; ++r) acc4(a, __ldg(x4 + s_row[r] * d4));
      double2* dst = reinterpret_cast<double2*>(p.partials + (c + seg) * p.dim) + 2 * q;
      dst[0] = make_double2(a[0], a[1]);
      dst[1] = make_double2(a[2], a[3]);
    }
    i = end;
  }
}

// grid (n_centroids, ceil(dim / blockDim.x)); thread <-> column
__global__ void __launch_bounds__(kKmUpdThreads) kmeans_update_finalize_kernel(const KmeansUpdateParams p) {
  const int c = blockIdx.x;
  const int col = blockIdx.y * blockDim.x + threadIdx.x;
  if (col >= p.dim) return;
  const long long a = __ldg(p.offsets + c), b = __ldg(p.offsets + c + 1);
  const long long o = static_cast<long long>(c) * p.dim + col;
  double s = 0.0;
  if (b > a) {
    const long long j0 = a / kKmUpdRows, j1 = (b - 1) / kKmUpdRows;
    const double* src = p.partials + (c + j0) * p.dim + col;
#pragma unroll 4
    for (long long j = j0; j <= j1; ++j, src += p.dim) s += *src;
    p.centroids[o] = __double2float_rn(s / static_cast<double>(b - a));
  }
  if (p.sums != nullptr) p.sums[o] = s;
}

}  // namespace edm
