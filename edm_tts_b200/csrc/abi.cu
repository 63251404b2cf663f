// C ABI of libedm_s2a.so: stateless operators + the S2A decoder context. See include/edm_s2a.h for the contract.
// Host code here only validates arguments, builds TMA descriptors and enqueues kernels on the caller's stream.
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <algorithm>
#include <utility>
#include <vector>

#include "../../include/edm_s2a.h"
#include "attention.cuh"
#include "elementwise.cuh"
#include "conv_stream.cuh"
#include "dac_conv.cuh"
#include "gemm.cuh"
#include "kmeans.cuh"
#include "rvq_tc.cuh"

using namespace edm;

namespace {

thread_local char g_err[512] = "";
std::atomic<unsigned long long> g_launches{0};

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define EDM_CUDA(expr)                                                                              \
  do {                                                                                              \
    cudaError_t e__ = (expr);                                                                       \
    if (e__ != cudaSuccess) return fail(EDM_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(e__));    \
  } while (0)
#define EDM_LAUNCH_CHECK(name)                                                                       \
  do {                                                                                               \
    g_launches.fetch_add(1, std::memory_order_relaxed);                                              \
    cudaError_t e__ = cudaGetLastError();                                                            \
    if (e__ != cudaSuccess) return fail(EDM_ERR_CUDA, "launch %s: %s", name, cudaGetErrorString(e__)); \
  } while (0)

// ---------------------------------------------------------------------------------------------- per-kernel timing
// bench.py brackets every launch of a kernel class with CUDA events on the launching stream (edm_prof_enable) so the
// roofline numbers come from the timed region itself, not from a profiler run.
enum ProfKind { PK_GEMM = 0, PK_ATTN, PK_LN, PK_CONV, PK_OTHER, PK_COUNT };
struct ProfEntry {
  cudaEvent_t a, b;
  int kind;
  double work;
};
// thread-local: the launching thread owns its timing state (a context is driven by one thread at a time)
thread_local bool g_prof_on = false;
thread_local std::vector<ProfEntry> g_prof;
thread_local std::vector<cudaEvent_t> g_event_pool;

cudaEvent_t prof_event() {
  if (!g_event_pool.empty()) {
    cudaEvent_t e = g_event_pool.back();
    g_event_pool.pop_back();
    return e;
  }
  cudaEvent_t e;
  cudaEventCreate(&e);
  return e;
}
struct ProfScope {
  bool on;
  ProfEntry e;
  cudaStream_t st;
  ProfScope(int kind, double work, cudaStream_t s) : on(g_prof_on), st(s) {
    if (on) {
      e.kind = kind;
      e.work = work;
      e.a = prof_event();
      e.b = prof_event();
      cudaEventRecord(e.a, st);
    }
  }
  ~ProfScope() {
    if (on) {
      cudaEventRecord(e.b, st);
      g_prof.push_back(e);
    }
  }
};

// Everything cached about "the device" is keyed by the current device: one process may drive several GPUs (a context per device),
// and cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is a per-device setting.
constexpr int kMaxDevices = 64;
int cur_device() {
  int dev = 0;
  cudaGetDevice(&dev);
  return dev >= 0 && dev < kMaxDevices ? dev : 0;
}

int check_arch() {
  static std::atomic<int> cached[kMaxDevices];  // 0 = unknown, 1 = sm_100, 2 = something else
  const int dev = cur_device();
  int st = cached[dev].load(std::memory_order_relaxed);
  if (st == 0) {
    int major = 0, minor = 0;
    if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev) != cudaSuccess)
      return fail(EDM_ERR_CUDA, "no CUDA device");
    st = major == 10 ? 1 : 2;
    cached[dev].store(st, std::memory_order_relaxed);
    if (st == 2) return fail(EDM_ERR_ARCH, "device sm_%d%d is not sm_100: this library has no fallback path", major, minor);
  }
  return st == 1 ? 0 : fail(EDM_ERR_ARCH, "device is not sm_100: this library has no fallback path");
}

int num_sms() {
  static std::atomic<int> n[kMaxDevices];
  const int dev = cur_device();
  int v = n[dev].load(std::memory_order_relaxed);
  if (v == 0) {
    cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    n[dev].store(v, std::memory_order_relaxed);
  }
  return v;
}

// "has this call site configured its kernels on the current device yet?"
struct DeviceOnce {
  std::atomic<unsigned long long> mask{0};
  bool needed() const { return (mask.load(std::memory_order_acquire) >> cur_device() & 1ull) == 0; }
  void done() { mask.fetch_or(1ull << cur_device(), std::memory_order_release); }
};

// Bring-up switches (environment variables) exist only in a -DEDM_BRINGUP build (tools/); the product library has none.
#ifdef EDM_BRINGUP
bool env_switch(const char* name, bool dflt) {
  const char* e = getenv(name);
  return e == nullptr ? dflt : e[0] != '0';
}
int env_int(const char* name, int dflt) {
  const char* e = getenv(name);
  return e == nullptr ? dflt : atoi(e);
}
#else
constexpr bool env_switch(const char*, bool dflt) { return dflt; }
constexpr int env_int(const char*, int dflt) { return dflt; }
#endif

// ---------------------------------------------------------------------------------------------- launches
// Every kernel of the decode paths is launched with programmatic stream serialisation (PDL): its CTAs may be scheduled while the
// previous kernel of the stream is still draining, run their prologue (barrier init, TMEM allocation, descriptor prefetch, bias /
// table staging from constant weights) and then block in griddepcontrol.wait until the previous kernel has completed and flushed its
// memory. Each such kernel executes griddepcontrol.wait in every CTA before it touches anything another kernel wrote (pdl_wait() in
// ptx.cuh), so completion stays transitive along the chain; a launch after a non-PDL kernel (torch's, a memcpy) simply serialises.
// Measured on the decode (tools/gpu_ab.sh, 854 launches): a constant ~1.7 ms less per decode up to 8 000 rows (B=1 x 150 frames: 8.4 ->
// 6.6 ms, B=16 x 500: 31.9 -> 30.5 ms), neutral at 16 000 rows and 0.5-1 % *slower* at the 32 000 rows of the bench step, where the
// kernels run for 100+ us and the early-resident CTAs of the next kernel only compete with the draining one. The decoder contexts
// therefore switch it off above kPdlMaxRows rows (PdlScope); the stateless operators keep it on.
constexpr int kPdlMaxRows = 16384;
thread_local bool t_pdl_allow = true;
struct PdlScope {
  bool prev;
  explicit PdlScope(bool allow) : prev(t_pdl_allow) { t_pdl_allow = allow; }
  ~PdlScope() { t_pdl_allow = prev; }
};
bool pdl_enabled() {
  static const int mode = env_int("EDM_PDL", -1);  // bring-up switch: 0 = never, 1 = always, default = by size
  return mode < 0 ? t_pdl_allow : mode != 0;
}

template <typename... KArgs, typename... Args>
void launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);  // the error is picked up by EDM_LAUNCH_CHECK (cudaGetLastError)
}

// ---------------------------------------------------------------------------------------------- TMA descriptors
typedef CUresult (*PFN_tmapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                        const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                        CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
PFN_tmapEncodeTiled get_encode() {
  static PFN_tmapEncodeTiled fn = nullptr;
  if (fn == nullptr) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_tmapEncodeTiled>(p);
  }
  return fn;
}

// bf16 row-major [rows, cols] with row pitch ld (elements); box = 64 columns (128 B, swizzle-128B) x box_rows
int make_tmap_2d(CUtensorMap* m, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows) {
  PFN_tmapEncodeTiled enc = get_encode();
  if (enc == nullptr) return fail(EDM_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) != 0 || (ld * 2) % 16 != 0) return fail(EDM_ERR_INVALID, "TMA operand must be 16-byte aligned (ptr %p, ld %llu)", ptr, (unsigned long long)ld);
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld * 2};
  cuuint32_t box[2] = {64, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(EDM_ERR_CUDA, "cuTensorMapEncodeTiled(2d rows=%llu cols=%llu ld=%llu) failed: %d", (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)ld, (int)r);
  return 0;
}
// fp32 row-major [rows, cols] with row pitch ld (elements); box = 32 columns (128 B, swizzle-128B) x box_rows
int make_tmap_f32_2d(CUtensorMap* m, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows,
                     CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B) {
  PFN_tmapEncodeTiled enc = get_encode();
  if (enc == nullptr) return fail(EDM_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) != 0 || (ld * 4) % 16 != 0) return fail(EDM_ERR_INVALID, "TMA operand must be 16-byte aligned (ptr %p, ld %llu)", ptr, (unsigned long long)ld);
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld * 4};
  cuuint32_t box[2] = {32, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(EDM_ERR_CUDA, "cuTensorMapEncodeTiled(f32 rows=%llu cols=%llu ld=%llu) failed: %d", (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)ld, (int)r);
  return 0;
}

// ---------------------------------------------------------------------------------------------- launch helpers
// Boustrophedon traversal: consecutive launches walk their rows / tiles in opposite directions, so a kernel starts with the part
// of its input that its producer wrote last and that is still in the 126 MB L2 (the hand-offs of the decoder are 66-262 MB).
int next_direction() {
  static const bool enabled = env_switch("EDM_FLIP", true);
  thread_local int dir = 0;
  if (!enabled) return 0;
  dir ^= 1;
  return dir;
}

// Weight operand of a GEMM: the tensor map of the CTA-pair kernel (each CTA of a pair loads half of the 256-row weight tile) and the
// 64-row-box map of the small-M kernel
struct WMap {
  CUtensorMap big, small;
};
int make_wmap(WMap* m, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld) {
  if (rows % kGemmBN == 0) {
    if (int rc = make_tmap_2d(&m->big, ptr, rows, cols, ld, kGemmBN / 2)) return rc;
  } else {
    memset(&m->big, 0, sizeof(m->big));  // N is not a multiple of 256: only the small-M kernel can take this weight
  }
  return make_tmap_2d(&m->small, ptr, rows, cols, ld, kSmBN);
}
bool gemm_small_m() { static const bool v = env_switch("EDM_GEMM_SMALL", true); return v; }
bool gemm_resid_tma() { static const bool v = env_switch("EDM_RESID_TMA", true); return v; }
int resid_tma_max_k() { static const int v = env_int("EDM_RESID_TMA_MAXK", 2048); return v; }
bool gemm_out_tma() { static const bool v = env_switch("EDM_OUT_TMA", true); return v; }

template <int EPI>
int launch_gemm_t(const CUtensorMap& ma, const WMap& wm, const GemmParams& p_in, cudaStream_t st) {
  const CUtensorMap& mb = wm.big;
  GemmParams p = p_in;
  p.reverse = next_direction();
  static DeviceOnce attr_once;
  if (attr_once.needed()) {
    EDM_CUDA(cudaFuncSetAttribute(gemm_bf16_tn_pair_kernel<EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPairSmemBytes));
    EDM_CUDA(cudaFuncSetAttribute(gemm_bf16_tn_small_kernel<EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmSmemBytes));
    if (EPI == EPI_RESID_F32)
      EDM_CUDA(cudaFuncSetAttribute(gemm_bf16_tn_pair_kernel<EPI_RESID_TMA>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPairSmemBytes));
    if (EPI == EPI_SWISH_BF16)
      EDM_CUDA(cudaFuncSetAttribute(gemm_bf16_tn_pair_kernel<EPI_SWISH_TMA>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPairSmemBytes));
    if (EPI == EPI_GELU_BF16)
      EDM_CUDA(cudaFuncSetAttribute(gemm_bf16_tn_pair_kernel<EPI_GELU_TMA>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPairSmemBytes));
    if (EPI == EPI_QKV_ROPE)
      EDM_CUDA(cudaFuncSetAttribute(gemm_bf16_tn_pair_kernel<EPI_ROPE_TMA>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPairSmemBytes));
    if (EPI == EPI_F32)
      EDM_CUDA(cudaFuncSetAttribute(gemm_bf16_tn_pair_kernel<EPI_F32_TMA>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPairSmemBytes));
    attr_once.done();
  }
  ProfScope prof(PK_GEMM, 2.0 * p.M * p.N * p.K, st);
  const int sms = num_sms();
  {
    // small M: the large tiles would leave most SMs without work while a few stream the weights (see gemm.cuh, small-M variant);
    // N not a multiple of 256 (hidden sizes 384 / 512 of the text-to-semantic model): only the 64-column tiles fit
    const int pair_tiles = ((p.M + 2 * kGemmBM - 1) / (2 * kGemmBM)) * ((p.N + kGemmBN - 1) / kGemmBN);
    if (p.N % kGemmBN != 0 || (gemm_small_m() && pair_tiles * 4 <= sms)) {
      p.reverse = 0;
      const int tiles = ((p.M + kGemmBM - 1) / kGemmBM) * (p.N / kSmBN);
      launch_pdl(gemm_bf16_tn_small_kernel<EPI>, dim3(tiles < sms ? tiles : sms), dim3(kSmThreads), kSmSmemBytes, st, ma, wm.small, p);
      EDM_LAUNCH_CHECK("gemm_bf16_tn_small");
      return 0;
    }
  }
  const int tiles = ((p.M + 2 * kGemmBM - 1) / (2 * kGemmBM)) * (p.N / kGemmBN);
  const int pairs = tiles < sms / 2 ? tiles : sms / 2;
  // short-K residual GEMMs are epilogue-bound: their add leaves as TMA reduce boxes (0.113 -> 0.081 ms at K = 1024); at
  // K = 4096 the mainloop hides the register-issued reductions and the 6-stage ring is worth more (0.202 vs 0.208 ms)
  if (EPI == EPI_RESID_F32 && gemm_resid_tma() && p.K <= resid_tma_max_k() && (reinterpret_cast<uintptr_t>(p.out) & 15) == 0 && (p.ldo * 4) % 16 == 0) {
    CUtensorMap mc;
    if (int rc = make_tmap_f32_2d(&mc, p.out, p.M, p.N, p.ldo, 32, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    launch_pdl(gemm_bf16_tn_pair_kernel<EPI_RESID_TMA>, dim3(2 * pairs), dim3(kGemmThreads), kPairSmemBytes, st, ma, mb, mc, p);
  } else if (EPI == EPI_F32 && gemm_out_tma() && (reinterpret_cast<uintptr_t>(p.out) & 15) == 0 && (p.ldo * 4) % 16 == 0) {
    CUtensorMap mc;  // fp32 logits leave as 32 x 32 TMA store boxes
    if (int rc = make_tmap_f32_2d(&mc, p.out, p.M, p.N, p.ldo, 32, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    launch_pdl(gemm_bf16_tn_pair_kernel<EPI_F32_TMA>, dim3(2 * pairs), dim3(kGemmThreads), kPairSmemBytes, st, ma, mb, mc, p);
  } else if ((EPI == EPI_SWISH_BF16 || EPI == EPI_GELU_BF16 || EPI == EPI_QKV_ROPE) && gemm_out_tma() && (reinterpret_cast<uintptr_t>(p.out) & 15) == 0 &&
             (p.ldo * 2) % 16 == 0) {
    // bf16 tiles leave as TMA store boxes (whole 128-byte lines) instead of 16-byte stores from registers
    CUtensorMap mc;
    if (int rc = make_tmap_2d(&mc, p.out, p.M, p.N, p.ldo, 32)) return rc;
    if (EPI == EPI_SWISH_BF16)
      launch_pdl(gemm_bf16_tn_pair_kernel<EPI_SWISH_TMA>, dim3(2 * pairs), dim3(kGemmThreads), kPairSmemBytes, st, ma, mb, mc, p);
    else if (EPI == EPI_GELU_BF16)
      launch_pdl(gemm_bf16_tn_pair_kernel<EPI_GELU_TMA>, dim3(2 * pairs), dim3(kGemmThreads), kPairSmemBytes, st, ma, mb, mc, p);
    else
      launch_pdl(gemm_bf16_tn_pair_kernel<EPI_ROPE_TMA>, dim3(2 * pairs), dim3(kGemmThreads), kPairSmemBytes, st, ma, mb, mc, p);
  } else {
    launch_pdl(gemm_bf16_tn_pair_kernel<EPI>, dim3(2 * pairs), dim3(kGemmThreads), kPairSmemBytes, st, ma, mb, ma, p);
  }
  EDM_LAUNCH_CHECK("gemm_bf16_tn_pair");
  return 0;
}
int launch_gemm(int epi, const CUtensorMap& ma, const WMap& mb, const GemmParams& p, cudaStream_t st) {
  if (p.M <= 0 || p.N <= 0 || p.N % kSmBN != 0 || p.N > kGemmMaxN || p.K % kGemmBK != 0 || p.K <= 0) return fail(EDM_ERR_INVALID, "gemm shape M=%d N=%d K=%d unsupported (N %% 64, N <= 8192, K %% 64)", p.M, p.N, p.K);
  switch (epi) {
    case EPI_BF16: return launch_gemm_t<EPI_BF16>(ma, mb, p, st);
    case EPI_SWISH_BF16: return launch_gemm_t<EPI_SWISH_BF16>(ma, mb, p, st);
    case EPI_QKV_ROPE: return launch_gemm_t<EPI_QKV_ROPE>(ma, mb, p, st);
    case EPI_RESID_F32: return launch_gemm_t<EPI_RESID_F32>(ma, mb, p, st);
    case EPI_F32: return launch_gemm_t<EPI_F32>(ma, mb, p, st);
    case EPI_GLU_BF16: return launch_gemm_t<EPI_GLU_BF16>(ma, mb, p, st);
    case EPI_ARGMAX: return launch_gemm_t<EPI_ARGMAX>(ma, mb, p, st);
    case EPI_GELU_BF16: return launch_gemm_t<EPI_GELU_BF16>(ma, mb, p, st);
  }
  return fail(EDM_ERR_INVALID, "unknown epilogue %d", epi);
}

#ifdef EDM_ATTN_TRACE
unsigned long long* g_attn_trace = nullptr;
#endif
// qkv map: make_tmap_2d over all rows, 128-row boxes. pairs: the packed layout's (sequence << 16 | query pair) list, longest first
// (nullptr for a uniform layout); flops: the algorithmic work, for the measurement hooks.
int launch_attention(const CUtensorMap& mqkv, const SeqLayout& lay, const int* pairs, int n_pairs, double flops, int H, void* out, uint32_t lbo,
                     uint32_t sbo, uint32_t kstep, cudaStream_t st, float scale = 0.125f) {
  static DeviceOnce attr_once;
  if (attr_once.needed()) {
    EDM_CUDA(cudaFuncSetAttribute(attention_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kAttnSmemBytes));
    attr_once.done();
  }
  AttnParams p;
  p.lay = lay; p.H = H; p.pairs = pairs;
  p.n_items = (pairs != nullptr ? n_pairs : lay.n_seq * ((lay.N + 255) / 256)) * H;
  p.q_col0 = 0; p.k_col0 = H * 64; p.v_col0 = 2 * H * 64;
  p.out = static_cast<__nv_bfloat16*>(out);
  p.ldo = static_cast<long long>(H) * 64;
  p.scale_log2e = scale * 1.4426950408889634f;  // softmax scale = dim_head^-1/2 (0.125 for the 64-wide heads of the S2A model)
  p.v_lbo = lbo; p.v_sbo = sbo; p.v_kstep = kstep; p.reverse = next_direction();
#ifdef EDM_ATTN_TRACE
  p.trace = g_attn_trace;
#endif
  if (p.n_items <= 0) return 0;
  dim3 grid(p.n_items < num_sms() ? p.n_items : num_sms());
  ProfScope prof(PK_ATTN, flops, st);
  launch_pdl(attention_fwd_kernel, dim3(grid), dim3(kAttnThreads), kAttnSmemBytes, st, mqkv, p);
  EDM_LAUNCH_CHECK("attention_fwd");
  return 0;
}

int launch_ln(const LnParams& p_in, cudaStream_t st) {
  if (p_in.rows <= 0) return 0;
  LnParams p = p_in;
  p.reverse = next_direction();
  // algorithmic bytes: one read of the row + each requested output
  ProfScope prof(PK_LN, static_cast<double>(p.rows) * kD * ((p.in_is_bf16 ? 2 : 4) + (p.y_out ? 4 : 0)) +
                            (p.z_out ? static_cast<double>(p.compact ? p.lay.t_rows : p.rows) * kD * 2 : 0.0), st);
  launch_pdl(layernorm_kernel, dim3((p.rows + 7) / 8), dim3(256), 0, st, p);
  EDM_LAUNCH_CHECK("layernorm");
  return 0;
}

// Residual GEMM x += scale * bf16(A W^T + b) followed by the LayerNorm of the updated rows (every residual branch of the conformer
// block is followed by one: conformer.py:229-234 with PreNorm :102-110). splits > 1 (low-latency mode of a context, few rows): a long-K
// GEMM on few tiles is bound by what one SM's TMA pulls in (~100 GB/s: 250 ns per 24 KB k-step, tools/ktrace.py) while most SMs idle,
// so K is cut into `splits` ranges that run as separate work items writing raw partial sums to `part`, and the LayerNorm launch adds
// them up (layernorm_splitk_kernel): no extra launch, deterministic (fixed order), the bf16 rounding point of the Linear output kept.
// The fp32 summation order differs from the unsplit kernels, which is why this is an opt-in: by default a row's bits do not depend on
// the batch it is decoded in. splits <= 1 or an unsuitable shape: the two plain launches.
int gemm_splitk_min_k() { static const int v = env_int("EDM_SPLITK_MINK", 2048); return v; }  // bring-up switch
int choose_splits(int M, int K) {
  const int tiles = ((M + kGemmBM - 1) / kGemmBM) * (kD / kSmBN), num_kb = K / kGemmBK, sms = num_sms();
  if (K < gemm_splitk_min_k()) return 1;
  for (int s = 4; s >= 2; s >>= 1)
    if (tiles * s <= sms && num_kb % s == 0 && num_kb / s >= 4) return s;
  return 1;
}
int launch_gemm_resid_ln(const CUtensorMap& ma, const WMap& wm, const GemmParams& p, const LnParams& ln, float* part, int splits, cudaStream_t st) {
  const int sms = num_sms();
  const int pair_tiles = ((p.M + 2 * kGemmBM - 1) / (2 * kGemmBM)) * ((p.N + kGemmBN - 1) / kGemmBN);
  const bool small = p.N % kGemmBN != 0 || (gemm_small_m() && pair_tiles * 4 <= sms);
  if (!small || part == nullptr || splits < 2 || splits > 4 || p.K % (kGemmBK * splits) != 0 || p.N != kD || p.ldo != kD || ln.in != p.out ||
      ln.rows != p.M || p.a_k_offset != 0) {
    if (int rc = launch_gemm(EPI_RESID_F32, ma, wm, p, st)) return rc;
    return launch_ln(ln, st);
  }
  static DeviceOnce attr_once;
  if (attr_once.needed()) {
    EDM_CUDA(cudaFuncSetAttribute(gemm_bf16_tn_small_kernel<EPI_F32>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmSmemBytes));
    attr_once.done();
  }
  {
    GemmParams q = p;
    q.bias = nullptr; q.out = part; q.ldo = kD; q.scale = 1.0f; q.reverse = 0;
    q.splits = splits; q.split_stride = static_cast<long long>(p.M) * kD;
    next_direction();
    ProfScope prof(PK_GEMM, 2.0 * p.M * p.N * p.K, st);
    const int work = ((p.M + kGemmBM - 1) / kGemmBM) * (p.N / kSmBN) * splits;
    launch_pdl(gemm_bf16_tn_small_kernel<EPI_F32>, dim3(work < sms ? work : sms), dim3(kSmThreads), kSmSmemBytes, st, ma, wm.small, q);
    EDM_LAUNCH_CHECK("gemm_bf16_tn_small (split-K)");
  }
  LnParams l = ln;
  l.partials = part; l.n_partials = splits; l.partial_stride = static_cast<long long>(p.M) * kD; l.lin_bias = p.bias; l.lin_scale = p.scale;
  l.x_io = static_cast<float*>(p.out); l.reverse = 0;
  next_direction();
  ProfScope prof(PK_LN, static_cast<double>(l.rows) * kD * (4.0 * (splits + 2) + (l.y_out ? 4 : 0) + (l.z_out ? 2 : 0)), st);
  launch_pdl(layernorm_splitk_kernel, dim3((l.rows + 7) / 8), dim3(256), 0, st, l);
  EDM_LAUNCH_CHECK("layernorm_splitk");
  return 0;
}

// Run length of the streaming conv kernel: every sequence is split into runs so that the persistent CTAs are evenly loaded and few
// halo rows are re-read (run lengths are multiples of the 16-token statistics group, so only a sequence's last run has a partial
// group). lens: the n_seq sequence lengths, or nullptr when every sequence has n rows.
int conv_run_len(int n_seq, const int* lens, int n, int sms) {
  long long rows = 0;
  int max_n = n;
  if (lens != nullptr) {
    max_n = 0;
    for (int i = 0; i < n_seq; ++i) {
      rows += lens[i];
      max_n = std::max(max_n, lens[i]);
    }
  } else {
    rows = static_cast<long long>(n_seq) * n;
  }
  int best_len = (max_n + 15) / 16 * 16;
  double best = -1.0;
  for (int len = 16; len <= (max_n + 15) / 16 * 16; len += 16) {
    long long units = 0;
    if (lens != nullptr)
      for (int i = 0; i < n_seq; ++i) units += (lens[i] + len - 1) / len;
    else
      units = static_cast<long long>(n_seq) * ((n + len - 1) / len);
    const long long rounds = (units + sms - 1) / sms;
    const double eff = static_cast<double>(rows) / (static_cast<double>(rounds * sms) * len) * len / (len + 4.0);
    if (eff > best + 1e-9) {
      best = eff;
      best_len = len;
    }
  }
  return best_len;
}
// Runs of a packed layout (built once at bind: the run length and the first run of every sequence)
struct ConvRuns {
  int run_len = 0, num_units = 0;
  const int* cu_runs = nullptr;  // device [n_seq + 1]
};

// glu_input: the kernel reads [rows, 4096] and applies the GLU itself; otherwise the input is the already gated [rows, 2048]
// (the decoder's path: the GLU runs in the pointwise-conv GEMM epilogue) and the streaming kernel of conv_stream.cuh is used.
// runs: required for a packed layout on the streaming kernel.
int launch_conv(const ConvModParams& p, bool glu_input, cudaStream_t st, const ConvRuns* runs = nullptr) {
  static DeviceOnce attr_once;
  if (attr_once.needed()) {
    EDM_CUDA(cudaFuncSetAttribute(conv_module_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kConvSmemBytes));
    EDM_CUDA(cudaFuncSetAttribute(conv_module_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kConvSmemBytes));
    EDM_CUDA(cudaFuncSetAttribute(conv_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kCsSmemBytes));
    attr_once.done();
  }
  if (p.lay.n_seq <= 0 || p.max_n <= 0) return 0;
  ProfScope prof(PK_CONV, static_cast<double>(p.lay.rows) * (glu_input ? 12288.0 : 8192.0), st);
  static const bool legacy = env_switch("EDM_CONV_LEGACY", false);  // bring-up switch: tiled kernel on the gated input as well
  if (glu_input || legacy) {
    dim3 grid((p.max_n + kConvTT - 1) / kConvTT, p.lay.n_seq);
    if (glu_input)
      launch_pdl(conv_module_kernel<true>, dim3(grid), dim3(kConvThreads), kConvSmemBytes, st, p);
    else
      launch_pdl(conv_module_kernel<false>, dim3(grid), dim3(kConvThreads), kConvSmemBytes, st, p);
  } else {
    const int sms = num_sms();
    ConvStreamParams q;
    q.in = p.in; q.out = p.out; q.dw_w = p.dw_w; q.dw_b = p.dw_b; q.cln_w = p.cln_w; q.lay = p.lay;
    q.reverse = next_direction();
    if (p.lay.cu_n != nullptr) {
      if (runs == nullptr || runs->cu_runs == nullptr) return fail(EDM_ERR_INVALID, "conv module: a packed layout needs its runs");
      q.run_len = runs->run_len; q.runs_per_seq = 0; q.cu_runs = runs->cu_runs; q.num_units = runs->num_units;
    } else {
      q.run_len = conv_run_len(p.lay.n_seq, nullptr, p.lay.N, sms);
      q.runs_per_seq = (p.lay.N + q.run_len - 1) / q.run_len; q.cu_runs = nullptr; q.num_units = p.lay.n_seq * q.runs_per_seq;
    }
    const long long units = q.num_units;
    launch_pdl(conv_stream_kernel, dim3(static_cast<unsigned>(units < sms ? units : sms)), dim3(kCsThreads), kCsSmemBytes, st, q);
  }
  EDM_LAUNCH_CHECK("conv_module");
  return 0;
}

int launch_sample(const SampleParams& p, cudaStream_t st) {
  if (p.rows <= 0) return 0;
  launch_pdl(sample_kernel, dim3((p.rows + 7) / 8), dim3(256), 0, st, p);
  EDM_LAUNCH_CHECK("sample");
  return 0;
}

__global__ void fill_u8_kernel(uint8_t* p, long long n, uint8_t v) {
  pdl_sync();
  long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}
// codes of sequence b: [Q, T_b] at Q * t_start(b), from the coarse ids ([4, T_b] blocks) and the fine ids ([n_fine, T_b] blocks)
__global__ void assemble_codes_kernel(const int* coarse, int n_coarse, const int* fine, int n_fine, long long* out, SeqLayout lay) {
  pdl_sync();
  const int Q = n_coarse + n_fine;
  long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(lay.t_rows) * Q) return;
  int b, t0;
  lay.tgt_pos(static_cast<int>(i / Q), b, t0);  // Q t_start(b) <= i < Q t_start(b + 1)
  const int tl = lay.t_len(b);
  const int local = static_cast<int>(i - static_cast<long long>(Q) * lay.t_start(b));
  const int q = local / tl, t = local - q * tl;
  out[i] = q < n_coarse ? coarse[lay.out_offset(b, q, 4, t)] : fine[lay.out_offset(b, q - n_coarse, n_fine, t)];
}

}  // namespace

// ================================================================================================ stateless ops
extern "C" int edm_abi_version(void) { return EDM_ABI_VERSION; }
extern "C" const char* edm_last_error(void) { return g_err; }
extern "C" unsigned long long edm_launch_count(void) { return g_launches.load(); }

extern "C" void edm_prof_enable(int on) {
  for (auto& e : g_prof) {
    g_event_pool.push_back(e.a);
    g_event_pool.push_back(e.b);
  }
  g_prof.clear();
  g_prof_on = on != 0;
}
// ms / work / count arrays of length 5: gemm (flops), attention (flops), layernorm (bytes), conv module (bytes), other.
// Synchronises on the recorded events, so call it after the timed region.
extern "C" int edm_prof_collect(double* ms, double* work, int* count) {
  for (int k = 0; k < PK_COUNT; ++k) {
    ms[k] = 0.0;
    work[k] = 0.0;
    count[k] = 0;
  }
  for (auto& e : g_prof) {
    EDM_CUDA(cudaEventSynchronize(e.b));
    float t = 0.f;
    EDM_CUDA(cudaEventElapsedTime(&t, e.a, e.b));
    ms[e.kind] += t;
    work[e.kind] += e.work;
    count[e.kind] += 1;
  }
  return 0;
}

#ifdef EDM_KTRACE
// bring-up build only: copies the kernel timeline (8 x uint64 per traced launch) to the host and resets it; returns the launch count
extern "C" int edm_ktrace_dump(unsigned long long* host, int max_slots) {
  unsigned n = 0;
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(&n, g_ktrace_n, sizeof(n));
  const int m = static_cast<int>(n) < max_slots ? static_cast<int>(n) : max_slots;
  if (host != nullptr && m > 0) cudaMemcpyFromSymbol(host, g_ktrace, sizeof(unsigned long long) * 8 * (m < 4096 ? m : 4096));
  const unsigned zero = 0;
  cudaMemcpyToSymbol(g_ktrace_n, &zero, sizeof(zero));
  return static_cast<int>(n);
}
#endif

extern "C" int edm_gemm_bf16(const void* a, long long lda, const void* b, long long ldb, int M, int N, int K, int epilogue,
                             const float* bias, void* out, long long ldo, float scale, const float* rope_cos,
                             const float* rope_sin, int seq_len, int rope_cols, void* stream) {
  if (int rc = check_arch()) return rc;
  CUtensorMap ma;
  WMap mb;
  if (int rc = make_tmap_2d(&ma, a, M, K, lda, kGemmBM)) return rc;
  if (int rc = make_wmap(&mb, b, N, K, ldb)) return rc;
  GemmParams p;
  p.M = M; p.N = N; p.K = K; p.a_k_offset = 0; p.b_row_offset = 0;
  p.bias = bias; p.out = out; p.ldo = ldo; p.scale = scale;
  seq_len = seq_len > 0 ? seq_len : 1;
  p.rope_cos = rope_cos; p.rope_sin = rope_sin; p.rope_lay = uniform_layout((M + seq_len - 1) / seq_len, seq_len, seq_len); p.rope_cols = rope_cols;
  p.reverse = 0; p.splits = 1; p.split_stride = 0;
  if (epilogue == EPI_QKV_ROPE && (rope_cos == nullptr || rope_sin == nullptr)) return fail(EDM_ERR_INVALID, "rope tables required");
  return launch_gemm(epilogue, ma, mb, p, static_cast<cudaStream_t>(stream));
}

extern "C" int edm_gemm_resid_layernorm(const void* a, long long lda, const void* b, long long ldb, int M, int K, const float* bias, float* x,
                                        float scale, const float* w1, const float* b1, const float* w2, const float* b2, float* y_out, void* z_out,
                                        int seq_len, int z_skip, float eps, float* scratch, int splits, void* stream) {
  if (int rc = check_arch()) return rc;
  if (M <= 0 || K <= 0 || K % kGemmBK != 0 || x == nullptr) return fail(EDM_ERR_INVALID, "gemm_resid_layernorm shape M=%d K=%d", M, K);
  CUtensorMap ma;
  WMap mb;
  if (int rc = make_tmap_2d(&ma, a, M, K, lda, kGemmBM)) return rc;
  if (int rc = make_wmap(&mb, b, kD, K, ldb)) return rc;
  GemmParams p;
  p.M = M; p.N = kD; p.K = K; p.a_k_offset = 0; p.b_row_offset = 0; p.bias = bias; p.out = x; p.ldo = kD; p.scale = scale;
  p.rope_cos = nullptr; p.rope_sin = nullptr; p.rope_lay = uniform_layout(M, 1, 1); p.rope_cols = 0; p.reverse = 0; p.splits = 1; p.split_stride = 0;
  LnParams ln;
  ln.in = x; ln.in_is_bf16 = 0; ln.rows = M; ln.w1 = w1; ln.b1 = b1; ln.w2 = w2; ln.b2 = b2; ln.y_out = y_out;
  ln.z_out = static_cast<__nv_bfloat16*>(z_out); ln.eps = eps; ln.reverse = 0;
  seq_len = seq_len > 0 ? seq_len : 1;
  ln.lay = uniform_layout(M / seq_len, seq_len, seq_len - z_skip); ln.compact = z_skip > 0;
  return launch_gemm_resid_ln(ma, mb, p, ln, scratch, splits, static_cast<cudaStream_t>(stream));
}

#ifdef EDM_ATTN_TRACE
extern "C" void edm_attn_set_trace(unsigned long long* p) { g_attn_trace = p; }
#endif
namespace {
int attention_entry(const void* qkv, int B, int N, int H, void* out, unsigned v_lbo, unsigned v_sbo, unsigned v_kstep, void* stream) {
  if (int rc = check_arch()) return rc;
  if (B <= 0 || N <= 0 || H <= 0) return fail(EDM_ERR_INVALID, "attention shape");
  CUtensorMap m;
  if (int rc = make_tmap_2d(&m, qkv, static_cast<uint64_t>(B) * N, 3ull * H * 64, 3ull * H * 64, 128)) return rc;
  return launch_attention(m, uniform_layout(B, N, N), nullptr, 0, 4.0 * B * H * static_cast<double>(N) * N * 64, H, out, v_lbo, v_sbo, v_kstep,
                          static_cast<cudaStream_t>(stream));
}
}  // namespace
#ifdef EDM_BRINGUP
// bring-up build only: the MN-major V descriptor fields (bytes) as arguments
extern "C" int edm_attention_dbg(const void* qkv, int B, int N, int H, void* out, unsigned v_lbo, unsigned v_sbo,
                                 unsigned v_kstep, void* stream) {
  return attention_entry(qkv, B, N, H, out, v_lbo, v_sbo, v_kstep, stream);
}
#endif
extern "C" int edm_attention(const void* qkv, int B, int N, int H, void* out, void* stream) {
  return attention_entry(qkv, B, N, H, out, 1024, 1024, 2048, stream);
}

extern "C" int edm_layernorm(const void* in, int in_is_bf16, int rows, const float* w1, const float* b1, const float* w2,
                             const float* b2, float* y_out, void* z_out, int seq_len, int z_skip, float eps, void* stream) {
  if (int rc = check_arch()) return rc;
  LnParams p;
  p.in = in; p.in_is_bf16 = in_is_bf16; p.rows = rows; p.w1 = w1; p.b1 = b1; p.w2 = w2; p.b2 = b2;
  p.y_out = y_out; p.z_out = static_cast<__nv_bfloat16*>(z_out); p.eps = eps;
  seq_len = seq_len > 0 ? seq_len : 1;
  p.lay = uniform_layout(rows / seq_len, seq_len, seq_len - z_skip); p.compact = z_skip > 0;
  return launch_ln(p, static_cast<cudaStream_t>(stream));
}

extern "C" int edm_conv_module(const void* in, int glu_input, void* out, const float* dw_w, const float* dw_b, const float* cln_w, int B, int N, void* stream) {
  if (int rc = check_arch()) return rc;
  ConvModParams p;
  p.in = static_cast<const __nv_bfloat16*>(in); p.out = static_cast<__nv_bfloat16*>(out);
  p.dw_w = dw_w; p.dw_b = dw_b; p.cln_w = cln_w; p.lay = uniform_layout(B, N, N); p.max_n = N;
  return launch_conv(p, glu_input != 0, static_cast<cudaStream_t>(stream));
}

// Op-level entry points of a packed batch (the context builds its layout once at bind; these build it per call).
namespace {
// reads the n_seq + 1 offsets back (the launch shapes depend on them) and checks them
int read_offsets(const int* cu_dev, int n_seq, std::vector<int>* cu, cudaStream_t st) {
  if (cu_dev == nullptr || n_seq <= 0 || n_seq >= (1 << 15)) return fail(EDM_ERR_INVALID, "varlen offsets (n_seq=%d)", n_seq);
  cu->assign(n_seq + 1, 0);
  EDM_CUDA(cudaMemcpyAsync(cu->data(), cu_dev, sizeof(int) * (n_seq + 1), cudaMemcpyDeviceToHost, st));
  EDM_CUDA(cudaStreamSynchronize(st));
  if ((*cu)[0] != 0) return fail(EDM_ERR_INVALID, "varlen offsets must start at 0");
  for (int i = 0; i < n_seq; ++i)
    if ((*cu)[i + 1] <= (*cu)[i]) return fail(EDM_ERR_INVALID, "varlen offsets: sequence %d is empty or negative", i);
  return 0;
}
// a stream-ordered device copy of `h` that lives until the work enqueued after it on `st` has run
struct StreamArray {
  int* p = nullptr;
  cudaStream_t st;
  explicit StreamArray(cudaStream_t s) : st(s) {}
  int put(const std::vector<int>& h) {
    EDM_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&p), h.size() * sizeof(int), st));
    EDM_CUDA(cudaMemcpyAsync(p, h.data(), h.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    return 0;
  }
  ~StreamArray() {
    if (p != nullptr) cudaFreeAsync(p, st);
  }
};
// Work items of the attention kernel on a packed layout, appended to `out`: (sequence << 16 | query pair) for every 256-row query
// pair of every sequence, longest sequence first (ties in sequence order), so that the static round-robin hands out the long items
// first. lens: rows per sequence.
void append_attention_pairs(const std::vector<int>& lens, std::vector<int>* out) {
  std::vector<int> order(lens.size());
  for (size_t i = 0; i < lens.size(); ++i) order[i] = static_cast<int>(i);
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return lens[a] > lens[b]; });
  for (int s : order)
    for (int q2 = 0; q2 < (lens[s] + 255) / 256; ++q2) out->push_back((s << 16) | q2);
}
SeqLayout packed_layout(int n_seq, const int* cu_dev, const std::vector<int>& cu) {
  SeqLayout l;
  l.n_seq = n_seq; l.N = 0; l.T = 0; l.cu_n = cu_dev; l.cu_t = cu_dev; l.rows = cu[n_seq]; l.t_rows = cu[n_seq];
  return l;
}
}  // namespace

extern "C" int edm_attention_varlen(const void* qkv, int n_seq, const int* cu_seqlens, int H, void* out, void* stream) {
  if (int rc = check_arch()) return rc;
  if (H <= 0) return fail(EDM_ERR_INVALID, "attention heads");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  std::vector<int> cu;
  if (int rc = read_offsets(cu_seqlens, n_seq, &cu, st)) return rc;
  std::vector<int> lens(n_seq), pairs;
  double flops = 0.0;
  for (int i = 0; i < n_seq; ++i) {
    lens[i] = cu[i + 1] - cu[i];
    flops += 4.0 * H * static_cast<double>(lens[i]) * lens[i] * 64;
  }
  append_attention_pairs(lens, &pairs);
  CUtensorMap m;
  if (int rc = make_tmap_2d(&m, qkv, cu[n_seq], 3ull * H * 64, 3ull * H * 64, 128)) return rc;
  StreamArray dp(st);
  if (int rc = dp.put(pairs)) return rc;
  return launch_attention(m, packed_layout(n_seq, cu_seqlens, cu), dp.p, static_cast<int>(pairs.size()), flops, H, out, 1024, 1024, 2048, st);
}

extern "C" int edm_conv_module_varlen(const void* in, int glu_input, void* out, const float* dw_w, const float* dw_b, const float* cln_w, int n_seq,
                                      const int* cu_seqlens, void* stream) {
  if (int rc = check_arch()) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  std::vector<int> cu;
  if (int rc = read_offsets(cu_seqlens, n_seq, &cu, st)) return rc;
  std::vector<int> lens(n_seq);
  int max_n = 0;
  for (int i = 0; i < n_seq; ++i) {
    lens[i] = cu[i + 1] - cu[i];
    max_n = std::max(max_n, lens[i]);
  }
  ConvModParams p;
  p.in = static_cast<const __nv_bfloat16*>(in); p.out = static_cast<__nv_bfloat16*>(out);
  p.dw_w = dw_w; p.dw_b = dw_b; p.cln_w = cln_w; p.lay = packed_layout(n_seq, cu_seqlens, cu); p.max_n = max_n;
  ConvRuns runs;
  runs.run_len = conv_run_len(n_seq, lens.data(), 0, num_sms());
  std::vector<int> cu_runs(n_seq + 1, 0);
  for (int i = 0; i < n_seq; ++i) cu_runs[i + 1] = cu_runs[i] + (lens[i] + runs.run_len - 1) / runs.run_len;
  runs.num_units = cu_runs[n_seq];
  StreamArray dr(st);
  if (!glu_input) {
    if (int rc = dr.put(cu_runs)) return rc;
    runs.cu_runs = dr.p;
  }
  return launch_conv(p, glu_input != 0, st, &runs);
}

extern "C" int edm_sample(const float* logits, long long ld, int rows, const float* noise, int use_philox, unsigned long long seed,
                          unsigned step, const int* forced_ids, int* ids, float* logp, int T, int Q, int out_q_stride, int out_q0, void* stream) {
  if (int rc = check_arch()) return rc;
  SampleParams p;
  if (T <= 0 || Q <= 0) return fail(EDM_ERR_INVALID, "sample: T=%d Q=%d", T, Q);
  p.logits = logits; p.ld = ld; p.rows = rows; p.noise = noise; p.use_philox = use_philox; p.seed = seed; p.seed_dev = nullptr; p.step = step; p.seq0 = 0;
  p.forced_ids = forced_ids; p.ids = ids; p.ids_raw = nullptr; p.logp = logp; p.lay = uniform_layout(rows / (T * Q), T, T); p.Q = Q;
  p.out_q_stride = out_q_stride; p.out_q0 = out_q0;
  return launch_sample(p, static_cast<cudaStream_t>(stream));
}

extern "C" int edm_remask(const float* logp, const float* gumbel, const uint8_t* mask_old, uint8_t* mask_new, const uint8_t* forced_mask,
                          int B, int T, float ratio, float temp_ratio, unsigned long long seed, unsigned step, void* stream) {
  if (int rc = check_arch()) return rc;
  if (T > kRemaskMaxT) return fail(EDM_ERR_INVALID, "remask supports T <= %d", kRemaskMaxT);
  RemaskParams p;
  p.logp = logp; p.gumbel = gumbel; p.mask_old = mask_old; p.mask_new = mask_new; p.mask_raw = nullptr; p.forced_mask = forced_mask;
  p.lay = uniform_layout(B, T, T); p.init_count = 0; p.init_counts = nullptr; p.ratio = ratio; p.temp_ratio = temp_ratio; p.seed = seed; p.seed_dev = nullptr; p.step = step; p.seq0 = 0;
  launch_pdl(remask_kernel, dim3(B), dim3(256), 0, static_cast<cudaStream_t>(stream), p);
  EDM_LAUNCH_CHECK("remask");
  return 0;
}

// descriptor strides (bytes) of the projection's MN-major tf32 A operand
#ifdef EDM_BRINGUP
// bring-up build only (tools/bringup_ops.py rvqtc): stride sweep, search kernel alone on given latents, scan without compare work
unsigned g_rvq_a_lbo = 4096, g_rvq_a_sbo = 512;
int g_rvq_skip_project = 0, g_rvq_scan_probe = 0;
extern "C" void edm_rvq_tc_debug(unsigned lbo, unsigned sbo, int skip_project, int scan_probe) {
  g_rvq_a_lbo = lbo;
  g_rvq_a_sbo = sbo;
  g_rvq_skip_project = skip_project;
  g_rvq_scan_probe = scan_probe;
}
#else
constexpr unsigned g_rvq_a_lbo = 4096, g_rvq_a_sbo = 512;
constexpr int g_rvq_skip_project = 0, g_rvq_scan_probe = 0;
#endif

extern "C" int edm_rvq_encode_tc(const void* z, int z_is_bf16, int B, int T, int n_levels, const float* w_hi, const float* w_lo, const float* b_in,
                                 const float* cb_packed, const float* g, float* e_ws, long long* codes, const long long* forced,
                                 float* latents, void* stream) {
  if (int rc = check_arch()) return rc;
  if (n_levels < 1 || n_levels > kRvqLevels || B <= 0 || T <= 0) return fail(EDM_ERR_INVALID, "rvq shape B=%d T=%d levels=%d", B, T, n_levels);
  if (T % (z_is_bf16 ? 8 : 4) != 0)
    return fail(EDM_ERR_INVALID, "rvq_encode_tc needs 16-byte rows for TMA (T %% %d == 0), got T=%d: pad the time axis", z_is_bf16 ? 8 : 4, T);
  static DeviceOnce attr_once;
  if (attr_once.needed()) {
    EDM_CUDA(cudaFuncSetAttribute(rvq_project_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRpSmemBytes));
    EDM_CUDA(cudaFuncSetAttribute(rvq_project_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRpSmemBytes));
    EDM_CUDA(cudaFuncSetAttribute(rvq_search_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRsSmemBytes));
    EDM_CUDA(cudaFuncSetAttribute(rvq_search_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRsSmemBytes));
    attr_once.done();
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CUtensorMap mz, mwh, mwl, mcb;
  if (z_is_bf16) {
    if (int rc = make_tmap_2d(&mz, z, static_cast<uint64_t>(B) * kRtLatent, T, T, 32)) return rc;
  } else {
    if (int rc = make_tmap_f32_2d(&mz, z, static_cast<uint64_t>(B) * kRtLatent, T, T, 32, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B)) return rc;
  }
  if (int rc = make_tmap_f32_2d(&mwh, w_hi, kRtE, kRtLatent, kRtLatent, kRtE)) return rc;
  if (int rc = make_tmap_f32_2d(&mwl, w_lo, kRtE, kRtLatent, kRtLatent, kRtE)) return rc;
  if (int rc = make_tmap_f32_2d(&mcb, cb_packed, 12 * 1024, 32, 32, kRsChunk)) return rc;
  const int tiles = ((T + kRtFrames - 1) / kRtFrames) * B;
  RvqProjParams pp;
  pp.B = B; pp.T = T; pp.b_in = b_in; pp.e_out = e_ws; pp.a_lbo = g_rvq_a_lbo; pp.a_sbo = g_rvq_a_sbo; pp.dbg = g_rvq_skip_project >> 4;
  if (!(g_rvq_skip_project & 1)) {
      const int ptiles = ((T + kRpFrames - 1) / kRpFrames) * B;
    if (z_is_bf16)
      rvq_project_kernel<true><<<ptiles < num_sms() ? ptiles : num_sms(), kRpThreads, kRpSmemBytes, st>>>(mz, mwh, mwl, pp);
    else
      rvq_project_kernel<false><<<ptiles < num_sms() ? ptiles : num_sms(), kRpThreads, kRpSmemBytes, st>>>(mz, mwh, mwl, pp);
    EDM_LAUNCH_CHECK("rvq_project");
  }
  RvqSearchParams sp;
  sp.B = B; sp.T = T; sp.n_levels = n_levels; sp.e = e_ws; sp.g = g; sp.codes = codes; sp.forced = forced; sp.latents = latents;
  sp.one = 1.0f; sp.onei = 1; sp.n_mma = (g_rvq_scan_probe >> 4) ? (g_rvq_scan_probe >> 4) : 4;
  const int s_ctas = (g_rvq_scan_probe & 8) ? num_sms() : 2 * num_sms();  // bring-up probe: one CTA per SM (how much the two co-resident tiles overlap)
  const int sgrid = tiles < s_ctas ? tiles : s_ctas;
#ifdef EDM_BRINGUP
  if ((g_rvq_scan_probe & 3) == 2) {
    static DeviceOnce once2;
    if (once2.needed()) {
      EDM_CUDA(cudaFuncSetAttribute(rvq_search_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRsSmemBytes));
      once2.done();
    }
    rvq_search_kernel<2><<<sgrid, kRsThreads, kRsSmemBytes, st>>>(mcb, sp);
  } else
#endif
  if (g_rvq_scan_probe & 1)
    rvq_search_kernel<1><<<sgrid, kRsThreads, kRsSmemBytes, st>>>(mcb, sp);
  else
    rvq_search_kernel<0><<<sgrid, kRsThreads, kRsSmemBytes, st>>>(mcb, sp);
  EDM_LAUNCH_CHECK("rvq_search");
  return 0;
}

extern "C" int edm_codes_to_features(const long long* codes, const float* proj, float* out, int B, int L, int T, int unreduced, void* stream) {
  if (int rc = check_arch()) return rc;
  if (L < 1 || L > kRvqLevels) return fail(EDM_ERR_INVALID, "codes_to_features levels=%d", L);
  CodesToFeatParams p;
  p.codes = codes; p.proj = proj; p.out = out; p.B = B; p.L = L; p.T = T; p.unreduced = unreduced;
  dim3 grid((T + 31) / 32, B);
  codes_to_features_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(p);
  EDM_LAUNCH_CHECK("codes_to_features");
  return 0;
}

extern "C" int edm_kmeans_assign(const float* x, long long n_frames, int dim, const float* c_hi, const float* c_lo, const float* half_neg_norm,
                                 int n_centroids, long long* idx_out, float* score_out, void* stream) {
  if (int rc = check_arch()) return rc;
  if (n_frames <= 0) return 0;
  if (dim <= 0 || dim % kKmKc != 0 || n_centroids <= 0 || n_centroids % kKmCodes != 0 || n_centroids > kKmMaxCentroids || n_frames > 0x7fffffffLL)
    return fail(EDM_ERR_INVALID, "kmeans_assign shape frames=%lld dim=%d centroids=%d unsupported (dim %% 32, centroids %% 256, <= 4096)", n_frames, dim, n_centroids);
  static DeviceOnce attr_once;
  if (attr_once.needed()) {
    EDM_CUDA(cudaFuncSetAttribute(kmeans_assign_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kKmSmemBytes));
    attr_once.done();
  }
  CUtensorMap mx, mh, ml;
  if (int rc = make_tmap_f32_2d(&mx, x, static_cast<uint64_t>(n_frames), dim, dim, kKmFrames)) return rc;
  if (int rc = make_tmap_f32_2d(&mh, c_hi, n_centroids, dim, dim, kKmCodes)) return rc;
  if (int rc = make_tmap_f32_2d(&ml, c_lo, n_centroids, dim, dim, kKmCodes)) return rc;
  KmeansParams p;
  p.n_frames = static_cast<int>(n_frames); p.dim = dim; p.n_centroids = n_centroids; p.half_neg_norm = half_neg_norm; p.idx_out = idx_out; p.score_out = score_out;
  const int tiles = (p.n_frames + kKmFrames - 1) / kKmFrames;
  kmeans_assign_kernel<<<tiles < num_sms() ? tiles : num_sms(), kKmThreads, kKmSmemBytes, static_cast<cudaStream_t>(stream)>>>(mx, mh, ml, p);
  EDM_LAUNCH_CHECK("kmeans_assign");
  return 0;
}

extern "C" size_t edm_kmeans_update_workspace_bytes(long long n, int dim, int n_centroids) {
  if (n < 0 || dim <= 0 || n_centroids <= 0) return 0;
  return static_cast<size_t>(n_centroids + (n + kKmUpdRows - 1) / kKmUpdRows) * static_cast<size_t>(dim) * sizeof(double);
}

extern "C" int edm_kmeans_update(const float* x, long long n, int dim, const long long* idx, const long long* perm, const long long* offsets,
                                 int n_centroids, double* partials, float* centroids, double* sums_out, void* stream) {
  if (int rc = check_arch()) return rc;
  if (dim <= 0 || dim % kKmKc != 0 || n_centroids <= 0 || n_centroids > kKmMaxCentroids || n < 0 || n > 0x7fffffffLL)
    return fail(EDM_ERR_INVALID, "kmeans_update shape n=%lld dim=%d centroids=%d unsupported (dim %% 32, 1 <= centroids <= 4096)", n, dim, n_centroids);
  if ((reinterpret_cast<uintptr_t>(x) & 15) != 0 || (reinterpret_cast<uintptr_t>(partials) & 15) != 0)
    return fail(EDM_ERR_INVALID, "kmeans_update: x and partials must be 16-byte aligned");
  if (n == 0) {
    if (sums_out != nullptr) EDM_CUDA(cudaMemsetAsync(sums_out, 0, static_cast<size_t>(n_centroids) * dim * sizeof(double), static_cast<cudaStream_t>(stream)));
    return 0;
  }
  KmeansUpdateParams p;
  p.x = x; p.idx = idx; p.perm = perm; p.offsets = offsets; p.partials = partials; p.centroids = centroids; p.sums = sums_out;
  p.n = n; p.dim = dim; p.n_centroids = n_centroids;
  const cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int d4 = dim / 4;
  const int t1 = d4 < kKmUpdThreads ? (d4 + 31) / 32 * 32 : kKmUpdThreads;
  const dim3 g1(static_cast<unsigned>((n + kKmUpdRows - 1) / kKmUpdRows), (d4 + t1 - 1) / t1);
  kmeans_update_partial_kernel<<<g1, t1, 0, st>>>(p);
  EDM_LAUNCH_CHECK("kmeans_update_partial");
  const int t2 = dim < kKmUpdThreads ? dim : kKmUpdThreads;
  kmeans_update_finalize_kernel<<<dim3(n_centroids, (dim + t2 - 1) / t2), t2, 0, st>>>(p);
  EDM_LAUNCH_CHECK("kmeans_update_finalize");
  return 0;
}

// ---------------------------------------------------------------------------------------------- DAC encoder convolutions
namespace {
// bf16 operand [B][rows][cols] with an explicit batch stride (elements): box = 64 channels x 128 rows x 1 batch; rows outside
// [0, rows) are zero-filled (the conv's zero padding)
int make_tmap_conv_a(CUtensorMap* m, const void* ptr, uint64_t B, uint64_t rows, uint64_t cols, uint64_t batch_stride, uint32_t box_rows = 128) {
  PFN_tmapEncodeTiled enc = get_encode();
  if (enc == nullptr) return fail(EDM_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) != 0 || (cols * 2) % 16 != 0 || (batch_stride * 2) % 16 != 0)
    return fail(EDM_ERR_INVALID, "conv operand must be 16-byte aligned");
  cuuint64_t dims[3] = {cols, rows, B};
  cuuint64_t strides[2] = {cols * 2, batch_stride * 2};
  cuuint32_t box[3] = {64, box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(EDM_ERR_CUDA, "cuTensorMapEncodeTiled(conv operand rows=%llu cols=%llu) failed: %d", (unsigned long long)rows, (unsigned long long)cols, (int)r);
  return 0;
}

// output boxes of the conv epilogue: 32 columns x 32 rows x 1 batch of [B][rows][cols]; fp32 (128 B rows, swizzle 128B) or bf16
// (64 B rows, swizzle 64B). Rows >= `rows` are clipped by TMA (ragged last tile, end of the padded operand).
int make_tmap_conv_out(CUtensorMap* m, const void* ptr, bool f32, uint64_t B, uint64_t rows, uint64_t cols, uint64_t batch_stride) {
  PFN_tmapEncodeTiled enc = get_encode();
  if (enc == nullptr) return fail(EDM_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  const uint64_t es = f32 ? 4 : 2;
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) != 0 || (cols * es) % 16 != 0 || (batch_stride * es) % 16 != 0)
    return fail(EDM_ERR_INVALID, "conv output must be 16-byte aligned");
  cuuint64_t dims[3] = {cols, rows, B};
  cuuint64_t strides[2] = {cols * es, batch_stride * es};
  cuuint32_t box[3] = {32, 32, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(m, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, f32 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(EDM_ERR_CUDA, "cuTensorMapEncodeTiled(conv output rows=%llu cols=%llu) failed: %d", (unsigned long long)rows, (unsigned long long)cols, (int)r);
  return 0;
}

template <int NT>
int launch_dac_conv(const CUtensorMap& ma, const CUtensorMap& mw, const CUtensorMap& my, const CUtensorMap& ms, DacConvParams& p, cudaStream_t st) {
  static DeviceOnce attr_once;
  if (attr_once.needed()) {
    EDM_CUDA(cudaFuncSetAttribute(dac_conv_kernel<NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, dac_conv_smem_bytes<NT>()));
    attr_once.done();
  }
  p.n_tiles_n = p.c_out / NT;
  const long long tiles = static_cast<long long>(p.B) * p.tiles_per_batch * p.n_tiles_n;
  if (tiles > 0x7fffffffLL) return fail(EDM_ERR_INVALID, "dac_conv: too many tiles");
  const int grid = tiles < num_sms() ? static_cast<int>(tiles) : num_sms();
  dac_conv_kernel<NT><<<grid, kDcThreads, dac_conv_smem_bytes<NT>(), st>>>(ma, mw, my, ms, p);
  EDM_LAUNCH_CHECK("dac_conv");
  return 0;
}
}  // namespace

extern "C" int edm_dac_conv(const void* a, long long a_rows, int a_cols, long long a_batch_stride, int B, const void* w, int c_out,
                            int n_taps, int tap_step, int row_off, int rows_out, const float* bias, const float* alpha, int bias_period,
                            const float* x_res, float* y, long long y_batch_stride, void* s_out, long long s_batch_stride,
                            int s_row_off, int s_rows, void* zt_out, int zt_is_f32, void* stream) {
  if (int rc = check_arch()) return rc;
  if (B <= 0 || rows_out <= 0) return 0;
  const int c_mod = bias_period > 0 ? bias_period : c_out;
  if (a_cols <= 0 || a_cols % 64 != 0 || c_out < 64 || c_out % 64 != 0 || c_mod > kDcMaxCout || c_mod % 32 != 0 || c_out % c_mod != 0 || n_taps <= 0 || a_rows <= 0)
    return fail(EDM_ERR_INVALID, "dac_conv shape cin=%d cout=%d period=%d taps=%d unsupported (channels %% 64, period <= 1536)", a_cols, c_out, c_mod, n_taps);
  if (zt_out != nullptr && c_mod != c_out) return fail(EDM_ERR_INVALID, "dac_conv: the transposed output needs bias_period == c_out");
  if (bias == nullptr) return fail(EDM_ERR_INVALID, "dac_conv: bias is required");
  CUtensorMap ma, mw;
  if (int rc = make_tmap_conv_a(&ma, a, B, static_cast<uint64_t>(a_rows), a_cols, static_cast<uint64_t>(a_batch_stride))) return rc;
  const int nt = c_out % 256 == 0 ? 256 : (c_out % 192 == 0 ? 192 : (c_out % 128 == 0 ? 128 : 64));
  const uint64_t k_total = static_cast<uint64_t>(n_taps) * a_cols;
  if (int rc = make_tmap_2d(&mw, w, c_out, k_total, k_total, nt)) return rc;
  DacConvParams p;
  p.B = B; p.rows_out = rows_out; p.tiles_per_batch = (rows_out + kDcBM - 1) / kDcBM; p.c_out = c_out; p.n_tiles_n = 0;
  p.n_taps = n_taps; p.tap_step = tap_step; p.row_off = row_off; p.k_chunks = a_cols / 64;
  p.c_mod = c_mod; p.bias = bias; p.alpha = alpha; p.x_res = x_res; p.y = y; p.y_batch_stride = y_batch_stride;
  p.s_out = static_cast<__nv_bfloat16*>(s_out); p.s_batch_stride = s_batch_stride; p.s_row_off = s_row_off; p.s_rows = s_rows;
  p.zt_out = zt_out; p.zt_is_f32 = zt_is_f32;
  if (x_res != nullptr && x_res != y) return fail(EDM_ERR_INVALID, "dac_conv: the residual input must be the stream that is updated (x_res == y)");
  CUtensorMap my = ma, ms = ma;  // placeholders when the output is absent (never dereferenced by the kernel)
  if (y != nullptr)
    if (int rc = make_tmap_conv_out(&my, y, true, B, rows_out, c_out, static_cast<uint64_t>(y_batch_stride))) return rc;
  if (s_out != nullptr) {
    const long long lim = static_cast<long long>(rows_out) + s_row_off;
    const long long s_eff = s_rows < lim ? s_rows : lim;
    if (s_eff <= 0 || s_row_off < 0) return fail(EDM_ERR_INVALID, "dac_conv: operand output rows");
    if (int rc = make_tmap_conv_out(&ms, s_out, false, B, static_cast<uint64_t>(s_eff), c_out, static_cast<uint64_t>(s_batch_stride))) return rc;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (nt == 256) return launch_dac_conv<256>(ma, mw, my, ms, p, st);
  if (nt == 192) return launch_dac_conv<192>(ma, mw, my, ms, p, st);
  if (nt == 128) return launch_dac_conv<128>(ma, mw, my, ms, p, st);
  return launch_dac_conv<64>(ma, mw, my, ms, p, st);
}

namespace {
template <int C>
int launch_dac_resunit(const CUtensorMap& ma, const CUtensorMap& m7, const CUtensorMap& m1, const CUtensorMap& my, const CUtensorMap& ms,
                       const DacResUnitParams& p, int s_row_off, cudaStream_t st) {
  static DeviceOnce attr_once;
  if (attr_once.needed()) {
    EDM_CUDA(cudaFuncSetAttribute(dac_resunit_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, DacResUnitCfg<C>::kSmemBytes));
    attr_once.done();
  }
  const long long tiles = static_cast<long long>(p.B) * p.tiles_per_batch;
  if (tiles > 0x7fffffffLL) return fail(EDM_ERR_INVALID, "dac_resunit: too many tiles");
  const int grid = tiles < num_sms() ? static_cast<int>(tiles) : num_sms();
  dac_resunit_kernel<C><<<grid, kRuThreads, DacResUnitCfg<C>::kSmemBytes, st>>>(ma, m7, m1, my, ms, p, s_row_off);
  EDM_LAUNCH_CHECK("dac_resunit");
  return 0;
}
}  // namespace

#ifdef EDM_DAC_TRACE
unsigned long long* g_dac_trace = nullptr;
extern "C" void edm_dac_set_trace(unsigned long long* p) { g_dac_trace = p; }
#endif
extern "C" int edm_dac_resunit(const void* a, long long a_batch_stride, int B, int rows, int channels, int dilation, const void* w7,
                               const void* w1, const float* b7, const float* a_mid, const float* b1, const float* a_next, float* y,
                               long long y_batch_stride, void* s_out, long long s_batch_stride, int s_row_off, int s_rows, void* stream) {
  if (int rc = check_arch()) return rc;
  if (B <= 0 || rows <= 0) return 0;
  if (channels != 64 && channels != 128 && channels != 192) return fail(EDM_ERR_INVALID, "dac_resunit: fused kernel exists for 64, 128 and 192 channels (got %d)", channels);
  if (a == s_out) return fail(EDM_ERR_INVALID, "dac_resunit: s_out must not alias the input operand (neighbouring tiles still read its halo)");
  if (!b7 || !a_mid || !b1 || !a_next || !y || !s_out || s_row_off < 0) return fail(EDM_ERR_INVALID, "dac_resunit: null argument");
  CUtensorMap ma, m7, m1, my, ms;
  if (int rc = make_tmap_conv_a(&ma, a, B, rows, channels, static_cast<uint64_t>(a_batch_stride))) return rc;
  if (int rc = make_tmap_2d(&m7, w7, channels, 7ull * channels, 7ull * channels, channels)) return rc;
  if (int rc = make_tmap_2d(&m1, w1, channels, channels, channels, channels)) return rc;
  if (int rc = make_tmap_conv_out(&my, y, true, B, rows, channels, static_cast<uint64_t>(y_batch_stride))) return rc;
  const long long lim = static_cast<long long>(rows) + s_row_off;
  const long long s_eff = s_rows < lim ? s_rows : lim;
  if (s_eff <= 0) return fail(EDM_ERR_INVALID, "dac_resunit: operand output rows");
  if (int rc = make_tmap_conv_out(&ms, s_out, false, B, static_cast<uint64_t>(s_eff), channels, static_cast<uint64_t>(s_batch_stride))) return rc;
  DacResUnitParams p;
  p.B = B; p.rows = rows; p.tiles_per_batch = (rows + kDcBM - 1) / kDcBM; p.dilation = dilation;
  p.b7 = b7; p.a_mid = a_mid; p.b1 = b1; p.a_next = a_next; p.y = y; p.y_batch_stride = y_batch_stride;
#ifdef EDM_DAC_TRACE
  p.trace = g_dac_trace;
#endif
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (channels == 192) {
    static DeviceOnce attr_once;
    if (attr_once.needed()) {
      EDM_CUDA(cudaFuncSetAttribute(dac_resunit_wide_kernel<192>, cudaFuncAttributeMaxDynamicSharedMemorySize, DacResUnitWideCfg<192>::kSmemBytes));
      attr_once.done();
    }
    const long long tiles = static_cast<long long>(p.B) * p.tiles_per_batch;
    const int grid = tiles < num_sms() ? static_cast<int>(tiles) : num_sms();
    dac_resunit_wide_kernel<192><<<grid, kRuThreads, DacResUnitWideCfg<192>::kSmemBytes, st>>>(ma, m7, m1, my, ms, p, s_row_off);
    EDM_LAUNCH_CHECK("dac_resunit_wide");
    return 0;
  }
  static const bool halo_mode = env_switch("EDM_DAC_HALO", true);  // bring-up switch, 0: seven shifted TMA boxes per tile (first form) for 64 channels too
  if (channels == 64 && halo_mode && dilation >= 1 && 128 + 6 * dilation <= kRu64HaloRows) {
    static DeviceOnce attr_once;
    if (attr_once.needed()) {
      EDM_CUDA(cudaFuncSetAttribute(dac_resunit64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kRu64SmemBytes));
      attr_once.done();
    }
    CUtensorMap mh, m7b;
    if (int rc = make_tmap_conv_a(&mh, a, B, rows, channels, static_cast<uint64_t>(a_batch_stride), 128 + 6 * dilation)) return rc;
    if (int rc = make_tmap_2d(&m7b, w7, channels, 7ull * channels, 7ull * channels, 64)) return rc;
    const long long tiles = static_cast<long long>(p.B) * p.tiles_per_batch;
    const int grid = tiles < num_sms() ? static_cast<int>(tiles) : num_sms();
    dac_resunit64_kernel<<<grid, kRuThreads, kRu64SmemBytes, st>>>(mh, m7b, m1, my, ms, p, s_row_off);
    EDM_LAUNCH_CHECK("dac_resunit64");
    return 0;
  }
  if (dilation < 1 || 128 + 6 * dilation > kRu64HaloRows) return fail(EDM_ERR_INVALID, "dac_resunit: dilation %d unsupported (halo tile of at most 192 rows)", dilation);
  CUtensorMap mh;
  if (int rc = make_tmap_conv_a(&mh, a, B, rows, channels, static_cast<uint64_t>(a_batch_stride), 128 + 6 * dilation)) return rc;
  if (channels == 64) return launch_dac_resunit<64>(mh, m7, m1, my, ms, p, s_row_off, st);
  return launch_dac_resunit<128>(mh, m7, m1, my, ms, p, s_row_off, st);
}

extern "C" int edm_dac_conv_last(const void* a, long long a_batch_stride, int B, int rows, int c_pad, const float* w, float bias, float* out,
                                 int apply_tanh, void* stream) {
  if (int rc = check_arch()) return rc;
  if (B <= 0 || rows <= 0) return 0;
  if (c_pad <= 0 || c_pad % 8 != 0 || c_pad > 256) return fail(EDM_ERR_INVALID, "dac_conv_last: padded channels %d unsupported (%% 8, <= 256)", c_pad);
  DacConvLastParams p;
  p.a = static_cast<const __nv_bfloat16*>(a); p.a_batch_stride = a_batch_stride; p.rows = rows; p.c_pad = c_pad; p.B = B; p.w = w; p.bias = bias;
  p.out = out; p.apply_tanh = apply_tanh;
  const long long runs = static_cast<long long>(B) * ((rows + 31) / 32);
  const long long blocks = (runs + 7) / 8;
  const int grid = static_cast<int>(blocks < 16LL * num_sms() ? blocks : 16LL * num_sms());
  dac_conv_last_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(p);
  EDM_LAUNCH_CHECK("dac_conv_last");
  return 0;
}

extern "C" int edm_dac_zero_rows(void* buf, long long row_pitch_bytes, const int* ranges, int n_ranges, int max_range_rows, void* stream) {
  if (int rc = check_arch()) return rc;
  if (n_ranges <= 0 || max_range_rows <= 0) return 0;
  if (buf == nullptr || ranges == nullptr || (reinterpret_cast<uintptr_t>(buf) & 15) != 0 || (reinterpret_cast<uintptr_t>(ranges) & 7) != 0 ||
      row_pitch_bytes <= 0 || row_pitch_bytes % 16 != 0)
    return fail(EDM_ERR_INVALID, "dac_zero_rows: buffer and row pitch must be 16-byte aligned, ranges 8-byte aligned");
  const long long blocks = (static_cast<long long>(max_range_rows) * row_pitch_bytes / 16 + kZeroRowsThreads - 1) / kZeroRowsThreads;
  const dim3 grid(static_cast<unsigned>(blocks < 1024 ? blocks : 1024), static_cast<unsigned>(n_ranges < 65535 ? n_ranges : 65535));
  dac_zero_rows_kernel<<<grid, kZeroRowsThreads, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<uint8_t*>(buf), row_pitch_bytes,
                                                                                        reinterpret_cast<const int2*>(ranges), n_ranges);
  EDM_LAUNCH_CHECK("dac_zero_rows");
  return 0;
}

extern "C" int edm_dac_conv_first(const float* audio, int B, int L, const float* w, const float* bias, const float* alpha, int c0,
                                  float* y, void* s_out, void* stream) {
  if (int rc = check_arch()) return rc;
  if (B <= 0 || L <= 0) return 0;
  if (c0 <= 0 || c0 % 64 != 0 || c0 > 512) return fail(EDM_ERR_INVALID, "dac_conv_first: channels %d unsupported (%% 64, <= 512)", c0);
  DacConv0Params p;
  p.audio = audio; p.w = w; p.bias = bias; p.alpha = alpha; p.y = y; p.s_out = static_cast<__nv_bfloat16*>(s_out); p.B = B; p.L = L; p.C0 = c0;
  const long long runs = static_cast<long long>(B) * ((L + kDc0Run - 1) / kDc0Run);
  const long long blocks = (runs + 15) / 16;
  dim3 grid(static_cast<unsigned>(blocks < 16LL * num_sms() ? blocks : 16LL * num_sms()), c0 / 64);
  dac_conv0_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(p);
  EDM_LAUNCH_CHECK("dac_conv_first");
  return 0;
}

// ================================================================================================ S2A context
namespace {

const char* const kBlockFields[] = {
    "ff1_ln_w", "ff1_ln_b", "ff1_w1", "ff1_b1", "ff1_w2", "ff1_b2",                       //
    "attn_ln_w", "attn_ln_b", "wqkv", "wo", "bo",                                        //
    "conv_ln_w", "conv_ln_b", "pw1_w", "pw1_b", "dw_w", "dw_b", "cln_w", "pw2_w", "pw2_b",  //
    "ff2_ln_w", "ff2_ln_b", "ff2_w1", "ff2_b1", "ff2_w2", "ff2_b2",                       //
    "post_ln_w", "post_ln_b"};
enum BlockField {
  F_FF1_LN_W, F_FF1_LN_B, F_FF1_W1, F_FF1_B1, F_FF1_W2, F_FF1_B2,
  F_ATTN_LN_W, F_ATTN_LN_B, F_WQKV, F_WO, F_BO,
  F_CONV_LN_W, F_CONV_LN_B, F_PW1_W, F_PW1_B, F_DW_W, F_DW_B, F_CLN_W, F_PW2_W, F_PW2_B,
  F_FF2_LN_W, F_FF2_LN_B, F_FF2_W1, F_FF2_B1, F_FF2_W2, F_FF2_B2,
  F_POST_LN_W, F_POST_LN_B, F_BLOCK_COUNT
};
const char* const kGlobalFields[] = {"sem_emb", "mask_token", "feat_table", "feat_const", "fp_ln_w", "fp_ln_b",
                                     "inj_table", "inj_const", "inj_ln_w", "inj_ln_b", "tl_ln_w", "tl_ln_b",
                                     "head_w", "head_b", "fine_w", "fine_b", "rope_cos", "rope_sin"};
enum GlobalField {
  G_SEM_EMB, G_MASK_TOKEN, G_FEAT_TABLE, G_FEAT_CONST, G_FP_LN_W, G_FP_LN_B,
  G_INJ_TABLE, G_INJ_CONST, G_INJ_LN_W, G_INJ_LN_B, G_TL_LN_W, G_TL_LN_B,
  G_HEAD_W, G_HEAD_B, G_FINE_W, G_FINE_B, G_ROPE_COS, G_ROPE_SIN, G_COUNT
};

struct BlockMaps {
  WMap ff1_w1, ff1_w2, wqkv, wo, pw1, pw2, ff2_w1, ff2_w2;
};

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

}  // namespace

struct edm_s2a_ctx {
  edm_s2a_config cfg;
  std::vector<const void*> w;  // depth * F_BLOCK_COUNT + G_COUNT
  std::vector<BlockMaps> bmaps;
  WMap head_map, fine_map;
  int n_fine;

  // bound shapes. B = sequences; T / P / N: the common lengths of a uniform bind (0 after edm_s2a_bind_varlen)
  bool bound = false;
  int B = 0, T = 0, P = 0, N = 0, M = 0, Mt = 0, Mp = 0, max_n = 0, min_t = 0;
  bool varlen = false;
  SeqLayout lay;                   // where the sequences are (device arrays in the workspace after a varlen bind)
  const int* pairs = nullptr;      // varlen: attention (sequence, query pair) list in the workspace, longest first
  int n_pairs = 0;
  double attn_flops = 0.0;
  ConvRuns conv_runs;              // varlen: runs of the streaming conv kernel
  int* layout_dev = nullptr;       // varlen: the layout arrays in the workspace (cu_n | cu_t | cu_runs | pairs)
  std::vector<int> host_layout;    // varlen: their host image
  uint8_t* ws = nullptr;
  size_t ws_bytes = 0;
  // workspace views
  float *x_in, *x, *coarse_out[4], *logits, *coarse_logits, *fine_logits, *logp;
  float2* arg_part;          // [Mt, n_fine, 16] partial arg-max of the fused heads (keep_logits == false)
  bool keep_logits = false;  // true: coarse / fine logits are materialised (parity runs, the eval-mode loss); false: arg-max in the GEMM epilogue
  __nv_bfloat16 *z, *h, *qkv, *g, *zt, *fine_h, *fine_z;
  int *ids, *ids_raw, *pred_codes, *pred_raw, *fine_codes, *sem_tokens, *sem_prompt, *ac_prompt;
  uint8_t *mask_a, *mask_b, *mask_raw;
  const float* prompt_proj = nullptr;            // optional caller-projected prompt injections [n_inj, B*P, 1024] (edm_s2a_set_prompt_injections)
  const unsigned long long* seed_dev = nullptr;  // optional device-resident seed offset (edm_s2a_set_seed_buffer)
  int ac_levels = 0;
  long long batch_offset = 0;  // global index of this context's first sequence (Philox counters)
  bool mask_in_a = true;  // which buffer holds the current mask
  CUtensorMap m_z, m_h, m_g, m_zt, m_fine_z, m_qkv;
  float* part = nullptr;  // [4, M, 1024] partial sums of the split-K residual GEMMs (low-latency mode; carved only for M <= kSplitMaxRows)
  bool low_latency = false;  // edm_s2a_set_low_latency

  const void* bw(int layer, int f) const { return w[static_cast<size_t>(layer) * F_BLOCK_COUNT + f]; }
  const float* bwf(int layer, int f) const { return static_cast<const float*>(bw(layer, f)); }
  const void* gw(int f) const { return w[static_cast<size_t>(cfg.depth) * F_BLOCK_COUNT + f]; }
  const float* gwf(int f) const { return static_cast<const float*>(gw(f)); }
  uint8_t* mask_cur() { return mask_in_a ? mask_a : mask_b; }
  uint8_t* mask_next() { return mask_in_a ? mask_b : mask_a; }
};

namespace {

int validate_cfg(const edm_s2a_config* c) {
  if (c == nullptr) return fail(EDM_ERR_INVALID, "null config");
  if (c->hidden != 1024 || c->heads != 16 || c->ff_mult != 4 || c->conv_kernel != 5 || c->num_codes != 1024)
    return fail(EDM_ERR_INVALID, "kernels are specialised for hidden=1024 heads=16 ff_mult=4 conv_kernel=5 codes=1024 (got %d %d %d %d %d)", c->hidden,
                c->heads, c->ff_mult, c->conv_kernel, c->num_codes);
  if (c->depth < 1 || c->depth > 64 || c->n_injection < 1 || c->n_injection > 4 || c->num_quantizers <= c->n_injection || c->num_quantizers > 12)
    return fail(EDM_ERR_INVALID, "unsupported depth / injection / quantizer counts");
  for (int i = 0; i < c->n_injection; ++i) {
    if (c->injection_layers[i] < 0 || c->injection_layers[i] >= c->depth) return fail(EDM_ERR_INVALID, "injection layer out of range");
    if (i > 0 && c->injection_layers[i] <= c->injection_layers[i - 1]) return fail(EDM_ERR_INVALID, "injection layers must increase");
  }
  return 0;
}

int injection_index(const edm_s2a_config& c, int layer) {
  for (int i = 0; i < c.n_injection; ++i)
    if (c.injection_layers[i] == layer) return i;
  return -1;
}

GemmParams gp(int M, int N, int K, const float* bias, void* out, long long ldo, float scale = 1.0f) {
  GemmParams p;
  p.M = M; p.N = N; p.K = K; p.a_k_offset = 0; p.b_row_offset = 0; p.bias = bias; p.out = out; p.ldo = ldo; p.scale = scale;
  p.rope_cos = nullptr; p.rope_sin = nullptr; p.rope_lay = uniform_layout(M, 1, 1); p.rope_cols = 0; p.reverse = 0; p.splits = 1; p.split_stride = 0;
  return p;
}

// One conformer block on the bound workspace. In: x (fp32 residual stream) and z = LN_ff1(x) (bf16). Out: `post` applied to the
// block's sum (post_norm and whatever the call site chains after it: the next block's pre-norm, the heads' LayerNorm, row compaction).
// Every residual GEMM goes out together with the LayerNorm that follows it (launch_gemm_resid_ln).
int run_block_body(edm_s2a_ctx* c, int l, const LnParams& post, cudaStream_t st) {
  const int M = c->M;
  const float eps = 1e-5f;
  LnParams ln;
  ln.in = c->x; ln.in_is_bf16 = 0; ln.rows = M; ln.w2 = nullptr; ln.b2 = nullptr;
  ln.y_out = nullptr; ln.z_out = c->z; ln.lay = c->lay; ln.compact = 0; ln.eps = eps;
  // ff1: x += 0.5 * W2 swish(W1 z + b1) + b2; then the attention pre-norm
  if (int rc = launch_gemm(EPI_SWISH_BF16, c->m_z, c->bmaps[l].ff1_w1, gp(M, 4096, 1024, c->bwf(l, F_FF1_B1), c->h, 4096), st)) return rc;
  ln.w1 = c->bwf(l, F_ATTN_LN_W); ln.b1 = c->bwf(l, F_ATTN_LN_B);
  if (int rc = launch_gemm_resid_ln(c->m_h, c->bmaps[l].ff1_w2, gp(M, 1024, 4096, c->bwf(l, F_FF1_B2), c->x, 1024, 0.5f), ln, c->part, c->low_latency ? choose_splits(M, 4096) : 1, st)) return rc;
  // attention
  {
    GemmParams p = gp(M, 3072, 1024, nullptr, c->qkv, 3072);
    p.rope_cos = c->gwf(G_ROPE_COS); p.rope_sin = c->gwf(G_ROPE_SIN); p.rope_lay = c->lay; p.rope_cols = 2048;
    if (int rc = launch_gemm(EPI_QKV_ROPE, c->m_z, c->bmaps[l].wqkv, p, st)) return rc;
  }
  if (int rc = launch_attention(c->m_qkv, c->lay, c->pairs, c->n_pairs, c->attn_flops, 16, c->z, 1024, 1024, 2048, st)) return rc;
  ln.w1 = c->bwf(l, F_CONV_LN_W); ln.b1 = c->bwf(l, F_CONV_LN_B);
  if (int rc = launch_gemm_resid_ln(c->m_z, c->bmaps[l].wo, gp(M, 1024, 1024, c->bwf(l, F_BO), c->x, 1024, 1.0f), ln, c->part, c->low_latency ? choose_splits(M, 1024) : 1, st)) return rc;
  // conv module. pointwise conv 1 + GLU in one pass: the packed weight interleaves 32 value rows with their 32 gate rows
  if (int rc = launch_gemm(EPI_GLU_BF16, c->m_z, c->bmaps[l].pw1, gp(M, 4096, 1024, c->bwf(l, F_PW1_B), c->h, 2048), st)) return rc;
  {
    ConvModParams p;
    p.in = c->h; p.out = c->g; p.dw_w = c->bwf(l, F_DW_W); p.dw_b = c->bwf(l, F_DW_B); p.cln_w = c->bwf(l, F_CLN_W); p.lay = c->lay; p.max_n = c->max_n;
    if (int rc = launch_conv(p, false, st, &c->conv_runs)) return rc;
  }
  ln.w1 = c->bwf(l, F_FF2_LN_W); ln.b1 = c->bwf(l, F_FF2_LN_B);
  if (int rc = launch_gemm_resid_ln(c->m_g, c->bmaps[l].pw2, gp(M, 1024, 2048, c->bwf(l, F_PW2_B), c->x, 1024, 1.0f), ln, c->part, c->low_latency ? choose_splits(M, 2048) : 1, st)) return rc;
  // ff2, then post_norm (+ what the caller chains after it)
  if (int rc = launch_gemm(EPI_SWISH_BF16, c->m_z, c->bmaps[l].ff2_w1, gp(M, 4096, 1024, c->bwf(l, F_FF2_B1), c->h, 4096), st)) return rc;
  return launch_gemm_resid_ln(c->m_h, c->bmaps[l].ff2_w2, gp(M, 1024, 4096, c->bwf(l, F_FF2_B2), c->x, 1024, 0.5f), post, c->part, c->low_latency ? choose_splits(M, 4096) : 1, st);
}

// pass prologue: x = copy of the encoder input, z = LN_ff1[0](x)
int pass_prologue(edm_s2a_ctx* c, const float* x_src, cudaStream_t st) {
  LnParams ln;
  ln.in = x_src; ln.in_is_bf16 = 0; ln.rows = c->M; ln.w1 = nullptr; ln.b1 = nullptr;
  ln.w2 = c->bwf(0, F_FF1_LN_W); ln.b2 = c->bwf(0, F_FF1_LN_B);
  ln.y_out = c->x; ln.z_out = c->z; ln.lay = c->lay; ln.compact = 0; ln.eps = 1e-5f;
  return launch_ln(ln, st);
}

}  // namespace

extern "C" int edm_s2a_num_weights(const edm_s2a_config* cfg) {
  if (validate_cfg(cfg)) return EDM_ERR_INVALID;
  return cfg->depth * F_BLOCK_COUNT + G_COUNT;
}

extern "C" const char* edm_s2a_weight_name(const edm_s2a_config* cfg, int index) {
  thread_local char buf[64];
  if (validate_cfg(cfg)) return nullptr;
  const int nb = cfg->depth * F_BLOCK_COUNT;
  if (index < 0 || index >= nb + G_COUNT) return nullptr;
  if (index < nb)
    snprintf(buf, sizeof(buf), "blocks.%d.%s", index / F_BLOCK_COUNT, kBlockFields[index % F_BLOCK_COUNT]);
  else
    snprintf(buf, sizeof(buf), "%s", kGlobalFields[index - nb]);
  return buf;
}

extern "C" edm_s2a_ctx* edm_s2a_create(const edm_s2a_config* cfg, const void* const* weights, int n_weights) {
  if (check_arch()) return nullptr;
  if (validate_cfg(cfg)) return nullptr;
  const int expect = cfg->depth * F_BLOCK_COUNT + G_COUNT;
  if (weights == nullptr || n_weights != expect) {
    fail(EDM_ERR_INVALID, "expected %d weight pointers, got %d", expect, n_weights);
    return nullptr;
  }
  for (int i = 0; i < expect; ++i)
    if (weights[i] == nullptr) {
      fail(EDM_ERR_INVALID, "weight %s is null", edm_s2a_weight_name(cfg, i));
      return nullptr;
    }
  edm_s2a_ctx* c = new edm_s2a_ctx();
  c->cfg = *cfg;
  c->w.assign(weights, weights + expect);
  c->n_fine = cfg->num_quantizers - cfg->n_injection;
  c->bmaps.resize(cfg->depth);
  int rc = 0;
  for (int l = 0; l < cfg->depth && rc == 0; ++l) {
    BlockMaps& m = c->bmaps[l];
    rc = rc ? rc : make_wmap(&m.ff1_w1, c->bw(l, F_FF1_W1), 4096, 1024, 1024);
    rc = rc ? rc : make_wmap(&m.ff1_w2, c->bw(l, F_FF1_W2), 1024, 4096, 4096);
    rc = rc ? rc : make_wmap(&m.wqkv, c->bw(l, F_WQKV), 3072, 1024, 1024);
    rc = rc ? rc : make_wmap(&m.wo, c->bw(l, F_WO), 1024, 1024, 1024);
    rc = rc ? rc : make_wmap(&m.pw1, c->bw(l, F_PW1_W), 4096, 1024, 1024);
    rc = rc ? rc : make_wmap(&m.pw2, c->bw(l, F_PW2_W), 1024, 2048, 2048);
    rc = rc ? rc : make_wmap(&m.ff2_w1, c->bw(l, F_FF2_W1), 4096, 1024, 1024);
    rc = rc ? rc : make_wmap(&m.ff2_w2, c->bw(l, F_FF2_W2), 1024, 4096, 4096);
  }
  rc = rc ? rc : make_wmap(&c->head_map, c->gw(G_HEAD_W), static_cast<uint64_t>(cfg->num_quantizers) * 1024, 1024, 1024);
  rc = rc ? rc : make_wmap(&c->fine_map, c->gw(G_FINE_W), static_cast<uint64_t>(c->n_fine) * 1024, 1024, 1024);
  if (rc) {
    delete c;
    return nullptr;
  }
  return c;
}

extern "C" void edm_s2a_destroy(edm_s2a_ctx* ctx) { delete ctx; }

namespace {
struct Carver {
  uint8_t* base;
  size_t off = 0;
  template <typename T>
  T* take(size_t count) {
    off = align_up(off, 1024);
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += count * sizeof(T);
    return p;
  }
};

constexpr size_t kSplitMaxRows = 1024;  // choose_splits never splits beyond 4 row tiles (148 SMs / 16 column tiles / 2)
// n_seq sequences, M encoder rows, Mt target rows, Mp prompt rows; layout_ints: ints of the varlen layout arrays (0 for a uniform bind)
size_t carve(edm_s2a_ctx* c, uint8_t* base, int B, size_t M, size_t Mt, size_t Mp, size_t layout_ints, bool assign) {
  const int nf = c->n_fine;
  Carver k{base};
  float* x_in = k.take<float>(M * 1024);
  float* x = k.take<float>(M * 1024);
  float* co[4];
  for (int i = 0; i < 4; ++i) co[i] = k.take<float>(M * 1024);
  __nv_bfloat16* z = k.take<__nv_bfloat16>(M * 1024);
  __nv_bfloat16* h = k.take<__nv_bfloat16>(M * 4096);
  __nv_bfloat16* qkv = k.take<__nv_bfloat16>(M * 3072);
  __nv_bfloat16* g = k.take<__nv_bfloat16>(M * 2048);
  __nv_bfloat16* zt = k.take<__nv_bfloat16>(Mt * 1024);
  float* logits = k.take<float>(Mt * 1024);
  // the [B, 12, T, 1024] logits exist only when a caller asks for them (1.5 GB at the bench shape); the decode keeps 64-column partial arg-maxes
  float* coarse_logits = c->keep_logits ? k.take<float>(4 * Mt * 1024) : nullptr;
  __nv_bfloat16* fine_h = k.take<__nv_bfloat16>(Mt * nf * 1024);
  __nv_bfloat16* fine_z = k.take<__nv_bfloat16>(Mt * nf * 1024);
  float* fine_logits = c->keep_logits ? k.take<float>(Mt * nf * 1024) : nullptr;
  float2* arg_part = k.take<float2>(Mt * nf * 16);
  float* logp = k.take<float>(Mt);
  int* ids = k.take<int>(Mt);
  int* ids_raw = k.take<int>(Mt);
  int* pred = k.take<int>(Mt * 4);
  int* pred_raw = k.take<int>(Mt * 4);
  int* fine_codes = k.take<int>(Mt * nf);
  int* sem_tokens = k.take<int>(Mt);
  int* sem_prompt = k.take<int>(Mp > 0 ? Mp : static_cast<size_t>(B));
  int* ac_prompt = k.take<int>(12 * (Mp > 0 ? Mp : static_cast<size_t>(B)));
  uint8_t* mask_a = k.take<uint8_t>(Mt);
  uint8_t* mask_b = k.take<uint8_t>(Mt);
  uint8_t* mask_raw = k.take<uint8_t>(Mt);
  float* part = M <= kSplitMaxRows ? k.take<float>(4 * M * 1024) : nullptr;
  int* layout = layout_ints > 0 ? k.take<int>(layout_ints) : nullptr;
  if (assign) {
    c->layout_dev = layout;
    c->part = part;
    c->x_in = x_in; c->x = x;
    for (int i = 0; i < 4; ++i) c->coarse_out[i] = co[i];
    c->z = z; c->h = h; c->qkv = qkv; c->g = g; c->zt = zt; c->logits = logits; c->coarse_logits = coarse_logits;
    c->fine_h = fine_h; c->fine_z = fine_z; c->fine_logits = fine_logits; c->arg_part = arg_part; c->logp = logp; c->ids = ids; c->ids_raw = ids_raw;
    c->pred_codes = pred; c->pred_raw = pred_raw; c->fine_codes = fine_codes; c->sem_tokens = sem_tokens; c->sem_prompt = sem_prompt;
    c->ac_prompt = ac_prompt; c->mask_a = mask_a; c->mask_b = mask_b; c->mask_raw = mask_raw;
  }
  return align_up(k.off, 1024);
}


// Lengths of a varlen bind: checked per sequence against the limits of a uniform bind; totals and the attention pair count out
int varlen_shape(const edm_s2a_ctx* c, int n_seq, const int* T, const int* P, size_t* M, size_t* Mt, size_t* Mp, int* n_pairs) {
  if (c == nullptr || n_seq <= 0 || n_seq >= (1 << 15) || T == nullptr) return fail(EDM_ERR_INVALID, "bind_varlen arguments (n_seq=%d)", n_seq);
  size_t m = 0, mt = 0, mp = 0;
  long long pairs = 0;
  for (int i = 0; i < n_seq; ++i) {
    const int t = T[i], pl = P != nullptr ? P[i] : 0;
    if (t <= 0 || pl < 0) return fail(EDM_ERR_INVALID, "sequence %d: T=%d P=%d", i, t, pl);
    if (t > kRemaskMaxT) return fail(EDM_ERR_INVALID, "sequence %d: T=%d exceeds %d", i, t, kRemaskMaxT);
    if (static_cast<long long>(pl) + t > c->cfg.max_positions) return fail(EDM_ERR_INVALID, "sequence %d: P+T=%lld exceeds rotary table (%d)", i, static_cast<long long>(pl) + t, c->cfg.max_positions);
    m += static_cast<size_t>(pl) + t;
    mt += t;
    mp += pl;
    pairs += (pl + t + 255) / 256;
  }
  if (m > 0x7fffffffull / 16) return fail(EDM_ERR_INVALID, "bind_varlen: %zu rows", m);
  *M = m; *Mt = mt; *Mp = mp; *n_pairs = static_cast<int>(pairs);
  return 0;
}
}  // namespace

extern "C" size_t edm_s2a_workspace_bytes(const edm_s2a_ctx* ctx, int B, int T, int P) {
  if (ctx == nullptr || B <= 0 || T <= 0 || P < 0) return 0;
  const size_t N = static_cast<size_t>(P) + T;
  return carve(const_cast<edm_s2a_ctx*>(ctx), nullptr, B, B * N, static_cast<size_t>(B) * T, static_cast<size_t>(B) * P, 0, false);
}

extern "C" size_t edm_s2a_workspace_bytes_varlen(const edm_s2a_ctx* ctx, int n_seq, const int* T, const int* P) {
  size_t M, Mt, Mp;
  int n_pairs;
  if (varlen_shape(ctx, n_seq, T, P, &M, &Mt, &Mp, &n_pairs)) return 0;
  return carve(const_cast<edm_s2a_ctx*>(ctx), nullptr, n_seq, M, Mt, Mp, 3 * (static_cast<size_t>(n_seq) + 1) + n_pairs, false);
}

extern "C" int edm_s2a_bind(edm_s2a_ctx* c, void* workspace, size_t bytes, int B, int T, int P) {
  if (c == nullptr || workspace == nullptr || B <= 0 || T <= 0 || P < 0) return fail(EDM_ERR_INVALID, "bind arguments");
  if (T > kRemaskMaxT) return fail(EDM_ERR_INVALID, "T=%d exceeds %d", T, kRemaskMaxT);
  if (P + T > c->cfg.max_positions) return fail(EDM_ERR_INVALID, "P+T=%d exceeds rotary table (%d)", P + T, c->cfg.max_positions);
  if ((reinterpret_cast<uintptr_t>(workspace) & 1023) != 0) return fail(EDM_ERR_INVALID, "workspace must be 1024-byte aligned");
  const size_t N = static_cast<size_t>(P) + T;
  const size_t need = carve(c, nullptr, B, B * N, static_cast<size_t>(B) * T, static_cast<size_t>(B) * P, 0, false);
  if (bytes < need) return fail(EDM_ERR_INVALID, "workspace too small: %zu < %zu", bytes, need);
  carve(c, static_cast<uint8_t*>(workspace), B, B * N, static_cast<size_t>(B) * T, static_cast<size_t>(B) * P, 0, true);
  c->ws = static_cast<uint8_t*>(workspace); c->ws_bytes = bytes;
  c->B = B; c->T = T; c->P = P; c->N = P + T; c->M = B * (P + T); c->Mt = B * T; c->Mp = B * P; c->max_n = P + T; c->min_t = T;
  c->varlen = false; c->lay = uniform_layout(B, P + T, T); c->pairs = nullptr; c->n_pairs = 0; c->conv_runs = ConvRuns();
  c->attn_flops = 4.0 * B * 16 * static_cast<double>(c->N) * c->N * 64;
  c->host_layout.clear();
  c->prompt_proj = nullptr;
  int rc = 0;
  rc = rc ? rc : make_tmap_2d(&c->m_z, c->z, c->M, 1024, 1024, kGemmBM);
  rc = rc ? rc : make_tmap_2d(&c->m_h, c->h, c->M, 4096, 4096, kGemmBM);
  rc = rc ? rc : make_tmap_2d(&c->m_g, c->g, c->M, 2048, 2048, kGemmBM);
  rc = rc ? rc : make_tmap_2d(&c->m_zt, c->zt, c->Mt, 1024, 1024, kGemmBM);
  rc = rc ? rc : make_tmap_2d(&c->m_fine_z, c->fine_z, c->Mt, static_cast<uint64_t>(c->n_fine) * 1024, static_cast<uint64_t>(c->n_fine) * 1024, kGemmBM);
  rc = rc ? rc : make_tmap_2d(&c->m_qkv, c->qkv, c->M, 3072, 3072, 128);
  if (rc) return rc;
  c->bound = true;
  return 0;
}

extern "C" int edm_s2a_bind_varlen(edm_s2a_ctx* c, void* workspace, size_t bytes, int n_seq, const int* T, const int* P, void* stream) {
  if (c == nullptr || workspace == nullptr) return fail(EDM_ERR_INVALID, "bind arguments");
  if ((reinterpret_cast<uintptr_t>(workspace) & 1023) != 0) return fail(EDM_ERR_INVALID, "workspace must be 1024-byte aligned");
  size_t M, Mt, Mp;
  int n_pairs;
  if (int rc = varlen_shape(c, n_seq, T, P, &M, &Mt, &Mp, &n_pairs)) return rc;
  const size_t n1 = static_cast<size_t>(n_seq) + 1, layout_ints = 3 * n1 + n_pairs;
  const size_t need = carve(c, nullptr, n_seq, M, Mt, Mp, layout_ints, false);
  if (bytes < need) return fail(EDM_ERR_INVALID, "workspace too small: %zu < %zu", bytes, need);
  c->bound = false;
  carve(c, static_cast<uint8_t*>(workspace), n_seq, M, Mt, Mp, layout_ints, true);
  int* dev = c->layout_dev;
  // host image of the layout arrays: cu_n | cu_t | cu_runs | pairs
  std::vector<int> lens(n_seq);
  std::vector<int>& h = c->host_layout;
  h.assign(3 * n1, 0);
  int max_n = 0, min_t = kRemaskMaxT;
  double flops = 0.0;
  for (int i = 0; i < n_seq; ++i) {
    const int pl = P != nullptr ? P[i] : 0;
    lens[i] = pl + T[i];
    h[i + 1] = h[i] + lens[i];
    h[n1 + i + 1] = h[n1 + i] + T[i];
    max_n = std::max(max_n, lens[i]);
    min_t = std::min(min_t, T[i]);
    flops += 4.0 * 16 * static_cast<double>(lens[i]) * lens[i] * 64;
  }
  const int run_len = conv_run_len(n_seq, lens.data(), 0, num_sms());
  for (int i = 0; i < n_seq; ++i) h[2 * n1 + i + 1] = h[2 * n1 + i] + (lens[i] + run_len - 1) / run_len;
  append_attention_pairs(lens, &h);
  EDM_CUDA(cudaMemcpyAsync(dev, h.data(), layout_ints * sizeof(int), cudaMemcpyHostToDevice, static_cast<cudaStream_t>(stream)));
  c->ws = static_cast<uint8_t*>(workspace); c->ws_bytes = bytes;
  c->B = n_seq; c->T = 0; c->P = 0; c->N = 0;
  c->M = static_cast<int>(M); c->Mt = static_cast<int>(Mt); c->Mp = static_cast<int>(Mp); c->max_n = max_n; c->min_t = min_t;
  c->varlen = true;
  c->lay.n_seq = n_seq; c->lay.N = 0; c->lay.T = 0; c->lay.cu_n = dev; c->lay.cu_t = dev + n1; c->lay.rows = c->M; c->lay.t_rows = c->Mt;
  c->conv_runs.run_len = run_len; c->conv_runs.cu_runs = dev + 2 * n1; c->conv_runs.num_units = h[2 * n1 + n_seq];
  c->pairs = dev + 3 * n1; c->n_pairs = n_pairs;
  c->attn_flops = flops;
  c->prompt_proj = nullptr;
  int rc = 0;
  rc = rc ? rc : make_tmap_2d(&c->m_z, c->z, c->M, 1024, 1024, kGemmBM);
  rc = rc ? rc : make_tmap_2d(&c->m_h, c->h, c->M, 4096, 4096, kGemmBM);
  rc = rc ? rc : make_tmap_2d(&c->m_g, c->g, c->M, 2048, 2048, kGemmBM);
  rc = rc ? rc : make_tmap_2d(&c->m_zt, c->zt, c->Mt, 1024, 1024, kGemmBM);
  rc = rc ? rc : make_tmap_2d(&c->m_fine_z, c->fine_z, c->Mt, static_cast<uint64_t>(c->n_fine) * 1024, static_cast<uint64_t>(c->n_fine) * 1024, kGemmBM);
  rc = rc ? rc : make_tmap_2d(&c->m_qkv, c->qkv, c->M, 3072, 3072, 128);
  if (rc) return rc;
  c->bound = true;
  return 0;
}

extern "C" void* edm_s2a_buffer(edm_s2a_ctx* c, const char* name, size_t* bytes) {
  if (c == nullptr || !c->bound || name == nullptr) return nullptr;
  const size_t M = c->M, Mt = c->Mt;
  struct { const char* n; void* p; size_t b; } tab[] = {
      {"x_in", c->x_in, M * 1024 * 4}, {"x", c->x, M * 1024 * 4}, {"z", c->z, M * 1024 * 2}, {"h", c->h, M * 4096 * 2},
      {"qkv", c->qkv, M * 3072 * 2}, {"g", c->g, M * 2048 * 2}, {"zt", c->zt, Mt * 1024 * 2},
      {"coarse_out0", c->coarse_out[0], M * 1024 * 4}, {"coarse_out1", c->coarse_out[1], M * 1024 * 4},
      {"coarse_out2", c->coarse_out[2], M * 1024 * 4}, {"coarse_out3", c->coarse_out[3], M * 1024 * 4},
      {"logits", c->logits, Mt * 1024 * 4}, {"coarse_logits", c->coarse_logits, c->keep_logits ? 4 * Mt * 1024 * 4 : 0},
      {"fine_logits", c->fine_logits, c->keep_logits ? Mt * c->n_fine * 1024 * 4 : 0}, {"logp", c->logp, Mt * 4}, {"ids", c->ids, Mt * 4},
      {"ids_raw", c->ids_raw, Mt * 4}, {"pred_codes", c->pred_codes, Mt * 16}, {"pred_raw", c->pred_raw, Mt * 16},
      {"fine_codes", c->fine_codes, Mt * c->n_fine * 4}, {"mask", c->mask_cur(), Mt}, {"mask_raw", c->mask_raw, Mt}};
  for (auto& e : tab)
    if (strcmp(e.n, name) == 0) {
      if (bytes) *bytes = e.b;
      return e.p;
    }
  return nullptr;
}

extern "C" int edm_s2a_build_input(edm_s2a_ctx* c, const int* sem_tokens, const int* sem_prompt, const int* ac_prompt, int ac_levels, void* stream) {
  if (c == nullptr || !c->bound) return fail(EDM_ERR_STATE, "context not bound");
  PdlScope pdl(c->M <= kPdlMaxRows);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (sem_tokens == nullptr) return fail(EDM_ERR_INVALID, "semantic tokens required");
  if (c->Mp > 0) {
    if (sem_prompt == nullptr || ac_prompt == nullptr) return fail(EDM_ERR_INVALID, "bound with %d prompt frames but no prompt given", c->Mp);
    if (ac_levels < c->cfg.n_injection || ac_levels > 12) return fail(EDM_ERR_INVALID, "acoustic prompt needs >= %d levels (got %d)", c->cfg.n_injection, ac_levels);
    EDM_CUDA(cudaMemcpyAsync(c->sem_prompt, sem_prompt, sizeof(int) * c->Mp, cudaMemcpyDeviceToDevice, st));
    EDM_CUDA(cudaMemcpyAsync(c->ac_prompt, ac_prompt, sizeof(int) * ac_levels * static_cast<size_t>(c->Mp), cudaMemcpyDeviceToDevice, st));
  }
  c->ac_levels = ac_levels;
  EDM_CUDA(cudaMemcpyAsync(c->sem_tokens, sem_tokens, sizeof(int) * c->Mt, cudaMemcpyDeviceToDevice, st));
  BuildInputParams p;
  p.x = c->x_in; p.sem_tokens = c->sem_tokens; p.sem_prompt = c->Mp > 0 ? c->sem_prompt : nullptr; p.ac_prompt = c->Mp > 0 ? c->ac_prompt : nullptr;
  p.ac_prompt_levels = ac_levels; p.sem_emb = c->gwf(G_SEM_EMB); p.mask_token = c->gwf(G_MASK_TOKEN); p.feat_table = c->gwf(G_FEAT_TABLE);
  p.feat_const = c->gwf(G_FEAT_CONST); p.fp_ln_w = c->gwf(G_FP_LN_W); p.fp_ln_b = c->gwf(G_FP_LN_B); p.lay = c->lay; p.rows = c->M; p.eps = 1e-5f;
  p.num_semantic = c->cfg.num_semantic;
  launch_pdl(build_input_kernel, dim3((c->M + 7) / 8), dim3(256), 0, st, p);
  EDM_LAUNCH_CHECK("build_input");
  c->mask_in_a = true;
  launch_pdl(fill_u8_kernel, dim3((c->Mt + 255) / 256), dim3(256), 0, st, c->mask_a, c->Mt, 1);
  EDM_LAUNCH_CHECK("fill_mask");
  return 0;
}

extern "C" int edm_s2a_first_level(edm_s2a_ctx* c, const float* x_in, void* stream) {
  if (c == nullptr || !c->bound) return fail(EDM_ERR_STATE, "context not bound");
  PdlScope pdl(c->M <= kPdlMaxRows);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int rc = pass_prologue(c, x_in ? x_in : c->x_in, st)) return rc;
  const int last = c->cfg.injection_layers[0];
  for (int l = 0; l <= last; ++l) {
    LnParams ln;
    ln.in = c->x; ln.in_is_bf16 = 0; ln.rows = c->M; ln.w1 = c->bwf(l, F_POST_LN_W); ln.b1 = c->bwf(l, F_POST_LN_B); ln.eps = 1e-5f;
    if (l < last) {
      ln.w2 = c->bwf(l + 1, F_FF1_LN_W); ln.b2 = c->bwf(l + 1, F_FF1_LN_B);
      ln.y_out = c->x; ln.z_out = c->z; ln.lay = c->lay; ln.compact = 0;
    } else {
      ln.w2 = c->gwf(G_TL_LN_W); ln.b2 = c->gwf(G_TL_LN_B);
      ln.y_out = nullptr; ln.z_out = c->zt; ln.lay = c->lay; ln.compact = c->Mp > 0;
    }
    if (int rc = run_block_body(c, l, ln, st)) return rc;
  }
  GemmParams p = gp(c->Mt, 1024, 1024, c->gwf(G_HEAD_B), c->logits, 1024);
  return launch_gemm(EPI_F32, c->m_zt, c->head_map, p, st);
}

extern "C" int edm_s2a_set_keep_logits(edm_s2a_ctx* c, int keep) {
  if (c == nullptr) return fail(EDM_ERR_INVALID, "null context");
  if ((keep != 0) != c->keep_logits) c->bound = false;  // the workspace layout changes: bind again
  c->keep_logits = keep != 0;
  return 0;
}

extern "C" int edm_s2a_set_low_latency(edm_s2a_ctx* c, int on) {
  if (c == nullptr) return fail(EDM_ERR_INVALID, "null context");
  c->low_latency = on != 0;
  return 0;
}

extern "C" int edm_s2a_set_prompt_injections(edm_s2a_ctx* c, const float* proj) {
  if (c == nullptr) return fail(EDM_ERR_INVALID, "null context");
  if (c->varlen && proj != nullptr) return fail(EDM_ERR_STATE, "feature-valued prompt injections need a uniform bind (edm_s2a_bind)");
  c->prompt_proj = proj;
  return 0;
}

extern "C" int edm_s2a_set_seed_buffer(edm_s2a_ctx* c, const unsigned long long* seed_dev) {
  if (c == nullptr) return fail(EDM_ERR_INVALID, "null context");
  c->seed_dev = seed_dev;
  return 0;
}

extern "C" int edm_s2a_set_batch_offset(edm_s2a_ctx* c, long long batch_offset) {
  if (c == nullptr || batch_offset < 0) return fail(EDM_ERR_INVALID, "batch offset");
  c->batch_offset = batch_offset;
  return 0;
}

extern "C" int edm_s2a_step(edm_s2a_ctx* c, int step, int steps, float temperature, unsigned long long seed, const float* cat_noise,
                            const float* remask_noise, const int* forced_ids, const uint8_t* forced_mask, void* stream) {
  if (c == nullptr || !c->bound) return fail(EDM_ERR_STATE, "context not bound");
  if (steps < 2 || step < 0 || step >= steps) return fail(EDM_ERR_INVALID, "step %d of %d", step, steps);
  PdlScope pdl(c->M <= kPdlMaxRows);
  // the reference's take_along_dim(sorted_confidence, mask_len >= 1) is out of range for a single frame (utils/utils.py:56)
  if (c->min_t < 2 && step < steps - 1 && forced_mask == nullptr) return fail(EDM_ERR_INVALID, "re-masking needs T >= 2 frames (T=%d, steps=%d)", c->min_t, steps);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool last = step == steps - 1;
  SampleParams sp;
  sp.logits = c->logits; sp.ld = 1024; sp.rows = c->Mt; sp.noise = last ? nullptr : cat_noise; sp.use_philox = last ? 0 : 1; sp.seed = seed; sp.seed_dev = c->seed_dev;
  sp.step = static_cast<unsigned>(step); sp.seq0 = c->batch_offset; sp.forced_ids = forced_ids; sp.ids = c->ids; sp.ids_raw = c->ids_raw; sp.logp = last ? nullptr : c->logp;
  sp.lay = c->lay; sp.Q = 1; sp.out_q_stride = 1; sp.out_q0 = 0;
  if (int rc = launch_sample(sp, st)) return rc;
  uint8_t* m_old = c->mask_cur();
  uint8_t* m_new = nullptr;
  if (!last) {
    // python: mask_ratio is a double; torch multiplies float32 tensors by float32(ratio)
    const double ratio_d = std::cos(M_PI / 2.0 * (static_cast<double>(step + 1) / static_cast<double>(steps)));
    RemaskParams rp;
    rp.logp = c->logp; rp.gumbel = remask_noise; rp.mask_old = m_old; rp.mask_new = c->mask_next(); rp.mask_raw = c->mask_raw; rp.forced_mask = forced_mask;
    rp.lay = c->lay; rp.init_count = 0; rp.init_counts = nullptr; rp.ratio = static_cast<float>(ratio_d); rp.temp_ratio = static_cast<float>(static_cast<double>(temperature) * ratio_d);
    rp.seed = seed; rp.seed_dev = c->seed_dev; rp.step = static_cast<unsigned>(step); rp.seq0 = c->batch_offset;
    launch_pdl(remask_kernel, dim3(c->lay.n_seq), dim3(256), 0, st, rp);
    EDM_LAUNCH_CHECK("remask");
    m_new = c->mask_next();
  }
  UpdateInputParams up;
  up.x = c->x_in; up.sem_tokens = c->sem_tokens; up.ids = c->ids; up.mask_old = m_old; up.mask_new = m_new; up.sem_emb = c->gwf(G_SEM_EMB);
  up.mask_token = c->gwf(G_MASK_TOKEN); up.feat_table = c->gwf(G_FEAT_TABLE); up.feat_const = c->gwf(G_FEAT_CONST);
  up.fp_ln_w = c->gwf(G_FP_LN_W); up.fp_ln_b = c->gwf(G_FP_LN_B); up.lay = c->lay; up.rows = c->Mt; up.eps = 1e-5f; up.num_semantic = c->cfg.num_semantic;
  launch_pdl(update_input_kernel, dim3((c->Mt + 7) / 8), dim3(256), 0, st, up);
  EDM_LAUNCH_CHECK("update_input");
  if (!last) c->mask_in_a = !c->mask_in_a;
  return 0;
}

extern "C" int edm_s2a_full_pass(edm_s2a_ctx* c, const float* x_in, const int* forced_coarse, long long* codes_out, void* stream) {
  if (c == nullptr || !c->bound) return fail(EDM_ERR_STATE, "context not bound");
  PdlScope pdl(c->M <= kPdlMaxRows);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const edm_s2a_config& cfg = c->cfg;
  if (int rc = pass_prologue(c, x_in ? x_in : c->x_in, st)) return rc;
  for (int l = 0; l < cfg.depth; ++l) {
    const int k = injection_index(cfg, l);
    const bool is_last = l == cfg.depth - 1;
    LnParams ln;
    ln.in = c->x; ln.in_is_bf16 = 0; ln.rows = c->M; ln.w1 = c->bwf(l, F_POST_LN_W); ln.b1 = c->bwf(l, F_POST_LN_B); ln.eps = 1e-5f;
    if (k < 0) {
      if (!is_last) {
        ln.w2 = c->bwf(l + 1, F_FF1_LN_W); ln.b2 = c->bwf(l + 1, F_FF1_LN_B); ln.y_out = c->x; ln.z_out = c->z; ln.lay = c->lay; ln.compact = 0;
      } else {
        ln.w2 = nullptr; ln.b2 = nullptr; ln.y_out = nullptr; ln.z_out = c->zt; ln.lay = c->lay; ln.compact = c->Mp > 0;  // bf16 copy of the target rows
      }
      if (int rc = run_block_body(c, l, ln, st)) return rc;
      continue;
    }
    // injection layer k: keep the block output, predict level k on the target rows, inject
    ln.w2 = c->gwf(G_TL_LN_W); ln.b2 = c->gwf(G_TL_LN_B); ln.y_out = c->coarse_out[k]; ln.z_out = c->zt; ln.lay = c->lay; ln.compact = c->Mp > 0;
    if (int rc = run_block_body(c, l, ln, st)) return rc;
    if (c->keep_logits) {
      float* lk = c->coarse_logits + static_cast<size_t>(k) * c->Mt * 1024;
      GemmParams p = gp(c->Mt, 1024, 1024, c->gwf(G_HEAD_B) + k * 1024, lk, 1024);
      p.b_row_offset = k * 1024;
      if (int rc = launch_gemm(EPI_F32, c->m_zt, c->head_map, p, st)) return rc;
      SampleParams sp;
      sp.logits = lk; sp.ld = 1024; sp.rows = c->Mt; sp.noise = nullptr; sp.use_philox = 0; sp.seed = 0; sp.seed_dev = nullptr; sp.step = 0; sp.seq0 = 0; sp.forced_ids = forced_coarse;
      sp.ids = c->pred_codes; sp.ids_raw = c->pred_raw; sp.logp = nullptr; sp.lay = c->lay; sp.Q = 1; sp.out_q_stride = 4; sp.out_q0 = k;
      if (int rc = launch_sample(sp, st)) return rc;
    } else {
      // head k with the arg-max in the GEMM epilogue: 16 (max, index) partials per row instead of 1024 fp32 logits
      GemmParams p = gp(c->Mt, 1024, 1024, c->gwf(G_HEAD_B) + k * 1024, c->arg_part, 16);
      p.b_row_offset = k * 1024;
      if (int rc = launch_gemm(EPI_ARGMAX, c->m_zt, c->head_map, p, st)) return rc;
      ArgmaxCombineParams ap;
      ap.part = c->arg_part; ap.rows = c->Mt; ap.parts = 16; ap.forced_ids = forced_coarse; ap.ids = c->pred_codes; ap.ids_raw = c->pred_raw;
      ap.lay = c->lay; ap.Q = 1; ap.out_q_stride = 4; ap.out_q0 = k;
      launch_pdl(argmax_combine_kernel, dim3((c->Mt + 255) / 256), dim3(256), 0, st, ap);
      EDM_LAUNCH_CHECK("argmax_combine");
    }
    InjectParams ip;
    ip.x = c->x; ip.cur_out = c->coarse_out[k]; ip.prev_out = (k > 0 && cfg.residual) ? c->coarse_out[k - 1] : nullptr;
    ip.pred_codes = c->pred_codes; ip.ac_prompt = c->Mp > 0 ? c->ac_prompt : nullptr; ip.ac_prompt_levels = c->ac_levels;
    ip.prompt_proj = (c->Mp > 0 && c->prompt_proj != nullptr) ? c->prompt_proj + static_cast<size_t>(k) * c->Mp * 1024 : nullptr;
    for (int i = 0; i < 4; ++i) ip.tables[i] = c->gwf(G_INJ_TABLE) + (static_cast<size_t>(k) * 4 + i) * 1024 * 1024;
    ip.inj_const = c->gwf(G_INJ_CONST) + k * 1024; ip.ln_w = c->gwf(G_INJ_LN_W) + k * 1024; ip.ln_b = c->gwf(G_INJ_LN_B) + k * 1024;
    ip.level = k; ip.lay = c->lay; ip.rows = c->M; ip.eps = 1e-5f;
    launch_pdl(inject_kernel, dim3((c->M + 7) / 8), dim3(256), 0, st, ip);
    EDM_LAUNCH_CHECK("inject");
    LnParams nx;
    nx.in = c->x; nx.in_is_bf16 = 0; nx.rows = c->M; nx.w1 = nullptr; nx.b1 = nullptr; nx.eps = 1e-5f; nx.y_out = nullptr;
    if (!is_last) {
      nx.w2 = c->bwf(l + 1, F_FF1_LN_W); nx.b2 = c->bwf(l + 1, F_FF1_LN_B); nx.z_out = c->z; nx.lay = c->lay; nx.compact = 0;
    } else {
      nx.w2 = nullptr; nx.b2 = nullptr; nx.z_out = c->zt; nx.lay = c->lay; nx.compact = c->Mp > 0;
    }
    if (int rc = launch_ln(nx, st)) return rc;
  }
  // fine levels: fine_head (wrapper :38-41) -> per-(token, level) LayerNorm -> per-codebook heads (:43-54)
  const int nf = c->n_fine;
  if (int rc = launch_gemm(EPI_BF16, c->m_zt, c->fine_map, gp(c->Mt, nf * 1024, 1024, c->gwf(G_FINE_B), c->fine_h, static_cast<long long>(nf) * 1024), st)) return rc;
  {
    LnParams ln;
    ln.in = c->fine_h; ln.in_is_bf16 = 1; ln.rows = c->Mt * nf; ln.w1 = c->gwf(G_TL_LN_W); ln.b1 = c->gwf(G_TL_LN_B); ln.w2 = nullptr; ln.b2 = nullptr;
    ln.y_out = nullptr; ln.z_out = c->fine_z; ln.lay = c->lay; ln.compact = 0; ln.eps = 1e-5f;
    if (int rc = launch_ln(ln, st)) return rc;
  }
  for (int q = 0; q < nf; ++q) {
    const int lvl = cfg.n_injection + q;
    if (c->keep_logits) {
      GemmParams p = gp(c->Mt, 1024, 1024, c->gwf(G_HEAD_B) + lvl * 1024, c->fine_logits + q * 1024, static_cast<long long>(nf) * 1024);
      p.a_k_offset = q * 1024; p.b_row_offset = lvl * 1024;
      if (int rc = launch_gemm(EPI_F32, c->m_fine_z, c->head_map, p, st)) return rc;
    } else {
      // partials of (token, level q) at arg_part[(token * nf + q) * 16 ..]: row pitch nf * 16, level offset q * 16
      GemmParams p = gp(c->Mt, 1024, 1024, c->gwf(G_HEAD_B) + lvl * 1024, c->arg_part + q * 16, static_cast<long long>(nf) * 16);
      p.a_k_offset = q * 1024; p.b_row_offset = lvl * 1024;
      if (int rc = launch_gemm(EPI_ARGMAX, c->m_fine_z, c->head_map, p, st)) return rc;
    }
  }
  if (c->keep_logits) {
    SampleParams sp;
    sp.logits = c->fine_logits; sp.ld = 1024; sp.rows = c->Mt * nf; sp.noise = nullptr; sp.use_philox = 0; sp.seed = 0; sp.seed_dev = nullptr; sp.step = 0; sp.seq0 = 0; sp.forced_ids = nullptr;
    sp.ids = c->fine_codes; sp.ids_raw = nullptr; sp.logp = nullptr; sp.lay = c->lay; sp.Q = nf; sp.out_q_stride = nf; sp.out_q0 = 0;
    if (int rc = launch_sample(sp, st)) return rc;
  } else {
    ArgmaxCombineParams ap;
    ap.part = c->arg_part; ap.rows = c->Mt * nf; ap.parts = 16; ap.forced_ids = nullptr; ap.ids = c->fine_codes; ap.ids_raw = nullptr;
    ap.lay = c->lay; ap.Q = nf; ap.out_q_stride = nf; ap.out_q0 = 0;
    launch_pdl(argmax_combine_kernel, dim3((c->Mt * nf + 255) / 256), dim3(256), 0, st, ap);
    EDM_LAUNCH_CHECK("argmax_combine");
  }
  if (codes_out != nullptr) {
    const long long total = static_cast<long long>(c->Mt) * cfg.num_quantizers;
    launch_pdl(assemble_codes_kernel, dim3(static_cast<unsigned>((total + 255) / 256)), dim3(256), 0, st, c->pred_raw, cfg.n_injection, c->fine_codes, nf, codes_out, c->lay);
    EDM_LAUNCH_CHECK("assemble_codes");
  }
  return 0;
}

extern "C" int edm_s2a_decode(edm_s2a_ctx* c, const int* sem_tokens, const int* sem_prompt, const int* ac_prompt, int ac_levels, int steps,
                              float temperature, unsigned long long seed, const float* cat_noise, const float* remask_noise,
                              const int* forced_ids, const uint8_t* forced_masks, const int* forced_coarse, long long* codes_out, void* stream) {
  if (c == nullptr || !c->bound) return fail(EDM_ERR_STATE, "context not bound");
  if (steps < 1) return fail(EDM_ERR_INVALID, "steps must be >= 1");
  if (int rc = edm_s2a_build_input(c, sem_tokens, sem_prompt, ac_prompt, ac_levels, stream)) return rc;
  if (steps > 1) {
    const size_t Mt = c->Mt;
    for (int s = 0; s < steps; ++s) {
      if (int rc = edm_s2a_first_level(c, nullptr, stream)) return rc;
      const bool last = s == steps - 1;
      if (int rc = edm_s2a_step(c, s, steps, temperature, seed, (cat_noise && !last) ? cat_noise + s * Mt * 1024 : nullptr,
                                (remask_noise && !last) ? remask_noise + s * Mt : nullptr, forced_ids ? forced_ids + s * Mt : nullptr,
                                (forced_masks && !last) ? forced_masks + s * Mt : nullptr, stream))
        return rc;
    }
  }
  return edm_s2a_full_pass(c, nullptr, forced_coarse, codes_out, stream);
}

// ================================================================================================ text-to-semantic context
// TextToSemanticWLen.infer (edm_tts/models/text_to_semantic/modeling_text_to_semantic.py:184-267): length predictor + `pred_iters`
// iterations of (embed -> conformer -> pred_transform -> pred_head -> sample -> re-mask). The reference's infer decodes one sequence;
// edm_t2s_begin does the same, edm_t2s_begin_batch decodes several of different lengths packed back to back (SeqLayout). Hidden sizes 128..1024 in steps of 128, heads of <= 64 dims: the fused QKV projection is packed with every head
// zero-padded to 64 columns (first half of the rotary pair in columns [0, dh/2), second half in [32, 32 + dh/2)), so the GEMM's
// rotary epilogue and the tcgen05 attention kernel of the S2A path run unchanged; only the softmax scale dh^-1/2 differs.
#include "t2s.cuh"

namespace {
const char* const kT2sGlobalFields[] = {"emb", "length_token", "pt_w", "pt_b", "pt_ln_w", "pt_ln_b", "head_w", "head_b",
                                        "len_w", "len_b", "rope_cos", "rope_sin", "lp_rope_cos", "lp_rope_sin"};
enum T2sGlobal { TG_EMB, TG_LENGTH_TOKEN, TG_PT_W, TG_PT_B, TG_PT_LN_W, TG_PT_LN_B, TG_HEAD_W, TG_HEAD_B,
                 TG_LEN_W, TG_LEN_B, TG_ROPE_COS, TG_ROPE_SIN, TG_LP_ROPE_COS, TG_LP_ROPE_SIN, TG_COUNT };
}  // namespace

struct edm_t2s_ctx {
  edm_t2s_config cfg;
  std::vector<const void*> w;      // (depth + lp_depth) * F_BLOCK_COUNT + TG_COUNT; main blocks first, then the length predictor's
  std::vector<BlockMaps> bmaps;
  WMap pt_map, head_map;
  int d = 0, ff = 0, C = 0, hp = 0, lp_hp = 0, hp_max = 0, total_tokens = 0;
  bool low_latency = true;     // edm_t2s_set_low_latency
  long long batch_offset = 0;  // edm_t2s_set_batch_offset
  // bound workspace: max_len rows (all sequences of a request together), at most max_seq sequences
  bool bound = false;
  int max_len = 0, max_seq = 0;
  size_t layout_cap = 0;       // ints of layout_dev
  float *x, *y, *logits, *logp, *raw_len, *part = nullptr;  // part: split-K partial sums, carved by edm_t2s_bind only
  __nv_bfloat16 *z, *h, *qkv, *att, *g, *zt;
  int *ids, *ids_raw, *tokens, *input_ids, *text, *layout_dev;
  uint8_t *full_mask, *mask_a, *mask_b, *mask_raw;
  std::vector<int> host_layout;
  // current pass (length predictor or decode): where its sequences are. A single sequence is a uniform layout without arrays.
  T2sSeqs seqs;
  const int* pairs = nullptr;  // attention items of a packed layout
  int n_pairs = 0, max_n = 0, out_len = 0;
  double sum_sq = 0.0;         // sum of L_s^2 (attention work)
  const int* init_counts = nullptr;  // packed decode: length_s per sequence (re-masking)
  float* part_use = nullptr;   // split-K partials of this pass, nullptr: the unsplit launches
  bool begun = false, mask_in_a = true;
  CUtensorMap m_z, m_h, m_att, m_g, m_zt, m_qkv;

  const void* bw(int blk, int f) const { return w[static_cast<size_t>(blk) * F_BLOCK_COUNT + f]; }
  const float* bwf(int blk, int f) const { return static_cast<const float*>(bw(blk, f)); }
  const void* gw(int f) const { return w[static_cast<size_t>(cfg.depth + cfg.lp_depth) * F_BLOCK_COUNT + f]; }
  const float* gwf(int f) const { return static_cast<const float*>(gw(f)); }
  uint8_t* mask_cur() { return mask_in_a ? mask_a : mask_b; }
  uint8_t* mask_next() { return mask_in_a ? mask_b : mask_a; }
};

namespace {

int t2s_validate(const edm_t2s_config* c) {
  if (c == nullptr) return fail(EDM_ERR_INVALID, "null config");
  const int d = c->hidden;
  if (d != 128 && d != 256 && d != 384 && d != 512 && d != 1024)
    return fail(EDM_ERR_INVALID, "text-to-semantic kernels are built for hidden 128 / 256 / 384 / 512 / 1024 (got %d)", d);
  if (c->ff_mult != 4 || c->conv_kernel != 5) return fail(EDM_ERR_INVALID, "kernels are specialised for ff_mult=4 conv_kernel=5 (got %d %d)", c->ff_mult, c->conv_kernel);
  for (int heads : {c->heads, c->lp_heads}) {
    if (heads < 1 || d % heads != 0) return fail(EDM_ERR_INVALID, "hidden %d is not divisible by %d heads", d, heads);
    const int dh = d / heads;
    if (dh > 64 || dh % 8 != 0) return fail(EDM_ERR_INVALID, "head dim %d unsupported (multiple of 8, <= 64)", dh);
  }
  if (c->depth < 1 || c->depth > 64 || c->lp_depth < 1 || c->lp_depth > 64) return fail(EDM_ERR_INVALID, "unsupported depth");
  if (c->semantic_vocab != 1024) return fail(EDM_ERR_INVALID, "the sampling kernel is built for 1024 semantic tokens (got %d)", c->semantic_vocab);
  if (c->text_vocab < 1 || c->num_special != 5) return fail(EDM_ERR_INVALID, "unsupported vocabulary (text %d, special %d)", c->text_vocab, c->num_special);
  if (c->max_positions < 8 || c->max_positions > kRemaskMaxT) return fail(EDM_ERR_INVALID, "max_positions must be in [8, %d]", kRemaskMaxT);
  return 0;
}

int launch_ln_g(int d, const LnGParams& p, cudaStream_t st) {
  if (p.rows <= 0) return 0;
  const int grid = (p.rows + 7) / 8;
  switch (d) {
    case 128: launch_pdl(layernorm_g_kernel<1>, dim3(grid), dim3(256), 0, st, p); break;
    case 256: launch_pdl(layernorm_g_kernel<2>, dim3(grid), dim3(256), 0, st, p); break;
    case 384: launch_pdl(layernorm_g_kernel<3>, dim3(grid), dim3(256), 0, st, p); break;
    case 512: launch_pdl(layernorm_g_kernel<4>, dim3(grid), dim3(256), 0, st, p); break;
    case 1024: launch_pdl(layernorm_g_kernel<8>, dim3(grid), dim3(256), 0, st, p); break;
    default: return fail(EDM_ERR_INVALID, "layernorm: hidden %d", d);
  }
  EDM_LAUNCH_CHECK("layernorm_g");
  return 0;
}

// Residual GEMM + the LayerNorm that follows it, text-to-semantic form (any hidden size 128 * NV): with `part` and a K that divides into
// 2 / 4 ranges of >= 4 k-blocks on few enough tiles, split-K partial sums reduced by layernorm_g_splitk_kernel (see launch_gemm_resid_ln);
// otherwise the two plain launches. `part` is given only to a single-sequence pass in low-latency mode (the default): the split changes
// the fp32 summation order, so a packed batch never splits and a row's bits do not depend on the batch it is decoded in.
int launch_gemm_resid_ln_g(int d, const CUtensorMap& ma, const WMap& wm, const GemmParams& p, const LnGParams& ln, float* part, cudaStream_t st) {
  const int sms = num_sms();
  const int tiles = ((p.M + kGemmBM - 1) / kGemmBM) * (p.N / kSmBN), num_kb = p.K / kGemmBK;
  const int pair_tiles = ((p.M + 2 * kGemmBM - 1) / (2 * kGemmBM)) * ((p.N + kGemmBN - 1) / kGemmBN);
  const bool small = p.N % kGemmBN != 0 || (gemm_small_m() && pair_tiles * 4 <= sms);
  int splits = 1;
  if (small && part != nullptr && p.K % kGemmBK == 0 && p.N == d && p.ldo == d && ln.in == p.out && ln.rows == p.M && p.a_k_offset == 0 &&
      ln.gather == nullptr && ln.override_row == nullptr && !ln.pre_gelu && p.K >= 768)
    for (int s = 4; s >= 2 && splits == 1; s >>= 1)
      if (tiles * s <= sms && num_kb % s == 0 && num_kb / s >= 3) splits = s;
  if (splits == 1) {
    if (int rc = launch_gemm(EPI_RESID_F32, ma, wm, p, st)) return rc;
    return launch_ln_g(d, ln, st);
  }
  static DeviceOnce attr_once;
  if (attr_once.needed()) {
    EDM_CUDA(cudaFuncSetAttribute(gemm_bf16_tn_small_kernel<EPI_F32>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmSmemBytes));
    attr_once.done();
  }
  {
    GemmParams q = p;
    q.bias = nullptr; q.out = part; q.ldo = d; q.scale = 1.0f; q.reverse = 0;
    q.splits = splits; q.split_stride = static_cast<long long>(p.M) * d;
    next_direction();
    ProfScope prof(PK_GEMM, 2.0 * p.M * p.N * p.K, st);
    const int work = tiles * splits;
    launch_pdl(gemm_bf16_tn_small_kernel<EPI_F32>, dim3(work < sms ? work : sms), dim3(kSmThreads), kSmSmemBytes, st, ma, wm.small, q);
    EDM_LAUNCH_CHECK("gemm_bf16_tn_small (split-K)");
  }
  LnGParams l = ln;
  l.partials = part; l.n_partials = splits; l.partial_stride = static_cast<long long>(p.M) * d; l.lin_bias = p.bias; l.lin_scale = p.scale;
  l.x_io = static_cast<float*>(p.out);
  const int grid = (l.rows + 7) / 8;
  switch (d) {
    case 128: launch_pdl(layernorm_g_splitk_kernel<1>, dim3(grid), dim3(256), 0, st, l); break;
    case 256: launch_pdl(layernorm_g_splitk_kernel<2>, dim3(grid), dim3(256), 0, st, l); break;
    case 384: launch_pdl(layernorm_g_splitk_kernel<3>, dim3(grid), dim3(256), 0, st, l); break;
    case 512: launch_pdl(layernorm_g_splitk_kernel<4>, dim3(grid), dim3(256), 0, st, l); break;
    case 1024: launch_pdl(layernorm_g_splitk_kernel<8>, dim3(grid), dim3(256), 0, st, l); break;
    default: return fail(EDM_ERR_INVALID, "layernorm: hidden %d", d);
  }
  EDM_LAUNCH_CHECK("layernorm_g_splitk");
  return 0;
}

template <int kC>
int launch_conv_tiled_t(const ConvModParams& p, cudaStream_t st) {
  static DeviceOnce attr_once;
  if (attr_once.needed()) {
    EDM_CUDA((cudaFuncSetAttribute(conv_module_kernel<false, kC>, cudaFuncAttributeMaxDynamicSharedMemorySize, conv_smem_bytes(kC))));
    attr_once.done();
  }
  dim3 grid((p.max_n + kConvTT - 1) / kConvTT, p.lay.n_seq);
  launch_pdl(conv_module_kernel<false, kC>, dim3(grid), dim3(kC / 4), conv_smem_bytes(kC), st, p);
  EDM_LAUNCH_CHECK("conv_module");
  return 0;
}
// gated input [B*N, C] -> depthwise conv, Swish, ChanLayerNorm for C inner channels (tiled kernel; sequences here are a few hundred tokens)
int launch_conv_tiled(int C, const ConvModParams& p, cudaStream_t st) {
  switch (C) {
    case 256: return launch_conv_tiled_t<256>(p, st);
    case 512: return launch_conv_tiled_t<512>(p, st);
    case 768: return launch_conv_tiled_t<768>(p, st);
    case 1024: return launch_conv_tiled_t<1024>(p, st);
    case 2048: return launch_conv_tiled_t<2048>(p, st);
  }
  return fail(EDM_ERR_INVALID, "conv module: %d inner channels", C);
}

LnGParams lng(const void* in, int rows, const float* w1, const float* b1, const float* w2, const float* b2, float* y, __nv_bfloat16* z) {
  LnGParams p;
  p.in = in; p.in_is_bf16 = 0; p.gather = nullptr; p.gather_rows = 0; p.override_row = nullptr; p.rows = rows;
  p.w1 = w1; p.b1 = b1; p.w2 = w2; p.b2 = b2; p.y_out = y; p.z_out = z; p.eps = 1e-5f; p.pre_gelu = 0;
  return p;
}

// tensor maps of the activation buffers for a pass over M rows with padded head width hp
int t2s_maps(edm_t2s_ctx* c, int M, int hp) {
  int rc = 0;
  rc = rc ? rc : make_tmap_2d(&c->m_z, c->z, M, c->d, c->d, kGemmBM);
  rc = rc ? rc : make_tmap_2d(&c->m_h, c->h, M, c->ff, c->ff, kGemmBM);
  rc = rc ? rc : make_tmap_2d(&c->m_att, c->att, M, hp, hp, kGemmBM);
  rc = rc ? rc : make_tmap_2d(&c->m_g, c->g, M, c->C, c->C, kGemmBM);
  rc = rc ? rc : make_tmap_2d(&c->m_zt, c->zt, M, c->d, c->d, kGemmBM);
  rc = rc ? rc : make_tmap_2d(&c->m_qkv, c->qkv, M, 3ull * hp, 3ull * hp, 128);
  return rc;
}

// One ConformerBlock (conformer/conformer.py:219-235) on the rows of the current pass (c->seqs.lay). In: x (fp32 stream), z = LN_ff1(x).
// Out: `post` applied to the block's sum (post_norm + the next block's pre-norm), or x = pre-post_norm sum when post == nullptr (the
// last block of a stack).
int t2s_block_body(edm_t2s_ctx* c, int blk, int H, int hp, const float* rope_cos, const float* rope_sin, const LnGParams* post, cudaStream_t st) {
  const int d = c->d, ff = c->ff, C = c->C;
  const SeqLayout& lay = c->seqs.lay;
  const int M = lay.rows;
  const BlockMaps& bm = c->bmaps[blk];
  if (int rc = launch_gemm(EPI_SWISH_BF16, c->m_z, bm.ff1_w1, gp(M, ff, d, c->bwf(blk, F_FF1_B1), c->h, ff), st)) return rc;
  if (int rc = launch_gemm_resid_ln_g(d, c->m_h, bm.ff1_w2, gp(M, d, ff, c->bwf(blk, F_FF1_B2), c->x, d, 0.5f),
                                      lng(c->x, M, c->bwf(blk, F_ATTN_LN_W), c->bwf(blk, F_ATTN_LN_B), nullptr, nullptr, nullptr, c->z), c->part_use, st)) return rc;
  {
    GemmParams p = gp(M, 3 * hp, d, nullptr, c->qkv, 3 * hp);
    p.rope_cos = rope_cos; p.rope_sin = rope_sin; p.rope_lay = lay; p.rope_cols = 2 * hp;
    if (int rc = launch_gemm(EPI_QKV_ROPE, c->m_z, bm.wqkv, p, st)) return rc;
  }
  const float scale = 1.0f / sqrtf(static_cast<float>(d / H));
  if (int rc = launch_attention(c->m_qkv, lay, c->pairs, c->n_pairs, 4.0 * H * c->sum_sq * 64, H, c->att, 1024, 1024, 2048, st, scale)) return rc;
  if (int rc = launch_gemm_resid_ln_g(d, c->m_att, bm.wo, gp(M, d, hp, c->bwf(blk, F_BO), c->x, d, 1.0f),
                                      lng(c->x, M, c->bwf(blk, F_CONV_LN_W), c->bwf(blk, F_CONV_LN_B), nullptr, nullptr, nullptr, c->z), c->part_use, st)) return rc;
  if (int rc = launch_gemm(EPI_GLU_BF16, c->m_z, bm.pw1, gp(M, 2 * C, d, c->bwf(blk, F_PW1_B), c->h, C), st)) return rc;
  {
    ConvModParams p;
    p.in = c->h; p.out = c->g; p.dw_w = c->bwf(blk, F_DW_W); p.dw_b = c->bwf(blk, F_DW_B); p.cln_w = c->bwf(blk, F_CLN_W); p.lay = lay; p.max_n = c->max_n;
    if (int rc = launch_conv_tiled(C, p, st)) return rc;
  }
  if (int rc = launch_gemm_resid_ln_g(d, c->m_g, bm.pw2, gp(M, d, C, c->bwf(blk, F_PW2_B), c->x, d, 1.0f),
                                      lng(c->x, M, c->bwf(blk, F_FF2_LN_W), c->bwf(blk, F_FF2_LN_B), nullptr, nullptr, nullptr, c->z), c->part_use, st)) return rc;
  if (int rc = launch_gemm(EPI_SWISH_BF16, c->m_z, bm.ff2_w1, gp(M, ff, d, c->bwf(blk, F_FF2_B1), c->h, ff), st)) return rc;
  if (post == nullptr) return launch_gemm(EPI_RESID_F32, c->m_h, bm.ff2_w2, gp(M, d, ff, c->bwf(blk, F_FF2_B2), c->x, d, 0.5f), st);
  return launch_gemm_resid_ln_g(d, c->m_h, bm.ff2_w2, gp(M, d, ff, c->bwf(blk, F_FF2_B2), c->x, d, 0.5f), *post, c->part_use, st);
}

// blocks [blk0, blk0 + n) on the rows of the current pass; x / z prepared by the caller; after the last block x holds the pre-post_norm sum
int t2s_stack(edm_t2s_ctx* c, int blk0, int n, int H, int hp, const float* rope_cos, const float* rope_sin, cudaStream_t st) {
  const int M = c->seqs.lay.rows;
  for (int i = 0; i < n; ++i) {
    const int blk = blk0 + i;
    if (i + 1 < n) {
      // post_norm of this block fused with the first pre-norm of the next one
      const LnGParams post = lng(c->x, M, c->bwf(blk, F_POST_LN_W), c->bwf(blk, F_POST_LN_B), c->bwf(blk + 1, F_FF1_LN_W), c->bwf(blk + 1, F_FF1_LN_B), c->x, c->z);
      if (int rc = t2s_block_body(c, blk, H, hp, rope_cos, rope_sin, &post, st)) return rc;
    } else {
      if (int rc = t2s_block_body(c, blk, H, hp, rope_cos, rope_sin, nullptr, st)) return rc;
    }
  }
  return 0;
}

// The current pass is one sequence of `rows` rows (text n_text, speech `length`): the uniform layout, split-K in low-latency mode.
void t2s_pass_single(edm_t2s_ctx* c, int rows, int n_text, int length) {
  c->seqs.lay = uniform_layout(1, rows, rows);
  c->seqs.cu_text = nullptr; c->seqs.cu_len = nullptr; c->seqs.n_text = n_text; c->seqs.length = length;
  c->pairs = nullptr; c->n_pairs = 0; c->max_n = rows; c->out_len = length;
  c->sum_sq = static_cast<double>(rows) * rows;
  c->init_counts = nullptr;
  c->part_use = c->low_latency ? c->part : nullptr;
}

// The current pass is n_seq packed sequences: n_text[s] + 1 rows each for the length predictor (length == nullptr), n_text[s] +
// length[s] + 4 for the decode. Checks the lengths against the bound capacity and the rotary tables, then uploads the layout arrays
// with one copy on `st`:  cu_n [n_seq + 1] | cu_text [n_seq + 1] | cu_len [n_seq + 1] | length [n_seq] | attention pairs.
int t2s_pass_batch(edm_t2s_ctx* c, int n_seq, const int* n_text, const int* length, cudaStream_t st) {
  if (n_seq < 1 || n_seq > c->max_seq) return fail(EDM_ERR_INVALID, "%d sequences for a workspace bound for %d", n_seq, c->max_seq);
  if (n_text == nullptr) return fail(EDM_ERR_INVALID, "per-sequence text lengths required");
  const size_t n1 = static_cast<size_t>(n_seq) + 1;
  std::vector<int>& h = c->host_layout;
  h.assign(3 * n1 + n_seq, 0);
  std::vector<int> rows(n_seq);
  long long total = 0;
  int max_n = 0;
  double sum_sq = 0.0;
  for (int s = 0; s < n_seq; ++s) {
    const int len = length != nullptr ? length[s] : 0;
    if (n_text[s] < 0 || (length != nullptr && len < 1)) return fail(EDM_ERR_INVALID, "sequence %d: n_text=%d length=%d", s, n_text[s], len);
    const long long r = length != nullptr ? static_cast<long long>(n_text[s]) + len + 4 : static_cast<long long>(n_text[s]) + 1;
    if (r > c->cfg.max_positions) return fail(EDM_ERR_INVALID, "sequence %d of %lld tokens exceeds max_positions=%d", s, r, c->cfg.max_positions);
    total += r;
    if (total > c->max_len) return fail(EDM_ERR_INVALID, "sequences of %lld+ rows exceed the bound workspace (%d rows)", total, c->max_len);
    rows[s] = static_cast<int>(r);
    h[s + 1] = h[s] + rows[s];
    h[n1 + s + 1] = h[n1 + s] + n_text[s];
    h[2 * n1 + s + 1] = h[2 * n1 + s] + len;
    h[3 * n1 + s] = len;
    max_n = std::max(max_n, rows[s]);
    sum_sq += static_cast<double>(r) * r;
  }
  append_attention_pairs(rows, &h);
  if (h.size() > c->layout_cap) return fail(EDM_ERR_INVALID, "layout of %zu ints exceeds the bound workspace (%zu)", h.size(), c->layout_cap);
  int* dev = c->layout_dev;
  EDM_CUDA(cudaMemcpyAsync(dev, h.data(), h.size() * sizeof(int), cudaMemcpyHostToDevice, st));
  SeqLayout& l = c->seqs.lay;
  l.n_seq = n_seq; l.N = 0; l.T = 0; l.cu_n = dev; l.cu_t = dev; l.rows = static_cast<int>(total); l.t_rows = l.rows;
  c->seqs.cu_text = dev + n1; c->seqs.cu_len = dev + 2 * n1; c->seqs.n_text = 0; c->seqs.length = 0;
  c->pairs = dev + 3 * n1 + n_seq; c->n_pairs = static_cast<int>(h.size() - (3 * n1 + n_seq));
  c->max_n = max_n; c->out_len = h[3 * n1 - 1]; c->sum_sq = sum_sq;
  c->init_counts = dev + 3 * n1;
  c->part_use = nullptr;
  return 0;
}

// ints of the layout arrays of t2s_pass_batch for max_seq sequences of max_len rows in all: 3 (max_seq + 1) offsets, max_seq lengths
// and at most max_len / 256 + max_seq attention pairs
size_t t2s_layout_ints(int max_len, int max_seq) { return 4 * (static_cast<size_t>(max_seq) + 1) + static_cast<size_t>(max_len) / 256 + max_seq; }

// max_len rows, max_seq sequences; with_part: the split-K partial sums of a single-sequence bind
size_t t2s_carve(edm_t2s_ctx* c, uint8_t* base, int max_len, int max_seq, bool with_part, bool assign) {
  const size_t M = static_cast<size_t>(max_len);
  Carver k{base};
  float* x = k.take<float>(M * c->d);
  float* y = k.take<float>(M * c->d);
  __nv_bfloat16* z = k.take<__nv_bfloat16>(M * c->d);
  __nv_bfloat16* h = k.take<__nv_bfloat16>(M * c->ff);
  __nv_bfloat16* qkv = k.take<__nv_bfloat16>(M * 3 * c->hp_max);
  __nv_bfloat16* att = k.take<__nv_bfloat16>(M * c->hp_max);
  __nv_bfloat16* g = k.take<__nv_bfloat16>(M * c->C);
  __nv_bfloat16* zt = k.take<__nv_bfloat16>(M * c->d);
  float* logits = k.take<float>(M * 1024);
  float* logp = k.take<float>(M);
  float* raw_len = k.take<float>(std::max(4, max_seq));
  int* ids = k.take<int>(M);
  int* ids_raw = k.take<int>(M);
  int* tokens = k.take<int>(M);
  int* input_ids = k.take<int>(M);
  int* text = k.take<int>(M);
  uint8_t* full_mask = k.take<uint8_t>(M);
  uint8_t* mask_a = k.take<uint8_t>(M);
  uint8_t* mask_b = k.take<uint8_t>(M);
  uint8_t* mask_raw = k.take<uint8_t>(M);
  float* part = with_part ? k.take<float>(4 * M * c->d) : nullptr;   // K-range partial sums of the split-K residual GEMMs
  int* layout = k.take<int>(t2s_layout_ints(max_len, max_seq));
  if (assign) {
    c->part = part;
    c->layout_dev = layout; c->layout_cap = t2s_layout_ints(max_len, max_seq);
    c->x = x; c->y = y; c->z = z; c->h = h; c->qkv = qkv; c->att = att; c->g = g; c->zt = zt; c->logits = logits; c->logp = logp; c->raw_len = raw_len;
    c->ids = ids; c->ids_raw = ids_raw; c->tokens = tokens; c->input_ids = input_ids; c->text = text;
    c->full_mask = full_mask; c->mask_a = mask_a; c->mask_b = mask_b; c->mask_raw = mask_raw;
  }
  return align_up(k.off, 1024);
}

}  // namespace

extern "C" int edm_t2s_num_weights(const edm_t2s_config* cfg) {
  if (t2s_validate(cfg)) return EDM_ERR_INVALID;
  return (cfg->depth + cfg->lp_depth) * F_BLOCK_COUNT + TG_COUNT;
}

extern "C" const char* edm_t2s_weight_name(const edm_t2s_config* cfg, int index) {
  thread_local char buf[64];
  if (t2s_validate(cfg)) return nullptr;
  const int nb = (cfg->depth + cfg->lp_depth) * F_BLOCK_COUNT;
  if (index < 0 || index >= nb + TG_COUNT) return nullptr;
  if (index < nb) {
    const int blk = index / F_BLOCK_COUNT;
    if (blk < cfg->depth)
      snprintf(buf, sizeof(buf), "blocks.%d.%s", blk, kBlockFields[index % F_BLOCK_COUNT]);
    else
      snprintf(buf, sizeof(buf), "lp_blocks.%d.%s", blk - cfg->depth, kBlockFields[index % F_BLOCK_COUNT]);
  } else {
    snprintf(buf, sizeof(buf), "%s", kT2sGlobalFields[index - nb]);
  }
  return buf;
}

extern "C" edm_t2s_ctx* edm_t2s_create(const edm_t2s_config* cfg, const void* const* weights, int n_weights) {
  if (check_arch()) return nullptr;
  if (t2s_validate(cfg)) return nullptr;
  const int expect = (cfg->depth + cfg->lp_depth) * F_BLOCK_COUNT + TG_COUNT;
  if (weights == nullptr || n_weights != expect) {
    fail(EDM_ERR_INVALID, "expected %d weight pointers, got %d", expect, n_weights);
    return nullptr;
  }
  for (int i = 0; i < expect; ++i)
    if (weights[i] == nullptr) {
      fail(EDM_ERR_INVALID, "weight %s is null", edm_t2s_weight_name(cfg, i));
      return nullptr;
    }
  edm_t2s_ctx* c = new edm_t2s_ctx();
  c->cfg = *cfg;
  c->w.assign(weights, weights + expect);
  c->d = cfg->hidden; c->ff = cfg->hidden * cfg->ff_mult; c->C = cfg->hidden * 2;
  c->hp = cfg->heads * 64; c->lp_hp = cfg->lp_heads * 64; c->hp_max = c->hp > c->lp_hp ? c->hp : c->lp_hp;
  c->total_tokens = cfg->text_vocab + cfg->semantic_vocab + cfg->num_special;
  const int nblk = cfg->depth + cfg->lp_depth;
  c->bmaps.resize(nblk);
  int rc = 0;
  for (int b = 0; b < nblk && rc == 0; ++b) {
    BlockMaps& m = c->bmaps[b];
    const int hp = b < cfg->depth ? c->hp : c->lp_hp;
    rc = rc ? rc : make_wmap(&m.ff1_w1, c->bw(b, F_FF1_W1), c->ff, c->d, c->d);
    rc = rc ? rc : make_wmap(&m.ff1_w2, c->bw(b, F_FF1_W2), c->d, c->ff, c->ff);
    rc = rc ? rc : make_wmap(&m.wqkv, c->bw(b, F_WQKV), 3ull * hp, c->d, c->d);
    rc = rc ? rc : make_wmap(&m.wo, c->bw(b, F_WO), c->d, hp, hp);
    rc = rc ? rc : make_wmap(&m.pw1, c->bw(b, F_PW1_W), 2ull * c->C, c->d, c->d);
    rc = rc ? rc : make_wmap(&m.pw2, c->bw(b, F_PW2_W), c->d, c->C, c->C);
    rc = rc ? rc : make_wmap(&m.ff2_w1, c->bw(b, F_FF2_W1), c->ff, c->d, c->d);
    rc = rc ? rc : make_wmap(&m.ff2_w2, c->bw(b, F_FF2_W2), c->d, c->ff, c->ff);
  }
  rc = rc ? rc : make_wmap(&c->pt_map, c->gw(TG_PT_W), c->d, c->d, c->d);
  rc = rc ? rc : make_wmap(&c->head_map, c->gw(TG_HEAD_W), 1024, c->d, c->d);
  if (rc) {
    delete c;
    return nullptr;
  }
  return c;
}

extern "C" void edm_t2s_destroy(edm_t2s_ctx* ctx) { delete ctx; }

namespace {
int t2s_bind(edm_t2s_ctx* c, void* workspace, size_t bytes, int max_len, int max_seq, bool with_part) {
  if ((reinterpret_cast<uintptr_t>(workspace) & 1023) != 0) return fail(EDM_ERR_INVALID, "workspace must be 1024-byte aligned");
  const size_t need = t2s_carve(c, nullptr, max_len, max_seq, with_part, false);
  if (bytes < need) return fail(EDM_ERR_INVALID, "workspace too small: %zu < %zu", bytes, need);
  t2s_carve(c, static_cast<uint8_t*>(workspace), max_len, max_seq, with_part, true);
  c->max_len = max_len;
  c->max_seq = max_seq;
  c->bound = true;
  c->begun = false;
  return 0;
}
}  // namespace

extern "C" size_t edm_t2s_workspace_bytes(const edm_t2s_ctx* ctx, int max_len) {
  if (ctx == nullptr || max_len <= 0) return 0;
  return t2s_carve(const_cast<edm_t2s_ctx*>(ctx), nullptr, max_len, 1, true, false);
}

extern "C" int edm_t2s_bind(edm_t2s_ctx* c, void* workspace, size_t bytes, int max_len) {
  if (c == nullptr || workspace == nullptr || max_len <= 0) return fail(EDM_ERR_INVALID, "bind arguments");
  if (max_len > c->cfg.max_positions) return fail(EDM_ERR_INVALID, "max_len=%d exceeds the rotary tables (%d)", max_len, c->cfg.max_positions);
  return t2s_bind(c, workspace, bytes, max_len, 1, true);
}

extern "C" size_t edm_t2s_workspace_bytes_batch(const edm_t2s_ctx* ctx, int max_rows, int max_seq) {
  if (ctx == nullptr || max_rows <= 0 || max_seq <= 0 || max_seq >= (1 << 15)) return 0;
  return t2s_carve(const_cast<edm_t2s_ctx*>(ctx), nullptr, max_rows, max_seq, false, false);
}

extern "C" int edm_t2s_bind_batch(edm_t2s_ctx* c, void* workspace, size_t bytes, int max_rows, int max_seq) {
  if (c == nullptr || workspace == nullptr || max_rows <= 0 || max_seq <= 0 || max_seq >= (1 << 15)) return fail(EDM_ERR_INVALID, "bind arguments");
  if (max_rows > 0x7fffffff / 1024) return fail(EDM_ERR_INVALID, "max_rows=%d", max_rows);
  return t2s_bind(c, workspace, bytes, max_rows, max_seq, false);
}

extern "C" int edm_t2s_set_low_latency(edm_t2s_ctx* c, int on) {
  if (c == nullptr) return fail(EDM_ERR_INVALID, "null context");
  c->low_latency = on != 0;
  return 0;
}

extern "C" int edm_t2s_set_batch_offset(edm_t2s_ctx* c, long long batch_offset) {
  if (c == nullptr || batch_offset < 0) return fail(EDM_ERR_INVALID, "batch offset");
  c->batch_offset = batch_offset;
  return 0;
}

extern "C" void* edm_t2s_buffer(edm_t2s_ctx* c, const char* name, size_t* bytes) {
  if (c == nullptr || !c->bound || name == nullptr) return nullptr;
  const size_t M = c->max_len;
  struct { const char* n; void* p; size_t b; } tab[] = {
      {"x", c->x, M * c->d * 4}, {"logits", c->logits, M * 1024 * 4}, {"logp", c->logp, M * 4},
      {"raw_len", c->raw_len, static_cast<size_t>(std::max(4, c->max_seq)) * 4},
      {"ids", c->ids, M * 4}, {"ids_raw", c->ids_raw, M * 4}, {"tokens", c->tokens, M * 4}, {"input_ids", c->input_ids, M * 4},
      {"full_mask", c->full_mask, M}, {"mask", c->mask_cur(), M}, {"mask_raw", c->mask_raw, M}};
  for (auto& e : tab)
    if (strcmp(e.n, name) == 0) {
      if (bytes) *bytes = e.b;
      return e.p;
    }
  return nullptr;
}

namespace {
// length predictor on the current pass (c->seqs.lay: n_text_s + 1 rows per sequence) over the packed text tokens
int t2s_length_predictor(edm_t2s_ctx* c, const int* text_tokens, float* raw_out, cudaStream_t st) {
  const edm_t2s_config& cfg = c->cfg;
  const SeqLayout& lay = c->seqs.lay;
  const int M = lay.rows;
  launch_pdl(t2s_lp_gather_kernel, dim3((M + 255) / 256), dim3(256), 0, st, c->seqs, text_tokens, c->text);
  EDM_LAUNCH_CHECK("t2s_lp_gather");
  if (int rc = t2s_maps(c, M, c->lp_hp)) return rc;
  const int b0 = cfg.depth;
  LnGParams p = lng(c->gw(TG_EMB), M, nullptr, nullptr, c->bwf(b0, F_FF1_LN_W), c->bwf(b0, F_FF1_LN_B), c->x, c->z);
  p.gather = c->text; p.gather_rows = c->total_tokens; p.override_row = c->gwf(TG_LENGTH_TOKEN);
  if (int rc = launch_ln_g(c->d, p, st)) return rc;
  if (int rc = t2s_stack(c, b0, cfg.lp_depth, cfg.lp_heads, c->lp_hp, c->gwf(TG_LP_ROPE_COS), c->gwf(TG_LP_ROPE_SIN), st)) return rc;
  const int last = b0 + cfg.lp_depth - 1;
  float* out = raw_out != nullptr ? raw_out : c->raw_len;
  const dim3 grid(lay.n_seq);
  const float *lw = c->bwf(last, F_POST_LN_W), *lb = c->bwf(last, F_POST_LN_B), *w = c->gwf(TG_LEN_W), *b = c->gwf(TG_LEN_B);
  switch (c->d) {
    case 128: launch_pdl(t2s_length_head_kernel<1>, grid, dim3(32), 0, st, c->x, lay.cu_n, lw, lb, w, b, 1e-5f, out); break;
    case 256: launch_pdl(t2s_length_head_kernel<2>, grid, dim3(32), 0, st, c->x, lay.cu_n, lw, lb, w, b, 1e-5f, out); break;
    case 384: launch_pdl(t2s_length_head_kernel<3>, grid, dim3(32), 0, st, c->x, lay.cu_n, lw, lb, w, b, 1e-5f, out); break;
    case 512: launch_pdl(t2s_length_head_kernel<4>, grid, dim3(32), 0, st, c->x, lay.cu_n, lw, lb, w, b, 1e-5f, out); break;
    default: launch_pdl(t2s_length_head_kernel<8>, grid, dim3(32), 0, st, c->x, lay.cu_n, lw, lb, w, b, 1e-5f, out); break;
  }
  EDM_LAUNCH_CHECK("t2s_length_head");
  c->begun = false;  // the activation buffers were reused
  return 0;
}
}  // namespace

// :198-203: length predictor on [length_token, text embeddings]; raw_out[0] (device) = log of the predicted length. The caller reads it
// back (the sequence length decides every later shape), applies exp / ceil as the reference does, and passes `length` to edm_t2s_begin.
extern "C" int edm_t2s_predict_length(edm_t2s_ctx* c, const int* text_tokens, int n_text, float* raw_out, void* stream) {
  if (c == nullptr || !c->bound) return fail(EDM_ERR_STATE, "context not bound");
  if (n_text < 0 || n_text + 1 > c->max_len) return fail(EDM_ERR_INVALID, "text of %d tokens does not fit the bound workspace (%d rows)", n_text, c->max_len);
  if (n_text + 1 > c->cfg.max_positions) return fail(EDM_ERR_INVALID, "text of %d tokens exceeds max_positions=%d", n_text, c->cfg.max_positions);
  if (n_text > 0 && text_tokens == nullptr) return fail(EDM_ERR_INVALID, "text tokens required");
  t2s_pass_single(c, n_text + 1, n_text, 0);
  return t2s_length_predictor(c, text_tokens, raw_out, static_cast<cudaStream_t>(stream));
}

// the length predictor on n_seq texts packed back to back (n_text_host[s] tokens each) in one pass: raw_out[s] = log length of text s
extern "C" int edm_t2s_predict_length_batch(edm_t2s_ctx* c, int n_seq, const int* text_tokens, const int* n_text_host, float* raw_out, void* stream) {
  if (c == nullptr || !c->bound) return fail(EDM_ERR_STATE, "context not bound");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int rc = t2s_pass_batch(c, n_seq, n_text_host, nullptr, st)) return rc;
  if (c->seqs.lay.rows > n_seq && text_tokens == nullptr) return fail(EDM_ERR_INVALID, "text tokens required");
  return t2s_length_predictor(c, text_tokens, raw_out, st);
}

namespace {
// token sequences and mask state of the current pass (:205-222); text: the packed text tokens in c->text
int t2s_begin_pass(edm_t2s_ctx* c, cudaStream_t st) {
  c->mask_in_a = true;
  T2sBeginParams p;
  p.seqs = c->seqs; p.text_tokens = c->text; p.tok_text = 1; p.tok_sep = 3; p.tok_speech = 2; p.tok_mask = 4;
  p.input_ids = c->input_ids; p.tokens = c->tokens; p.full_mask = c->full_mask; p.mask = c->mask_a;
  launch_pdl(t2s_begin_kernel, dim3((c->seqs.lay.rows + 255) / 256), dim3(256), 0, st, p);
  EDM_LAUNCH_CHECK("t2s_begin");
  if (int rc = t2s_maps(c, c->seqs.lay.rows, c->hp)) return rc;
  c->begun = true;
  return 0;
}
}  // namespace

// :205-222: the token sequence of one request and its mask state
extern "C" int edm_t2s_begin(edm_t2s_ctx* c, const int* text_tokens, int n_text, int length, void* stream) {
  if (c == nullptr || !c->bound) return fail(EDM_ERR_STATE, "context not bound");
  if (n_text < 0 || length < 1) return fail(EDM_ERR_INVALID, "n_text=%d length=%d", n_text, length);
  const long long L = static_cast<long long>(n_text) + length + 4;
  if (L > c->max_len) return fail(EDM_ERR_INVALID, "sequence of %lld tokens exceeds the bound workspace (%d rows)", L, c->max_len);
  if (L > c->cfg.max_positions) return fail(EDM_ERR_INVALID, "sequence of %lld tokens exceeds max_positions=%d", L, c->cfg.max_positions);
  if (n_text > 0 && text_tokens == nullptr) return fail(EDM_ERR_INVALID, "text tokens required");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (n_text > 0) EDM_CUDA(cudaMemcpyAsync(c->text, text_tokens, sizeof(int) * n_text, cudaMemcpyDeviceToDevice, st));
  t2s_pass_single(c, static_cast<int>(L), n_text, length);
  return t2s_begin_pass(c, st);
}

// n_seq requests packed back to back: text s has n_text_host[s] tokens (packed in text_tokens), length_host[s] speech positions
extern "C" int edm_t2s_begin_batch(edm_t2s_ctx* c, int n_seq, const int* text_tokens, const int* n_text_host, const int* length_host, void* stream) {
  if (c == nullptr || !c->bound) return fail(EDM_ERR_STATE, "context not bound");
  if (length_host == nullptr) return fail(EDM_ERR_INVALID, "per-sequence lengths required");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  c->begun = false;
  if (int rc = t2s_pass_batch(c, n_seq, n_text_host, length_host, st)) return rc;
  const int total_text = c->host_layout[2 * (static_cast<size_t>(n_seq) + 1) - 1];
  if (total_text > 0) {
    if (text_tokens == nullptr) return fail(EDM_ERR_INVALID, "text tokens required");
    EDM_CUDA(cudaMemcpyAsync(c->text, text_tokens, sizeof(int) * total_text, cudaMemcpyDeviceToDevice, st));
  }
  return t2s_begin_pass(c, st);
}

// embeddings_to_logits (:135-152, mask = None) -> buffer "logits" [rows, 1024] fp32 over the rows of what was begun. x_in: fp32
// [rows, hidden] embeddings, or NULL to embed the context's running tokens (input_embedding lookup fused into the first LayerNorm pass).
extern "C" int edm_t2s_logits(edm_t2s_ctx* c, const float* x_in, void* stream) {
  if (c == nullptr || !c->bound || !c->begun) return fail(EDM_ERR_STATE, "no sequence: call edm_t2s_begin first");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const edm_t2s_config& cfg = c->cfg;
  const int M = c->seqs.lay.rows, d = c->d;
  LnGParams p = lng(x_in != nullptr ? static_cast<const void*>(x_in) : c->gw(TG_EMB), M, nullptr, nullptr, c->bwf(0, F_FF1_LN_W), c->bwf(0, F_FF1_LN_B), c->x, c->z);
  if (x_in == nullptr) {
    p.gather = c->tokens;
    p.gather_rows = c->total_tokens;
  }
  if (int rc = launch_ln_g(d, p, st)) return rc;
  if (int rc = t2s_stack(c, 0, cfg.depth, cfg.heads, c->hp, c->gwf(TG_ROPE_COS), c->gwf(TG_ROPE_SIN), st)) return rc;
  const int last = cfg.depth - 1;
  // post_norm -> bf16 operand of pred_transform.0; Linear -> fp32; GELU + LayerNorm -> bf16 operand of pred_head -> fp32 logits
  if (int rc = launch_ln_g(d, lng(c->x, M, c->bwf(last, F_POST_LN_W), c->bwf(last, F_POST_LN_B), nullptr, nullptr, nullptr, c->zt), st)) return rc;
  if (int rc = launch_gemm(EPI_F32, c->m_zt, c->pt_map, gp(M, d, d, c->gwf(TG_PT_B), c->y, d), st)) return rc;
  {
    LnGParams q = lng(c->y, M, c->gwf(TG_PT_LN_W), c->gwf(TG_PT_LN_B), nullptr, nullptr, nullptr, c->zt);
    q.pre_gelu = 1;
    if (int rc = launch_ln_g(d, q, st)) return rc;
  }
  return launch_gemm(EPI_F32, c->m_zt, c->head_map, gp(M, 1024, d, c->gwf(TG_HEAD_B), c->logits, 1024), st);
}

// one iteration's decisions (:229-260) on the logits of edm_t2s_logits: sample / arg-max, confidence re-masking over the speech
// positions of every sequence, token update. Noise / forcing arrays are those of this iteration ([rows, 1024], [rows], [rows], [rows])
// or NULL. Row t of sequence s draws the Philox counter (batch_offset + s) * L_s + t.
extern "C" int edm_t2s_step(edm_t2s_ctx* c, int iter, int iters, float temperature, unsigned long long seed, const float* cat_noise,
                            const float* remask_noise, const int* forced_ids, const uint8_t* forced_mask, void* stream) {
  if (c == nullptr || !c->bound || !c->begun) return fail(EDM_ERR_STATE, "no sequence: call edm_t2s_begin first");
  if (iters < 1 || iter < 0 || iter >= iters) return fail(EDM_ERR_INVALID, "iteration %d of %d", iter, iters);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool last = iter == iters - 1;
  const SeqLayout& lay = c->seqs.lay;
  const int rows = lay.rows;
  SampleParams sp;
  sp.logits = c->logits; sp.ld = 1024; sp.rows = rows; sp.noise = last ? nullptr : cat_noise; sp.use_philox = last ? 0 : 1; sp.seed = seed; sp.seed_dev = nullptr;
  sp.step = static_cast<unsigned>(iter); sp.seq0 = c->batch_offset; sp.forced_ids = forced_ids; sp.ids = c->ids; sp.ids_raw = c->ids_raw; sp.logp = last ? nullptr : c->logp;
  sp.lay = lay; sp.Q = 1; sp.out_q_stride = 1; sp.out_q0 = 0;
  if (int rc = launch_sample(sp, st)) return rc;
  T2sUpdateParams up;
  up.ids = c->ids; up.next_mask = nullptr; up.full_mask = c->full_mask; up.input_ids = c->input_ids; up.tokens = c->tokens; up.rows = rows;
  up.offset = c->cfg.num_special + c->cfg.text_vocab; up.tok_mask = 4;
  if (!last) {
    const double ratio_d = std::cos(M_PI / 2.0 * (static_cast<double>(iter + 1) / static_cast<double>(iters)));
    RemaskParams rp;
    rp.logp = c->logp; rp.gumbel = remask_noise; rp.mask_old = c->mask_cur(); rp.mask_new = c->mask_next(); rp.mask_raw = c->mask_raw; rp.forced_mask = forced_mask;
    rp.lay = lay; rp.init_count = c->seqs.length; rp.init_counts = c->init_counts;
    rp.ratio = static_cast<float>(ratio_d); rp.temp_ratio = static_cast<float>(static_cast<double>(temperature) * ratio_d);
    rp.seed = seed; rp.seed_dev = nullptr; rp.step = static_cast<unsigned>(iter); rp.seq0 = c->batch_offset;
    launch_pdl(remask_kernel, dim3(lay.n_seq), dim3(256), 0, st, rp);
    EDM_LAUNCH_CHECK("remask");
    up.next_mask = c->mask_next();
  }
  launch_pdl(t2s_update_kernel, dim3((rows + 255) / 256), dim3(256), 0, st, up);
  EDM_LAUNCH_CHECK("t2s_update");
  if (!last) c->mask_in_a = !c->mask_in_a;
  return 0;
}

// speech_pred_tokens (:267): int64, semantic vocabulary; [length] of the one sequence, or [sum length_s] packed for a batch
extern "C" int edm_t2s_result(edm_t2s_ctx* c, long long* tokens_out, void* stream) {
  if (c == nullptr || !c->bound || !c->begun) return fail(EDM_ERR_STATE, "no sequence: call edm_t2s_begin first");
  if (tokens_out == nullptr) return fail(EDM_ERR_INVALID, "output required");
  launch_pdl(t2s_gather_out_kernel, dim3((c->out_len + 255) / 256), dim3(256), 0, static_cast<cudaStream_t>(stream), c->seqs, c->tokens, c->out_len, tokens_out);
  EDM_LAUNCH_CHECK("t2s_gather_out");
  return 0;
}

namespace {
// pred_iters x (logits, step) + result on what was begun. Noise / forcing arrays are laid out [iteration][rows (x 1024)].
int t2s_iterate(edm_t2s_ctx* c, int pred_iters, float temperature, unsigned long long seed, const float* cat_noise, const float* remask_noise,
                const int* forced_ids, const uint8_t* forced_masks, long long* tokens_out, void* stream) {
  const size_t L = c->seqs.lay.rows;
  for (int i = 0; i < pred_iters; ++i) {
    const bool last = i == pred_iters - 1;
    if (int rc = edm_t2s_logits(c, nullptr, stream)) return rc;
    if (int rc = edm_t2s_step(c, i, pred_iters, temperature, seed, (cat_noise && !last) ? cat_noise + i * L * 1024 : nullptr,
                              (remask_noise && !last) ? remask_noise + i * L : nullptr, forced_ids ? forced_ids + i * L : nullptr,
                              (forced_masks && !last) ? forced_masks + i * L : nullptr, stream))
      return rc;
  }
  return edm_t2s_result(c, tokens_out, stream);
}
}  // namespace

// whole infer loop for a known length. Noise / forcing arrays are laid out [iteration][...] over L = n_text + length + 4 positions.
extern "C" int edm_t2s_decode(edm_t2s_ctx* c, const int* text_tokens, int n_text, int length, int pred_iters, float temperature,
                              unsigned long long seed, const float* cat_noise, const float* remask_noise, const int* forced_ids,
                              const uint8_t* forced_masks, long long* tokens_out, void* stream) {
  if (pred_iters < 1) return fail(EDM_ERR_INVALID, "pred_iters must be >= 1");
  if (int rc = edm_t2s_begin(c, text_tokens, n_text, length, stream)) return rc;
  return t2s_iterate(c, pred_iters, temperature, seed, cat_noise, remask_noise, forced_ids, forced_masks, tokens_out, stream);
}

// edm_t2s_decode for n_seq packed requests (edm_t2s_begin_batch); noise / forcing arrays [iteration][sum L_s (x 1024)], tokens_out
// [sum length_s]
extern "C" int edm_t2s_decode_batch(edm_t2s_ctx* c, int n_seq, const int* text_tokens, const int* n_text_host, const int* length_host, int pred_iters,
                                    float temperature, unsigned long long seed, const float* cat_noise, const float* remask_noise,
                                    const int* forced_ids, const uint8_t* forced_masks, long long* tokens_out, void* stream) {
  if (pred_iters < 1) return fail(EDM_ERR_INVALID, "pred_iters must be >= 1");
  if (int rc = edm_t2s_begin_batch(c, n_seq, text_tokens, n_text_host, length_host, stream)) return rc;
  return t2s_iterate(c, pred_iters, temperature, seed, cat_noise, remask_noise, forced_ids, forced_masks, tokens_out, stream);
}

// ================================================================================================ HuBERT feature extractor
#include "hubert.cuh"

extern "C" int edm_hubert_conv0(const float* audio, long long n_samples, int rows, const float* w, const float* bias, const float* ln_w,
                                const float* ln_b, void* out, void* stream) {
  if (int rc = check_arch()) return rc;
  if (rows <= 0) return 0;
  if (!audio || !w || !bias || !ln_w || !ln_b || !out || n_samples <= 0) return fail(EDM_ERR_INVALID, "hubert_conv0: null argument");
  HbConv0Params p;
  p.audio = audio; p.n_samples = n_samples; p.rows = rows; p.w = w; p.bias = bias; p.ln_w = ln_w; p.ln_b = ln_b;
  p.out = static_cast<__nv_bfloat16*>(out);
  const long long blocks = (static_cast<long long>(rows) + 7) / 8;
  hubert_conv0_kernel<<<static_cast<int>(blocks < 8LL * num_sms() ? blocks : 8LL * num_sms()), 256, 0, static_cast<cudaStream_t>(stream)>>>(p);
  EDM_LAUNCH_CHECK("hubert_conv0");
  return 0;
}

extern "C" int edm_hubert_ln512(const void* in, const int* gather, int rows, const float* w, const float* b, int gelu, void* out, void* stream) {
  if (int rc = check_arch()) return rc;
  if (rows <= 0) return 0;
  if (!in || !w || !b || !out) return fail(EDM_ERR_INVALID, "hubert_ln512: null argument");
  if (gather != nullptr && in == out) return fail(EDM_ERR_INVALID, "hubert_ln512: a gathering call cannot run in place");
  HbLnParams p;
  p.in = static_cast<const __nv_bfloat16*>(in); p.gather = gather; p.rows = rows; p.w = w; p.b = b; p.gelu = gelu;
  p.out = static_cast<__nv_bfloat16*>(out);
  hubert_ln512_kernel<<<(rows + 7) / 8, 256, 0, static_cast<cudaStream_t>(stream)>>>(p);
  EDM_LAUNCH_CHECK("hubert_ln512");
  return 0;
}

extern "C" int edm_hubert_pad_rows(const float* x, const int* map, int rows, void* out, void* stream) {
  if (int rc = check_arch()) return rc;
  if (rows <= 0) return 0;
  if (!x || !map || !out) return fail(EDM_ERR_INVALID, "hubert_pad_rows: null argument");
  hubert_pad_rows_kernel<<<(rows + 7) / 8, 256, 0, static_cast<cudaStream_t>(stream)>>>(x, map, rows, static_cast<__nv_bfloat16*>(out));
  EDM_LAUNCH_CHECK("hubert_pad_rows");
  return 0;
}

extern "C" int edm_hubert_pos_conv(const void* xp, const int* map, int rows, const void* w, const float* bias, float* x, void* stream) {
  if (int rc = check_arch()) return rc;
  if (rows <= 0) return 0;
  if (!xp || !map || !w || !bias || !x) return fail(EDM_ERR_INVALID, "hubert_pos_conv: null argument");
  if ((reinterpret_cast<uintptr_t>(x) & 15) != 0) return fail(EDM_ERR_INVALID, "hubert_pos_conv: x must be 16-byte aligned");
  static DeviceOnce attr_once;
  if (attr_once.needed()) {
    EDM_CUDA(cudaFuncSetAttribute(hubert_pos_conv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kPcSmemBytes));
    attr_once.done();
  }
  CUtensorMap ma, mw;
  if (int rc = make_tmap_2d(&ma, xp, rows, kD, kD, 128)) return rc;
  if (int rc = make_tmap_2d(&mw, w, kD, 64ull * kPcTaps, 64ull * kPcTaps, 64)) return rc;
  HbPosConvParams p;
  p.rows = rows; p.bias = bias; p.map = map; p.x = x;
  const long long tiles = (static_cast<long long>(rows) + 127) / 128 * 16;
  if (tiles > 0x7fffffffLL) return fail(EDM_ERR_INVALID, "hubert_pos_conv: too many rows");
  ProfScope prof(PK_CONV, 2.0 * rows * kD * 64 * kPcTaps, static_cast<cudaStream_t>(stream));
  hubert_pos_conv_kernel<<<static_cast<int>(tiles < num_sms() ? tiles : num_sms()), kPcThreads, kPcSmemBytes, static_cast<cudaStream_t>(stream)>>>(ma, mw, p);
  EDM_LAUNCH_CHECK("hubert_pos_conv");
  return 0;
}
