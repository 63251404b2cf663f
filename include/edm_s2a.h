/* edm_s2a.h — C ABI of the B200-native S2A decode path (libedm_s2a.so).
 *
 * The reference (naba89/EDM-TTS) has no FFI boundary: its hot path is a chain of torch.nn.Module calls. Each entry
 * point below names the reference code it replaces (path:line relative to the reference repo). Conventions:
 *   - every pointer is a CUDA device pointer unless the name ends in _host; `stream` is a cudaStream_t passed as void*;
 *   - calls only enqueue work on `stream` (no device synchronisation, no allocation after edm_s2a_bind);
 *   - return value 0 = ok, negative = error; edm_last_error() gives a thread-local message;
 *   - bf16 buffers are raw 16-bit storage; "f32" is IEEE float; token / code ids are int32 unless stated;
 *   - the library refuses to run on anything but compute capability 10.x (no fallback path exists).
 */
#ifndef EDM_S2A_H_
#define EDM_S2A_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EDM_ABI_VERSION 1

enum edm_status {
  EDM_OK = 0,
  EDM_ERR_INVALID = -1,    /* bad argument / unsupported shape */
  EDM_ERR_CUDA = -2,       /* CUDA runtime / driver error */
  EDM_ERR_ARCH = -3,       /* device is not sm_100 */
  EDM_ERR_STATE = -4       /* call order violated (e.g. decode before bind) */
};

/* GEMM epilogues (edm_gemm_bf16) */
enum edm_epilogue {
  EDM_EPI_BF16 = 0,        /* out_bf16 = acc + bias */
  EDM_EPI_SWISH_BF16 = 1,  /* conformer.py:54-56,152-154  Linear -> Swish */
  EDM_EPI_QKV_ROPE = 2,    /* conformer.py:132-138       to_q/to_kv + rotary embedding on q,k */
  EDM_EPI_RESID_F32 = 3,   /* conformer.py:222-233       x += scale * (Linear(...)) on the fp32 residual stream */
  EDM_EPI_F32 = 4,         /* injection_conformer_wrapper.py:56-63   logits head */
  EDM_EPI_GLU_BF16 = 5,    /* conformer.py:59-66,170-171  pointwise conv + GLU; weight rows interleaved 32 value | 32 gate */
  EDM_EPI_GELU_BF16 = 11,  /* transformers HubertFeedForward: intermediate_dense -> GELU (erf); out_bf16 = GELU(bf16(acc + bias)) */
  EDM_EPI_ARGMAX = 10      /* logits head followed by argmax(-1) (wrapper :119-121, modeling :228): out = float2 [M, ldo] partials,
                              out[r, c / 64] = (max, first arg-max as int bits) of logits[r, c .. c + 64); N % 64 == 0 */
};

int edm_abi_version(void);
const char* edm_last_error(void);

/* ---------------------------------------------------------------------------------------------------------------
 * Stateless operators (unit-parity surface)
 * ------------------------------------------------------------------------------------------------------------- */

/* out[M,N] = epilogue(A[M,K] (bf16, row pitch lda) x B[N,K]^T (bf16, row pitch ldb)), tcgen05 + TMA.
 * Replaces nn.Linear / 1x1 nn.Conv1d calls: conformer.py:124-126,152-154,170,175; wrapper :38-63. N % 64 == 0
 * (N % 256 == 0 for the CTA-pair kernel that large M selects), K % 64 == 0. */
int edm_gemm_bf16(const void* a, long long lda, const void* b, long long ldb, int M, int N, int K, int epilogue,
                  const float* bias, void* out, long long ldo, float scale, const float* rope_cos,
                  const float* rope_sin, int seq_len, int rope_cols, void* stream);

/* softmax(q k^T / 8) v for H heads of 64; qkv is the fused projection [B*N, 3*H*64] (q | k | v), out [B*N, H*64] bf16.
 * Replaces Attend.flash_attn, attend.py:63-115 (non-causal, no mask, dropout 0). */
int edm_attention(const void* qkv, int B, int N, int H, void* out, void* stream);

/* edm_attention on a packed batch: n_seq sequences of different lengths back to back, sequence i = rows [cu_seqlens[i],
 * cu_seqlens[i + 1]) of qkv [sum N_i, 3*H*64] and out [sum N_i, H*64]; cu_seqlens int32 [n_seq + 1] on the device, starting at 0.
 * Each sequence attends only to itself. Reads the offsets back to size the launch (one synchronisation of `stream`). */
int edm_attention_varlen(const void* qkv, int n_seq, const int* cu_seqlens, int H, void* out, void* stream);

/* y = LN(in; w1,b1) [optional fp32 store], z = LN(y; w2,b2) or y [optional bf16 store, rows n < z_skip of every
 * seq_len-long sequence dropped]. 1024 channels. Replaces nn.LayerNorm at conformer.py:106,168,216 and wrapper :44. */
int edm_layernorm(const void* in, int in_is_bf16, int rows, const float* w1, const float* b1, const float* w2,
                  const float* b2, float* y_out, void* z_out, int seq_len, int z_skip, float eps, void* stream);

/* x[M,1024] += scale * bf16(A[M,K] x B[1024,K]^T + bias), then edm_layernorm(x, ...) on the updated rows: a residual branch of the
 * conformer block and the pre-norm of the next one (conformer.py:229-234 with PreNorm :102-110). splits = 2 or 4 with few rows (the
 * small-M kernel's regime, M <= 2304): the GEMM runs as that many K ranges whose raw partial sums go to `scratch`
 * ([splits, M, 1024] fp32) and are added, in range order, by the LayerNorm launch (what a context in low-latency mode does for
 * single utterances). splits <= 1, scratch NULL or a larger M: edm_gemm_bf16(EDM_EPI_RESID_F32) followed by edm_layernorm. */
int edm_gemm_resid_layernorm(const void* a, long long lda, const void* b, long long ldb, int M, int K, const float* bias, float* x,
                             float scale, const float* w1, const float* b1, const float* w2, const float* b2, float* y_out,
                             void* z_out, int seq_len, int z_skip, float eps, float* scratch, int splits, void* stream);

/* GLU -> depthwise conv (k=5, zero pad 2|2 per sequence) -> Swish -> ChanLayerNorm -> out [B*N,2048] bf16.
 * glu_input != 0: in is [B*N,4096] bf16 (value | gate) and the GLU runs here; glu_input == 0: in is [B*N,2048] bf16 already
 * gated by the pointwise-conv GEMM (EDM_EPI_GLU_BF16), which is what the decoder context uses.
 * Replaces conformer.py:171-174 (GLU :59-66, DepthWiseConv1d :69-77, Swish :54-56, ChanLayerNorm :90-99). */
int edm_conv_module(const void* in, int glu_input, void* out, const float* dw_w, const float* dw_b, const float* cln_w,
                    int B, int N, void* stream);
/* edm_conv_module on a packed batch (sequences as in edm_attention_varlen, zero padding at both ends of each sequence, any length
 * >= 1). Reads the offsets back to size the launch (one synchronisation of `stream`). */
int edm_conv_module_varlen(const void* in, int glu_input, void* out, const float* dw_w, const float* dw_b, const float* cln_w,
                           int n_seq, const int* cu_seqlens, void* stream);

/* Per-row arg-max / Gumbel-max sampling over 1024 logits + log-softmax of the chosen id.
 * rows = B*T*Q; ids land at ids[(b*out_q_stride + out_q0 + q)*T + t]. noise: [rows,1024] Gumbel or NULL;
 * use_philox: in-kernel noise when noise == NULL. Replaces modeling_injection_conformer.py:185,192,203-207,228. */
int edm_sample(const float* logits, long long ld, int rows, const float* noise, int use_philox,
               unsigned long long seed, unsigned step, const int* forced_ids, int* ids, float* logp, int T, int Q,
               int out_q_stride, int out_q0, void* stream);

/* Confidence re-masking of one step (modeling_injection_conformer.py:199-213 + utils/utils.py:49-60). */
int edm_remask(const float* logp, const float* gumbel, const uint8_t* mask_old, uint8_t* mask_new,
               const uint8_t* forced_mask, int B, int T, float ratio, float temp_ratio, unsigned long long seed,
               unsigned step, void* stream);

/* DAC residual VQ on the tcgen05 tensor cores (csrc/rvq_tc.cuh): z [B,1024,T] -> codes int64 [B,n_levels,T] (codes only; eval mode).
 * A 3xTF32 projection GEMM z -> e_ws [B*T,96] followed by the 12-level search with TMEM-resident score tiles. z [B,1024,T] fp32 with T % 4 == 0 or bf16 with T % 8 == 0 (TMA needs
 * 16-byte rows; the host side pads other lengths). bf16 z is expanded to tf32-exact fp32 tiles on chip (half the HBM bytes). Tables (pack_rvq_weights): w_hi / w_lo [96,1024] tf32-split stacked in_proj weights,
 * b_in [96], cb_packed [12,1024,32] = [c^_hi | c^_hi | c^_lo | -|c^|^2/2 hi, lo, 0...], g [12,12,1024,8]. e_ws is caller
 * scratch of B*T*96 floats. Replaces ResidualVectorQuantize.forward, dac/vector_quantizer.py:146-210. */
int edm_rvq_encode_tc(const void* z, int z_is_bf16, int B, int T, int n_levels, const float* w_hi, const float* w_lo, const float* b_in,
                      const float* cb_packed, const float* g, float* e_ws, long long* codes, const long long* forced,
                      float* latents, void* stream);

/* codes int64 [B,L,T] -> features fp32 [B,1024,T] (or [B,L,1024,T] when unreduced); proj = [12,1024,1024] projected
 * codebooks incl. bias. Replaces from_codes / from_codes_unreduced, dac/vector_quantizer.py:212-252. */
int edm_codes_to_features(const long long* codes, const float* proj, float* out, int B, int L, int T, int unreduced,
                          void* stream);

/* Nearest-centroid assignment (HuBERT k-means step of the semantic tokenizer): x [n_frames, dim] fp32 -> idx int64 [n_frames],
 * idx = argmax_c (x . c - |c|^2 / 2) = argmin_c |x - c|_2, first maximum on ties. c_hi / c_lo [n_centroids, dim]: tf32 split of
 * the centroids, half_neg_norm [n_centroids] = -|c|^2 / 2 (edm_tts_b200/kmeans.py packs them); dim % 32 == 0, n_centroids % 256
 * == 0 and <= 4096. score_out (nullable) receives the winning score. Replaces `(-torch.cdist(embed, centers)).argmax(-1)`,
 * edm_tts/models/audio_tokenizer/semantic_tokenizer_hubert/semantic_tokenizer_hubert.py:74-90. */
int edm_kmeans_assign(const float* x, long long n_frames, int dim, const float* c_hi, const float* c_lo,
                      const float* half_neg_norm, int n_centroids, long long* idx_out, float* score_out, void* stream);

/* Centroid update of one Lloyd iteration (the k-means fit of the semantic tokenizer; the reference fits offline with faiss,
 * utility_scripts/hubert_kmeans/): centroids[c] = (sum of rows x[r] with idx[r] == c) / count_c, accumulated in fp64 and rounded once
 * to fp32, written in place; clusters with count 0 keep their row. perm [n] lists the rows cluster by cluster (e.g. the indices of
 * a stable sort of idx), offsets [n_centroids + 1] the first position of each cluster in perm (offsets[n_centroids] = n). Every idx
 * must lie in [0, n_centroids): for an id outside it nothing is read or written out of bounds, but a segment stops summing there, so
 * the centroids of the clusters after it in that segment are wrong (edm_tts_b200/kmeans.py checks the ids first). The sum of
 * each cluster is taken in a fixed order that depends on n only, so the result is the same bits for any device and run.
 * partials: fp64 scratch of edm_kmeans_update_workspace_bytes(n, dim, n_centroids) bytes. sums_out (nullable) [n_centroids, dim]
 * receives the fp64 sums of the clusters (0 for empty ones). dim % 32 == 0, 1 <= n_centroids <= 4096; x and partials 16-byte aligned. */
size_t edm_kmeans_update_workspace_bytes(long long n, int dim, int n_centroids);
int edm_kmeans_update(const float* x, long long n, int dim, const long long* idx, const long long* perm, const long long* offsets,
                      int n_centroids, double* partials, float* centroids, double* sums_out, void* stream);

/* One convolution of the DAC encoder as an implicit GEMM on tcgen05 (bf16 operands, fp32 accumulate), channel-last activations.
 * Replaces each WNConv1d (+ the Snake1d in front of the NEXT conv, + the ResidualUnit add) of edm_tts/models/dac/encoder.py:11-58 /
 * nn_layers.py:8-47 (run under bf16 autocast by utility_scripts/dump_tokens/dump_tokens.py:213).
 *   a        bf16 operand view [B][a_rows][a_cols] (batch stride a_batch_stride elements) that already holds Snake(x); rows outside
 *            [0, a_rows) read as zero (the conv padding)
 *   w        bf16 [c_out][n_taps * a_cols], weight-norm folded, K index = tap * a_cols + channel
 *   out[t]   = bias + sum_j a[t + row_off + j * tap_step] . w[:, j]   for t in [0, rows_out)
 *   x_res    nullable fp32 [B][rows_out][c_out] added to out (ResidualUnit skip; may alias y)
 *   y        nullable fp32 stream out, batch stride y_batch_stride
 *   s_out    nullable bf16 operand out = Snake_alpha(out) (alpha nullable = identity), row t + s_row_off, rows >= s_rows dropped
 *   zt_out   nullable [B][c_out][rows_out] (fp32 if zt_is_f32 else bf16): the latent z in the reference's [B, D, T] layout
 * bias_period: 0, or the period C of bias / alpha along the output columns when the columns are s phases x C channels -- a
 * ConvTranspose1d(kernel 2s, stride s) of the decoder (decoder.py:15-23) is the 2-tap conv out_view[q, r * C + co] =
 * sum_u a[q - u] . w[:, co, r + u s] whose output view [L_in + 1][s * C] is the channel-last output shifted by `padding` rows.
 * a_cols % 64 == 0, c_out % 64 == 0, period % 32 == 0 and <= 1536. */
int edm_dac_conv(const void* a, long long a_rows, int a_cols, long long a_batch_stride, int B, const void* w, int c_out,
                 int n_taps, int tap_step, int row_off, int rows_out, const float* bias, const float* alpha, int bias_period, const float* x_res,
                 float* y, long long y_batch_stride, void* s_out, long long s_batch_stride, int s_row_off, int s_rows,
                 void* zt_out, int zt_is_f32, void* stream);

/* One whole ResidualUnit (nn_layers.py:33-47) of the 64- / 128- / 192-channel stages in one launch:
 *   h = Snake_mid(conv7_dilated(a) + b7) (kept in shared memory);  y += conv1x1(h) + b1 (in place);  s_out = bf16(Snake_next(y)).
 * a: bf16 [B][rows][channels] = Snake_in(x) (batch stride a_batch_stride); w7 bf16 [channels][7 * channels], w1 bf16
 * [channels][channels]; s_out as in edm_dac_conv and must not alias a. channels in {64, 128, 192}. */
int edm_dac_resunit(const void* a, long long a_batch_stride, int B, int rows, int channels, int dilation, const void* w7,
                    const void* w1, const float* b7, const float* a_mid, const float* b1, const float* a_next, float* y,
                    long long y_batch_stride, void* s_out, long long s_batch_stride, int s_row_off, int s_rows, void* stream);

/* Last conv of the decoder (C -> 1 channel, k = 7, padding 3) + tanh (decoder.py:55-59): a bf16 [B][rows][c_pad] = Snake(x) with
 * zero-padded channels, w fp32 [7][c_pad], out fp32 [B][rows]. */
int edm_dac_conv_last(const void* a, long long a_batch_stride, int B, int rows, int c_pad, const float* w, float bias, float* out,
                      int apply_tanh, void* stream);

/* Clears row ranges of a channel-last buffer in one launch (16-byte stores): the gap rows of a packed encoder or decoder batch
 * (DACEncoder.forward_batch, DACDecoder.forward_batch), which every conv producer overwrites with bias / Snake(bias) and which the
 * next multi-tap conv must read as its zero padding. buf: row 0 of the buffer, 16-byte aligned; row_pitch_bytes: bytes per row, a multiple of 16; ranges: device
 * array of n_ranges int pairs (start, end), 0 <= start <= end rows, each [start, end) cleared; max_range_rows >= the longest
 * end - start (sizes the grid only). */
int edm_dac_zero_rows(void* buf, long long row_pitch_bytes, const int* ranges, int n_ranges, int max_range_rows, void* stream);

/* First conv of the encoder (1 -> c0 channels, k = 7, padding 3; encoder.py:38) on CUDA cores: audio fp32 [B][L] ->
 * y fp32 [B][L][c0] and s_out bf16 = Snake_alpha(y). w fp32 [c0][7]; c0 % 64 == 0. */
int edm_dac_conv_first(const float* audio, int B, int L, const float* w, const float* bias, const float* alpha, int c0, float* y,
                       void* s_out, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * HuBERT-large backbone of the semantic tokenizer (semantic_tokenizer_hubert.py:74-90: transformers HubertModel, layer-norm
 * feature extractor, stable-layer-norm encoder, features = hidden_states[output_layer]). The transformer layers are edm_layernorm,
 * edm_gemm_bf16 (EDM_EPI_BF16 fused q|k|v, EDM_EPI_RESID_F32 out_proj / output_dense, EDM_EPI_GELU_BF16 intermediate_dense) and
 * edm_attention_varlen (scale 1/8 = 64^-1/2); the strided convs 1-6 of the feature extractor are edm_dac_conv on the [rows / 2][1024]
 * view of their 512-channel input. The calls below are the rest. Clips are packed as described in csrc/hubert.cuh. */

/* HubertLayerNormConvLayer 0 (conv_layers[0]: Conv1d(1, 512, k 10, s 5) -> LayerNorm(512) -> GELU): audio fp32 [n_samples] ->
 * out bf16 [rows][512], frame f reading samples 5f .. 5f + 9 (zero at or past n_samples). w fp32 [10][512] (tap-major). */
int edm_hubert_conv0(const float* audio, long long n_samples, int rows, const float* w, const float* bias, const float* ln_w,
                     const float* ln_b, void* out, void* stream);

/* LayerNorm(512, eps 1e-5) on bf16 rows, then GELU (erf) when gelu != 0: out[r] = act(LN(in[gather ? gather[r] : r])). Replaces the
 * LayerNorm + GELU of HubertLayerNormConvLayer 1-6 (in place, gather NULL) and the LayerNorm of HubertFeatureProjection (gathering the
 * valid frames of the packed conv output). */
int edm_hubert_ln512(const void* in, const int* gather, int rows, const float* w, const float* b, int gelu, void* out, void* stream);

/* Operand of the positional conv: out bf16 [rows][1024], row r = bf16(x[map[r]]) or zeros when map[r] < 0 (x fp32 [N][1024]). */
int edm_hubert_pad_rows(const float* x, const int* map, int rows, void* out, void* stream);

/* HubertPositionalConvEmbedding + residual add (HubertEncoderStableLayerNorm.forward: x = x + GELU(SamePad(conv(x)))), grouped conv
 * k 128, padding 64, 16 groups of 64 channels, tcgen05 implicit GEMM: x[map[t]] += bf16(GELU(bf16(conv(xp)[t] + bias))) for every padded
 * row t with map[t] >= 0, where xp is edm_hubert_pad_rows' output with >= 64 zero rows on both sides of every sequence. w bf16
 * [1024][128 * 64] (row 64 g + n, column 64 j + c = weight-normed weight[64 g + n, c, j]). */
int edm_hubert_pos_conv(const void* xp, const int* map, int rows, const void* w, const float* bias, float* x, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * S2A decoder context: InjectionConformerModel.infer_special, modeling_injection_conformer.py:130-230, and
 * InjectionConformerWrapper.forward_first_level / forward, injection_conformer_wrapper.py:65-150.
 * ------------------------------------------------------------------------------------------------------------- */
typedef struct edm_s2a_ctx edm_s2a_ctx;

typedef struct edm_s2a_config {
  int hidden;             /* 1024 */
  int heads;              /* 16 (head dim 64) */
  int depth;              /* <= 16 */
  int ff_mult;            /* 4 */
  int conv_kernel;        /* 5 */
  int num_quantizers;     /* 12 */
  int num_codes;          /* 1024 */
  int num_semantic;       /* rows of the semantic embedding */
  int n_injection;        /* <= 4 */
  int injection_layers[4];
  int residual;           /* config.residual */
  int max_positions;      /* rows of the rotary tables */
} edm_s2a_config;

/* Weight table: names are fixed by the library; the host passes one device pointer per name, in order. */
int edm_s2a_num_weights(const edm_s2a_config* cfg);
const char* edm_s2a_weight_name(const edm_s2a_config* cfg, int index);

edm_s2a_ctx* edm_s2a_create(const edm_s2a_config* cfg, const void* const* weights, int n_weights);
void edm_s2a_destroy(edm_s2a_ctx* ctx);

size_t edm_s2a_workspace_bytes(const edm_s2a_ctx* ctx, int B, int T, int P);
/* workspace must be 1024-byte aligned; shapes stay bound until the next bind */
int edm_s2a_bind(edm_s2a_ctx* ctx, void* workspace, size_t bytes, int B, int T, int P);

/* Variable-length batch: n_seq utterances, utterance i with P[i] >= 0 prompt frames and T[i] >= 1 target frames (host arrays;
 * P may be NULL = no prompts), each within the limits of edm_s2a_bind (T[i] <= 4096, P[i] + T[i] <= max_positions). The utterances
 * are packed back to back without padding; every later call takes and returns its buffers in that layout:
 *   semantic tokens [sum T_i] (utterance i at cu_t[i] = T_0 + .. + T_{i-1}), semantic prompt [sum P_i] (at cu_p[i]),
 *   acoustic prompt: utterance i is [q, P_i] at q * cu_p[i], forced_coarse: [4, T_i] at 4 * cu_t[i],
 *   codes out: [12, T_i] at 12 * cu_t[i], per-step noise / forcing [step][sum T_i (x 1024)], workspace buffers by packed rows.
 * With equal lengths this is byte for byte the layout of edm_s2a_bind. Row t of utterance i draws the Philox counter
 * (batch_offset + i) * T_i + t, what a single-utterance call with batch offset batch_offset + i draws, so utterance i decodes to the
 * same bits as edm_s2a_bind(1, T_i, P_i) with that offset (outside low-latency mode). Copies the layout arrays into the workspace
 * on `stream`. edm_s2a_set_prompt_injections(non-NULL) is refused (EDM_ERR_STATE) under this bind (edm_s2a_bind_masked takes it). */
size_t edm_s2a_workspace_bytes_varlen(const edm_s2a_ctx* ctx, int n_seq, const int* T, const int* P);
int edm_s2a_bind_varlen(edm_s2a_ctx* ctx, void* workspace, size_t bytes, int n_seq, const int* T, const int* P, void* stream);

/* Masked bind (speech editing: regenerate any chosen frames of an utterance given the others). Sequence i has N[i] encoder rows
 * packed back to back; target[row] != 0 (host array, sum N[i] bytes) marks the T_i >= 1 rows to regenerate, the other
 * P_i = N[i] - T_i rows are known rows and are treated exactly as prompt rows: input sem + LN(Linear(feat_0(code))), never sampled or
 * re-masked, injected with the cumulative ground-truth features of their levels. Everything per target row (semantic tokens, noise,
 * forced ids and masks, output codes) is laid out as under edm_s2a_bind_varlen with T_i targets, in time order; everything per known row
 * (semantic prompt tokens, [q, P_i] acoustic codes, edm_s2a_set_prompt_injections rows) as its prompt of P_i frames, in time order.
 * The Philox counter of target t is (batch_offset + i) * T_i + t, so with the known rows in front this is edm_s2a_bind_varlen with
 * P = N - T, bit for bit. The workspace is edm_s2a_workspace_bytes_varlen(n_seq, T, P = N - T). Sequences with no target row or with
 * N[i] > max_positions are refused. Copies the layout arrays into the workspace on `stream`. */
int edm_s2a_bind_masked(edm_s2a_ctx* ctx, void* workspace, size_t bytes, int n_seq, const int* N, const unsigned char* target, void* stream);

/* named views into the bound workspace (for parity tests / the Python mirror): returns device pointer or NULL. "tgt_enc" / "enc_slot"
 * are the row maps of a masked bind (target row -> encoder row; encoder row -> target index t, or -1 - k for the k-th known row). */
void* edm_s2a_buffer(edm_s2a_ctx* ctx, const char* name, size_t* bytes);

/* Global index of this context's first sequence inside the caller's whole batch. The in-kernel Philox counters are
 * offset by it so the sampled tokens do not depend on how the batch is chunked or sharded over GPUs. */
int edm_s2a_set_batch_offset(edm_s2a_ctx* ctx, long long batch_offset);

/* keep != 0: edm_s2a_full_pass materialises the per-level logits (buffers "coarse_logits" [4,B*T,1024] and "fine_logits"
 * [B*T,n_fine,1024], fp32) as InjectionConformerWrapper.forward returns them (injection_conformer_wrapper.py:143-150). keep == 0 (the
 * default, what infer_special needs: it only takes the arg-max, modeling_injection_conformer.py:228): the head GEMMs reduce their logits
 * to (max, arg-max) partials in the epilogue and the [B,12,T,1024] tensor never exists. Changes the workspace layout: query
 * edm_s2a_workspace_bytes and bind again after switching. */
int edm_s2a_set_keep_logits(edm_s2a_ctx* ctx, int keep);

/* on != 0: single-utterance serving mode. The reference's own call site decodes ONE utterance (inference.py:43-48); with a few hundred
 * rows every kernel is latency-bound and the long-K residual GEMMs (FeedForward down-projection K = 4096, pointwise-conv-2 K = 2048)
 * leave most SMs idle, so for <= 512 rows they are split over K (2 or 4 ranges, reduced in a fixed order inside the LayerNorm launch
 * that follows: deterministic, same bf16 rounding points). The fp32 summation order then differs from the unsplit kernels, i.e. the
 * rounding noise of a row depends on how many rows are decoded together; with on == 0 (the default) a row's bits never do. */
int edm_s2a_set_low_latency(edm_s2a_ctx* ctx, int on);

/* Feature-valued prompt injections (the `injections` argument of InjectionConformerWrapper.forward, injection_conformer_wrapper.py:92-131):
 * proj = fp32 [n_injection, B*P, 1024], row (k, b, n) = project_injection[k].0 applied to the caller's cumulative DAC feature of
 * prompt frame n (Linear only; the LayerNorm runs in the kernel). While set, edm_s2a_full_pass injects these on the prompt rows
 * instead of the rows looked up from the acoustic prompt codes. NULL (the default, and after every edm_s2a_bind) restores the codes. */
int edm_s2a_set_prompt_injections(edm_s2a_ctx* ctx, const float* proj);

/* Optional device-resident seed offset: when set (non-NULL), the sampling / re-masking kernels add *seed_dev to the seed argument
 * of edm_s2a_step / edm_s2a_decode at run time. A decode captured in a CUDA graph bakes its scalar arguments into the capture; the
 * caller bumps this word before each replay so that every replay draws fresh noise, as Categorical.sample() /
 * Gumbel.sample() do per call in the reference (modeling_injection_conformer.py:192, utils/utils.py:52). NULL detaches. */
int edm_s2a_set_seed_buffer(edm_s2a_ctx* ctx, const unsigned long long* seed_dev);

/* modeling_injection_conformer.py:139-168: build encoder input + mask state (all target rows masked). */
int edm_s2a_build_input(edm_s2a_ctx* ctx, const int* sem_tokens, const int* sem_prompt, const int* ac_prompt,
                        int ac_prompt_levels, void* stream);
/* wrapper :65-90: blocks 0..first injection layer + head 0 on the target rows -> buffer "logits" [B*T,1024] fp32.
 * x_in (fp32 [B,N,1024]) replaces the context's encoder input when not NULL. */
int edm_s2a_first_level(edm_s2a_ctx* ctx, const float* x_in, void* stream);
/* modeling_injection_conformer.py:184-219 for step `step` of `steps`: sample/argmax, feature re-embed, re-mask. */
int edm_s2a_step(edm_s2a_ctx* ctx, int step, int steps, float temperature, unsigned long long seed,
                 const float* cat_noise, const float* remask_noise, const int* forced_ids, const uint8_t* forced_mask,
                 void* stream);
/* wrapper :92-150 + modeling :228: full pass -> codes int64 [B,12,T]. forced_coarse int32 [B,4,T] teacher-forces the
 * tokens injected at the coarse levels (the emitted codes are still the model's own arg-max). Per-level logits are kept in the
 * buffers "coarse_logits" / "fine_logits" only after edm_s2a_set_keep_logits(ctx, 1). x_in as above. */
int edm_s2a_full_pass(edm_s2a_ctx* ctx, const float* x_in, const int* forced_coarse, long long* codes_out,
                      void* stream);
/* whole infer_special: build_input, `steps` first-level passes (skipped when steps == 1), full pass. Noise / forcing
 * arrays are laid out [step][...] and may be NULL (Philox noise from `seed`). */
int edm_s2a_decode(edm_s2a_ctx* ctx, const int* sem_tokens, const int* sem_prompt, const int* ac_prompt,
                   int ac_prompt_levels, int steps, float temperature, unsigned long long seed, const float* cat_noise,
                   const float* remask_noise, const int* forced_ids, const uint8_t* forced_masks,
                   const int* forced_coarse, long long* codes_out, void* stream);
/* ---------------------------------------------------------------------------------------------------------------
 * Text-to-semantic decoder context: TextToSemanticWLen.infer, edm_tts/models/text_to_semantic/modeling_text_to_semantic.py:184-267.
 * One sequence per call as in the reference (edm_t2s_begin / edm_t2s_decode), or several of different lengths packed back to back
 * (the *_batch entry points). Same conventions as the S2A context: weights by name, caller-owned workspace, stream-ordered, no host
 * synchronisation inside the library.
 * ------------------------------------------------------------------------------------------------------------- */
typedef struct edm_t2s_ctx edm_t2s_ctx;

typedef struct edm_t2s_config {
  int hidden;          /* 128 / 256 / 384 / 512 / 1024 (configuration.py:16; train_config.yaml:15 uses 384) */
  int heads;           /* main encoder heads, head dim = hidden / heads <= 64 */
  int depth;           /* main encoder blocks */
  int lp_heads;        /* length predictor heads */
  int lp_depth;        /* length predictor blocks */
  int ff_mult;         /* 4 */
  int conv_kernel;     /* 5 */
  int text_vocab;      /* 256 byte tokens */
  int semantic_vocab;  /* 1024 */
  int num_special;     /* 5: pad, text, speech, sep, mask (configuration.py:45-51) */
  int max_positions;   /* rows of the rotary tables = longest sequence (text + speech + 4), <= 4096 */
} edm_t2s_config;

/* Weight names: "blocks.{i}.<field>" / "lp_blocks.{i}.<field>" with the S2A block fields (wqkv / wo packed with 64-column padded
 * heads, see edm_tts_b200/t2s.py), then emb, length_token, pt_w, pt_b, pt_ln_w, pt_ln_b, head_w, head_b, len_w, len_b,
 * rope_cos, rope_sin, lp_rope_cos, lp_rope_sin. */
int edm_t2s_num_weights(const edm_t2s_config* cfg);
const char* edm_t2s_weight_name(const edm_t2s_config* cfg, int index);
edm_t2s_ctx* edm_t2s_create(const edm_t2s_config* cfg, const void* const* weights, int n_weights);
void edm_t2s_destroy(edm_t2s_ctx* ctx);
size_t edm_t2s_workspace_bytes(const edm_t2s_ctx* ctx, int max_len);
int edm_t2s_bind(edm_t2s_ctx* ctx, void* workspace, size_t bytes, int max_len);
/* Workspace of a packed batch: up to max_seq sequences of max_rows rows in all (each sequence still within max_positions, the
 * rotary tables; the total is not). Such a workspace has no room for split-K partial sums, so nothing decoded on it splits. */
size_t edm_t2s_workspace_bytes_batch(const edm_t2s_ctx* ctx, int max_rows, int max_seq);
int edm_t2s_bind_batch(edm_t2s_ctx* ctx, void* workspace, size_t bytes, int max_rows, int max_seq);
void* edm_t2s_buffer(edm_t2s_ctx* ctx, const char* name, size_t* bytes);
/* on != 0 (the default): a single sequence decoded on an edm_t2s_bind workspace splits its long-K residual GEMMs over K, which is
 * faster for one utterance but changes the fp32 summation order. on == 0: the unsplit launches a packed batch always takes, so an
 * utterance decodes to the same bits alone (with batch offset b + s) as at index s of a batch with offset b. */
int edm_t2s_set_low_latency(edm_t2s_ctx* ctx, int on);
/* Global index of the first sequence of the next decodes (default 0): row t of sequence s draws the Philox counter
 * (batch_offset + s) * L_s + t, so the tokens do not depend on how a batch is chunked. */
int edm_t2s_set_batch_offset(edm_t2s_ctx* ctx, long long batch_offset);

/* :198-203 length predictor; text_tokens int32 [n_text] on the device (bytes + num_special). raw_out[0] (device, or the buffer
 * "raw_len" when NULL) = log(length); the caller applies exp / ceil (the sequence length fixes every later shape). */
int edm_t2s_predict_length(edm_t2s_ctx* ctx, const int* text_tokens, int n_text, float* raw_out, void* stream);
/* The length predictor on n_seq texts in one pass: text s is n_text_host[s] tokens (host array) of the packed device array
 * text_tokens; raw_out[s] (device, or the buffer "raw_len" when NULL) = log(length_s). */
int edm_t2s_predict_length_batch(edm_t2s_ctx* ctx, int n_seq, const int* text_tokens, const int* n_text_host, float* raw_out, void* stream);
/* :205-222 sequence [text] bytes [sep] [speech] [mask]*length [sep] + mask state. */
int edm_t2s_begin(edm_t2s_ctx* ctx, const int* text_tokens, int n_text, int length, void* stream);
/* n_seq sequences packed back to back: sequence s is text s (n_text_host[s] tokens of the packed text_tokens) with length_host[s]
 * speech positions, L_s = n_text_s + length_s + 4 rows starting at L_0 + .. + L_{s-1}. edm_t2s_logits / step / result then work on
 * all of them: buffers and per-iteration noise / forcing by packed rows, result [sum length_s] packed. Copies the layout arrays into
 * the workspace on `stream`. */
int edm_t2s_begin_batch(edm_t2s_ctx* ctx, int n_seq, const int* text_tokens, const int* n_text_host, const int* length_host, void* stream);
/* embeddings_to_logits :135-152 on the running tokens (x_in == NULL) or on given embeddings fp32 [L, hidden] -> buffer "logits". */
int edm_t2s_logits(edm_t2s_ctx* ctx, const float* x_in, void* stream);
/* :229-260 decisions of iteration `iter` of `iters`: sample (arg-max on the last), confidence re-masking, token update. */
int edm_t2s_step(edm_t2s_ctx* ctx, int iter, int iters, float temperature, unsigned long long seed, const float* cat_noise,
                 const float* remask_noise, const int* forced_ids, const uint8_t* forced_mask, void* stream);
/* :267 speech_pred_tokens int64 [length] ([sum length_s] after edm_t2s_begin_batch). */
int edm_t2s_result(edm_t2s_ctx* ctx, long long* tokens_out, void* stream);
/* begin + pred_iters x (logits, step) + result. */
int edm_t2s_decode(edm_t2s_ctx* ctx, const int* text_tokens, int n_text, int length, int pred_iters, float temperature,
                   unsigned long long seed, const float* cat_noise, const float* remask_noise, const int* forced_ids,
                   const uint8_t* forced_masks, long long* tokens_out, void* stream);
/* begin_batch + pred_iters x (logits, step) + result; noise / forcing arrays [iteration][sum L_s (x 1024)] or NULL. */
int edm_t2s_decode_batch(edm_t2s_ctx* ctx, int n_seq, const int* text_tokens, const int* n_text_host, const int* length_host, int pred_iters,
                         float temperature, unsigned long long seed, const float* cat_noise, const float* remask_noise, const int* forced_ids,
                         const uint8_t* forced_masks, long long* tokens_out, void* stream);

/* number of kernels launched by this library since load (bench.py's gpu_launches) */
unsigned long long edm_launch_count(void);
/* Measurement hooks (bench.py): while enabled, every GEMM / attention / LayerNorm / conv-module launch is bracketed by
 * CUDA events on its stream. edm_prof_collect fills 5-element arrays (gemm, attention, layernorm, conv module, other):
 * summed milliseconds, summed algorithmic work (FLOPs for the first two, bytes for the rest) and launch counts. */
void edm_prof_enable(int on);
int edm_prof_collect(double* ms, double* work, int* count);

#ifdef __cplusplus
}
#endif
#endif /* EDM_S2A_H_ */
