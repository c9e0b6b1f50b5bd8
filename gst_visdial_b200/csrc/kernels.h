// Host-side launch interface of the gstvd kernels.  Every launcher enqueues on `stream` and returns the number of
// kernels it launched (the engine accumulates that into gstvd_launch_count) or throws std::runtime_error.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <utility>

namespace gstvd {

// Set by the engine around the decode step: launch with the programmatic-stream-serialization attribute (PDL).
bool& pdl_flag();
bool carveout_max_flag();   // env GSTVD_CARVEOUT_MAX=1: pin the shared-memory carve-out of every launch_k kernel (measured: no gain)

template <typename... KArgs, typename... Args>
inline void launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = pdl_flag() ? 1 : 0;
  // Optional experiment: identical L1/shared-memory carve-out for every kernel of the decode chain (measured: no effect).
  static thread_local const void* configured[64];
  static thread_local int n_configured = 0;
  bool seen = false;
  for (int i = 0; i < n_configured; ++i) seen |= (configured[i] == (const void*)kernel);
  if (!seen && n_configured < 64) {
    if (carveout_max_flag()) cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    configured[n_configured++] = (const void*)kernel;
  }
  cudaLaunchKernelEx(&cfg, kernel, KArgs(std::forward<Args>(args))...);
}

enum DType { kF32 = 0, kBF16 = 1 };

struct GemmArgs {
  const void* A = nullptr; int64_t lda = 0;   // [M,K] row-major; fp32 (SIMT f32) or bf16
  const void* W = nullptr; int64_t ldw = 0;   // [N,K] row-major (nn.Linear layout), same dtype as A
  const float* bias = nullptr;                // [N] or null
  void* C = nullptr; int64_t ldc = 0;         // [M,N]
  int out_f32 = 0;                            // 1: C is fp32 regardless of the compute dtype
  int act = 0;                                // 0 none, 1 erf-GELU
  int M = 0, N = 0, K = 0;
  // head-major scatter epilogue (cross-attention K/V prefill): active when hm_D > 0.
  //   row -> (b = row / hm_L, pos = row % hm_L);  col -> (g = col / hm_D, d = col % hm_D);
  //   layer = g / hm_G, r = g % hm_G;   C index = (((layer*hm_B + b)*hm_G + r)*hm_L + pos)*hm_D + d
  int hm_D = 0, hm_L = 0, hm_G = 0, hm_B = 0;
  int hm_tpi = 0;      // set by launch_gemm_tc: head-major TMA mode, M tiles per image (tiles never straddle images)
  int tma_store = 0;   // set by launch_gemm_tc: 1 = epilogue stores through a TMA tensor map, 2 = direct 16-byte row stores (skinny problems)
  // ---- deferred LayerNorm (decode step, direct-store epilogue only; DESIGN.md section 4) ----
  // The decoder's dense -> LayerNorm(x + input) pairs (HF BertSelfOutput / BertOutput, call site models/visual_dialog_decoder.py:300-311)
  // run without a LayerNorm kernel: the producing GEMM stores the RAW sum x = A W^T + b + residual (bf16) and, per 32-column block,
  // the row's (mean, M2) of the stored values; every consumer of LN(x) applies it on the fly from the merged statistics:
  //   as the next GEMM's A operand:  LN(x) W^T + b = rstd (x W'^T - mean c) + d   with W' = W * gamma (columns), c_n = sum_k W'_nk,
  //                                  d_n = sum_k beta_k W_nk + b_n  (W', c, d are prepared once by launch_fold_ln_weights);
  //   as the next residual:          (x - mean) rstd gamma + beta, evaluated in the epilogue.
  int64_t stats_ld = 0;                 // row capacity of every statistics buffer below: layout [part][stats_ld rows]
  const float2* fold_stats = nullptr;   // partial (mean, M2) of the raw A rows; non-null: W is W', bias is d
  int fold_parts = 0;                   // partials per row (= raw width / 32)
  const float* fold_c = nullptr;        // [N]
  const void* res = nullptr; int64_t ldr = 0;       // bf16 residual added before the activation / rounding (null: none)
  const float2* res_stats = nullptr; int res_parts = 0;   // non-null: `res` is raw, the residual is its LayerNorm
  const float* res_gamma = nullptr; const float* res_beta = nullptr;
  float2* stats_out = nullptr;          // (mean, M2) of this launch's stored values per 32-column block
  unsigned long long* dbg_times = nullptr;   // measurement aid: per-CTA globaltimer stamps (8 per CTA)
  int dbg = 0;   // measurement aid (env GSTVD_GEMM_DBG): 1 = epilogue without global stores, 2 = epilogue skipped, 3 = no MMA
};

constexpr int kLnStatStride = 32;   // partial statistics per row (rows of at most 1024 columns)
constexpr float kLnEpsDeferred = 1e-12f;

// SIMT GEMM: dtype kF32 (all fp32) or kBF16 (bf16 operands, fp32 accumulate; debugging aid)
int launch_gemm_simt(const GemmArgs& a, int dtype, cudaStream_t stream);
// tcgen05 / TMEM / TMA GEMM, bf16 operands, fp32 accumulate.
// Skinny (M <= 512) problems use the 6-warp / ~100 KB configuration of which two CTAs fit one SM.
int launch_gemm_tc(const GemmArgs& a, int num_sms, cudaStream_t stream);
void gemm_tc_init();  // resolves cuTensorMapEncodeTiled, sets kernel attributes
struct AttnArgs {
  const void* q = nullptr; int64_t q_bs = 0, q_hs = 0, q_rs = 0;   // element strides: batch, head, row
  const void* k = nullptr; int64_t k_bs = 0, k_hs = 0, k_rs = 0;
  const void* v = nullptr; int64_t v_bs = 0, v_hs = 0, v_rs = 0;
  void* o = nullptr;       int64_t o_bs = 0, o_hs = 0, o_rs = 0;
  const float* kmask = nullptr; int64_t kmask_bs = 0;              // [Bkv, Lk] 1 keep / 0 masked, or null
  float neg = -10000.0f;                                          // additive value for masked keys
  int causal = 0;                                                 // key j allowed for query i iff j <= i
  int B = 0, H = 0, Lq = 0, Lk = 0, D = 0;
  int kv_batch_div = 1;                                           // kv batch index = b / kv_batch_div
};
// Generic exact-softmax attention (any Lq/Lk, D <= 128, Lk <= 512), SIMT, fp32 math.
int launch_attention_generic(const AttnArgs& a, int dtype, cudaStream_t stream);
// Tensor-core (mma.sync bf16) attention for the encoder / teacher-forced shapes; D in {64,128}.
int launch_attention_mma(const AttnArgs& a, cudaStream_t stream);
bool attention_mma_supported(const AttnArgs& a);

// y = LN(x + residual) ; rows x width ; dtype of x/residual/y = dtype ; gamma/beta fp32
int launch_add_layernorm(int dtype, int rows, int width, const void* x, int64_t ldx, const void* residual, int64_t ldr,
                         const float* gamma, const float* beta, void* y, int64_t ldy, cudaStream_t stream);
// deferred LayerNorm (see GemmArgs): folded weight preparation (fp32 W [N,K] -> bf16 W' + c[N] + d[N]) and the materialising
// normalisation of a raw bf16 tensor from its stored partial statistics (width = 32 * parts)
int launch_fold_ln_weights(int N, int K, const float* W, const float* gamma, const float* beta, const float* bias, void* Wf, float* c,
                           float* d, cudaStream_t stream);
int launch_ln_apply_stats(int rows, int width, const void* x, const float2* stats, int64_t stats_ld, int parts, const float* gamma,
                          const float* beta, void* y, cudaStream_t stream);
// text embeddings: y[row] = LN(word[id] + pos[p] + type[seg]);  positions = row % L + pos_offset(*d_pos_offset if non-null)
// eos_to_pad: [SEP] and negative ids (the end marker of a shorter decoder prefix) are embedded as [PAD]
int launch_embed_text(int dtype, int rows, int L, int width, const int64_t* ids, const int64_t* seg, const int* d_pos_offset,
                      int eos_to_pad, const float* word, const float* pos, const float* type, const float* type_ext,
                      int type_vocab, const float* gamma, const float* beta, void* y, cudaStream_t stream);
// decode-step embeddings from int32 current tokens (EOS -> PAD applied), position P0 + *d_step with P0 = p0s[row / rows_per_image]
// (per-image decoder prefix lengths - 1) or pos0 when p0s is null
int launch_embed_step(int dtype, int rows, int width, const int32_t* tokens, int pos0, const int* p0s, int rows_per_image, const int* d_step,
                      const float* word, const float* pos, const float* type, const float* gamma, const float* beta, void* y,
                      cudaStream_t stream);
// image embeddings: y = LN(x(+bias already) + loc * Wloc^T + bloc)
int launch_image_embed_ln(int dtype, int rows, int width, const void* x, const float* loc, const float* wloc,
                          const float* bloc, const float* gamma, const float* beta, void* y, cudaStream_t stream);
// dtype conversions / copies
int launch_cast_f32_to(int dtype, const float* src, void* dst, int64_t n, cudaStream_t stream);
int launch_cast_to_f32(int dtype, const void* src, float* dst, int64_t n, cudaStream_t stream);
// strided row copies (concat for VLFusion etc.): dst[r, :width] = src[r, :width] ; all in dtype
int launch_copy_rows(int dtype, int rows, int width, const void* src, int64_t lds, void* dst, int64_t ldd, cudaStream_t stream);
// fused = cat(image rows, text rows) per batch, mask likewise
int launch_concat_fused(int dtype, int B, int Lv, int Lt, int width, const void* v, const void* t, void* fused,
                        const float* imask, const float* tmask, float* fmask, cudaStream_t stream);
// pooled = relu(a) * relu(b)  (fp32 in/out)
int launch_relu_mul(int dtype, int64_t n, const void* a, const void* b, void* out, cudaStream_t stream);
// gather row 0 of each batch: dst[b,:] = src[b*L*width ...]
int launch_gather_first_rows(int dtype, int B, int L, int width, const void* src, void* dst, cudaStream_t stream);

// ---- decode-step kernels (persistent KV cache) ------------------------------------------------------------
struct DecodeGeom {
  int B, K, H, heads, D, layers, T;   // T = max positions in the self cache (P0 + new tokens)
  int Le;                             // encoder length (cross keys)
  int P0 = 0;                         // decoder prefix length - 1: cache positions 0..P0-1 hold the prefix (launch_prefix_kv_store)
  // Per-image decoder prefixes of different lengths: int32 [B], image b's own P0 (<= P0; its prefix holds P0s[b] + 1 tokens), read
  // by the kernels of the decode step.  Null: every image has P0.  Cache positions P0s[b] .. P0 - 1 of image b hold the prefill's
  // padding rows until its decode steps overwrite them; a step never reads a position at or past its own.
  const int* P0s = nullptr;
  __host__ __device__ int p0(int b) const { return P0s ? P0s[b] : P0; }
};
// Forced kernel choices of the decode attention launchers (`force` argument; kDecDefault keeps the launcher's own choice,
// environment switches included).  The single-kernel test entries use them; the decode step always passes kDecDefault.
constexpr int kDecDefault = -1;
enum SelfAttnKernel { kSelfFirst = 0, kSelfV2 = 1 };
enum CrossAttnKernel { kCrossWarpTma = 0, kCrossCtaTma = 1, kCrossMma = 2, kCrossSimt = 3, kCrossGeneric = 4 };

// self-attention for one new position per row: appends k/v at position g.p0(b) + *d_step and attends over 0..g.p0(b) + *d_step
// qkv [M, 3H]; cache layout [layer][kv][b][t][k][H]
// step_host >= 0: the caller knows the step index (must equal *d_step); the lean kernel then only loads positions <= step
// force: kDecDefault, kSelfFirst or kSelfV2 (dec_self_attn_supports must hold)
int launch_dec_self_attn(int dtype, const DecodeGeom& g, int layer, const void* qkv, void* self_cache, const int* d_step, int step_host,
                         const uint8_t* anc, void* out, cudaStream_t stream, int force);
// the lean bf16 / 64-dim kernel will run for these arguments (default on; env GSTVD_SELF_V2=0 disables it)
bool dec_self_attn_v2_active(int dtype, const DecodeGeom& g, const void* qkv, const void* self_cache, const void* out);
// kernel (kSelfFirst / kSelfV2) can run these arguments (anc != null: only the lean kernel reads an ancestry table)
bool dec_self_attn_supports(int kernel, int dtype, const DecodeGeom& g, const void* qkv, const void* self_cache, const void* out,
                            const uint8_t* anc);
// anc: uint8 [B*K][32] (rows of 64 when g.T > 32) ancestry table (slot that holds position t of beam k's history), permuted instead of gathering the cache;
// only the lean kernel reads it - pass null to the self-attention and call launch_reorder_cache otherwise
int launch_anc_update(const DecodeGeom& g, const int32_t* beam_idx, const int* d_step, uint8_t* anc, cudaStream_t stream);
// decoder prefix prefill: stores layer `layer`'s K / V of the qkv rows [B * P0][3H] (teacher-forced pass over the first P0 prefix
// positions) into every beam slot of cache positions 0..P0-1; launches nothing when P0 = 0.  With g.P0s the rows of image b past
// its own g.p0(b) are padding, stored like the others and never read.
int launch_prefix_kv_store(int dtype, const DecodeGeom& g, int layer, const void* qkv, void* self_cache, cudaStream_t stream);
// cross-attention of every beam row over its image's cross K/V. cross layout [layer][b][kv*heads+h][Le][D]
// force: kDecDefault, kCrossMma, kCrossSimt or kCrossGeneric (dec_cross_supports must hold)
int launch_dec_cross_attn(int dtype, const DecodeGeom& g, int layer, const void* q, const void* cross_cache,
                          const float* enc_mask, void* out, cudaStream_t stream, int force);
// TMA-streamed bf16 variant (cross_tma.cu); cross_len [B] = keys to fetch per image (launch_cross_len), may be null
// dec_cross_tma_supported: the decode step's choice (honours env GSTVD_CROSS_NO_TMA); force: kDecDefault, kCrossWarpTma or kCrossCtaTma
bool dec_cross_tma_supported(int dtype, const DecodeGeom& g);
bool dec_cross_tma_fits(int dtype, const DecodeGeom& g);   // the same without the environment switch
int launch_dec_cross_tma(const DecodeGeom& g, int layer, const void* q, const void* cross_cache, const float* enc_mask,
                         const int* cross_len, void* out, int num_sms, cudaStream_t stream, int force);
// kernel (a CrossAttnKernel) can run this geometry, whatever the environment says
bool dec_cross_supports(int kernel, int dtype, const DecodeGeom& g);
int launch_cross_len(int B, int Le, const float* mask, int* out, cudaStream_t stream);
void dec_cross_print_times();   // measurement aid (env GSTVD_CROSS_TIMES=1): per-CTA phase stamps of the last cross-attention launch
// cached CUtensorMap (returned as an opaque pointer) over [groups][L][D] bf16 rows, box = D x box_rows (gemm_tc.cu)
const void* tma_map_rows3(const void* ptr, int D, int L, int64_t groups, int box_rows);
// in-place beam gather of the self cache over the generated positions g.p0(b) .. g.p0(b) + len - 1 of image b;
// len = *d_len + 1 if d_len else len_host
int launch_reorder_cache(int dtype, const DecodeGeom& g, void* self_cache, const int32_t* beam_idx, const int* d_len,
                         int len_host, const uint8_t* d_skip, cudaStream_t stream);

// ---- token selection -------------------------------------------------------------------------------------
constexpr int kSelMax = 16;   // per-row candidates kept (>= 2*max_beams, >= max top_k)
constexpr int kProcMaxLen = 64;   // longest decoder input the logits processors read (= the cached positions of the decode kernels)

// HF logits processors on a row's score s (include/gstvd.h gstvd_generate; CPU oracle: oracle/processors.py), applied where the
// selection kernels apply their ban lists.  d = the row's decoder input of cur_len = P + t ids: the image's decoder prefix ([SEP] read
// as [PAD]; [CLS] when null), then the row's t generated tokens.
//   repetition_penalty p (1 = off): every distinct id of d gets s < 0 ? fp32(s * p) : fp32(s / p)
//   no_repeat_ngram n (0 = off): the id that follows an earlier occurrence of the last n-1 ids of d gets -inf
//   min_length m (0 = off): [SEP] gets -inf while cur_len < m
// d is read either from an int32 key buffer (sampling: keys [rows, key_stride], [SEP] already [PAD]) or from the int64 decoder prefix
// [rows / rows_per_image, P] (null: [CLS], P = 1) followed by the beam token buffer tokens [rows, tok_stride] of this step's parity.
// t = step, or *d_step when step < 0.  p0s (DecodeGeom::P0s, rows_per_image rows per image): image b's prefix is its first p0s[b] + 1
// ids (cur_len = p0s[b] + 1 + t); a key row then holds it right-aligned, columns P - 1 - p0s[b] .. P - 1, before the generated tokens.
struct LogitsProcs {
  float repetition_penalty = 1.f;
  int no_repeat_ngram = 0, min_length = 0;
  const int32_t* keys = nullptr; int key_stride = 0;
  const int64_t* prefix = nullptr; const int32_t* tokens = nullptr; int tok_stride = 0; int rows_per_image = 1;
  int P = 1, step = -1;
  const int* d_step = nullptr;
  const int* p0s = nullptr;
  __host__ __device__ bool active() const { return repetition_penalty != 1.f || no_repeat_ngram > 0 || min_length > 0; }
};

// Per row: logZ (fp64 accumulate) and the top `nsel` entries of  score_j by (score desc, index asc), where
//   mode 0 (beam):   score_j = fp32(proc(fp32(x_j - logZ)) + row_bias[row])   (mode 2: the same with the exp terms of logZ in fp32)
//   mode 1 (sample): score_j = proc(fp32(x_j / temperature))
//   proc = the logits processors of `procs` (identity when inactive); banned tokens (every mode) = -inf, applied after the transform:
//   logZ is over the full, unprocessed row
// logits [rows, ldl] fp32.  ban_tokens [rows, ban_stride] / ban_count [rows] may be null.
int launch_row_select(int rows, int V, const float* logits, int64_t ldl, int mode, const float* row_bias, float temperature,
                      const int32_t* ban_tokens, const int32_t* ban_count, int ban_stride, int nsel,
                      float* sel_val, int32_t* sel_idx, float* logz, const LogitsProcs& procs, cudaStream_t stream);

struct BeamBuffers {
  float* beam_scores;      // [B,K]
  int32_t* tokens;         // [2][B,K,T] double buffered token history
  int32_t* cur_tokens;     // [B*K] input token of the next step
  int32_t* beam_idx;       // [B,K] parent of every new beam (this step)
  uint8_t* done;           // [B]
  double* hyp_score;       // [B,K]
  int32_t* hyp_len;        // [B,K]
  int32_t* hyp_tokens;     // [B,K,T]
  int32_t* hyp_count;      // [B]
  double* hyp_worst;       // [B]
  int* d_step;             // device step counter
};
// prefix: int64 [B, P] decoder prefix (null: start_token, P = 1); len0 = P, the prefix length counted in every hypothesis length.
// G beam groups of K / G beams (G | K; G = 1: plain beam search): the first beam of every group starts with score 0 (G = K: all beams).
// B = searches of K beams, N consecutive searches per image (beam sampling; 1 otherwise): search s reads prefix row s / N.
// Image b's prefix ends at its first negative id (prefix_len below); the first step's input is its last token.  p0s (may be null):
// receives every image's prefix length - 1 (DecodeGeom::P0s).  The kernels below that take p0s read the image's own length from it
// in place of len0 / P (null: len0 / P for every image).
int launch_beam_init(const BeamBuffers& bb, int B, int K, int G, int N, int T, int start_token, const int64_t* prefix, int P, int* p0s,
                     cudaStream_t stream);
// Beam sampling (oracle/beam_sample.py): S = B * N searches of K beams, rows search-major; sel_val / sel_idx = row_select mode 0 / 2
// output with nsel = kSelMax and the beam scores as row bias.  d_seed = {seed, row_offset} (device).  Parents are written image-local
// (n * K + parent, n = s % N), so the cache reorder runs with N * K rows per image.
int launch_beam_sample_step(const BeamBuffers& bb, int S, int N, int K, int T, int V, const float* sel_val, const int32_t* sel_idx, int top_k,
                            float temperature, float top_p, const uint64_t* d_seed, int eos, int len0, const int* p0s, cudaStream_t stream);
// G > 1: diverse beam search with the Hamming penalty `penalty` (oracle/beam_groups.py).  A candidate whose token earlier groups took
// at this step is re-scored from logits [B*K, ldl] fp32 and logz [B*K] (row_select's outputs for this step); needs nsel >= K + K / G.
// The re-score applies the repetition penalty rep_penalty after the Hamming term when the token occurs in the beam's decoder input
// (prefix: int64 [B, len0] decoder prefix, null: [CLS]; then the beam's tokens).  G = 1 reads none of these.
int launch_beam_step(const BeamBuffers& bb, int B, int K, int G, int T, int V, int nsel, const float* sel_val,
                     const int32_t* sel_idx, const float* logits, int64_t ldl, const float* logz, float penalty, float rep_penalty,
                     const int64_t* prefix, int eos, int len0, const int* p0s, int32_t* out_beam_idx, int32_t* out_tokens,
                     float* out_scores, cudaStream_t stream);
// out_ids [B*N, T] / out_scores [B*N]: the N <= K best finished hypotheses of every image, image-major, in the pop order of HF
// BeamSearchScorer.finalize (score descending, the later-inserted first among equal scores); N = 1 is the single best.
// Search b belongs to image b / per_image (p0s).
int launch_beam_finalize(const BeamBuffers& bb, int B, int K, int T, int eos, int len0, const int* p0s, int per_image, int N, int64_t* out_ids,
                         float* out_scores, cudaStream_t stream);

// n-gram blocking (utils/decoding_utils.py:38-78): ban list per row from the question history and the decoded prefix.
// prefix_tokens int32 [rows, P+T] (decoder prefix of len0 = P tokens, then the generated ones; EOS already replaced by PAD),
// prefix_len = *d_step + len0.  N rows per image (sampled candidates): row r reads the history of image r / N
int launch_ngram_ban(int rows, int N, int Lh, const int64_t* hist_ids, const int64_t* hist_seg, const int32_t* prefix,
                     int prefix_stride, const int* d_step, int len0, int n, int32_t* ban_tokens, int32_t* ban_count, int ban_stride,
                     cudaStream_t stream);
// the same for the B*K beam rows: key = the last n-1 tokens of prefix_b ([SEP] read as [PAD]; null: [CLS], P = 1) followed by beam
// row b*K+k of `tokens` [B, K, T] (the beam token buffer of this step's parity); history row = b.  Needs n - 1 <= P + step, step < T.
// p0s: prefix_b is the first p0s[b] + 1 ids of row b (stride P); an image whose decoder input is shorter than n - 1 bans nothing.
int launch_beam_ngram_ban(int B, int K, int T, int Lh, const int64_t* hist_ids, const int64_t* hist_seg, const int64_t* prefix, int P,
                          const int* p0s, const int32_t* tokens, int step, int n, int32_t* ban_tokens, int32_t* ban_count, int ban_stride,
                          cudaStream_t stream);
// sample-mode selection from row_select output; writes seq[row, step] and cur_tokens[row], prefix[row, step+1]
// top_k == 0: multinomial over the whole (optionally nucleus-filtered) vocabulary; writes the same state as launch_sample_step
// N rows per image (sampled candidates): row r draws as row r / N of a single-sample call seeded candidate_seed(seed, r % N)
// procs: the logits processors, applied after the temperature (their step is *d_step)
int launch_full_vocab_sample(int rows, int N, int V, const float* logits, int64_t ldl, float temperature, float top_p, const int32_t* ban_tokens,
                             const int32_t* ban_count, int ban_stride, int T, uint64_t seed, uint64_t row_offset, const uint64_t* d_seed,
                             const int* d_step, int eos, int32_t* seq, int32_t* cur_tokens, int32_t* prefix, int prefix_stride, int32_t* out_tokens,
                             const LogitsProcs& procs, cudaStream_t stream);
int launch_sample_step(int rows, int N, int T, int nsel, const float* sel_val, const int32_t* sel_idx, int top_k, float top_p,
                       uint64_t seed, uint64_t row_offset, const uint64_t* d_seed, const int* d_step, int eos, int32_t* seq, int32_t* cur_tokens, int32_t* prefix,
                       int prefix_stride, int32_t* out_tokens, cudaStream_t stream);
// dec_prefix: int64 [rows / N, P] decoder prefix (null: start_token, P = 1), shared by the N rows of an image; the key buffer
// `prefix` [rows, prefix_stride >= P + T].  An image's prefix ends at its first negative id; it is written right-aligned into
// columns P - P_b .. P - 1 of the key rows (zeros before it: [PAD], which no history n-gram holds), so the samplers append token t
// at column P + t for every row.  p0s (may be null): receives every image's P_b - 1 (DecodeGeom::P0s).
int launch_sample_init(int rows, int N, int T, int start_token, int32_t* seq, int32_t* cur_tokens, int32_t* prefix,
                       int prefix_stride, int* d_step, const int64_t* dec_prefix, int P, int* p0s, cudaStream_t stream);
int launch_sample_finalize(int rows, int T, int eos, const int32_t* seq, int64_t* out_ids, cudaStream_t stream);
int launch_step_advance(int* d_step, cudaStream_t stream);
// device-side scalar set (a pageable-memory cudaMemcpyAsync would synchronise the stream with the host)
int launch_set_u64(uint64_t* dst, uint64_t v, uint64_t v1, cudaStream_t stream);   // dst[0] = v, dst[1] = v1

// teacher-forced scoring helpers
int launch_shift_labels(int B, int L, int64_t* dec_ids, int64_t* labels, int eos, cudaStream_t stream);
int launch_ce_loss(int rows, int V, const float* logits, int64_t ldl, const int64_t* labels, float* loss, cudaStream_t stream);
// history splice (generate.py:145-160, :214-228)
int launch_splice(int B, int Lt, int Lu, int64_t* ids, int64_t* seg, float* mask, int32_t* enc_len, const int64_t* utt,
                  int segment_value, int strip_sep, int32_t* abnormal, int sep, cudaStream_t stream);
int launch_build_prefix_from_ids(int rows, int len, const int64_t* prefix_ids, int32_t* prefix, int prefix_stride, int eos,
                                 cudaStream_t stream);

}  // namespace gstvd
