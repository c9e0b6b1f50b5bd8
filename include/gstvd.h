/*
 * gstvd.h - C ABI of the B200-native generation hot path of gst-visdial.
 *
 * The reference (gicheonkang/gst-visdial) is pure Python/PyTorch and has no FFI of its own; this header is the
 * boundary that sits UNDER the reference's three nn.Module classes (which gst_visdial_b200/models/ mirrors and
 * binds through ctypes, see INTEGRATION.md).  Each entry point names the reference interface it replaces;
 * file:line citations are into the reference tree.
 *
 * Conventions
 *   - plain C symbols, no C++ types, no exceptions across the boundary;
 *   - every call returns 0 on success or a negative gstvd_status; the message is available from
 *     gstvd_last_error(ctx) (ctx may be NULL for errors raised before a context exists);
 *   - the caller owns every tensor it passes: raw DEVICE pointers (row-major, contiguous, fp32 / int64 as
 *     stated), explicit sizes, and the cudaStream_t (as void*) the work must be enqueued on.  Only
 *     gstvd_load_weight accepts host or device memory;
 *   - the library owns its context: packed weights, workspace, KV caches, CUDA graphs;
 *   - one context per (process, device); calls on one context must be serialised by the caller, different
 *     contexts are independent (one per DataParallel replica / per rank);
 *   - there is no CPU fallback: gstvd_create fails on anything that is not compute capability 10.x.
 */
#ifndef GSTVD_H_
#define GSTVD_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GSTVD_ABI_VERSION 5
#define GSTVD_MAX_CONNECTIONS 16

typedef enum {
  GSTVD_OK = 0,
  GSTVD_ERR_INVALID = -1,      /* bad argument / shape / unknown weight name */
  GSTVD_ERR_CUDA = -2,         /* CUDA runtime or driver error */
  GSTVD_ERR_UNSUPPORTED = -3,  /* device is not sm_100, or a feature is not implemented */
  GSTVD_ERR_STATE = -4         /* call order violated (e.g. generate before encode) */
} gstvd_status;

typedef enum { GSTVD_F32 = 0, GSTVD_BF16 = 1 } gstvd_dtype;

/* Token-selection modes of gstvd_generate. */
typedef enum {
  GSTVD_SELECT_SAMPLE = 0, /* temperature / top-k / top-p filtering + multinomial; top_k == 1 is greedy
                              (models/visual_dialog_model.py:86-110, utils/decoding_utils.py:4-35) */
  GSTVD_SELECT_BEAM = 1,   /* beam search, contract in oracle/beam.py (new behaviour, north_star) */
  GSTVD_SELECT_BEAM_SAMPLE = 2 /* beam sampling (HF num_beams > 1 with do_sample): num_beams, top_k, top_p, temperature and seed all
                                  apply; contract at gstvd_generate and in oracle/beam_sample.py */
} gstvd_select_mode;

/* Model geometry: the fields of config/bert_base_6layer_6conect_{enc,dec}.json that the path reads
 * (models/vilbert_dialog.py:131-250 BertConfig; models/visual_dialog_decoder.py:22 BertGenerationConfig). */
typedef struct {
  int32_t abi_version;        /* GSTVD_ABI_VERSION */
  int32_t compute_dtype;      /* gstvd_dtype: arithmetic of activations / GEMM inputs (accumulation is fp32) */
  /* text stream */
  int32_t vocab_size, hidden_size, num_hidden_layers, num_attention_heads, intermediate_size;
  int32_t max_position_embeddings, type_vocab_size;
  /* image stream */
  int32_t v_feature_size, v_hidden_size, v_num_hidden_layers, v_num_attention_heads, v_intermediate_size;
  /* co-attention */
  int32_t bi_hidden_size, bi_num_attention_heads;
  int32_t num_connections;
  int32_t v_biattention_id[GSTVD_MAX_CONNECTIONS];
  int32_t t_biattention_id[GSTVD_MAX_CONNECTIONS];
  /* decoder (hidden size == hidden_size, shares the embedding tables) ; 0 layers = encoder-only context */
  int32_t dec_num_hidden_layers, dec_num_attention_heads, dec_intermediate_size;
  /* capacity the workspace is sized for */
  int32_t max_batch;          /* images (encoder rows) per call */
  int32_t max_text_len;       /* 256 (options.py:78) */
  int32_t max_regions;        /* 37  (36 regions + global, utils/image_features_reader.py:126-128) */
  int32_t max_new_tokens;     /* 18  (models/visual_dialog_model.py:77) */
  int32_t max_beams;          /* beams per image for GSTVD_SELECT_BEAM */
  int32_t max_dec_len;        /* longest teacher-forced decoder input (25, options.py:79) */
  int32_t flags;              /* GSTVD_FLAG_* */
} gstvd_config;

#define GSTVD_FLAG_NO_CUDA_GRAPH 1   /* launch decode steps eagerly instead of replaying a captured graph */
#define GSTVD_FLAG_DEBUG_SIMT_GEMM 2 /* debugging aid: route bf16 GEMMs through the SIMT kernel */
#define GSTVD_FLAG_NO_PDL 8          /* decode-step kernels without programmatic dependent launch */
#define GSTVD_FLAG_GENERIC_ATTENTION 4 /* debugging aid: route bf16 attention through the generic SIMT kernel */

typedef struct {
  int32_t mode;               /* gstvd_select_mode */
  int32_t num_beams;          /* beam mode: K (<= max_beams); sample mode: ignored (num_return_sequences rows per image) */
  int32_t max_new_tokens;     /* <= config.max_new_tokens */
  int32_t top_k;              /* sample mode; 1 = greedy; 2..GSTVD_MAX_TOP_K = top-k set (ties kept); 0 = no top-k cut: multinomial over the
                                 whole - optionally nucleus-filtered - vocabulary (utils/decoding_utils.py:17 skips the cut) */
  float temperature;          /* sample mode: logits / temperature */
  float top_p;                /* sample mode: nucleus threshold applied inside the top-k set; 0 = off */
  int32_t ngram_blocking_size;/* sample and beam mode: 0 = off; n: ban tokens completing an n-gram of the question history (beam mode:
                                 per beam, on the log-softmax scores before the beam score is added; contract in oracle/beam_ngram.py) */
  uint64_t seed;              /* sample mode RNG seed (counter-based; reproducible per (seed, row_offset + row, step)) */
  int64_t row_offset;         /* global index of row 0 (e.g. the image index of the first sample of this batch / shard): the
                                 draws of an image do not depend on how the images were split into batches or ranks */
  int32_t num_return_sequences; /* N >= 1 sequences per image (HF num_return_sequences); contract at gstvd_generate */
  int32_t num_beam_groups;    /* G >= 1 (HF num_beam_groups): beam mode splits the K beams into G groups; 1 = plain beam search */
  float diversity_penalty;    /* Hamming penalty between beam groups (HF diversity_penalty), finite and >= 0 */
  float repetition_penalty;   /* HF repetition_penalty, finite and > 0; 1 = off.  Logits processors: contract at gstvd_generate */
  int32_t no_repeat_ngram_size; /* HF no_repeat_ngram_size (n-grams of the output itself), >= 0; 0 = off */
  int32_t min_length;         /* HF min_length: [SEP] banned while the decoder input (prefix included) is shorter, >= 0; 0 = off */
} gstvd_gen_params;

#define GSTVD_MAX_TOP_K 16

typedef struct gstvd_ctx gstvd_ctx;

/* ---- lifecycle ------------------------------------------------------------------------------------------- */
/* Replaces module construction: VisualDialogEncoder.__init__ (models/visual_dialog_encoder.py:9-17),
 * VisualDialogDecoder.__init__ (models/visual_dialog_decoder.py:19-27), EncoderDecoderModel.__init__
 * (models/visual_dialog_model.py:16-22). */
int gstvd_create(const gstvd_config* cfg, int device, gstvd_ctx** out);
void gstvd_destroy(gstvd_ctx* ctx);
const char* gstvd_last_error(const gstvd_ctx* ctx);
int gstvd_abi_version(void);

/* Replaces load_state_dict(ckpt['model_state_dict']) (generate.py:68-69,78-79): one call per state_dict key, names
 * in the EncoderDecoderModel namespace ("encoder.bert_pretrained.bert....", "decoder.decoder.bert....",
 * "vlfusion.fc_l.weight").  `data` is fp32, host or device, `numel` elements.  Returns 0 if stored, 1 if the key
 * is known but unused by the path (pre-training heads, q_dense1/2, sep_embeddings), <0 on error. */
int gstvd_load_weight(gstvd_ctx* ctx, const char* name, const float* data, int64_t numel, void* stream);
/* Packs weights for the compute dtype (bf16 copies of matrices). Must be called after the last load. */
int gstvd_finalize_weights(gstvd_ctx* ctx, void* stream);
/* Number of expected keys that were never loaded (debugging aid; 0 after a full checkpoint). */
int gstvd_missing_weights(const gstvd_ctx* ctx);

/* ---- encoder --------------------------------------------------------------------------------------------- */
/* Replaces VisualDialogEncoder.forward (models/visual_dialog_encoder.py:19-76) ->
 * BertForMultiModalPreTraining.forward (models/vilbert_dialog.py:1453-1519) -> BertModel.forward (:1325-1407)
 * and VLFusion.forward (models/visual_dialog_model.py:131-135).
 *   input_ids, token_type_ids : int64 [B, Lt]           attention_mask : fp32 [B, Lt] (1 keep / 0 masked)
 *   image_feat : fp32 [B, Lv, v_feature_size]           image_loc : fp32 [B, Lv, 5]     image_mask : fp32 [B, Lv]
 * Outputs (each may be NULL = not exported):
 *   out_t fp32 [B, Lt, hidden]   out_v fp32 [B, Lv, v_hidden]   out_fused fp32 [B, Lv+Lt, hidden] (image rows
 *   first)   out_fused_mask fp32 [B, Lv+Lt]   out_nsp fp32 [B, 2] (seq_relationship_score, :1030-1038).
 * The fused states stay resident in the context for gstvd_prefill_cross(ctx, B, NULL, NULL, ...). */
int gstvd_encode(gstvd_ctx* ctx, int B, int Lt, int Lv,
                 const int64_t* input_ids, const int64_t* token_type_ids, const float* attention_mask,
                 const float* image_feat, const float* image_loc, const float* image_mask,
                 float* out_t, float* out_v, float* out_fused, float* out_fused_mask, float* out_nsp,
                 void* stream);

/* ---- decoder --------------------------------------------------------------------------------------------- */
/* Projects the encoder states to every decoder layer's cross-attention K/V once (the reference re-projects
 * them on every step: HF BertLayer crossattention, call site models/visual_dialog_decoder.py:300-311).
 * enc_hidden fp32 [B, Le, hidden] / enc_mask fp32 [B, Le]; pass NULL,NULL to use the states left by gstvd_encode. */
int gstvd_prefill_cross(gstvd_ctx* ctx, int B, int Le, const float* enc_hidden, const float* enc_mask, void* stream);

/* Replaces the decode branch of EncoderDecoderModel.forward (models/visual_dialog_model.py:74-120) including
 * batch_ngram_blocking / batch_top_k_top_p_sampling (utils/decoding_utils.py:4-78), with a persistent KV cache.  The tensors are
 * positional; params holds the whole selection policy, including N = num_return_sequences, G = num_beam_groups and
 * diversity_penalty.
 *   prefix : int64 [B, P], 1 <= P <= max_dec_len: the decoder input to continue from, the reference's dec_input_ids
 *            (models/visual_dialog_model.py:86-110 continues from whatever the caller passes), shared by the rows of an image; NULL
 *            means one [CLS] per row (P must be 1).  At every step the decoder sees prefix + the tokens generated so far at positions
 *            0 .. P-1+t, without a padding mask; a [SEP] in the prefix is read as [PAD] (models/visual_dialog_decoder.py:57).  n-gram
 *            keys may reach into the prefix.  Beam hypotheses count the prefix in their length (HF beam_search input_ids.shape[-1]).
 *            The caller's tensor is not modified.  P - 1 + max_new_tokens must not exceed 64 (cached positions of the decode
 *            kernels) nor max_position_embeddings.
 *            Prefixes of different lengths in one call: a negative id ends an image's prefix.  Image b continues from
 *            prefix[b, :P_b], P_b = the column of the first negative id of row b, or P if it has none; the ids after it are not
 *            read as tokens.  P stays the row stride and the longest length, and the checks above apply to it.  Every output row of
 *            image b is exactly what a call holding image b alone with prefix[b, :P_b] returns, in every mode below (sampling with the
 *            same seed and row_offset + b): its cache positions run 0 .. P_b - 1 + t, step t is embedded at position P_b - 1 + t and
 *            starts from prefix[b, P_b - 1], its decoder input for n-gram keys and the logits processors is prefix[b, :P_b] followed by
 *            its tokens with cur_len = P_b + t, and hypothesis lengths, scores and is_done use P_b + t.  A row whose first id is
 *            negative is invalid input: its output is unspecified (the call stays memory-safe; no negative id is ever looked up).
 *   hist_ids, hist_segments : int64 [B, Lh] encoder input ids / segments (only read when ngram_blocking_size > 0, in sample and
 *                             beam mode; the question history is ids * (segments == 0), visual_dialog_model.py:98-99)
 *   out_ids    : int64 [B*N, max_new_tokens], image-major (row b*N + n): the new tokens only, PAD(0) after the first [SEP]
 *   out_scores : fp32 [B*N] (may be NULL; beam modes only) - hypothesis score (sum log-prob / length)
 *
 * Return sequences (HF num_return_sequences):
 *   beam mode, 1 <= N <= num_beams: the N best finished hypotheses of BeamSearchScorer.finalize (transformers 4.16.2) in its pop order -
 *     score descending, the later-inserted hypothesis first among equal scores; contract in oracle/beam_nbest.py.  Decoding is the same
 *     as with N = 1; only the finalisation differs.
 *   sample mode, 1 <= N <= min(8, max_beams): N independent continuations per image, decoded as N rows that share the image's cross
 *     K/V, decoder prefix and n-gram history.  Candidate n of image b draws exactly what an N = 1 call with seed
 *     candidate_seed(seed, n) draws for image b (the RNG row stays row_offset + b); candidate_seed(seed, 0) = seed and, for n >= 1,
 *     splitmix64(seed ^ splitmix64(n * 0xD1B54A32D192ED03)) (splitmix64 as in the sampler).  No scores are written.
 *   Other N are rejected with GSTVD_ERR_INVALID.
 *
 * Beam groups, diverse beam search (HF num_beam_groups / diversity_penalty; transformers 4.16.2 group_beam_search with
 * HammingDiversityLogitsProcessor; Vijayakumar et al., "Diverse Beam Search"; CPU oracle: oracle/beam_groups.py):
 *   The K beams form G groups of gs = K / G consecutive beams; beam k of an image starts with score 0 if k % gs == 0, else -1e9.
 *   Every step runs one decoder pass over all K rows; logZ is per row.  Within a step the groups run in order: the candidate (beam k
 *   of group g, token w) scores fp32(fp32(fp32(x - logZ) - fp32(diversity_penalty * c_w)) + beam_score_k), with c_w = the number of
 *   new beams of groups 0..g-1 of the same image that took w at this step (an [SEP] that closed a hypothesis does not count).
 *   n-gram-banned tokens are -inf and stay -inf.  Each group takes the top 2*gs of its gs*V candidates by (score desc,
 *   (k - g*gs)*V + w asc) and runs BeamSearchScorer.process with group_size = gs: [SEP] is added to the hypotheses only at rank < gs,
 *   the group gets gs new beams whose parents stay inside the group.  All groups share the image's hypothesis heap of capacity K; its
 *   done flag is tested before every group (a group of a done image is padded) and updated after every group with
 *   is_done(best of the group's 2*gs candidates, P + t).  Finalisation and the N-best order are those of beam mode above.
 *   With G = 1 the call is plain beam search, launch for launch, whatever diversity_penalty holds: the penalty only acts on groups
 *   after the first.
 *   Rejected with GSTVD_ERR_INVALID: num_beam_groups < 1, num_beams % num_beam_groups != 0, num_beam_groups > 1 outside beam mode,
 *   diversity_penalty negative or not finite.
 *
 * Beam sampling, mode GSTVD_SELECT_BEAM_SAMPLE (transformers 4.16.2 beam_sample + BeamSearchScorer, length_penalty 1, early_stopping
 * off; CPU oracle: oracle/beam_sample.py).  Per image the call runs N independent stochastic beam searches of K = num_beams beams and
 * returns the best hypothesis of search n as output row b*N + n (out_scores: its score).  Search n of image b is what an N = 1 call
 * with seed candidate_seed(seed, n) runs for that image.  Decode rows are search-major, row (b*N + n)*K + k; the N*K <= max_beams rows
 * of an image share its cross K/V, decoder prefix and n-gram history.  Per search and step t (P = prefix length):
 *   1. all K beams start at score 0 (unlike beam search, which starts beams 1..K-1 at -1e9; only the draw separates them);
 *   2. s = fp32(fp32(x - logZ) + beam_score) per (beam k, token w), logZ as in beam search; n-gram-banned tokens are -inf;
 *   3. the warpers act on s, i.e. AFTER the beam score is added, as in 4.16.2: w = fp32(s / temperature), so the temperature compounds
 *      through the beam scores (a beam's score is the sum of its warped steps, each divided by the temperature again at the next
 *      step); top-k keeps w >= the k'-th largest w of the row, k' = max(top_k, 2), ties as far as the row's 16 best reach; top-p
 *      (0 = off) inside that set keeps ranks 0 and 1 and drops rank r >= 2 once the probability mass before r exceeds top_p;
 *   4. 2K entries are drawn without replacement from softmax(w) over the search's K*V entries (HF torch.multinomial(probs, 2K)) by
 *      Gumbel-top-2K: the 2K largest of fp64(w) - log(-log u), u = ((h >> 11) + 0.5) * 2^-53 with
 *      h = splitmix64(splitmix64(sd ^ splitmix64(((row_offset + b) << 20) ^ t)) ^ (k*V + w)), sd = candidate_seed(seed, n);
 *      the draws of an image do not depend on how images are split across calls (row_offset);
 *   5. the drawn entries, ordered by (w desc, k*V + w asc), go through BeamSearchScorer.process as in beam search: [SEP] closes a
 *      hypothesis only at rank < K, a hypothesis scores its warped sum / (P + t), is_done uses the best drawn w.
 *   Rejected with GSTVD_ERR_INVALID: num_beams < 2 or > 8, N < 1, N*num_beams > max_beams, num_beam_groups > 1, a temperature that is
 *   not finite and > 0, top_p outside [0, 1].  Rejected with GSTVD_ERR_UNSUPPORTED: top_k = 0 or top_k > 16.
 *
 * Logits processors, every mode (HF RepetitionPenaltyLogitsProcessor, NoRepeatNGramLogitsProcessor, MinLengthLogitsProcessor;
 * CPU oracle: oracle/processors.py).  d = a row's decoder input (HF input_ids) at step t: the image's decoder prefix with [SEP] read
 * as [PAD] ([CLS] when prefix is NULL), then the row's own t generated tokens (a beam row: the tokens of that beam; a sample row's
 * generated [SEP] is read as [PAD] too) - the key the question-history blocking uses.  cur_len = P + t.  The processors act on each
 * row's score s at the point where the question-history bans act; -inf stays -inf:
 *   1. repetition_penalty p (1 = off): each distinct id of d gets s < 0 ? fp32(s * p) : fp32(s / p), once however often it occurs
 *      (HF's gather / scatter);
 *   2. no_repeat_ngram_size n (0 = off), only when cur_len + 1 >= n: wherever the last n-1 ids of d occur earlier in d, the id that
 *      follows them there gets -inf.  No special id is exempt (unlike the question-history rule): n = 1 bans every id of d, [CLS]
 *      included;
 *   3. min_length m (0 = off): [SEP] (102) gets -inf while cur_len < m; the unit is the HF 4.16.2 one, decoder-input length with the
 *      prefix, not a count of new tokens.
 *   What s is:
 *   - sampling (top-k and top_k = 0): s = fp32(x / temperature); the processors act before top-k / top-p and the nucleus mass is
 *     computed on the processed row.  (HF applies them before the temperature; the reference's loop divides first and then runs its
 *     blocking processor, and this follows the reference.  The two orders differ only in fp32 rounding.)
 *   - beam search and beam sampling: s = fp32(x - logZ), logZ over the unprocessed row; the processed value is what the beam score
 *     accumulates, and so what out_scores reports.  Beam sampling's warpers then act on fp32(s + beam_score) as above.
 *   - beam groups: the Hamming term first, then the repetition penalty (the order of HF _get_logits_processor): a penalised token
 *     scores fp32(fp32(fp32(fp32(x - logZ) - fp32(lambda * c_w)) * p) + beam_score) (s / p for s >= 0).  The per-row candidate lists
 *     are ranked by the processed score without the Hamming term; the Hamming term only lowers a score and the penalty is monotone,
 *     so the lists still hold each group's exact top 2*gs (argument at beam_step_kernel, csrc/select.cu).
 *   With p = 1, n = 0 and m = 0 a call launches the same kernels and gives the same results, bit for bit, as without the processors.
 *   Rejected with GSTVD_ERR_INVALID: repetition_penalty not finite or <= 0, no_repeat_ngram_size < 0, min_length < 0 (so a
 *   zero-filled params struct is rejected: fill every field). */
int gstvd_generate(gstvd_ctx* ctx, int B, const gstvd_gen_params* params, const int64_t* prefix, int P,
                   const int64_t* hist_ids, const int64_t* hist_segments, int Lh,
                   int64_t* out_ids, float* out_scores, void* stream);

/* One whole forward call of the decode branch of EncoderDecoderModel.forward (models/visual_dialog_model.py:24-120): the same work and
 * results as gstvd_encode (no exported outputs) + gstvd_prefill_cross(resident states) + gstvd_generate with the same params and
 * prefix, replayed from ONE CUDA graph per shape - the host enqueues a few device-to-device copies of the inputs and one graph launch.
 * params, prefix, P, out_ids and out_scores follow the contract of gstvd_generate.  The n-gram blocking history is the call's own
 * input_ids / token_type_ids.  Afterwards the encoder / cross-K/V state is resident exactly as after the three calls (e.g. for the
 * perplexity pass, gstvd_score). */
int gstvd_round(gstvd_ctx* ctx, int B, int Lt, int Lv,
                const int64_t* input_ids, const int64_t* token_type_ids, const float* attention_mask,
                const float* image_feat, const float* image_loc, const float* image_mask,
                const gstvd_gen_params* params, const int64_t* prefix, int P,
                int64_t* out_ids, float* out_scores, void* stream);

/* Replaces VisualDialogDecoder.forward in loss mode (models/visual_dialog_decoder.py:33-86) as driven by
 * generate.py:183-209 and evaluate_gen.py:94-106: teacher-forced pass over dec_ids [B, L].
 *   dec_ids  : int64 [B, L]; when labels == NULL it is MUTATED IN PLACE ([SEP] -> PAD) exactly like :57 and the
 *              labels are the ids shifted left (:54-56)
 *   dec_mask : fp32 [B, L] or NULL (all ones)
 *   out_loss : fp32 [B, L] per-position CE with ignore_index 0 (reduction 'none'); may be NULL
 *   out_logits : fp32 [B, L, vocab]; may be NULL */
int gstvd_score(gstvd_ctx* ctx, int B, int L, int64_t* dec_ids, const float* dec_mask, const int64_t* labels,
                float* out_loss, float* out_logits, void* stream);

/* Generative ranking (evaluate_gen.py:62-107): `options` candidate sequences per image are scored against ONE encoder pass /
 * cross-attention K/V of that image (the reference re-encodes the same image and history for every option).
 *   dec_ids / dec_mask / labels / out_loss / out_logits : as gstvd_score with B = n_images * options rows, option-major per image
 *   n_images must equal the B of the last gstvd_prefill_cross; n_images * options <= config.max_batch */
int gstvd_score_options(gstvd_ctx* ctx, int n_images, int options, int L, int64_t* dec_ids, const float* dec_mask,
                        const int64_t* labels, float* out_loss, float* out_logits, void* stream);

/* In-place beam reorder of the self-attention KV cache: cache[:, new_beam] = cache[:, beam_idx[new_beam]] for
 * every layer - the semantic of _reorder_cache / index_select(0, beam_idx) (models/visual_dialog_decoder.py:29-31,
 * :177-181).  beam_idx int32 [B, K] holds the parent beam (0..K-1) within each image; len = cached positions. */
int gstvd_reorder_cache(gstvd_ctx* ctx, int B, int K, int len, const int32_t* beam_idx, void* stream);

/* ---- dialog state (generate.py:145-160, :214-228) ----------------------------------------------------------- */
/* Appends utterance utt[b, :n_b] (n_b = count of non-zero ids) to row b of enc_input_ids at enc_len[b]; on
 * overflow past Lt writes a lone [SEP], n_b = 1 and sets abnormal[b] = 1.  segment_value >= 0 also writes that
 * value into enc_segments over the appended span (answers: 1).  strip_sep != 0 drops [SEP] tokens from utt first
 * (single-device reference behaviour for answers, SURVEY.md 8a).  Updates enc_len and attention_mask. */
int gstvd_splice(gstvd_ctx* ctx, int B, int Lt, int Lu, int64_t* enc_input_ids, int64_t* enc_segments,
                 float* attention_mask, int32_t* enc_len, const int64_t* utt, int segment_value, int strip_sep,
                 int32_t* abnormal, void* stream);

/* ---- single operators, exported for the parity tests ------------------------------------------------------ */
/* C[M,N] = act(A[M,K] * W[N,K]^T + bias).  a/w/c are fp32 device buffers; with dtype == GSTVD_BF16 the operands are
 * rounded to bf16 and the tcgen05 kernel runs, with GSTVD_F32 the SIMT fp32 kernel runs. act: 0 none, 1 erf-GELU. */
int gstvd_op_linear(gstvd_ctx* ctx, int dtype, int M, int N, int K, const float* a, const float* w, const float* bias,
                    int act, float* c, void* stream);
/* y = LayerNorm(x + residual) with eps 1e-12 inside the sqrt (models/vilbert_dialog.py:283-296). residual may be NULL */
int gstvd_op_add_layernorm(gstvd_ctx* ctx, int dtype, int rows, int width, const float* x, const float* residual,
                           const float* gamma, const float* beta, float* y, void* stream);
/* softmax(q k^T / sqrt(D) + (1-mask)*neg [+ causal]) v ; q [B,Lq,H*D], k/v [B,Lk,H*D], mask [B,Lk] or NULL */
int gstvd_op_attention(gstvd_ctx* ctx, int dtype, int B, int H, int Lq, int Lk, int D, const float* q, const float* k,
                       const float* v, const float* mask, float neg, int causal, float* out, void* stream);
/* One beam-search step on caller-supplied logits fp32 [B*K, V] (ldl = row stride).  State lives in the context:
 * call gstvd_op_beam_begin first, then step max_new times, then gstvd_op_beam_end.  Outputs per step:
 * beam_idx / next_tokens int32 [B, K], next_scores fp32 [B, K]. */
int gstvd_op_beam_begin(gstvd_ctx* ctx, int B, int K, int max_new, void* stream);
int gstvd_op_beam_step(gstvd_ctx* ctx, const float* logits, int64_t ldl, int32_t* beam_idx, int32_t* next_tokens,
                       float* next_scores, void* stream);
int gstvd_op_beam_end(gstvd_ctx* ctx, int64_t* out_ids, float* out_scores, void* stream);
/* top-k filter + greedy/multinomial on caller-supplied logits fp32 [rows, V]; prefix int64 [rows, prefix_len] holds
 * the decoded tokens so far (for n-gram blocking, may be NULL); out_tokens int32 [rows].  The logits processors of params act
 * with d = prefix ([SEP] read as [PAD]) and need prefix_len = step + 1 <= 64 */
int gstvd_op_sample(gstvd_ctx* ctx, int rows, const float* logits, int64_t ldl, const gstvd_gen_params* params,
                    const int64_t* hist_ids, const int64_t* hist_segments, int Lh, const int64_t* prefix, int prefix_len,
                    int step, int32_t* out_tokens, void* stream);

/* The deferred-LayerNorm chain of a decode step on caller-supplied operands (bf16 contexts; all buffers fp32 on the device,
 * rounded to bf16 inside): the dense -> LayerNorm(x + input) pairs of HF BertSelfOutput / BertOutput (call site
 * models/visual_dialog_decoder.py:300-311) without a LayerNorm kernel in between -
 *   x1 = a1 w1^T + b1 + res0            stored raw (bf16) with per-32-column row statistics
 *   x2 = LN1(x1) w2^T + b2 + LN1(x1)    LN1 applied inside the second GEMM (folded weights for the operand, on the fly for the residual)
 *   out = LN2(x2)                       materialised from the stored statistics
 * a1 [M,K1], w1 [N,K1], res0 [M,N], w2 [N,N]; N % 64 == 0, N <= 1024, K1 % 64 == 0, M <= 512.  out_x1 (raw x1, may be NULL). */
int gstvd_op_deferred_ln_chain(gstvd_ctx* ctx, int M, int N, int K1, const float* a1, const float* w1, const float* b1,
                               const float* res0, const float* gamma1, const float* beta1, const float* w2, const float* b2,
                               const float* gamma2, const float* beta2, float* out, float* out_x1, void* stream);

/* The decode step's attention kernels one at a time, on caller-supplied data (parity tests).  All float buffers are fp32 on the
 * device; dtype GSTVD_BF16 rounds them to bf16 inside and converts the results back.  Each call uses its own one-layer geometry,
 * not the context's caches.  `kernel` forces one kernel (-1: the decode step's own choice, environment switches included); a
 * forced kernel that cannot run the arguments is refused with GSTVD_ERR_UNSUPPORTED before anything is launched.
 *
 * Self-attention of one new position per (image, beam) row; kernel 0 = the first kernel (fp32 / bf16, D 64 or 128), 1 = the lean
 * bf16 / D = 64 kernel (the only reader of an ancestry table).
 *   qkv [B*K, 3*heads*D]; cache [2 (k, v)][B][T][K][heads*D] in/out: the new k / v are written at position P0_b + step of the row's
 *   own beam slot, P0_b = p0s[b] (int32 [B] on the device, 0 <= p0s[b] <= P0; per-image decoder prefix lengths - 1) or P0 when
 *   p0s is NULL; the row attends over positions 0 .. P0_b + step;
 *   prefix_qkv [B*P0, 3*heads*D] or NULL: its k / v are first stored at positions 0..P0-1 of every slot;
 *   anc uint8 [B*K][T <= 32 ? 32 : 64] or NULL: position t of row (b, k) is read from slot anc[b*K + k][t];
 *   step_known != 0 hands the step to the launch (loads bounded by it), else only through device memory (every row loaded, masked);
 *   out [B*K, heads*D].  K <= 8, T <= 64, P0 + step < T. */
int gstvd_op_dec_self_attn(gstvd_ctx* ctx, int dtype, int kernel, int B, int K, int heads, int D, int T, int P0, const int32_t* p0s,
                           int step, int step_known, const float* qkv, const float* prefix_qkv, float* cache, const uint8_t* anc,
                           float* out, void* stream);
/* Cross-attention of B*K rows (K per image) over cross_kv [B][2*heads (k heads, then v heads)][Le][D] with mask [B, Le] (NULL:
 * all ones; additive (1 - m) * -1e9).  kernel 0 = warp-per-item TMA, 1 = CTA-per-item TMA, 2 = mma.sync, 3 = SIMT, 4 = generic.
 * use_cross_len != 0 (needs the mask): the TMA kernels fetch keys up to cross_len[b] = last non-zero mask entry + 1 (Le for an
 * all-zero row), as in the decode step; out_cross_len int32 [B] (may be NULL) receives it.  q / out [B*K, heads*D]; K <= 8, Le <= 512. */
int gstvd_op_dec_cross_attn(gstvd_ctx* ctx, int dtype, int kernel, int B, int K, int heads, int D, int Le, const float* q,
                            const float* cross_kv, const float* mask, int use_cross_len, int32_t* out_cross_len, float* out,
                            void* stream);
/* One beam-ancestry update of a caller-supplied table anc uint8 [B*K][T <= 32 ? 32 : 64] (in place): beam_idx int32 [B, K] holds each
 * new beam's parent; row (b, k) becomes the parent's row over positions < P0_b + step and holds the parent at P0_b + step, with
 * P0_b = p0s[b] (int32 [B] on the device, 0 <= p0s[b] <= P0) or P0 when p0s is NULL. */
int gstvd_op_anc_update(gstvd_ctx* ctx, int B, int K, int T, int P0, const int32_t* p0s, int step, const int32_t* beam_idx, uint8_t* anc,
                        void* stream);

/* Test access to the self-attention KV cache in the layout a generate call with (B, K) uses: buf fp32 [B, max_new_tokens, K,
 * hidden] on the device for one (layer, kv in {0: key, 1: value}); write != 0 stores buf into the cache (rounded to the
 * compute dtype), else reads it back.  Lets the tests check gstvd_reorder_cache against index_select(0, beam_idx) directly. */
int gstvd_debug_self_cache(gstvd_ctx* ctx, int write, int B, int K, int layer, int kv, float* buf, void* stream);

/* Measurement aid (bench.py's decode-step roofline): out int32 [B] (device) = keys of each image's resident cross-attention K/V
 * that a decode step fetches (last unmasked key + 1, computed at gstvd_prefill_cross). */
int gstvd_cross_key_counts(gstvd_ctx* ctx, int B, int32_t* out, void* stream);

/* Number of kernels this context has launched since creation (bench.py's gpu_launches). */
int64_t gstvd_launch_count(const gstvd_ctx* ctx);

/* Measurement aid for bench.py's roofline: while enabled, every tcgen05 GEMM launch with at least `min_rows` rows that is
 * issued eagerly (not inside a captured decode graph) is bracketed by a CUDA event pair on its own stream.
 * gstvd_profile_read synchronises the device, returns the summed algorithmic FLOPs (2*M*N*K), algorithmic bytes
 * (operands read once + output written once), summed event time in ms and the number of launches, and resets. */
int gstvd_profile_gemm(gstvd_ctx* ctx, int enable, int min_rows);
int gstvd_profile_read(gstvd_ctx* ctx, double* flops, double* bytes, double* ms, int64_t* launches);

#ifdef __cplusplus
}
#endif
#endif /* GSTVD_H_ */
