// gstvd engine: context (packed weights, workspace, KV caches, CUDA graphs), orchestration of the encoder / decoder
// kernels and the extern "C" boundary declared in include/gstvd.h.
//
// Schedule and arithmetic follow SURVEY.md appendix A, i.e. models/vilbert_dialog.py:806-912 (interleaved text /
// image / connection layers), models/visual_dialog_model.py:131-135 (fusion) and the HF BertLayer decoder
// (call site models/visual_dialog_decoder.py:300-311).
#include <cuda_runtime.h>

#include <cmath>
#include <cstdarg>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <algorithm>
#include <map>
#include <mutex>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/gstvd.h"
#include "common.cuh"
#include "kernels.h"

using namespace gstvd;

namespace gstvd {
bool& pdl_flag() { static thread_local bool f = false; return f; }
bool carveout_max_flag() { static const bool on = getenv("GSTVD_CARVEOUT_MAX") != nullptr; return on; }
}  // namespace gstvd

namespace {

thread_local std::string g_last_error;

#define CUDA_CHECK(expr)                                                                          \
  do {                                                                                            \
    cudaError_t _e = (expr);                                                                      \
    if (_e != cudaSuccess)                                                                        \
      throw std::runtime_error(std::string("CUDA error: ") + cudaGetErrorString(_e) + " at " #expr); \
  } while (0)

struct InvalidArg : std::runtime_error { using std::runtime_error::runtime_error; };
struct StateError : std::runtime_error { using std::runtime_error::runtime_error; };
struct Unsupported : std::runtime_error { using std::runtime_error::runtime_error; };

std::string fmt(const char* f, ...) {
  char buf[512];
  va_list ap; va_start(ap, f); vsnprintf(buf, sizeof buf, f, ap); va_end(ap);
  return buf;
}

struct Linear { int out = 0, in = 0; float* w32 = nullptr; float* b = nullptr; bf16* w16 = nullptr; };
struct LNp { int n = 0; float* g = nullptr; float* b = nullptr; };
struct SelfLayer { Linear qkv, o, f1, f2; LNp ln_att, ln_out; };
struct ConnLayer { Linear qkv1, qkv2, dense1, dense2, v_f1, v_f2, t_f1, t_f2; LNp ln1, ln2, v_ln, t_ln; };
// Deferred LayerNorm (bf16 decode step): a projection whose input is LN(x) multiplies the RAW x by W' = W * gamma instead;
// c / d are the epilogue's correction vectors (GemmArgs::fold_*, launch_fold_ln_weights).
struct FoldLin { int out = 0, in = 0; bf16* w16 = nullptr; float* c = nullptr; float* d = nullptr; };
struct DecLayer { Linear qkv, o, cq, co, f1, f2; LNp ln_att, ln_cross, ln_out; FoldLin qkv_f, cq_f, f1_f; };
struct Slot { float* dst; int64_t numel; bool loaded; };

struct DevBuf {
  void* p = nullptr; size_t bytes = 0;
  void alloc(size_t n) { if (n == 0) n = 16; CUDA_CHECK(cudaMalloc(&p, n)); bytes = n; }
  void release() { if (p) cudaFree(p); p = nullptr; bytes = 0; }
};

// Key of a captured decode graph (gstvd_generate) or round graph (gstvd_round): shapes and selection parameters only, built by
// graph_key.  The n-gram blocking history, the decoder prefix and the round's inputs are copied into context-owned buffers before a
// replay, so the caller's tensor addresses are not part of the key (a caching allocator hands out a new address per batch).  seed and
// row_offset are not either: the graph reads them from device memory, so a replay can use a new seed.  Fields that do not apply to
// a kind of call are 0: Lh / Le for a generate graph; Lt / Lv and the has_* flags (optional inputs, out_scores) for a round graph.
// K = decode rows per image; P = decoder prefix length; has_prefix = 0 for the implicit [CLS] start.
struct GraphKey {
  int B, K, mode, T, top_k, ngram, P, has_prefix, N, G, Lh, Le, Lt, Lv, has_seg, has_att, has_imask, has_scores, no_repeat_ngram, min_length;
  float temperature, top_p, penalty, repetition_penalty;
  bool operator<(const GraphKey& o) const { return std::memcmp(this, &o, sizeof(GraphKey)) < 0; }
};
constexpr size_t kMaxGraphs = 24;      // least-recently-used graphs beyond this are destroyed (an 18-step graph holds ~2k kernel nodes)
struct GraphEntry { cudaGraphExec_t exec; int64_t kernels; uint64_t last_use; };   // kernels per replay, counted during capture
using GraphPool = std::map<GraphKey, GraphEntry>;

}  // namespace

struct gstvd_ctx {
  gstvd_config cfg;
  int device = 0, num_sms = 148, dtype = kF32;
  size_t esz = 4;
  std::string last_error;
  int64_t launches = 0;
  bool finalized = false;

  // geometry
  int H, Hv, Hb, heads, heads_v, heads_b, F, Fv, V, Vpad, Lt_max, Lv_max, Le_max, B_max, T_max, K_max, Ldec_max;
  int dec_layers, dec_heads, dec_F;

  // weights
  DevBuf mat32, mat16, vec32;
  size_t mat_elems = 0, vec_elems = 0;
  std::unordered_map<std::string, Slot> slots;
  float *word = nullptr, *pos = nullptr, *type = nullptr, *type_ext = nullptr; LNp emb_ln;
  Linear img_emb; float *loc_w = nullptr, *loc_b = nullptr; LNp img_ln;
  std::vector<SelfLayer> t_layers, v_layers;
  std::vector<ConnLayer> c_layers;
  Linear t_pool, v_pool, nsp_head, fc_l, fc_v;
  std::vector<DecLayer> d_layers;
  Linear cross_kv;      // all decoder layers' crossattention.self.{key,value}: [layers*2*H, H]
  Linear lm_head;

  // workspace (element type = compute dtype unless noted)
  DevBuf xt, yt, xv, yv, qkv_t, qkv_v, ctx_t, ctx_v, tmp_t, tmp_v, ffn_t, ffn_v, feat_cast, fused, pool;
  DevBuf fused_mask;                                  // fp32 [B, Le]
  DevBuf dh, da, db, dqkv, dctx, dtmp, dffn, dqc;      // decoder activations, rows = max(B*K, B*Ldec)
  DevBuf logits;                                      // fp32 [rows, Vpad]
  DevBuf cross_cache, self_cache;
  DevBuf cross_len;                                   // int32 [B]: keys up to the last unmasked one (launch_cross_len)
  DevBuf labels;                                      // int64 [B*Ldec]
  DevBuf sel_val, sel_idx, logz;                      // [rows, kSelMax]
  DevBuf ban_tokens, ban_count, prefix, seq;          // sample-mode state, one row per decode row (B*K: sampled candidates)
  DevBuf beam_scores, beam_tokens, cur_tokens, beam_idx, beam_done, hyp_score, hyp_len, hyp_tokens, hyp_count, hyp_worst;
  DevBuf d_step, d_seed;
  DevBuf anc;                                         // uint8 [B*K][64]: beam ancestry table (launch_anc_update; rows of 32 up to 32 positions)
  DevBuf dec_prefix_own, dec_prefix_head;             // int64 [B_max, max_dec_len]: decoder prefix of a call; [B, P-1]: its prefill ids
  DevBuf prefix_p0;                                   // int32 [B_max]: each image's decoder prefix length - 1 (DecodeGeom::P0s)
  DevBuf fold16, foldvec;                             // deferred LayerNorm: folded bf16 weights, c / d vectors
  DevBuf st1, st2, st3;                               // float2 [rows][kLnStatStride]: partial row statistics of the raw x1 / x2 / x3
  bool fold_ready = false;
  int64_t stats_ld = 0;                               // row capacity of st1 / st2 / st3 (layout [part][row])
  int enc_B = 0, enc_Le = 0;        // shape of the resident fused states
  int cross_B = 0, cross_Le = 0;    // shape of the resident cross K/V
  // beam op-test state
  int op_B = 0, op_K = 0, op_T = 0;

  GraphPool graphs;                   // decode graphs (gstvd_generate): every decode step of one call
  GraphPool round_graphs;             // whole-round graphs (gstvd_round): encoder + cross-K/V prefill + every decode step of one call
  uint64_t graph_clock = 0;
  DevBuf r_ids, r_seg, r_att, r_feat, r_loc, r_imask, r_out_ids, r_out_scores;   // context-owned copies of a round's inputs / outputs
  DevBuf hist_ids_own, hist_seg_own;                  // int64 [B_max, Lt_max]: n-gram blocking history read by captured graphs
  // optional event profiling of the tcgen05 GEMM launches (bench.py roofline): one event pair per launch
  bool profiling = false; int prof_min_rows = 0;
  struct ProfRec { cudaEvent_t a, b; double flops, bytes; };
  std::vector<ProfRec> prof_pool; size_t prof_used = 0;
  cudaStream_t own_stream = nullptr;     // decode steps run (and are graph-captured) here: the caller may be on the legacy stream
  cudaEvent_t ev_in = nullptr, ev_out = nullptr;

  size_t act_bytes(size_t elems) const { return elems * esz; }
};

namespace {

// ---- weight layout ----------------------------------------------------------------------------------------------
struct Planner {
  gstvd_ctx* c;
  std::vector<std::pair<float**, size_t>> mats, vecs;   // deferred pointer fix-ups: (where, offset)
  size_t mat_off = 0, vec_off = 0;
  struct Pending { std::string name; bool mat; size_t off; int64_t numel; };
  std::vector<Pending> pend;

  size_t take_mat(size_t n) { size_t o = mat_off; mat_off += (n + 63) & ~size_t(63); return o; }
  size_t take_vec(size_t n) { size_t o = vec_off; vec_off += (n + 63) & ~size_t(63); return o; }

  // Linear whose rows are the concatenation of several nn.Linear modules (fused q/k/v etc.)
  void linear(Linear& L, int in, const std::vector<std::pair<std::string, int>>& parts) {
    int out = 0;
    for (auto& p : parts) out += p.second;
    L.out = out; L.in = in;
    size_t wo = take_mat((size_t)out * in), bo = take_vec(out);
    mats.push_back({&L.w32, wo}); vecs.push_back({&L.b, bo});
    int r = 0;
    for (auto& p : parts) {
      pend.push_back({p.first + ".weight", true, wo + (size_t)r * in, (int64_t)p.second * in});
      pend.push_back({p.first + ".bias", false, bo + r, p.second});
      r += p.second;
    }
  }
  void linear1(Linear& L, const std::string& name, int out, int in) { linear(L, in, {{name, out}}); }
  void ln(LNp& l, const std::string& name, int n) {
    l.n = n;
    size_t go = take_vec(n), bo = take_vec(n);
    vecs.push_back({&l.g, go}); vecs.push_back({&l.b, bo});
    pend.push_back({name + ".weight", false, go, n});
    pend.push_back({name + ".bias", false, bo, n});
  }
  void table(float*& ptr, const std::string& name, int64_t numel) {
    size_t o = take_vec(numel);
    vecs.push_back({&ptr, o});
    pend.push_back({name, false, o, numel});
  }
};

void plan_weights(gstvd_ctx* c) {
  const gstvd_config& g = c->cfg;
  Planner P{c};
  const std::string E = "encoder.bert_pretrained.bert.";
  const int H = c->H, Hv = c->Hv, Hb = c->Hb;
  P.table(c->word, E + "embeddings.word_embeddings.weight", (int64_t)g.vocab_size * H);
  P.table(c->pos, E + "embeddings.position_embeddings.weight", (int64_t)g.max_position_embeddings * H);
  P.table(c->type, E + "embeddings.token_type_embeddings.weight", (int64_t)g.type_vocab_size * H);
  P.table(c->type_ext, E + "embeddings.token_type_embeddings_extension.weight", (int64_t)10 * H);
  P.ln(c->emb_ln, E + "embeddings.LayerNorm", H);
  P.linear1(c->img_emb, E + "v_embeddings.image_embeddings", Hv, g.v_feature_size);
  P.table(c->loc_w, E + "v_embeddings.image_location_embeddings.weight", (int64_t)Hv * 5);
  P.table(c->loc_b, E + "v_embeddings.image_location_embeddings.bias", Hv);
  P.ln(c->img_ln, E + "v_embeddings.LayerNorm", Hv);
  auto self_layer = [&](SelfLayer& L, const std::string& p, int h, int f) {
    P.linear(L.qkv, h, {{p + "attention.self.query", h}, {p + "attention.self.key", h}, {p + "attention.self.value", h}});
    P.linear1(L.o, p + "attention.output.dense", h, h);
    P.ln(L.ln_att, p + "attention.output.LayerNorm", h);
    P.linear1(L.f1, p + "intermediate.dense", f, h);
    P.linear1(L.f2, p + "output.dense", h, f);
    P.ln(L.ln_out, p + "output.LayerNorm", h);
  };
  c->t_layers.resize(g.num_hidden_layers);
  for (int i = 0; i < g.num_hidden_layers; ++i) self_layer(c->t_layers[i], E + "encoder.layer." + std::to_string(i) + ".", H, c->F);
  c->v_layers.resize(g.v_num_hidden_layers);
  for (int i = 0; i < g.v_num_hidden_layers; ++i) self_layer(c->v_layers[i], E + "encoder.v_layer." + std::to_string(i) + ".", Hv, c->Fv);
  c->c_layers.resize(g.num_connections);
  for (int i = 0; i < g.num_connections; ++i) {
    ConnLayer& L = c->c_layers[i];
    const std::string p = E + "encoder.c_layer." + std::to_string(i) + ".";
    P.linear(L.qkv1, Hv, {{p + "biattention.query1", Hb}, {p + "biattention.key1", Hb}, {p + "biattention.value1", Hb}});
    P.linear(L.qkv2, H, {{p + "biattention.query2", Hb}, {p + "biattention.key2", Hb}, {p + "biattention.value2", Hb}});
    P.linear1(L.dense1, p + "biOutput.dense1", Hv, Hb);
    P.ln(L.ln1, p + "biOutput.LayerNorm1", Hv);
    P.linear1(L.dense2, p + "biOutput.dense2", H, Hb);
    P.ln(L.ln2, p + "biOutput.LayerNorm2", H);
    P.linear1(L.v_f1, p + "v_intermediate.dense", c->Fv, Hv);
    P.linear1(L.v_f2, p + "v_output.dense", Hv, c->Fv);
    P.ln(L.v_ln, p + "v_output.LayerNorm", Hv);
    P.linear1(L.t_f1, p + "t_intermediate.dense", c->F, H);
    P.linear1(L.t_f2, p + "t_output.dense", H, c->F);
    P.ln(L.t_ln, p + "t_output.LayerNorm", H);
  }
  P.linear1(c->t_pool, E + "t_pooler.dense", Hb, H);
  P.linear1(c->v_pool, E + "v_pooler.dense", Hb, Hv);
  P.linear1(c->nsp_head, "encoder.bert_pretrained.cls.bi_seq_relationship", 2, Hb);
  if (c->dec_layers > 0) {
    P.linear1(c->fc_l, "vlfusion.fc_l", H, H);
    P.linear1(c->fc_v, "vlfusion.fc_v", H, Hv);
    const std::string D = "decoder.decoder.bert.encoder.layer.";
    c->d_layers.resize(c->dec_layers);
    std::vector<std::pair<std::string, int>> kv_parts;
    for (int i = 0; i < c->dec_layers; ++i) {
      DecLayer& L = c->d_layers[i];
      const std::string p = D + std::to_string(i) + ".";
      P.linear(L.qkv, H, {{p + "attention.self.query", H}, {p + "attention.self.key", H}, {p + "attention.self.value", H}});
      P.linear1(L.o, p + "attention.output.dense", H, H);
      P.ln(L.ln_att, p + "attention.output.LayerNorm", H);
      P.linear1(L.cq, p + "crossattention.self.query", H, H);
      kv_parts.push_back({p + "crossattention.self.key", H});
      kv_parts.push_back({p + "crossattention.self.value", H});
      P.linear1(L.co, p + "crossattention.output.dense", H, H);
      P.ln(L.ln_cross, p + "crossattention.output.LayerNorm", H);
      P.linear1(L.f1, p + "intermediate.dense", c->dec_F, H);
      P.linear1(L.f2, p + "output.dense", H, c->dec_F);
      P.ln(L.ln_out, p + "output.LayerNorm", H);
    }
    P.linear(c->cross_kv, H, kv_parts);
    // lm_head.decoder.weight / lm_head.bias (lm_head.decoder.bias is the same tensor, visual_dialog_decoder.py:333-335)
    c->lm_head.out = g.vocab_size; c->lm_head.in = H;
    size_t wo = P.take_mat((size_t)g.vocab_size * H), bo = P.take_vec(g.vocab_size);
    P.mats.push_back({&c->lm_head.w32, wo}); P.vecs.push_back({&c->lm_head.b, bo});
    P.pend.push_back({"decoder.decoder.lm_head.decoder.weight", true, wo, (int64_t)g.vocab_size * H});
    P.pend.push_back({"decoder.decoder.lm_head.bias", false, bo, g.vocab_size});
  }
  c->mat_elems = P.mat_off; c->vec_elems = P.vec_off;
  c->mat32.alloc(c->mat_elems * 4);
  c->vec32.alloc(c->vec_elems * 4);
  CUDA_CHECK(cudaMemset(c->mat32.p, 0, c->mat32.bytes));
  CUDA_CHECK(cudaMemset(c->vec32.p, 0, c->vec32.bytes));
  if (c->dtype == kBF16) c->mat16.alloc(c->mat_elems * 2);
  for (auto& m : P.mats) *m.first = (float*)c->mat32.p + m.second;
  for (auto& v : P.vecs) *v.first = (float*)c->vec32.p + v.second;
  for (auto& p : P.pend) {
    float* base = p.mat ? (float*)c->mat32.p : (float*)c->vec32.p;
    c->slots[p.name] = Slot{base + p.off, p.numel, false};
  }
}

void set_w16(gstvd_ctx* c, Linear& L) { if (L.w32) L.w16 = (bf16*)c->mat16.p + (L.w32 - (float*)c->mat32.p); }

void assign_w16(gstvd_ctx* c) {
  set_w16(c, c->img_emb);
  for (auto& L : c->t_layers) { set_w16(c, L.qkv); set_w16(c, L.o); set_w16(c, L.f1); set_w16(c, L.f2); }
  for (auto& L : c->v_layers) { set_w16(c, L.qkv); set_w16(c, L.o); set_w16(c, L.f1); set_w16(c, L.f2); }
  for (auto& L : c->c_layers) {
    set_w16(c, L.qkv1); set_w16(c, L.qkv2); set_w16(c, L.dense1); set_w16(c, L.dense2);
    set_w16(c, L.v_f1); set_w16(c, L.v_f2); set_w16(c, L.t_f1); set_w16(c, L.t_f2);
  }
  set_w16(c, c->t_pool); set_w16(c, c->v_pool); set_w16(c, c->nsp_head); set_w16(c, c->fc_l); set_w16(c, c->fc_v);
  for (auto& L : c->d_layers) { set_w16(c, L.qkv); set_w16(c, L.o); set_w16(c, L.cq); set_w16(c, L.co); set_w16(c, L.f1); set_w16(c, L.f2); }
  set_w16(c, c->cross_kv); set_w16(c, c->lm_head);
}

// Known checkpoint keys the path does not read.
bool is_ignored_key(const std::string& n) {
  static const char* pats[] = {".q_dense1.", ".q_dense2.", "sep_embeddings", "cls.predictions.", "cls.imagePredictions.",
                               "position_ids"};
  for (auto p : pats) if (n.find(p) != std::string::npos) return true;
  return false;
}

std::string canonical_name(const std::string& n) {
  const std::string de = "decoder.decoder.bert.embeddings.";
  if (n.compare(0, de.size(), de) == 0) return "encoder.bert_pretrained.bert.embeddings." + n.substr(de.size());
  if (n == "decoder.decoder.lm_head.decoder.bias") return "decoder.decoder.lm_head.bias";
  return n;
}

void alloc_workspace(gstvd_ctx* c) {
  const size_t B = c->B_max, Lt = c->Lt_max, Lv = c->Lv_max, Le = c->Le_max;
  const size_t Mt = B * Lt, Mv = B * Lv;
  const size_t H = c->H, Hv = c->Hv, Hb = c->Hb;
  auto A = [&](DevBuf& b, size_t elems) { b.alloc(c->act_bytes(elems)); };
  const size_t wt = std::max(H, Hb), wv = std::max(Hv, Hb);
  A(c->xt, Mt * H); A(c->yt, Mt * H); A(c->xv, Mv * Hv); A(c->yv, Mv * Hv);
  A(c->qkv_t, Mt * 3 * wt); A(c->qkv_v, Mv * 3 * wv);
  A(c->ctx_t, Mt * wt); A(c->ctx_v, Mv * wv);
  A(c->tmp_t, Mt * wt); A(c->tmp_v, Mv * std::max(wv, H));
  A(c->ffn_t, Mt * c->F); A(c->ffn_v, Mv * c->Fv);
  A(c->feat_cast, Mv * c->cfg.v_feature_size);
  A(c->fused, B * Le * H);
  A(c->pool, B * (H + Hv + 3 * Hb + 8));
  c->fused_mask.alloc(B * Le * 4);
  if (c->dec_layers > 0) {
    const size_t K = c->K_max, T = c->T_max;
    const size_t R = std::max(B * K, B * (size_t)c->Ldec_max);
    A(c->dh, R * H); A(c->da, R * H); A(c->db, R * H); A(c->dqkv, R * 3 * H); A(c->dctx, R * H); A(c->dtmp, R * H);
    A(c->dffn, R * c->dec_F); A(c->dqc, R * H);
    c->logits.alloc(R * (size_t)c->Vpad * 4);
    A(c->cross_cache, (size_t)c->dec_layers * B * 2 * H * Le);
    // max_new_tokens + max_dec_len - 1 positions per row: a decoder prefix of P tokens occupies P - 1 positions before the first
    // generated one.  A call's cache stride is its own position count (P - 1 + its max_new_tokens).
    A(c->self_cache, (size_t)c->dec_layers * 2 * B * (T + c->Ldec_max - 1) * K * H);
    c->labels.alloc(B * (size_t)c->Ldec_max * 8);
    c->cross_len.alloc(B * 4);
    c->sel_val.alloc(R * kSelMax * 4); c->sel_idx.alloc(R * kSelMax * 4); c->logz.alloc(R * 4);
    c->ban_tokens.alloc(B * K * Lt * 4); c->ban_count.alloc(B * K * 4);   // one ban list per decode row (beam rows included)
    c->hist_ids_own.alloc(B * Lt * 8); c->hist_seg_own.alloc(B * Lt * 8);
    c->r_ids.alloc(B * Lt * 8); c->r_seg.alloc(B * Lt * 8); c->r_att.alloc(B * Lt * 4);
    c->r_feat.alloc(B * Lv * (size_t)c->cfg.v_feature_size * 4); c->r_loc.alloc(B * Lv * 5 * 4); c->r_imask.alloc(B * Lv * 4);
    // outputs and sample-mode state hold up to K_max rows per image: N-best beams / N sampled candidates
    c->r_out_ids.alloc(B * K * T * 8); c->r_out_scores.alloc(B * K * 4);
    c->prefix.alloc(B * K * (T + c->Ldec_max) * 4); c->seq.alloc(B * K * T * 4);
    c->dec_prefix_own.alloc(B * c->Ldec_max * 8); c->dec_prefix_head.alloc(B * c->Ldec_max * 8); c->prefix_p0.alloc(B * 4);
    c->beam_scores.alloc(B * K * 4); c->beam_tokens.alloc(2 * B * K * T * 4); c->cur_tokens.alloc(R * 4);
    // hypothesis heaps: one per search of K beams with K + 1 slots.  Beam search: B searches of K <= K_max beams; beam sampling: B * N
    // searches of K >= 2 beams with N * K <= K_max, i.e. at most B * K_max / 2 searches and B * (K_max + K_max / 2) slots.
    const size_t S = B * std::max<size_t>(1, K / 2), HS = B * (K + std::max<size_t>(1, K / 2));
    c->beam_idx.alloc(B * K * 4); c->beam_done.alloc(S); c->hyp_score.alloc(HS * 8);
    c->hyp_len.alloc(HS * 4); c->hyp_tokens.alloc(HS * T * 4); c->hyp_count.alloc(S * 4);
    c->hyp_worst.alloc(S * 8);
    c->anc.alloc(B * K * 64);
    CUDA_CHECK(cudaMemset(c->anc.p, 0, B * K * 64));
    c->stats_ld = (int64_t)((R + 15) & ~size_t(15));
    c->st1.alloc(c->stats_ld * kLnStatStride * 8); c->st2.alloc(c->stats_ld * kLnStatStride * 8); c->st3.alloc(c->stats_ld * kLnStatStride * 8);
  }
  c->d_step.alloc(16); c->d_seed.alloc(16);
  CUDA_CHECK(cudaMemset(c->d_step.p, 0, 16));
}

// ---- op wrappers ---------------------------------------------------------------------------------------------------
struct Exec {
  gstvd_ctx* c; cudaStream_t s;
  int dt() const { return c->dtype; }

  void gemm(const void* A, int64_t lda, const Linear& L, void* C, int64_t ldc, int M, int act = 0, bool out_f32 = false,
            int hm_D = 0, int hm_L = 0, int hm_G = 0, int hm_B = 0) {
    GemmArgs a;
    a.A = A; a.lda = lda; a.ldw = L.in; a.bias = L.b; a.C = C; a.ldc = ldc; a.out_f32 = out_f32 ? 1 : 0; a.act = act;
    a.M = M; a.N = L.out; a.K = L.in; a.hm_D = hm_D; a.hm_L = hm_L; a.hm_G = hm_G; a.hm_B = hm_B;
    if (c->dtype == kF32) { a.W = L.w32; c->launches += launch_gemm_simt(a, kF32, s); }
    else {
      a.W = L.w16;
      if (c->cfg.flags & GSTVD_FLAG_DEBUG_SIMT_GEMM) c->launches += launch_gemm_simt(a, kBF16, s);
      else {
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        const bool prof = c->profiling && M >= c->prof_min_rows && c->prof_used < c->prof_pool.size() &&
                          cudaStreamIsCapturing(s, &cs) == cudaSuccess && cs == cudaStreamCaptureStatusNone;
        if (prof) cudaEventRecord(c->prof_pool[c->prof_used].a, s);
        c->launches += launch_gemm_tc(a, c->num_sms, s);
        if (prof) {
          auto& r = c->prof_pool[c->prof_used++];
          cudaEventRecord(r.b, s);
          r.flops = 2.0 * M * (double)L.out * L.in;
          r.bytes = 2.0 * ((double)M * L.in + (double)L.out * L.in) + (out_f32 ? 4.0 : 2.0) * M * (double)L.out;
        }
      }
    }
  }
  // Deferred-LayerNorm GEMM (bf16 decode step): C = act(LN?(A) W^T + b + LN?(res)) stored raw, with optional statistics out.
  //   fold != null : A holds RAW rows whose partial statistics are a_stats (GemmArgs::fold_*), the weights are fold's
  //   res_ln != null : the residual is LN(res) with that layer norm's affine and the partial statistics res_stats
  void gemm_ln(const void* A, int64_t lda, const Linear& L, const FoldLin* fold, const float2* a_stats, void* C, int M, int act,
               const void* res, const LNp* res_ln, const float2* res_stats, float2* stats_out) {
    GemmArgs a;
    a.A = A; a.lda = lda; a.ldw = L.in; a.C = C; a.ldc = L.out; a.act = act; a.M = M; a.N = L.out; a.K = L.in;
    if (fold) { a.W = fold->w16; a.bias = fold->d; a.fold_c = fold->c; a.fold_stats = a_stats; a.fold_parts = L.in / 32; }
    else { a.W = L.w16; a.bias = L.b; }
    a.res = res; a.ldr = L.out;
    if (res_ln) { a.res_stats = res_stats; a.res_parts = L.out / 32; a.res_gamma = res_ln->g; a.res_beta = res_ln->b; }
    a.stats_out = stats_out; a.stats_ld = c->stats_ld;
    c->launches += launch_gemm_tc(a, c->num_sms, s);
  }
  void add_ln(const void* x, const void* res, const LNp& l, void* y, int rows) {
    c->launches += launch_add_layernorm(dt(), rows, l.n, x, l.n, res, l.n, l.g, l.b, y, l.n, s);
  }
  // y = LN(A L^T + bias + res): GEMM into tmp, then add + LayerNorm (the bf16 decode step defers the LayerNorm instead: gemm_ln)
  void gemm_add_ln(const void* A, int64_t lda, const Linear& L, const void* res, const LNp& l, void* tmp, void* y, int M) {
    gemm(A, lda, L, tmp, L.out, M);
    add_ln(tmp, res, l, y, M);
  }
  // q/k/v: rows of `ld` elements holding all heads; one batch = L rows
  void attention(const void* q, int64_t ldq, int Lq, const void* k, const void* v, int64_t ldkv, int Lk, void* o, int64_t ldo,
                 int B, int heads, int D, const float* kmask, float neg, int causal) {
    AttnArgs a;
    a.q = q; a.q_bs = (int64_t)Lq * ldq; a.q_hs = D; a.q_rs = ldq;
    a.k = k; a.k_bs = (int64_t)Lk * ldkv; a.k_hs = D; a.k_rs = ldkv;
    a.v = v; a.v_bs = (int64_t)Lk * ldkv; a.v_hs = D; a.v_rs = ldkv;
    a.o = o; a.o_bs = (int64_t)Lq * ldo; a.o_hs = D; a.o_rs = ldo;
    a.kmask = kmask; a.kmask_bs = Lk; a.neg = neg; a.causal = causal;
    a.B = B; a.H = heads; a.Lq = Lq; a.Lk = Lk; a.D = D; a.kv_batch_div = 1;
    run_attention(a);
  }
  void run_attention(const AttnArgs& a) {
    if (c->dtype == kBF16 && !(c->cfg.flags & GSTVD_FLAG_GENERIC_ATTENTION) && attention_mma_supported(a)) c->launches += launch_attention_mma(a, s);
    else c->launches += launch_attention_generic(a, dt(), s);
  }
  char* off(void* p, size_t elems) const { return (char*)p + elems * c->esz; }
  const char* off(const void* p, size_t elems) const { return (const char*)p + elems * c->esz; }
};

void self_layer_fwd(Exec& X, const SelfLayer& L, void* x, void* y, void* qkv, void* ctx, void* tmp, void* ffn, int B, int Lq,
                    int heads, const float* mask) {
  gstvd_ctx* c = X.c;
  const int h = L.o.out, M = B * Lq, D = h / heads;
  X.gemm(x, h, L.qkv, qkv, 3 * h, M);
  X.attention(qkv, 3 * h, Lq, X.off(qkv, h), X.off(qkv, 2 * h), 3 * h, Lq, ctx, h, B, heads, D, mask, -10000.0f, 0);
  X.gemm(ctx, h, L.o, tmp, h, M);
  X.add_ln(tmp, x, L.ln_att, y, M);
  X.gemm(y, h, L.f1, ffn, L.f1.out, M, 1);
  X.gemm(ffn, L.f1.out, L.f2, tmp, h, M);
  X.add_ln(tmp, y, L.ln_out, x, M);
  (void)c;
}

// XT runs the text-stream work, XV the image-stream work (the same Exec: running the image stream on a second CUDA stream was
// measured slower once several batches are in flight, profiles/r2_switch_ab.txt).
void conn_layer_fwd(Exec& XT, Exec& XV, const ConnLayer& L, int B, int Lt, int Lv, const float* tmask, const float* vmask) {
  gstvd_ctx* c = XT.c;
  const int H = c->H, Hv = c->Hv, Hb = c->Hb, D = Hb / c->heads_b, Mt = B * Lt, Mv = B * Lv;
  void *xt = c->xt.p, *yt = c->yt.p, *xv = c->xv.p, *yv = c->yv.p;
  void *qv = c->qkv_v.p, *qt = c->qkv_t.p;
  XV.gemm(xv, Hv, L.qkv1, qv, 3 * Hb, Mv);      // query1 | key1 | value1  (image stream)
  XT.gemm(xt, H, L.qkv2, qt, 3 * Hb, Mt);       // query2 | key2 | value2  (text stream)
  // text queries over image keys/values -> ctx_t ; image queries over text keys/values -> ctx_v  (:671-710)
  XT.attention(qt, 3 * Hb, Lt, XT.off(qv, Hb), XT.off(qv, 2 * Hb), 3 * Hb, Lv, c->ctx_t.p, Hb, B, c->heads_b, D, vmask, -10000.0f, 0);
  XV.attention(qv, 3 * Hb, Lv, XV.off(qt, Hb), XV.off(qt, 2 * Hb), 3 * Hb, Lt, c->ctx_v.p, Hb, B, c->heads_b, D, tmask, -10000.0f, 0);
  // BertBiOutput with the contexts swapped into the opposite stream (:765, :732-744)
  XV.gemm(c->ctx_v.p, Hb, L.dense1, c->tmp_v.p, Hv, Mv);
  XV.add_ln(c->tmp_v.p, xv, L.ln1, yv, Mv);
  XT.gemm(c->ctx_t.p, Hb, L.dense2, c->tmp_t.p, H, Mt);
  XT.add_ln(c->tmp_t.p, xt, L.ln2, yt, Mt);
  XV.gemm(yv, Hv, L.v_f1, c->ffn_v.p, c->Fv, Mv, 1);
  XV.gemm(c->ffn_v.p, c->Fv, L.v_f2, c->tmp_v.p, Hv, Mv);
  XV.add_ln(c->tmp_v.p, yv, L.v_ln, xv, Mv);
  XT.gemm(yt, H, L.t_f1, c->ffn_t.p, c->F, Mt, 1);
  XT.gemm(c->ffn_t.p, c->F, L.t_f2, c->tmp_t.p, H, Mt);
  XT.add_ln(c->tmp_t.p, yt, L.t_ln, xt, Mt);
}

// Deferred LayerNorm weights of the decoder (bf16 contexts): per layer cq' = cq * gamma(ln_att), f1' = f1 * gamma(ln_cross) and,
// from layer 1 on, qkv' = qkv * gamma(ln_out of the layer below), each with its c / d vectors.  113 MB at the reference geometry.
void prepare_fold(gstvd_ctx* c, cudaStream_t s) {
  c->fold_ready = false;
  if (c->dtype != kBF16 || c->dec_layers == 0 || c->H % 64 != 0 || c->H > 32 * kLnStatStride) return;
  const size_t H = c->H, F = c->dec_F;
  const size_t per_layer_mat = (H + F + 3 * H) * H, per_layer_vec = 2 * (H + F + 3 * H);
  if (!c->fold16.p) { c->fold16.alloc(per_layer_mat * c->dec_layers * 2); c->foldvec.alloc(per_layer_vec * c->dec_layers * 4); }
  bf16* m = (bf16*)c->fold16.p; float* v = (float*)c->foldvec.p;
  auto prep = [&](FoldLin& f, const Linear& L, const LNp& ln) {
    f.out = L.out; f.in = L.in; f.w16 = m; f.c = v; f.d = v + L.out;
    m += (size_t)L.out * L.in; v += 2 * (size_t)L.out;
    c->launches += launch_fold_ln_weights(L.out, L.in, L.w32, ln.g, ln.b, L.b, f.w16, f.c, f.d, s);
  };
  for (int l = 0; l < c->dec_layers; ++l) {
    DecLayer& L = c->d_layers[l];
    prep(L.cq_f, L.cq, L.ln_att);
    prep(L.f1_f, L.f1, L.ln_cross);
    if (l > 0) prep(L.qkv_f, L.qkv, c->d_layers[l - 1].ln_out);
  }
  c->fold_ready = true;
}

void check_ready(gstvd_ctx* c) { if (!c->finalized) throw StateError("weights not finalized: call gstvd_finalize_weights first"); }

// Programmatic dependent launch for every launch_k kernel enqueued in the scope: each of them starts with its prologue
// (barrier init, TMEM allocation, weight / gamma prefetch) while the predecessor drains and calls griddepcontrol.wait before
// it touches the predecessor's output.  Kernels launched with <<<>>> inside the scope keep full stream ordering.
struct PdlScope {
  bool prev;
  explicit PdlScope(bool on) : prev(pdl_flag()) { pdl_flag() = on; }
  ~PdlScope() { pdl_flag() = prev; }
};

void do_encode(gstvd_ctx* c, int B, int Lt, int Lv, const int64_t* ids, const int64_t* seg, const float* att, const float* feat,
               const float* loc, const float* imask, float* out_t, float* out_v, float* out_fused, float* out_fused_mask,
               float* out_nsp, cudaStream_t s) {
  check_ready(c);
  if (B < 1 || B > c->B_max || Lt < 1 || Lt > c->Lt_max || Lv < 1 || Lv > c->Lv_max)
    throw InvalidArg(fmt("encode: shape B=%d Lt=%d Lv=%d exceeds capacity (%d, %d, %d)", B, Lt, Lv, c->B_max, c->Lt_max, c->Lv_max));
  if (!ids || !feat || !loc) throw InvalidArg("encode: input_ids / image_feat / image_loc must not be NULL");
  PdlScope pdl_scope(!(c->cfg.flags & GSTVD_FLAG_NO_PDL));
  if (Lt > c->cfg.max_position_embeddings) throw InvalidArg("encode: Lt exceeds max_position_embeddings");
  Exec X{c, s};
  Exec& XV = X;                               // image-stream work
  const int H = c->H, Hv = c->Hv, Mt = B * Lt, Mv = B * Lv;
  c->launches += launch_embed_text(c->dtype, Mt, Lt, H, ids, seg, nullptr, 0, c->word, c->pos, c->type, c->type_ext,
                                   c->cfg.type_vocab_size, c->emb_ln.g, c->emb_ln.b, c->xt.p, s);
  const void* feat_in = feat;
  if (c->dtype != kF32) {
    c->launches += launch_cast_f32_to(c->dtype, feat, c->feat_cast.p, (int64_t)Mv * c->cfg.v_feature_size, XV.s);
    feat_in = c->feat_cast.p;
  }
  XV.gemm(feat_in, c->cfg.v_feature_size, c->img_emb, c->tmp_v.p, Hv, Mv);
  c->launches += launch_image_embed_ln(c->dtype, Mv, Hv, c->tmp_v.p, loc, c->loc_w, c->loc_b, c->img_ln.g, c->img_ln.b, c->xv.p, XV.s);

  auto text_layer = [&](int i) { self_layer_fwd(X, c->t_layers[i], c->xt.p, c->yt.p, c->qkv_t.p, c->ctx_t.p, c->tmp_t.p, c->ffn_t.p, B, Lt, c->heads, att); };
  auto image_layer = [&](int i) { self_layer_fwd(XV, c->v_layers[i], c->xv.p, c->yv.p, c->qkv_v.p, c->ctx_v.p, c->tmp_v.p, c->ffn_v.p, B, Lv, c->heads_v, imask); };
  int v_start = 0, t_start = 0;
  for (int n = 0; n < c->cfg.num_connections; ++n) {          // models/vilbert_dialog.py:831-905
    const int v_end = c->cfg.v_biattention_id[n], t_end = c->cfg.t_biattention_id[n];
    for (int i = v_start; i < v_end; ++i) image_layer(i);
    for (int i = t_start; i < t_end; ++i) text_layer(i);
    conn_layer_fwd(X, XV, c->c_layers[n], B, Lt, Lv, att, imask);
    v_start = v_end; t_start = t_end;
  }
  for (int i = v_start; i < c->cfg.v_num_hidden_layers; ++i) image_layer(i);
  for (int i = t_start; i < c->cfg.num_hidden_layers; ++i) text_layer(i);

  if (out_t) c->launches += launch_cast_to_f32(c->dtype, c->xt.p, out_t, (int64_t)Mt * H, s);
  if (out_v) c->launches += launch_cast_to_f32(c->dtype, c->xv.p, out_v, (int64_t)Mv * Hv, s);
  if (out_nsp) {
    // poolers + bi_seq_relationship, fusion 'mul' (models/vilbert_dialog.py:915-941, :1030-1038)
    const int Hb = c->Hb;
    char* p = (char*)c->pool.p;
    void* t0 = p; void* v0 = X.off(t0, (size_t)B * H); void* pt = X.off(v0, (size_t)B * Hv);
    void* pv = X.off(pt, (size_t)B * Hb); void* pm = X.off(pv, (size_t)B * Hb);
    c->launches += launch_gather_first_rows(c->dtype, B, Lt, H, c->xt.p, t0, s);
    c->launches += launch_gather_first_rows(c->dtype, B, Lv, Hv, c->xv.p, v0, s);
    X.gemm(t0, H, c->t_pool, pt, Hb, B);
    X.gemm(v0, Hv, c->v_pool, pv, Hb, B);
    c->launches += launch_relu_mul(c->dtype, (int64_t)B * Hb, pt, pv, pm, s);
    X.gemm(pm, Hb, c->nsp_head, out_nsp, 2, B, 0, true);
  }
  if (c->dec_layers > 0) {
    // VLFusion: cat(fc_v(v), fc_l(t)) with image rows first (models/visual_dialog_model.py:131-135)
    X.gemm(c->xv.p, Hv, c->fc_v, c->tmp_v.p, H, Mv);
    X.gemm(c->xt.p, H, c->fc_l, c->tmp_t.p, H, Mt);
    c->launches += launch_concat_fused(c->dtype, B, Lv, Lt, H, c->tmp_v.p, c->tmp_t.p, c->fused.p, imask, att, (float*)c->fused_mask.p, s);
    c->enc_B = B; c->enc_Le = Lv + Lt;
    if (out_fused) c->launches += launch_cast_to_f32(c->dtype, c->fused.p, out_fused, (int64_t)B * (Lv + Lt) * H, s);
    if (out_fused_mask) CUDA_CHECK(cudaMemcpyAsync(out_fused_mask, c->fused_mask.p, (size_t)B * (Lv + Lt) * 4, cudaMemcpyDeviceToDevice, s));
  } else if (out_fused || out_fused_mask) {
    throw InvalidArg("encode: fused outputs requested from an encoder-only context");
  }
}

void do_prefill(gstvd_ctx* c, int B, int Le, const float* enc_hidden, const float* enc_mask, cudaStream_t s) {
  check_ready(c);
  if (c->dec_layers == 0) throw StateError("prefill_cross: encoder-only context");
  if (B < 1 || B > c->B_max || Le < 1 || Le > c->Le_max) throw InvalidArg("prefill_cross: shape exceeds capacity");
  PdlScope pdl_scope(!(c->cfg.flags & GSTVD_FLAG_NO_PDL));
  Exec X{c, s};
  const int H = c->H;
  if (enc_hidden) {
    c->launches += launch_cast_f32_to(c->dtype, enc_hidden, c->fused.p, (int64_t)B * Le * H, s);
    if (enc_mask) CUDA_CHECK(cudaMemcpyAsync(c->fused_mask.p, enc_mask, (size_t)B * Le * 4, cudaMemcpyDeviceToDevice, s));
    else {
      std::vector<float> ones((size_t)B * Le, 1.f);
      CUDA_CHECK(cudaMemcpyAsync(c->fused_mask.p, ones.data(), ones.size() * 4, cudaMemcpyHostToDevice, s));
      CUDA_CHECK(cudaStreamSynchronize(s));
    }
    c->enc_B = B; c->enc_Le = Le;
  } else if (c->enc_B != B || c->enc_Le != Le) {
    throw StateError(fmt("prefill_cross: resident encoder states are [%d, %d], asked for [%d, %d]", c->enc_B, c->enc_Le, B, Le));
  }
  const int D = H / c->dec_heads;
  // one GEMM for every layer's K and V, written head-major: [layer][image][kv*heads + h][Le][D]
  X.gemm(c->fused.p, H, c->cross_kv, c->cross_cache.p, 0, B * Le, 0, false, D, Le, 2 * c->dec_heads, B);
  c->launches += launch_cross_len(B, Le, (const float*)c->fused_mask.p, (int*)c->cross_len.p, s);
  c->cross_B = B; c->cross_Le = Le;
}

// T = new tokens; P = decoder prefix length (its first P - 1 positions are prefilled, the last one is the first step's input).
// ragged: a caller's prefix of P > 1 columns, whose rows may end early at a negative id; the decode kernels then read every image's
// own length from the context buffer decode_init fills (a P = 1 prefix has one length and keeps the uniform path).
DecodeGeom make_geom(gstvd_ctx* c, int B, int K, int T, int P = 1, bool ragged = false) {
  DecodeGeom g;
  g.B = B; g.K = K; g.H = c->H; g.heads = c->dec_heads; g.D = c->H / c->dec_heads; g.layers = c->dec_layers; g.T = P - 1 + T; g.Le = c->cross_Le;
  g.P0 = P - 1;
  if (ragged && P > 1) g.P0s = (const int*)c->prefix_p0.p;
  return g;
}

BeamBuffers beam_buffers(gstvd_ctx* c) {
  BeamBuffers bb;
  bb.beam_scores = (float*)c->beam_scores.p; bb.tokens = (int32_t*)c->beam_tokens.p; bb.cur_tokens = (int32_t*)c->cur_tokens.p;
  bb.beam_idx = (int32_t*)c->beam_idx.p; bb.done = (uint8_t*)c->beam_done.p; bb.hyp_score = (double*)c->hyp_score.p;
  bb.hyp_len = (int32_t*)c->hyp_len.p; bb.hyp_tokens = (int32_t*)c->hyp_tokens.p; bb.hyp_count = (int32_t*)c->hyp_count.p;
  bb.hyp_worst = (double*)c->hyp_worst.p; bb.d_step = (int*)c->d_step.p;
  return bb;
}

// Teacher-forced decoder layer stack (HF BertLayer: causal self-attention, cross-attention, FFN) over B sequences of L positions whose
// embeddings are in c->dh; `options` consecutive sequences share one image's cross K/V.  kv != null (decoder prefix prefill): after
// each layer's q|k|v GEMM that layer's K / V rows are stored into every beam slot of the self cache, and the last layer stops there
// (its output feeds nothing: no FFN, no LM head).
void dec_teacher_layers(gstvd_ctx* c, Exec& X, int B, int L, const float* dec_mask, int options, const DecodeGeom* kv) {
  const int H = c->H, M = B * L, D = H / c->dec_heads, Le = c->cross_Le;
  const int64_t per_image = (int64_t)2 * c->dec_heads * Le * D;
  for (int l = 0; l < c->dec_layers; ++l) {
    const DecLayer& Ly = c->d_layers[l];
    X.gemm(c->dh.p, H, Ly.qkv, c->dqkv.p, 3 * H, M);
    if (kv) {
      c->launches += launch_prefix_kv_store(c->dtype, *kv, l, c->dqkv.p, c->self_cache.p, X.s);
      if (l == c->dec_layers - 1) return;
    }
    X.attention(c->dqkv.p, 3 * H, L, X.off(c->dqkv.p, H), X.off(c->dqkv.p, 2 * H), 3 * H, L, c->dctx.p, H, B, c->dec_heads, D, dec_mask,
                -10000.0f, 1);
    X.gemm(c->dctx.p, H, Ly.o, c->dtmp.p, H, M);
    X.add_ln(c->dtmp.p, c->dh.p, Ly.ln_att, c->da.p, M);
    X.gemm(c->da.p, H, Ly.cq, c->dqc.p, H, M);
    {
      AttnArgs a;
      const char* kbase = (const char*)c->cross_cache.p + (size_t)l * (B / options) * per_image * c->esz;
      a.q = c->dqc.p; a.q_bs = (int64_t)L * H; a.q_hs = D; a.q_rs = H;
      a.k = kbase; a.k_bs = per_image; a.k_hs = (int64_t)Le * D; a.k_rs = D;
      a.v = kbase + (size_t)c->dec_heads * Le * D * c->esz; a.v_bs = per_image; a.v_hs = a.k_hs; a.v_rs = D;
      a.o = c->dctx.p; a.o_bs = (int64_t)L * H; a.o_hs = D; a.o_rs = H;
      a.kmask = (const float*)c->fused_mask.p; a.kmask_bs = Le; a.neg = -1e9f; a.causal = 0;
      a.B = B; a.H = c->dec_heads; a.Lq = L; a.Lk = Le; a.D = D; a.kv_batch_div = options;
      X.run_attention(a);
    }
    X.gemm(c->dctx.p, H, Ly.co, c->dtmp.p, H, M);
    X.add_ln(c->dtmp.p, c->da.p, Ly.ln_cross, c->db.p, M);
    X.gemm(c->db.p, H, Ly.f1, c->dffn.p, c->dec_F, M, 1);
    X.gemm(c->dffn.p, c->dec_F, Ly.f2, c->dtmp.p, H, M);
    X.add_ln(c->dtmp.p, c->db.p, Ly.ln_out, c->dh.p, M);
  }
}

// Decoder prefix prefill: a teacher-forced pass over the first P0 = P - 1 prefix positions of the g.B images (ids in
// c->dec_prefix_head, [SEP] embedded as [PAD] like the in-place replacement of models/visual_dialog_decoder.py:57) that leaves every
// layer's K / V of those positions in the self cache.  P = 1 launches nothing.  A shorter prefix (image b: P_b = g.p0(b) + 1 tokens)
// runs in the same pass with its negative ids embedded as [PAD]: the pass is causal, so positions below P_b - 1 see only the image's
// own prefix and are exact; the rest are padding that b's decode steps overwrite before they read them.
void prefix_prefill(gstvd_ctx* c, const DecodeGeom& g, cudaStream_t s) {
  if (g.P0 == 0) return;
  PdlScope pdl_scope(!(c->cfg.flags & GSTVD_FLAG_NO_PDL));
  Exec X{c, s};
  c->launches += launch_embed_text(c->dtype, g.B * g.P0, g.P0, c->H, (const int64_t*)c->dec_prefix_head.p, nullptr, nullptr, 1, c->word, c->pos,
                                   c->type, c->type_ext, c->cfg.type_vocab_size, c->emb_ln.g, c->emb_ln.b, c->dh.p, s);
  dec_teacher_layers(c, X, g.B, g.P0, nullptr, 1, &g);
}

// Copies the caller's decoder prefix [B, P] into the context (captured graphs read it there) and its first P - 1 columns, the prefill
// ids, into the compact [B, P - 1] buffer.  Returns the context copy, or null for the implicit [CLS] start (prefix == null).
const int64_t* stage_prefix(gstvd_ctx* c, int B, const int64_t* prefix, int P, cudaStream_t s) {
  if (!prefix) return nullptr;
  CUDA_CHECK(cudaMemcpyAsync(c->dec_prefix_own.p, prefix, (size_t)B * P * 8, cudaMemcpyDeviceToDevice, s));
  if (P > 1)
    CUDA_CHECK(cudaMemcpy2DAsync(c->dec_prefix_head.p, (size_t)(P - 1) * 8, prefix, (size_t)P * 8, (size_t)(P - 1) * 8, B,
                                 cudaMemcpyDeviceToDevice, s));
  return (const int64_t*)c->dec_prefix_own.p;
}

// Selection state of a decode call: beams / sample rows start from the last token of the prefix (the [CLS] when it is null).  The same
// launch writes every image's prefix length - 1 into g.P0s when the geometry has per-image lengths.
void decode_init(gstvd_ctx* c, const DecodeGeom& g, const gstvd_gen_params& gp, const int64_t* prefix, cudaStream_t s) {
  const int P = g.P0 + 1, T = gp.max_new_tokens;
  int* p0s = const_cast<int*>(g.P0s);
  if (gp.mode == GSTVD_SELECT_BEAM)
    c->launches += launch_beam_init(beam_buffers(c), g.B, g.K, gp.num_beam_groups, 1, T, 101, prefix, P, p0s, s);
  else if (gp.mode == GSTVD_SELECT_BEAM_SAMPLE) {
    const int K = gp.num_beams, N = g.K / K;      // N searches of K beams per image, all beams at score 0
    c->launches += launch_beam_init(beam_buffers(c), g.B * N, K, K, N, T, 101, prefix, P, p0s, s);
  } else c->launches += launch_sample_init(g.B * g.K, g.K, T, 101, (int32_t*)c->seq.p, (int32_t*)c->cur_tokens.p, (int32_t*)c->prefix.p, P + T, (int*)c->d_step.p,
                                         prefix, P, p0s, s);
}

// The request's logits processors; the caller fills in where the rows' decoder input lives.
LogitsProcs logits_procs(const gstvd_gen_params& gp) {
  LogitsProcs p;
  p.repetition_penalty = gp.repetition_penalty; p.no_repeat_ngram = gp.no_repeat_ngram_size; p.min_length = gp.min_length;
  return p;
}

// One decode step for all M = B*K rows: embeddings -> 12 x [self-attn over cache, cross-attn, FFN] -> LM head -> selection.
// step_host = index of this step when the caller knows it (it always does: eager loops and the captured graph both unroll the
// steps), so kernels that only need it to bound their loads take it as a launch parameter instead of reading *d_step first.
// prefix: int64 [B, P] decoder prefix (P = g.P0 + 1), null for the [CLS] start; image b's own length is g.p0(b) + 1.
void decode_step(gstvd_ctx* c, const DecodeGeom& g, const gstvd_gen_params& gp, const int64_t* prefix, const int64_t* hist_ids,
                 const int64_t* hist_seg, int Lh, cudaStream_t s, int step_host) {
  Exec X{c, s};
  PdlScope pdl_scope(!(c->cfg.flags & GSTVD_FLAG_NO_PDL));
  const int H = c->H, M = g.B * g.K;
  const int P = g.P0 + 1, Tn = g.T - g.P0;          // prefix length, new tokens (stride of the token buffers)
  const int* d_step = (const int*)c->d_step.p;
  // Beam mode with the lean self-attention kernel: the cache is never gathered, the kernel reads each history position from the
  // slot recorded in the ancestry table (token ids identical to the gather, +3 % dialogs/s; env GSTVD_SELF_ANC=0 restores the gather)
  const char* anc_env = getenv("GSTVD_SELF_ANC");
  const bool beams = gp.mode == GSTVD_SELECT_BEAM || gp.mode == GSTVD_SELECT_BEAM_SAMPLE;
  const bool use_anc = beams && (anc_env == nullptr || atoi(anc_env) != 0) &&
                       dec_self_attn_v2_active(c->dtype, g, c->dqkv.p, c->self_cache.p, c->dctx.p);
  const uint8_t* anc = use_anc ? (const uint8_t*)c->anc.p : nullptr;
  c->launches += launch_embed_step(c->dtype, M, H, (const int32_t*)c->cur_tokens.p, g.P0, g.P0s, g.K, d_step, c->word, c->pos, c->type,
                                   c->emb_ln.g, c->emb_ln.b, c->dh.p, s);
  // Deferred LayerNorm (default for bf16): no LayerNorm kernel inside the layer stack - the three dense -> LN(x + input) pairs of a
  // layer store raw sums + partial row statistics, their consumers normalise on the fly (GemmArgs::fold_* / res_*), and one
  // ln_apply_stats launch materialises the last layer's output for the LM head.  36 launches and 36 dependent stages per step less.
  static const bool defer_env = [] { const char* e = getenv("GSTVD_DEFER_LN"); return e == nullptr || atoi(e) != 0; }();
  const bool defer = defer_env && c->fold_ready && c->dtype == kBF16 && !(c->cfg.flags & GSTVD_FLAG_DEBUG_SIMT_GEMM) && M <= 512;
  if (defer) {
    float2 *st1 = (float2*)c->st1.p, *st2 = (float2*)c->st2.p, *st3 = (float2*)c->st3.p;
    void *x1 = c->da.p, *x2 = c->db.p, *x3 = c->dtmp.p;
    for (int l = 0; l < c->dec_layers; ++l) {
      const DecLayer& L = c->d_layers[l];
      const LNp* ln_below = l > 0 ? &c->d_layers[l - 1].ln_out : nullptr;
      // q|k|v from LN_out(x3 of the layer below) (layer 0: from the embedding output, already normalised)
      if (l == 0) X.gemm(c->dh.p, H, L.qkv, c->dqkv.p, 3 * H, M);
      else X.gemm_ln(x3, H, L.qkv, &L.qkv_f, st3, c->dqkv.p, M, 0, nullptr, nullptr, nullptr, nullptr);
      c->launches += launch_dec_self_attn(c->dtype, g, l, c->dqkv.p, c->self_cache.p, d_step, step_host, anc, c->dctx.p, s, kDecDefault);
      // x1 = o(ctx) + input
      X.gemm_ln(c->dctx.p, H, L.o, nullptr, nullptr, x1, M, 0, l == 0 ? c->dh.p : x3, ln_below, st3, st1);
      X.gemm_ln(x1, H, L.cq, &L.cq_f, st1, c->dqc.p, M, 0, nullptr, nullptr, nullptr, nullptr);
      if (dec_cross_tma_supported(c->dtype, g))
        c->launches += launch_dec_cross_tma(g, l, c->dqc.p, c->cross_cache.p, (const float*)c->fused_mask.p, (const int*)c->cross_len.p, c->dctx.p,
                                            c->num_sms, s, kDecDefault);
      else
        c->launches += launch_dec_cross_attn(c->dtype, g, l, c->dqc.p, c->cross_cache.p, (const float*)c->fused_mask.p, c->dctx.p, s, kDecDefault);
      // x2 = co(ctx) + LN_att(x1);  ffn = gelu(f1(LN_cross(x2)));  x3 = f2(ffn) + LN_cross(x2)
      X.gemm_ln(c->dctx.p, H, L.co, nullptr, nullptr, x2, M, 0, x1, &L.ln_att, st1, st2);
      X.gemm_ln(x2, H, L.f1, &L.f1_f, st2, c->dffn.p, M, 1, nullptr, nullptr, nullptr, nullptr);
      X.gemm_ln(c->dffn.p, c->dec_F, L.f2, nullptr, nullptr, x3, M, 0, x2, &L.ln_cross, st2, st3);
    }
    c->launches += launch_ln_apply_stats(M, H, x3, st3, c->stats_ld, H / 32, c->d_layers[c->dec_layers - 1].ln_out.g, c->d_layers[c->dec_layers - 1].ln_out.b,
                                         c->dh.p, s);
  } else
  for (int l = 0; l < c->dec_layers; ++l) {
    const DecLayer& L = c->d_layers[l];
    X.gemm(c->dh.p, H, L.qkv, c->dqkv.p, 3 * H, M);
    c->launches += launch_dec_self_attn(c->dtype, g, l, c->dqkv.p, c->self_cache.p, d_step, step_host, anc, c->dctx.p, s, kDecDefault);
    X.gemm_add_ln(c->dctx.p, H, L.o, c->dh.p, L.ln_att, c->dtmp.p, c->da.p, M);
    X.gemm(c->da.p, H, L.cq, c->dqc.p, H, M);
    if (dec_cross_tma_supported(c->dtype, g))
      c->launches += launch_dec_cross_tma(g, l, c->dqc.p, c->cross_cache.p, (const float*)c->fused_mask.p, (const int*)c->cross_len.p, c->dctx.p,
                                          c->num_sms, s, kDecDefault);
    else
      c->launches += launch_dec_cross_attn(c->dtype, g, l, c->dqc.p, c->cross_cache.p, (const float*)c->fused_mask.p, c->dctx.p, s, kDecDefault);
    X.gemm_add_ln(c->dctx.p, H, L.co, c->da.p, L.ln_cross, c->dtmp.p, c->db.p, M);
    X.gemm(c->db.p, H, L.f1, c->dffn.p, c->dec_F, M, 1);
    X.gemm_add_ln(c->dffn.p, c->dec_F, L.f2, c->db.p, L.ln_out, c->dtmp.p, c->dh.p, M);
  }
  X.gemm(c->dh.p, H, c->lm_head, c->logits.p, c->Vpad, M, 0, true);
  float* sv = (float*)c->sel_val.p; int32_t* si = (int32_t*)c->sel_idx.p;
  // the logits processors act inside the selection kernels; each reads its rows' decoder input (cur_len = P + step <= 64)
  LogitsProcs procs = logits_procs(gp);
  procs.P = P; procs.step = step_host; procs.d_step = d_step; procs.p0s = g.P0s; procs.rows_per_image = g.K;
  if (beams) {
    // beam sampling: g.K = N * K rows per image (N searches of K beams), each row's 16 best for the warpers and the draw
    const bool sampled = gp.mode == GSTVD_SELECT_BEAM_SAMPLE;
    const int nsel = sampled ? kSelMax : 2 * g.K;
    // bf16: log-sum-exp terms in fp32 (mode 2); the fp32 parity path keeps the fp64 terms of the bit-exact contract (mode 0)
    static const bool exact_lse = getenv("GSTVD_EXACT_LSE") != nullptr;
    BeamBuffers bb = beam_buffers(c);
    const int32_t* bt = nullptr; const int32_t* bc = nullptr;
    // n-gram blocking: nothing to launch while every key is shorter than n-1 tokens (P + t < n-1) or, for the [CLS] start, still
    // holds the [CLS], which no banned n-gram contains (t < n-1).  A caller's prefix may hold anything: no position is known special.
    // With per-image lengths the condition uses the longest, P; the kernel skips the images whose key is still too short.
    const int n = gp.ngram_blocking_size;
    if (n > 0 && step_host >= (prefix ? n - 1 - P : n - 1)) {
      c->launches += launch_beam_ngram_ban(g.B, g.K, Tn, Lh, hist_ids, hist_seg, prefix, P, g.P0s, bb.tokens + (int64_t)(step_host & 1) * M * Tn,
                                           step_host, n, (int32_t*)c->ban_tokens.p, (int32_t*)c->ban_count.p, Lh, s);
      bt = (const int32_t*)c->ban_tokens.p; bc = (const int32_t*)c->ban_count.p;
    }
    // beam groups: row_select also writes each row's logZ, from which the beam step re-scores the candidates a diversity penalty
    // lowers (the candidate lists stay ranked by the unpenalised score; launch_beam_step explains why nsel = 2K suffices)
    const int G = gp.num_beam_groups;
    float* lz = G > 1 ? (float*)c->logz.p : nullptr;
    // a beam row's decoder input: the image's prefix, then the beam's tokens in the token buffer of this step's parity
    procs.prefix = prefix; procs.tokens = bb.tokens + (int64_t)(step_host & 1) * M * Tn; procs.tok_stride = Tn;
    c->launches += launch_row_select(M, c->V, (const float*)c->logits.p, c->Vpad, (c->dtype == kBF16 && !exact_lse) ? 2 : 0,
                                     (const float*)c->beam_scores.p, 1.f, bt, bc, Lh, nsel, sv, si, lz, procs, s);
    if (sampled) {
      const int K = gp.num_beams;
      c->launches += launch_beam_sample_step(bb, M / K, g.K / K, K, Tn, c->V, sv, si, gp.top_k, gp.temperature, gp.top_p,
                                             (const uint64_t*)c->d_seed.p, 102, P, g.P0s, s);
    } else {
      c->launches += launch_beam_step(bb, g.B, g.K, G, Tn, c->V, nsel, sv, si, G > 1 ? (const float*)c->logits.p : nullptr, c->Vpad, lz,
                                      gp.diversity_penalty, gp.repetition_penalty, prefix, 102, P, g.P0s, nullptr, nullptr, nullptr, s);
    }
    if (use_anc) c->launches += launch_anc_update(g, bb.beam_idx, d_step, (uint8_t*)c->anc.p, s);
    else c->launches += launch_reorder_cache(c->dtype, g, c->self_cache.p, bb.beam_idx, d_step, 0, nullptr, s);
  } else {
    // g.K rows per image: the num_return_sequences sampled candidates, each with its own n-gram key and RNG stream
    const int nsel = kSelMax;
    const int32_t* bt = nullptr; const int32_t* bc = nullptr;
    // key buffer c->prefix [M, P + Tn]: the decoder prefix (right-aligned when it is shorter than P), then the generated tokens; the
    // samplers append token t at P + t
    const int kst = P + Tn;
    int32_t* key_next = (int32_t*)c->prefix.p + (P - 1);
    if (gp.ngram_blocking_size > 0) {
      c->launches += launch_ngram_ban(M, g.K, Lh, hist_ids, hist_seg, (const int32_t*)c->prefix.p, kst, d_step, P, gp.ngram_blocking_size,
                                      (int32_t*)c->ban_tokens.p, (int32_t*)c->ban_count.p, Lh, s);
      bt = (const int32_t*)c->ban_tokens.p; bc = (const int32_t*)c->ban_count.p;
    }
    procs.keys = (const int32_t*)c->prefix.p; procs.key_stride = kst;      // a sample row's decoder input is its n-gram key
    if (gp.top_k == 0) {
      // no top-k cut (utils/decoding_utils.py:17 skips it): multinomial over the whole, optionally nucleus-filtered, vocabulary
      c->launches += launch_full_vocab_sample(M, g.K, c->V, (const float*)c->logits.p, c->Vpad, gp.temperature, gp.top_p, bt, bc, Lh, Tn, 0, 0,
                                              (const uint64_t*)c->d_seed.p, d_step, 102, (int32_t*)c->seq.p, (int32_t*)c->cur_tokens.p,
                                              key_next, kst, nullptr, procs, s);
    } else {
      c->launches += launch_row_select(M, c->V, (const float*)c->logits.p, c->Vpad, 1, nullptr, gp.temperature, bt, bc, Lh, nsel, sv, si,
                                       nullptr, procs, s);
      c->launches += launch_sample_step(M, g.K, Tn, nsel, sv, si, gp.top_k, gp.top_p, 0, 0, (const uint64_t*)c->d_seed.p, d_step, 102, (int32_t*)c->seq.p,
                                        (int32_t*)c->cur_tokens.p, key_next, kst, nullptr, s);
    }
  }
  c->launches += launch_step_advance((int*)c->d_step.p, s);
}

// Argument checks of a generate call returning N = gp.num_return_sequences sequences per image; returns the decode rows per image
// (beam mode: the beams; sample mode: the N candidates; beam sampling: N searches of num_beams beams).
int check_generate(gstvd_ctx* c, const gstvd_gen_params& gp, const int64_t* prefix, int P, const int64_t* hist_ids, const int64_t* hist_seg,
                   int Lh, const int64_t* out_ids) {
  check_ready(c);
  if (c->dec_layers == 0) throw StateError("generate: encoder-only context");
  const int T = gp.max_new_tokens, N = gp.num_return_sequences, G = gp.num_beam_groups;
  const float penalty = gp.diversity_penalty;
  if (T < 1 || T > c->T_max) throw InvalidArg("generate: max_new_tokens out of range");
  if (P < 1 || P > c->Ldec_max) throw InvalidArg(fmt("generate: decoder prefix length %d outside 1..max_dec_len (%d)", P, c->Ldec_max));
  if (!prefix && P > 1) throw InvalidArg("generate: the decoder prefix is NULL but its length is above 1");
  if (P - 1 + T > 64)
    throw InvalidArg(fmt("generate: prefix length %d + %d new tokens need %d cached positions; the decode kernels hold at most 64", P, T, P - 1 + T));
  if (P - 1 + T > c->cfg.max_position_embeddings)
    throw InvalidArg(fmt("generate: prefix length %d + %d new tokens exceed max_position_embeddings (%d)", P, T, c->cfg.max_position_embeddings));
  if (!out_ids) throw InvalidArg("generate: out_ids is NULL");
  if (!(penalty >= 0.f) || !std::isfinite(penalty)) throw InvalidArg(fmt("generate: diversity_penalty %g must be finite and >= 0", (double)penalty));
  if (!(gp.repetition_penalty > 0.f) || !std::isfinite(gp.repetition_penalty))
    throw InvalidArg(fmt("generate: repetition_penalty %g must be finite and > 0 (1 = off)", (double)gp.repetition_penalty));
  if (gp.no_repeat_ngram_size < 0) throw InvalidArg(fmt("generate: no_repeat_ngram_size %d must be >= 0", gp.no_repeat_ngram_size));
  if (gp.min_length < 0) throw InvalidArg(fmt("generate: min_length %d must be >= 0", gp.min_length));
  if (G < 1) throw InvalidArg(fmt("generate: %d beam groups", G));
  if (G > 1 && gp.mode != GSTVD_SELECT_BEAM) throw InvalidArg("generate: beam groups need beam search");
  int K = 1;
  if (gp.mode == GSTVD_SELECT_BEAM) {
    K = gp.num_beams;
    if (K < 1 || K > c->K_max || 2 * K > kSelMax) throw InvalidArg("generate: num_beams out of range");
    if (N < 1 || N > K) throw InvalidArg(fmt("generate: %d return sequences outside 1..num_beams (%d)", N, K));
    if (K % G != 0) throw InvalidArg(fmt("generate: %d beam groups do not divide %d beams", G, K));
  } else if (gp.mode == GSTVD_SELECT_BEAM_SAMPLE) {
    K = gp.num_beams;
    if (K < 2 || 2 * K > kSelMax) throw InvalidArg(fmt("generate: beam sampling needs 2 <= num_beams <= %d, got %d", kSelMax / 2, K));
    if (N < 1 || N * K > c->K_max)
      throw InvalidArg(fmt("generate: %d beam-sampled searches of %d beams exceed max_beams (%d) rows per image", N, K, c->K_max));
    if (!(gp.temperature > 0.f) || !std::isfinite(gp.temperature)) throw InvalidArg("generate: temperature must be finite and > 0");
    if (!(gp.top_p >= 0.f && gp.top_p <= 1.f)) throw InvalidArg("generate: top_p must be in [0, 1]");
    if (gp.top_k < 1 || gp.top_k > GSTVD_MAX_TOP_K) throw Unsupported("generate: beam sampling needs top_k in 1..16");
    K *= N;
  } else if (gp.mode == GSTVD_SELECT_SAMPLE) {
    if (N < 1 || N > c->K_max || N > 8) throw InvalidArg(fmt("generate: %d sampled candidates outside 1..min(8, max_beams = %d)", N, c->K_max));
    K = N;
    if (gp.top_k < 0 || gp.top_k > GSTVD_MAX_TOP_K) throw Unsupported("generate: top_k must be 0 (no top-k cut) or in 1..16");
    if (gp.top_k == 0 && c->V > 32768) throw Unsupported("generate: top_k = 0 needs a vocabulary of at most 32768 entries");
    if (!(gp.temperature > 0.f)) throw InvalidArg("generate: temperature must be > 0");
  } else {
    throw InvalidArg("generate: unknown mode");
  }
  if (gp.ngram_blocking_size > 0 && (!hist_ids || !hist_seg || Lh < 1 || Lh > c->Lt_max)) throw InvalidArg("generate: n-gram blocking needs hist_ids / hist_segments");
  return K;
}

// out_ids [B*N, T] image-major (sample mode: N == K, one row per candidate)
void generate_finalize(gstvd_ctx* c, const DecodeGeom& g, const gstvd_gen_params& gp, int64_t* out_ids, float* out_scores, cudaStream_t s) {
  const int B = g.B, K = g.K, P = g.P0 + 1, T = gp.max_new_tokens, N = gp.num_return_sequences;
  if (gp.mode == GSTVD_SELECT_BEAM) c->launches += launch_beam_finalize(beam_buffers(c), B, K, T, 102, P, g.P0s, 1, N, out_ids, out_scores, s);
  else if (gp.mode == GSTVD_SELECT_BEAM_SAMPLE)   // search n of image b is search b * N + n: its best hypothesis is output row b * N + n
    c->launches += launch_beam_finalize(beam_buffers(c), B * N, gp.num_beams, T, 102, P, g.P0s, N, 1, out_ids, out_scores, s);
  else c->launches += launch_sample_finalize(B * K, T, 102, (const int32_t*)c->seq.p, out_ids, s);
}

// The key of a generate graph (Lh, Le set) or a round graph (Lt, Lv and the has_* flags set), from the request and the shapes.
GraphKey graph_key(const gstvd_gen_params& gp, int B, int K, int P, bool has_prefix, int Lh, int Le, int Lt, int Lv, bool has_seg,
                   bool has_att, bool has_imask, bool has_scores) {
  GraphKey k;
  std::memset(&k, 0, sizeof k);
  k.B = B; k.K = K; k.mode = gp.mode; k.T = gp.max_new_tokens; k.top_k = gp.top_k; k.ngram = gp.ngram_blocking_size;
  k.P = P; k.has_prefix = has_prefix; k.N = gp.num_return_sequences; k.G = gp.num_beam_groups;
  k.Lh = Lh; k.Le = Le; k.Lt = Lt; k.Lv = Lv; k.has_seg = has_seg; k.has_att = has_att; k.has_imask = has_imask; k.has_scores = has_scores;
  k.temperature = gp.temperature; k.top_p = gp.top_p; k.penalty = gp.diversity_penalty;
  k.repetition_penalty = gp.repetition_penalty; k.no_repeat_ngram = gp.no_repeat_ngram_size; k.min_length = gp.min_length;
  return k;
}

// Launches the graph of `key` from `pool`.  On a miss it first captures `body` into a new graph, destroying the least recently used
// graph of a full pool.  The launch counter advances by the kernels the capture counted, as if `body` had run eagerly.
template <class Body>
void replay_graph(gstvd_ctx* c, GraphPool& pool, const GraphKey& key, cudaStream_t s, Body&& body) {
  auto it = pool.find(key);
  if (it == pool.end()) {
    if (pool.size() >= kMaxGraphs) {
      auto victim = pool.begin();
      for (auto j = pool.begin(); j != pool.end(); ++j) if (j->second.last_use < victim->second.last_use) victim = j;
      CUDA_CHECK(cudaStreamSynchronize(s));             // it may still be executing on this stream
      cudaGraphExecDestroy(victim->second.exec);
      pool.erase(victim);
    }
    const int64_t before = c->launches;
    cudaGraph_t graph;
    CUDA_CHECK(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
    try {
      body();
    } catch (...) {
      cudaGraph_t dead; cudaStreamEndCapture(s, &dead);
      throw;
    }
    CUDA_CHECK(cudaStreamEndCapture(s, &graph));
    cudaGraphExec_t exec;
    CUDA_CHECK(cudaGraphInstantiate(&exec, graph, 0));
    CUDA_CHECK(cudaGraphDestroy(graph));
    it = pool.emplace(key, GraphEntry{exec, c->launches - before, 0}).first;
    c->launches = before;                           // capture itself launches nothing
  }
  it->second.last_use = ++c->graph_clock;
  CUDA_CHECK(cudaGraphLaunch(it->second.exec, s));
  c->launches += it->second.kernels;
}

void do_generate(gstvd_ctx* c, int B, const gstvd_gen_params& gp, const int64_t* prefix, int P, const int64_t* hist_ids,
                 const int64_t* hist_seg, int Lh, int64_t* out_ids, float* out_scores, cudaStream_t s) {
  const int K = check_generate(c, gp, prefix, P, hist_ids, hist_seg, Lh, out_ids);
  if (c->cross_B != B) throw StateError(fmt("generate: cross K/V prefilled for %d images, asked for %d", c->cross_B, B));
  const int T = gp.max_new_tokens;
  const int64_t* pre = stage_prefix(c, B, prefix, P, s);
  const DecodeGeom g = make_geom(c, B, K, T, P, pre != nullptr);
  // the sampling seed lives in device memory so that a captured graph can be replayed with a new seed
  c->launches += launch_set_u64((uint64_t*)c->d_seed.p, gp.seed, (uint64_t)gp.row_offset, s);
  decode_init(c, g, gp, pre, s);

  const bool use_graph = !(c->cfg.flags & GSTVD_FLAG_NO_CUDA_GRAPH);
  const int64_t* g_ids = hist_ids; const int64_t* g_seg = hist_seg;
  if (use_graph && gp.ngram_blocking_size > 0) {
    // the graph reads the history from the context's own buffers: refresh them (device-to-device, ordered on this stream)
    CUDA_CHECK(cudaMemcpyAsync(c->hist_ids_own.p, hist_ids, (size_t)B * Lh * 8, cudaMemcpyDeviceToDevice, s));
    CUDA_CHECK(cudaMemcpyAsync(c->hist_seg_own.p, hist_seg, (size_t)B * Lh * 8, cudaMemcpyDeviceToDevice, s));
    g_ids = (const int64_t*)c->hist_ids_own.p; g_seg = (const int64_t*)c->hist_seg_own.p;
  }
  auto body = [&] {
    prefix_prefill(c, g, s);
    for (int t = 0; t < T; ++t) decode_step(c, g, gp, pre, g_ids, g_seg, Lh, s, t);   // all T steps in ONE graph: no host round trip between steps
  };
  // the cross cache geometry (Le) is part of the captured launch parameters
  if (!use_graph) body();
  else replay_graph(c, c->graphs, graph_key(gp, B, K, P, pre, Lh, c->cross_Le, 0, 0, false, false, false, false), s, body);
  generate_finalize(c, g, gp, out_ids, out_scores, s);
}

// One forward call of the decode branch of EncoderDecoderModel.forward (models/visual_dialog_model.py:24-120) - encoder, fusion,
// cross-K/V prefill and every decode step - replayed from ONE CUDA graph per shape: the host enqueues a handful of device-to-device
// copies of the inputs into context-owned buffers and one graph launch instead of ~350 kernels per round.  Same kernels, same
// order, same results as gstvd_encode + gstvd_prefill_cross + gstvd_generate (asserted by the tests); eager when graphs are
// disabled or while the GEMM profiler is on (events cannot be recorded inside a graph).
void do_round(gstvd_ctx* c, int B, int Lt, int Lv, const int64_t* ids, const int64_t* seg, const float* att, const float* feat,
              const float* loc, const float* imask, const gstvd_gen_params& gp, const int64_t* prefix, int P, int64_t* out_ids,
              float* out_scores, cudaStream_t s) {
  const int K = check_generate(c, gp, prefix, P, ids, seg ? seg : ids, Lt, out_ids);
  if (B < 1 || B > c->B_max || Lt < 1 || Lt > c->Lt_max || Lv < 1 || Lv > c->Lv_max) throw InvalidArg("round: shape exceeds capacity");
  if (!ids || !feat || !loc) throw InvalidArg("round: input_ids / image_feat / image_loc must not be NULL");
  if (gp.ngram_blocking_size > 0 && !seg) throw InvalidArg("round: n-gram blocking needs token_type_ids");
  const int T = gp.max_new_tokens, N = gp.num_return_sequences, F = c->cfg.v_feature_size;
  auto d2d = [&](void* dst, const void* src, size_t bytes) { if (src) CUDA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, s)); };
  d2d(c->r_ids.p, ids, (size_t)B * Lt * 8); d2d(c->r_seg.p, seg, (size_t)B * Lt * 8); d2d(c->r_att.p, att, (size_t)B * Lt * 4);
  d2d(c->r_feat.p, feat, (size_t)B * Lv * F * 4); d2d(c->r_loc.p, loc, (size_t)B * Lv * 5 * 4); d2d(c->r_imask.p, imask, (size_t)B * Lv * 4);
  const int64_t* pre = stage_prefix(c, B, prefix, P, s);
  c->launches += launch_set_u64((uint64_t*)c->d_seed.p, gp.seed, (uint64_t)gp.row_offset, s);
  const int64_t* g_ids = (const int64_t*)c->r_ids.p;
  const int64_t* g_seg = seg ? (const int64_t*)c->r_seg.p : nullptr;
  auto body = [&] {
    do_encode(c, B, Lt, Lv, g_ids, g_seg, att ? (const float*)c->r_att.p : nullptr, (const float*)c->r_feat.p, (const float*)c->r_loc.p,
              imask ? (const float*)c->r_imask.p : nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, s);
    do_prefill(c, B, Lv + Lt, nullptr, nullptr, s);
    const DecodeGeom g = make_geom(c, B, K, T, P, pre != nullptr);
    decode_init(c, g, gp, pre, s);
    prefix_prefill(c, g, s);
    for (int t = 0; t < T; ++t) decode_step(c, g, gp, pre, g_ids, g_seg, Lt, s, t);
    generate_finalize(c, g, gp, (int64_t*)c->r_out_ids.p, out_scores ? (float*)c->r_out_scores.p : nullptr, s);
  };
  const bool use_graph = !(c->cfg.flags & GSTVD_FLAG_NO_CUDA_GRAPH) && !c->profiling;
  if (!use_graph) {
    body();
  } else {
    replay_graph(c, c->round_graphs, graph_key(gp, B, K, P, pre, 0, 0, Lt, Lv, seg, att, imask, out_scores), s, body);
    // host-side state the captured calls set (a replay does not run them again)
    c->enc_B = B; c->enc_Le = Lv + Lt; c->cross_B = B; c->cross_Le = Lv + Lt;
  }
  CUDA_CHECK(cudaMemcpyAsync(out_ids, c->r_out_ids.p, (size_t)B * N * T * 8, cudaMemcpyDeviceToDevice, s));
  if (out_scores) CUDA_CHECK(cudaMemcpyAsync(out_scores, c->r_out_scores.p, (size_t)B * N * 4, cudaMemcpyDeviceToDevice, s));
}

// `options` decoder sequences per image share that image's cross-attention K/V (evaluate_gen.py:62-107 re-encodes the same
// (image, history) once per answer option; here it is encoded once).  B = sequences = images * options.
void do_score(gstvd_ctx* c, int B, int L, int64_t* dec_ids, const float* dec_mask, const int64_t* labels, float* out_loss,
              float* out_logits, cudaStream_t s, int options = 1) {
  check_ready(c);
  if (c->dec_layers == 0) throw StateError("score: encoder-only context");
  if (options < 1 || B % options != 0) throw InvalidArg("score: sequences must be a multiple of options");
  if (B > c->B_max) throw InvalidArg(fmt("score: %d sequences exceed the context capacity %d", B, c->B_max));
  if (c->cross_B != B / options) throw StateError(fmt("score: cross K/V prefilled for %d images, asked for %d", c->cross_B, B / options));
  if (L < 1 || L > c->Ldec_max || L > c->cfg.max_position_embeddings) throw InvalidArg("score: L out of range");
  if (!dec_ids) throw InvalidArg("score: dec_ids is NULL");
  PdlScope pdl_scope(!(c->cfg.flags & GSTVD_FLAG_NO_PDL));
  Exec X{c, s};
  const int H = c->H, M = B * L;
  const int64_t* lab = labels;
  if (!labels) {
    c->launches += launch_shift_labels(B, L, dec_ids, (int64_t*)c->labels.p, 102, s);   // also [SEP] -> PAD in place (:53-57)
    lab = (const int64_t*)c->labels.p;
  }
  c->launches += launch_embed_text(c->dtype, M, L, H, dec_ids, nullptr, nullptr, 0, c->word, c->pos, c->type, c->type_ext,
                                   c->cfg.type_vocab_size, c->emb_ln.g, c->emb_ln.b, c->dh.p, s);
  dec_teacher_layers(c, X, B, L, dec_mask, options, nullptr);
  float* lg = out_logits ? out_logits : (float*)c->logits.p;
  const int64_t ldl = out_logits ? c->V : c->Vpad;
  X.gemm(c->dh.p, H, c->lm_head, lg, ldl, M, 0, true);
  if (out_loss) c->launches += launch_ce_loss(M, c->V, lg, ldl, lab, out_loss, s);
}

// scratch device buffer for the single-operator test entry points
struct Scratch {
  std::vector<void*> ptrs;
  void* get(size_t bytes) { void* p; CUDA_CHECK(cudaMalloc(&p, bytes ? bytes : 16)); ptrs.push_back(p); return p; }
  ~Scratch() { for (void* p : ptrs) cudaFree(p); }
};

template <typename F>
int guarded(gstvd_ctx* ctx, F&& f) {
  int prev = -1;
  cudaGetDevice(&prev);
  int rc = GSTVD_OK;
  try {
    if (ctx) CUDA_CHECK(cudaSetDevice(ctx->device));
    f();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) throw std::runtime_error(std::string("CUDA launch error: ") + cudaGetErrorString(e));
  } catch (const InvalidArg& e) { rc = GSTVD_ERR_INVALID; g_last_error = e.what(); }
  catch (const StateError& e) { rc = GSTVD_ERR_STATE; g_last_error = e.what(); }
  catch (const Unsupported& e) { rc = GSTVD_ERR_UNSUPPORTED; g_last_error = e.what(); }
  catch (const std::exception& e) {
    rc = std::strstr(e.what(), "CUDA") ? GSTVD_ERR_CUDA : GSTVD_ERR_INVALID;
    g_last_error = e.what();
  }
  if (rc != GSTVD_OK && ctx) ctx->last_error = g_last_error;
  if (prev >= 0) cudaSetDevice(prev);
  return rc;
}

}  // namespace

// =====================================================================================================================
extern "C" {

int gstvd_abi_version(void) { return GSTVD_ABI_VERSION; }

const char* gstvd_last_error(const gstvd_ctx* ctx) { return ctx ? ctx->last_error.c_str() : g_last_error.c_str(); }

int gstvd_create(const gstvd_config* cfg, int device, gstvd_ctx** out) {
  if (!cfg || !out) { g_last_error = "gstvd_create: NULL argument"; return GSTVD_ERR_INVALID; }
  *out = nullptr;
  gstvd_ctx* c = nullptr;
  int rc = guarded(nullptr, [&] {
    if (cfg->abi_version != GSTVD_ABI_VERSION) throw InvalidArg("gstvd_create: abi_version mismatch");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) throw Unsupported("gstvd_create: no CUDA device (there is no CPU fallback)");
    if (device < 0 || device >= ndev) throw InvalidArg("gstvd_create: bad device index");
    cudaDeviceProp prop;
    CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) throw Unsupported(fmt("gstvd_create: device %d is sm_%d%d; this library only runs on sm_100 (B200)", device, prop.major, prop.minor));
    CUDA_CHECK(cudaSetDevice(device));
    const gstvd_config& g = *cfg;
    if (g.compute_dtype != GSTVD_F32 && g.compute_dtype != GSTVD_BF16) throw InvalidArg("gstvd_create: compute_dtype");
    if (g.num_connections < 0 || g.num_connections > GSTVD_MAX_CONNECTIONS) throw InvalidArg("gstvd_create: num_connections");
    if (g.hidden_size % g.num_attention_heads || g.v_hidden_size % g.v_num_attention_heads || g.bi_hidden_size % g.bi_num_attention_heads)
      throw InvalidArg("gstvd_create: hidden sizes must be divisible by head counts");
    auto bad_dim = [](int n) { return n <= 0 || n % 8 != 0; };
    if (bad_dim(g.hidden_size) || bad_dim(g.v_hidden_size) || bad_dim(g.bi_hidden_size) || bad_dim(g.intermediate_size) ||
        bad_dim(g.v_intermediate_size) || bad_dim(g.v_feature_size))
      throw InvalidArg("gstvd_create: feature dimensions must be positive multiples of 8");
    if (g.hidden_size > 1024 || g.v_hidden_size > 1024) throw Unsupported("gstvd_create: hidden sizes above 1024 are not supported by the row kernels");
    if (g.max_batch < 1 || g.max_text_len < 1 || g.max_regions < 1) throw InvalidArg("gstvd_create: capacities must be positive");
    if (g.max_text_len + g.max_regions > 512) throw Unsupported("gstvd_create: at most 512 encoder positions");
    c = new gstvd_ctx();
    c->cfg = g; c->device = device; c->num_sms = prop.multiProcessorCount; c->dtype = g.compute_dtype; c->esz = g.compute_dtype == GSTVD_F32 ? 4 : 2;
    c->H = g.hidden_size; c->Hv = g.v_hidden_size; c->Hb = g.bi_hidden_size; c->heads = g.num_attention_heads; c->heads_v = g.v_num_attention_heads;
    c->heads_b = g.bi_num_attention_heads; c->F = g.intermediate_size; c->Fv = g.v_intermediate_size; c->V = g.vocab_size;
    c->Vpad = (g.vocab_size + 7) & ~7;
    c->Lt_max = g.max_text_len; c->Lv_max = g.max_regions; c->Le_max = g.max_text_len + g.max_regions; c->B_max = g.max_batch;
    c->T_max = g.max_new_tokens > 0 ? g.max_new_tokens : 18; c->K_max = g.max_beams > 0 ? g.max_beams : 1;
    c->Ldec_max = g.max_dec_len > 0 ? g.max_dec_len : 25;
    if (c->Ldec_max < c->T_max) c->Ldec_max = c->T_max;
    c->dec_layers = g.dec_num_hidden_layers; c->dec_heads = g.dec_num_attention_heads > 0 ? g.dec_num_attention_heads : 1;
    c->dec_F = g.dec_intermediate_size;
    if (c->dec_layers > 0) {
      if (c->H % c->dec_heads) throw InvalidArg("gstvd_create: decoder heads");
      const int D = c->H / c->dec_heads;
      if (D != 64 && D != 128) throw Unsupported("gstvd_create: decoder head_dim must be 64 or 128");
      if (c->T_max > 32 || c->K_max > 8) throw Unsupported("gstvd_create: at most 32 new tokens and 8 beams");
      if (bad_dim(c->dec_F)) throw InvalidArg("gstvd_create: dec_intermediate_size");
    }
    if (c->dtype == kBF16) gemm_tc_init();
    plan_weights(c);
    alloc_workspace(c);
    CUDA_CHECK(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
    CUDA_CHECK(cudaEventCreateWithFlags(&c->ev_in, cudaEventDisableTiming));
    CUDA_CHECK(cudaEventCreateWithFlags(&c->ev_out, cudaEventDisableTiming));
    CUDA_CHECK(cudaDeviceSynchronize());
  });
  if (rc != GSTVD_OK) { if (c) gstvd_destroy(c); return rc; }
  *out = c;
  return GSTVD_OK;
}

void gstvd_destroy(gstvd_ctx* c) {
  if (!c) return;
  if (getenv("GSTVD_CROSS_TIMES") != nullptr) dec_cross_print_times();
  int prev = -1; cudaGetDevice(&prev);
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  for (auto& kv : c->graphs) cudaGraphExecDestroy(kv.second.exec);
  for (auto& kv : c->round_graphs) cudaGraphExecDestroy(kv.second.exec);
  DevBuf* bufs[] = {&c->mat32, &c->mat16, &c->vec32, &c->xt, &c->yt, &c->xv, &c->yv, &c->qkv_t, &c->qkv_v, &c->ctx_t, &c->ctx_v, &c->tmp_t,
                    &c->tmp_v, &c->ffn_t, &c->ffn_v, &c->feat_cast, &c->fused, &c->pool, &c->fused_mask, &c->dh, &c->da, &c->db, &c->dqkv,
                    &c->dctx, &c->dtmp, &c->dffn, &c->dqc, &c->logits, &c->cross_cache, &c->self_cache, &c->cross_len, &c->labels, &c->sel_val, &c->sel_idx,
                    &c->logz, &c->ban_tokens, &c->ban_count, &c->prefix, &c->seq, &c->beam_scores, &c->beam_tokens, &c->cur_tokens,
                    &c->beam_idx, &c->beam_done, &c->hyp_score, &c->hyp_len, &c->hyp_tokens, &c->hyp_count, &c->hyp_worst, &c->d_step, &c->d_seed, &c->anc, &c->dec_prefix_own, &c->dec_prefix_head, &c->prefix_p0, &c->fold16, &c->foldvec,
                    &c->st1, &c->st2, &c->st3, &c->hist_ids_own, &c->hist_seg_own, &c->r_ids, &c->r_seg, &c->r_att,
                    &c->r_feat, &c->r_loc, &c->r_imask, &c->r_out_ids, &c->r_out_scores};
  for (DevBuf* b : bufs) b->release();
  for (auto& r : c->prof_pool) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  if (c->ev_in) cudaEventDestroy(c->ev_in);
  if (c->ev_out) cudaEventDestroy(c->ev_out);
  if (c->own_stream) cudaStreamDestroy(c->own_stream);
  delete c;
  if (prev >= 0) cudaSetDevice(prev);
}

int gstvd_load_weight(gstvd_ctx* c, const char* name, const float* data, int64_t numel, void* stream) {
  if (!c || !name || !data) { g_last_error = "gstvd_load_weight: NULL argument"; return GSTVD_ERR_INVALID; }
  int result = 0;
  int rc = guarded(c, [&] {
    const std::string n = canonical_name(name);
    auto it = c->slots.find(n);
    if (it == c->slots.end()) {
      if (is_ignored_key(n)) { result = 1; return; }
      throw InvalidArg(std::string("gstvd_load_weight: unknown key '") + name + "'");
    }
    if (it->second.numel != numel) throw InvalidArg(fmt("gstvd_load_weight: '%s' has %lld elements, expected %lld", name, (long long)numel, (long long)it->second.numel));
    CUDA_CHECK(cudaMemcpyAsync(it->second.dst, data, (size_t)numel * 4, cudaMemcpyDefault, (cudaStream_t)stream));
    it->second.loaded = true;
    c->finalized = false;
  });
  return rc != GSTVD_OK ? rc : result;
}

int gstvd_missing_weights(const gstvd_ctx* c) {
  if (!c) return -1;
  int n = 0;
  for (auto& kv : c->slots) if (!kv.second.loaded) ++n;
  return n;
}

int gstvd_finalize_weights(gstvd_ctx* c, void* stream) {
  if (!c) { g_last_error = "gstvd_finalize_weights: NULL context"; return GSTVD_ERR_INVALID; }
  return guarded(c, [&] {
    cudaStream_t s = (cudaStream_t)stream;
    if (c->dtype == kBF16) {
      c->launches += launch_cast_f32_to(kBF16, (const float*)c->mat32.p, c->mat16.p, (int64_t)c->mat_elems, s);
      assign_w16(c);
      prepare_fold(c, s);
    }
    for (auto& kv : c->graphs) cudaGraphExecDestroy(kv.second.exec);
    c->graphs.clear();
    for (auto& kv : c->round_graphs) cudaGraphExecDestroy(kv.second.exec);
    c->round_graphs.clear();
    c->finalized = true;
  });
}

int gstvd_encode(gstvd_ctx* c, int B, int Lt, int Lv, const int64_t* input_ids, const int64_t* token_type_ids, const float* attention_mask,
                 const float* image_feat, const float* image_loc, const float* image_mask, float* out_t, float* out_v, float* out_fused,
                 float* out_fused_mask, float* out_nsp, void* stream) {
  if (!c) { g_last_error = "gstvd_encode: NULL context"; return GSTVD_ERR_INVALID; }
  return guarded(c, [&] { do_encode(c, B, Lt, Lv, input_ids, token_type_ids, attention_mask, image_feat, image_loc, image_mask, out_t, out_v,
                                    out_fused, out_fused_mask, out_nsp, (cudaStream_t)stream); });
}

int gstvd_prefill_cross(gstvd_ctx* c, int B, int Le, const float* enc_hidden, const float* enc_mask, void* stream) {
  if (!c) { g_last_error = "gstvd_prefill_cross: NULL context"; return GSTVD_ERR_INVALID; }
  return guarded(c, [&] { do_prefill(c, B, Le, enc_hidden, enc_mask, (cudaStream_t)stream); });
}

int gstvd_generate(gstvd_ctx* c, int B, const gstvd_gen_params* params, const int64_t* prefix, int P, const int64_t* hist_ids,
                   const int64_t* hist_segments, int Lh, int64_t* out_ids, float* out_scores, void* stream) {
  if (!c || !params) { g_last_error = "gstvd_generate: NULL argument"; return GSTVD_ERR_INVALID; }
  return guarded(c, [&] {
    cudaStream_t user = (cudaStream_t)stream;
    CUDA_CHECK(cudaEventRecord(c->ev_in, user));
    CUDA_CHECK(cudaStreamWaitEvent(c->own_stream, c->ev_in, 0));
    do_generate(c, B, *params, prefix, P, hist_ids, hist_segments, Lh, out_ids, out_scores, c->own_stream);
    CUDA_CHECK(cudaEventRecord(c->ev_out, c->own_stream));
    CUDA_CHECK(cudaStreamWaitEvent(user, c->ev_out, 0));
  });
}

int gstvd_round(gstvd_ctx* c, int B, int Lt, int Lv, const int64_t* input_ids, const int64_t* token_type_ids, const float* attention_mask,
                const float* image_feat, const float* image_loc, const float* image_mask, const gstvd_gen_params* params,
                const int64_t* prefix, int P, int64_t* out_ids, float* out_scores, void* stream) {
  if (!c || !params) { g_last_error = "gstvd_round: NULL argument"; return GSTVD_ERR_INVALID; }
  return guarded(c, [&] {
    cudaStream_t user = (cudaStream_t)stream;
    CUDA_CHECK(cudaEventRecord(c->ev_in, user));
    CUDA_CHECK(cudaStreamWaitEvent(c->own_stream, c->ev_in, 0));
    do_round(c, B, Lt, Lv, input_ids, token_type_ids, attention_mask, image_feat, image_loc, image_mask, *params, prefix, P, out_ids,
             out_scores, c->own_stream);
    CUDA_CHECK(cudaEventRecord(c->ev_out, c->own_stream));
    CUDA_CHECK(cudaStreamWaitEvent(user, c->ev_out, 0));
  });
}

int gstvd_score(gstvd_ctx* c, int B, int L, int64_t* dec_ids, const float* dec_mask, const int64_t* labels, float* out_loss,
                float* out_logits, void* stream) {
  if (!c) { g_last_error = "gstvd_score: NULL context"; return GSTVD_ERR_INVALID; }
  return guarded(c, [&] { do_score(c, B, L, dec_ids, dec_mask, labels, out_loss, out_logits, (cudaStream_t)stream); });
}

int gstvd_score_options(gstvd_ctx* c, int n_images, int options, int L, int64_t* dec_ids, const float* dec_mask, const int64_t* labels,
                        float* out_loss, float* out_logits, void* stream) {
  if (!c) { g_last_error = "gstvd_score_options: NULL context"; return GSTVD_ERR_INVALID; }
  return guarded(c, [&] { do_score(c, n_images * options, L, dec_ids, dec_mask, labels, out_loss, out_logits, (cudaStream_t)stream, options); });
}

int gstvd_reorder_cache(gstvd_ctx* c, int B, int K, int len, const int32_t* beam_idx, void* stream) {
  if (!c || !beam_idx) { g_last_error = "gstvd_reorder_cache: NULL argument"; return GSTVD_ERR_INVALID; }
  return guarded(c, [&] {
    if (c->dec_layers == 0) throw StateError("reorder_cache: encoder-only context");
    if (B < 1 || B > c->B_max || K < 1 || K > c->K_max || len < 0 || len > c->T_max) throw InvalidArg("reorder_cache: shape out of range");
    DecodeGeom g = make_geom(c, B, K, c->T_max);
    c->launches += launch_reorder_cache(c->dtype, g, c->self_cache.p, beam_idx, nullptr, len, nullptr, (cudaStream_t)stream);
  });
}

int gstvd_splice(gstvd_ctx* c, int B, int Lt, int Lu, int64_t* enc_input_ids, int64_t* enc_segments, float* attention_mask,
                 int32_t* enc_len, const int64_t* utt, int segment_value, int strip_sep, int32_t* abnormal, void* stream) {
  if (!c || !enc_input_ids || !enc_len || !utt) { g_last_error = "gstvd_splice: NULL argument"; return GSTVD_ERR_INVALID; }
  return guarded(c, [&] {
    c->launches += launch_splice(B, Lt, Lu, enc_input_ids, enc_segments, attention_mask, enc_len, utt, segment_value, strip_sep, abnormal, 102,
                                 (cudaStream_t)stream);
  });
}

int gstvd_cross_key_counts(gstvd_ctx* c, int B, int32_t* out, void* stream) {
  if (!c || !out) return GSTVD_ERR_INVALID;
  return guarded(c, [&] {
    if (c->dec_layers == 0) throw StateError("cross_key_counts: encoder-only context");
    if (B < 1 || B != c->cross_B) throw StateError("cross_key_counts: B must equal the batch of the last gstvd_prefill_cross");
    CUDA_CHECK(cudaMemcpyAsync(out, c->cross_len.p, (size_t)B * 4, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  });
}

int64_t gstvd_launch_count(const gstvd_ctx* c) { return c ? c->launches : -1; }

int gstvd_profile_gemm(gstvd_ctx* c, int enable, int min_rows) {
  if (!c) return GSTVD_ERR_INVALID;
  return guarded(c, [&] {
    if (enable && c->prof_pool.empty()) {
      c->prof_pool.resize(8192);
      for (auto& r : c->prof_pool) { CUDA_CHECK(cudaEventCreate(&r.a)); CUDA_CHECK(cudaEventCreate(&r.b)); }
    }
    c->profiling = enable != 0; c->prof_min_rows = min_rows; c->prof_used = 0;
  });
}

int gstvd_profile_read(gstvd_ctx* c, double* flops, double* bytes, double* ms, int64_t* launches) {
  if (!c) return GSTVD_ERR_INVALID;
  return guarded(c, [&] {
    CUDA_CHECK(cudaDeviceSynchronize());
    double f = 0, by = 0, t = 0;
    for (size_t i = 0; i < c->prof_used; ++i) {
      float e = 0.f;
      CUDA_CHECK(cudaEventElapsedTime(&e, c->prof_pool[i].a, c->prof_pool[i].b));
      f += c->prof_pool[i].flops; by += c->prof_pool[i].bytes; t += e;
    }
    if (flops) *flops = f; if (bytes) *bytes = by; if (ms) *ms = t; if (launches) *launches = (int64_t)c->prof_used;
    c->prof_used = 0;
  });
}

// ---- single operators ------------------------------------------------------------------------------------------
int gstvd_op_linear(gstvd_ctx* c, int dtype, int M, int N, int K, const float* a, const float* w, const float* bias, int act, float* out,
                    void* stream) {
  if (!c) return GSTVD_ERR_INVALID;
  return guarded(c, [&] {
    cudaStream_t s = (cudaStream_t)stream;
    GemmArgs g;
    g.M = M; g.N = N; g.K = K; g.lda = K; g.ldw = K; g.ldc = N; g.bias = bias; g.act = act; g.C = out; g.out_f32 = 1;
    if (dtype == kF32) {
      g.A = a; g.W = w;
      c->launches += launch_gemm_simt(g, kF32, s);
    } else {
      Scratch sc;
      void* a16 = sc.get((size_t)M * K * 2); void* w16 = sc.get((size_t)N * K * 2);
      c->launches += launch_cast_f32_to(kBF16, a, a16, (int64_t)M * K, s);
      c->launches += launch_cast_f32_to(kBF16, w, w16, (int64_t)N * K, s);
      g.A = a16; g.W = w16;
      static const bool bf16_out = getenv("GSTVD_OP_LINEAR_BF16OUT") != nullptr;   // measurement aid: time the bf16-output epilogue
      void* c16 = nullptr;
      if (bf16_out) { c16 = sc.get((size_t)M * N * 2); g.C = c16; g.out_f32 = 0; }
      gemm_tc_init();
      static const bool want_times = getenv("GSTVD_GEMM_TIMES") != nullptr;   // measurement aid: per-CTA phase timestamps
      unsigned long long* d_times = nullptr;
      if (want_times) { d_times = (unsigned long long*)sc.get(256 * 8 * 8); CUDA_CHECK(cudaMemsetAsync(d_times, 0, 256 * 8 * 8, s)); g.dbg_times = d_times; }
      if (c->cfg.flags & GSTVD_FLAG_DEBUG_SIMT_GEMM) c->launches += launch_gemm_simt(g, kBF16, s);
      else {
        const bool prof = c->profiling && c->prof_used < c->prof_pool.size();
        if (prof) cudaEventRecord(c->prof_pool[c->prof_used].a, s);
        c->launches += launch_gemm_tc(g, c->num_sms, s);
        if (prof) {
          auto& r = c->prof_pool[c->prof_used++];
          cudaEventRecord(r.b, s);
          r.flops = 2.0 * M * (double)N * K;
          r.bytes = 2.0 * ((double)M * K + (double)N * K) + 4.0 * M * (double)N;
        }
      }
      if (c16) c->launches += launch_cast_to_f32(kBF16, c16, out, (int64_t)M * N, s);
      CUDA_CHECK(cudaStreamSynchronize(s));
      if (d_times) {
        std::vector<unsigned long long> h(256 * 8);
        CUDA_CHECK(cudaMemcpy(h.data(), d_times, h.size() * 8, cudaMemcpyDeviceToHost));
        unsigned long long t0 = ~0ull; int ctas = 0;
        for (int i = 0; i < 256; ++i) if (h[i * 8]) { t0 = std::min(t0, h[i * 8]); ++ctas; }
        double sum[8] = {0}, mx[8] = {0};
        for (int i = 0; i < 256; ++i) if (h[i * 8]) for (int j = 0; j < 8; ++j) { double v = h[i * 8 + j] ? (double)(h[i * 8 + j] - t0) : 0; sum[j] += v; mx[j] = std::max(mx[j], v); }
        fprintf(stderr, "[gemm times M=%d N=%d K=%d ctas=%d] mean/max ns since first CTA start: start %.0f/%.0f prologue %.0f/%.0f pdl_wait %.0f/%.0f first_full %.0f/%.0f last_commit %.0f/%.0f epi_begin %.0f/%.0f epi_end %.0f/%.0f end %.0f/%.0f\n",
                M, N, K, ctas, sum[0] / ctas, mx[0], sum[1] / ctas, mx[1], sum[2] / ctas, mx[2], sum[3] / ctas, mx[3], sum[4] / ctas, mx[4], sum[5] / ctas, mx[5], sum[6] / ctas, mx[6], sum[7] / ctas, mx[7]);
      }
    }
  });
}

int gstvd_op_add_layernorm(gstvd_ctx* c, int dtype, int rows, int width, const float* x, const float* residual, const float* gamma,
                           const float* beta, float* y, void* stream) {
  if (!c) return GSTVD_ERR_INVALID;
  return guarded(c, [&] {
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == kF32) {
      c->launches += launch_add_layernorm(kF32, rows, width, x, width, residual, width, gamma, beta, y, width, s);
    } else {
      Scratch sc;
      const int64_t n = (int64_t)rows * width;
      void* x16 = sc.get(n * 2); void* r16 = residual ? sc.get(n * 2) : nullptr; void* y16 = sc.get(n * 2);
      c->launches += launch_cast_f32_to(kBF16, x, x16, n, s);
      if (residual) c->launches += launch_cast_f32_to(kBF16, residual, r16, n, s);
      c->launches += launch_add_layernorm(kBF16, rows, width, x16, width, r16, width, gamma, beta, y16, width, s);
      c->launches += launch_cast_to_f32(kBF16, y16, y, n, s);
      CUDA_CHECK(cudaStreamSynchronize(s));
    }
  });
}

static void print_gemm_stamps(const char* tag, const unsigned long long* d_times, int M, int N, int K) {
  std::vector<unsigned long long> h(256 * 8);
  cudaMemcpy(h.data(), d_times, h.size() * 8, cudaMemcpyDeviceToHost);
  unsigned long long t0 = ~0ull; int ctas = 0;
  for (int i = 0; i < 256; ++i) if (h[i * 8]) { t0 = std::min(t0, h[i * 8]); ++ctas; }
  double sum[8] = {0}, mx[8] = {0};
  for (int i = 0; i < 256; ++i) if (h[i * 8]) for (int j = 0; j < 8; ++j) { double v = h[i * 8 + j] ? (double)(h[i * 8 + j] - t0) : 0; sum[j] += v; mx[j] = std::max(mx[j], v); }
  fprintf(stderr, "[%s M=%d N=%d K=%d ctas=%d] mean/max ns since first CTA start: start %.0f/%.0f prologue %.0f/%.0f pdl_wait %.0f/%.0f first_full|stats %.0f/%.0f last_commit %.0f/%.0f epi_begin %.0f/%.0f epi_end %.0f/%.0f end %.0f/%.0f\n",
          tag, M, N, K, ctas, sum[0] / ctas, mx[0], sum[1] / ctas, mx[1], sum[2] / ctas, mx[2], sum[3] / ctas, mx[3], sum[4] / ctas, mx[4], sum[5] / ctas, mx[5], sum[6] / ctas, mx[6], sum[7] / ctas, mx[7]);
}

int gstvd_op_deferred_ln_chain(gstvd_ctx* c, int M, int N, int K1, const float* a1, const float* w1, const float* b1, const float* res0,
                               const float* gamma1, const float* beta1, const float* w2, const float* b2, const float* gamma2,
                               const float* beta2, float* out, float* out_x1, void* stream) {
  if (!c) return GSTVD_ERR_INVALID;
  return guarded(c, [&] {
    cudaStream_t s = (cudaStream_t)stream;
    if (c->dtype != kBF16) throw Unsupported("op_deferred_ln_chain: bf16 contexts only");
    if (M < 1 || M > 512 || N < 64 || N > 32 * kLnStatStride || N % 64 != 0 || K1 < 64 || K1 % 64 != 0) throw InvalidArg("op_deferred_ln_chain: shape");
    if (!a1 || !w1 || !b1 || !res0 || !gamma1 || !beta1 || !w2 || !b2 || !gamma2 || !beta2 || !out) throw InvalidArg("op_deferred_ln_chain: NULL buffer");
    Scratch sc;
    void* a16 = sc.get((size_t)M * K1 * 2); void* w16 = sc.get((size_t)N * K1 * 2); void* r16 = sc.get((size_t)M * N * 2);
    void* w2f = sc.get((size_t)N * N * 2); float* cd = (float*)sc.get((size_t)2 * N * 4);
    void* x1 = sc.get((size_t)M * N * 2); void* x2 = sc.get((size_t)M * N * 2); void* y16 = sc.get((size_t)M * N * 2);
    const int64_t sld = (M + 15) & ~15;
    float2* st1 = (float2*)sc.get((size_t)sld * kLnStatStride * 8); float2* st2 = (float2*)sc.get((size_t)sld * kLnStatStride * 8);
    c->launches += launch_cast_f32_to(kBF16, a1, a16, (int64_t)M * K1, s);
    c->launches += launch_cast_f32_to(kBF16, w1, w16, (int64_t)N * K1, s);
    c->launches += launch_cast_f32_to(kBF16, res0, r16, (int64_t)M * N, s);
    c->launches += launch_fold_ln_weights(N, N, w2, gamma1, beta1, b2, w2f, cd, cd + N, s);
    gemm_tc_init();
    GemmArgs g1;
    g1.A = a16; g1.lda = K1; g1.W = w16; g1.ldw = K1; g1.bias = b1; g1.C = x1; g1.ldc = N; g1.M = M; g1.N = N; g1.K = K1;
    g1.res = r16; g1.ldr = N; g1.stats_out = st1; g1.stats_ld = sld;
    static const bool want_times = getenv("GSTVD_GEMM_TIMES") != nullptr;   // measurement aid: per-CTA phase timestamps
    unsigned long long* d_t1 = nullptr; unsigned long long* d_t2 = nullptr;
    if (want_times) {
      d_t1 = (unsigned long long*)sc.get(256 * 8 * 8); d_t2 = (unsigned long long*)sc.get(256 * 8 * 8);
      CUDA_CHECK(cudaMemsetAsync(d_t1, 0, 256 * 8 * 8, s)); CUDA_CHECK(cudaMemsetAsync(d_t2, 0, 256 * 8 * 8, s));
      g1.dbg_times = d_t1;
    }
    c->launches += launch_gemm_tc(g1, c->num_sms, s);
    GemmArgs g2;
    g2.A = x1; g2.lda = N; g2.W = w2f; g2.ldw = N; g2.bias = cd + N; g2.C = x2; g2.ldc = N; g2.M = M; g2.N = N; g2.K = N;
    g2.fold_stats = st1; g2.fold_parts = N / 32; g2.fold_c = cd;
    g2.res = x1; g2.ldr = N; g2.res_stats = st1; g2.res_parts = N / 32; g2.res_gamma = gamma1; g2.res_beta = beta1;
    g2.stats_out = st2; g2.stats_ld = sld; g2.dbg_times = d_t2;
    c->launches += launch_gemm_tc(g2, c->num_sms, s);
    c->launches += launch_ln_apply_stats(M, N, x2, st2, sld, N / 32, gamma2, beta2, y16, s);
    c->launches += launch_cast_to_f32(kBF16, y16, out, (int64_t)M * N, s);
    if (out_x1) c->launches += launch_cast_to_f32(kBF16, x1, out_x1, (int64_t)M * N, s);
    CUDA_CHECK(cudaStreamSynchronize(s));
    if (want_times) { print_gemm_stamps("ln gemm 1 (res + stats)", d_t1, M, N, K1); print_gemm_stamps("ln gemm 2 (fold + res + stats)", d_t2, M, N, N); }
  });
}

int gstvd_debug_self_cache(gstvd_ctx* c, int write, int B, int K, int layer, int kv, float* buf, void* stream) {
  if (!c || !buf) return GSTVD_ERR_INVALID;
  return guarded(c, [&] {
    if (c->dec_layers == 0) throw StateError("debug_self_cache: encoder-only context");
    if (B < 1 || B > c->B_max || K < 1 || K > c->K_max || layer < 0 || layer >= c->dec_layers || (kv != 0 && kv != 1))
      throw InvalidArg("debug_self_cache: argument out of range");
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t n = (int64_t)B * c->T_max * K * c->H;
    char* base = (char*)c->self_cache.p + ((int64_t)layer * 2 + kv) * n * c->esz;
    if (write) c->launches += launch_cast_f32_to(c->dtype, buf, base, n, s);
    else c->launches += launch_cast_to_f32(c->dtype, base, buf, n, s);
  });
}

int gstvd_op_attention(gstvd_ctx* c, int dtype, int B, int H, int Lq, int Lk, int D, const float* q, const float* k, const float* v,
                       const float* mask, float neg, int causal, float* out, void* stream) {
  if (!c) return GSTVD_ERR_INVALID;
  return guarded(c, [&] {
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t W = (int64_t)H * D;
    AttnArgs a;
    a.q_bs = Lq * W; a.q_hs = D; a.q_rs = W; a.k_bs = Lk * W; a.k_hs = D; a.k_rs = W; a.v_bs = Lk * W; a.v_hs = D; a.v_rs = W;
    a.o_bs = Lq * W; a.o_hs = D; a.o_rs = W; a.kmask = mask; a.kmask_bs = Lk; a.neg = neg; a.causal = causal;
    a.B = B; a.H = H; a.Lq = Lq; a.Lk = Lk; a.D = D;
    if (dtype == kF32) {
      a.q = q; a.k = k; a.v = v; a.o = out;
      c->launches += launch_attention_generic(a, kF32, s);
    } else {
      Scratch sc;
      const int64_t nq = (int64_t)B * Lq * W, nk = (int64_t)B * Lk * W;
      void* q16 = sc.get(nq * 2); void* k16 = sc.get(nk * 2); void* v16 = sc.get(nk * 2); void* o16 = sc.get(nq * 2);
      c->launches += launch_cast_f32_to(kBF16, q, q16, nq, s);
      c->launches += launch_cast_f32_to(kBF16, k, k16, nk, s);
      c->launches += launch_cast_f32_to(kBF16, v, v16, nk, s);
      a.q = q16; a.k = k16; a.v = v16; a.o = o16;
      if (!(c->cfg.flags & GSTVD_FLAG_GENERIC_ATTENTION) && attention_mma_supported(a)) c->launches += launch_attention_mma(a, s);
      else c->launches += launch_attention_generic(a, kBF16, s);
      c->launches += launch_cast_to_f32(kBF16, o16, out, nq, s);
      CUDA_CHECK(cudaStreamSynchronize(s));
    }
  });
}

// ---- decode-step attention kernels, one at a time (parity tests): own DecodeGeom with one layer, independent of the context's caches ----
// Per-image P0 values (int32 [B] on the device) are checked against 0 <= p0s[b] <= P0 on the host before any launch.
static void check_p0s(const int32_t* p0s, int B, int P0, cudaStream_t s, const char* who) {
  if (!p0s) return;
  std::vector<int32_t> h(B);
  CUDA_CHECK(cudaMemcpyAsync(h.data(), p0s, (size_t)B * 4, cudaMemcpyDeviceToHost, s));
  CUDA_CHECK(cudaStreamSynchronize(s));
  for (int b = 0; b < B; ++b)
    if (h[b] < 0 || h[b] > P0) throw InvalidArg(fmt("%s: p0s[%d] = %d outside 0..P0 (%d)", who, b, h[b], P0));
}

int gstvd_op_dec_self_attn(gstvd_ctx* c, int dtype, int kernel, int B, int K, int heads, int D, int T, int P0, const int32_t* p0s, int step,
                           int step_known, const float* qkv, const float* prefix_qkv, float* cache, const uint8_t* anc, float* out,
                           void* stream) {
  if (!c) return GSTVD_ERR_INVALID;
  return guarded(c, [&] {
    if (dtype != kF32 && dtype != kBF16) throw InvalidArg("op_dec_self_attn: dtype");
    if (kernel != kDecDefault && kernel != kSelfFirst && kernel != kSelfV2) throw InvalidArg("op_dec_self_attn: kernel must be -1, 0 or 1");
    if (B < 1 || K < 1 || K > 8 || heads < 1 || (D != 64 && D != 128) || T < 1 || T > 64 || P0 < 0 || step < 0 || P0 + step >= T)
      throw InvalidArg("op_dec_self_attn: shape out of range (K <= 8, D 64 or 128, T <= 64, P0 + step < T)");
    if (!qkv || !cache || !out) throw InvalidArg("op_dec_self_attn: NULL buffer");
    if (prefix_qkv && P0 < 1) throw InvalidArg("op_dec_self_attn: prefix_qkv needs P0 >= 1");
    cudaStream_t s = (cudaStream_t)stream;
    check_p0s(p0s, B, P0, s, "op_dec_self_attn");
    DecodeGeom g;
    g.B = B; g.K = K; g.H = heads * D; g.heads = heads; g.D = D; g.layers = 1; g.T = T; g.Le = 0; g.P0 = P0; g.P0s = p0s;
    const int64_t M = (int64_t)B * K, n_qkv = M * 3 * g.H, n_pre = (int64_t)B * P0 * 3 * g.H, n_cache = (int64_t)2 * B * T * K * g.H;
    Scratch sc;
    int* d_step = (int*)sc.get(4);
    const void* q_c = qkv; const void* pre_c = prefix_qkv; void* cache_c = cache; void* out_c = out;
    if (dtype == kBF16) {
      q_c = sc.get(n_qkv * 2); cache_c = sc.get(n_cache * 2); out_c = sc.get(M * g.H * 2);
      pre_c = prefix_qkv ? sc.get(n_pre * 2) : nullptr;
    }
    const bool fits = kernel == kDecDefault ? (anc == nullptr || dec_self_attn_v2_active(dtype, g, q_c, cache_c, out_c))
                                            : dec_self_attn_supports(kernel, dtype, g, q_c, cache_c, out_c, anc);
    if (!fits)
      throw Unsupported(fmt("op_dec_self_attn: kernel %d does not run dtype %d, D = %d, T = %d, K = %d%s", kernel, dtype, D, T, K,
                            anc ? " with an ancestry table" : ""));
    if (dtype == kBF16) {
      c->launches += launch_cast_f32_to(kBF16, qkv, (void*)q_c, n_qkv, s);
      c->launches += launch_cast_f32_to(kBF16, cache, cache_c, n_cache, s);
      if (prefix_qkv) c->launches += launch_cast_f32_to(kBF16, prefix_qkv, (void*)pre_c, n_pre, s);
    }
    CUDA_CHECK(cudaMemcpyAsync(d_step, &step, 4, cudaMemcpyHostToDevice, s));
    if (prefix_qkv) c->launches += launch_prefix_kv_store(dtype, g, 0, pre_c, cache_c, s);
    c->launches += launch_dec_self_attn(dtype, g, 0, q_c, cache_c, d_step, step_known ? step : -1, anc, out_c, s, kernel);
    if (dtype == kBF16) {
      c->launches += launch_cast_to_f32(kBF16, cache_c, cache, n_cache, s);
      c->launches += launch_cast_to_f32(kBF16, out_c, out, M * g.H, s);
    }
    CUDA_CHECK(cudaStreamSynchronize(s));
  });
}

int gstvd_op_dec_cross_attn(gstvd_ctx* c, int dtype, int kernel, int B, int K, int heads, int D, int Le, const float* q,
                            const float* cross_kv, const float* mask, int use_cross_len, int32_t* out_cross_len, float* out, void* stream) {
  if (!c) return GSTVD_ERR_INVALID;
  return guarded(c, [&] {
    if (dtype != kF32 && dtype != kBF16) throw InvalidArg("op_dec_cross_attn: dtype");
    if (kernel < kDecDefault || kernel > kCrossGeneric) throw InvalidArg("op_dec_cross_attn: kernel must be -1 .. 4");
    if (B < 1 || K < 1 || K > 8 || heads < 1 || D < 8 || D > 128 || D % 8 || Le < 1 || Le > 512)
      throw InvalidArg("op_dec_cross_attn: shape out of range (K <= 8, D % 8 == 0 and <= 128, Le <= 512)");
    if (!q || !cross_kv || !out) throw InvalidArg("op_dec_cross_attn: NULL buffer");
    if (use_cross_len && !mask) throw InvalidArg("op_dec_cross_attn: cross_len is computed from the mask");
    cudaStream_t s = (cudaStream_t)stream;
    DecodeGeom g;
    g.B = B; g.K = K; g.H = heads * D; g.heads = heads; g.D = D; g.layers = 1; g.T = 1; g.Le = Le; g.P0 = 0;
    const bool tma = kernel == kDecDefault ? dec_cross_tma_supported(dtype, g) : (kernel == kCrossWarpTma || kernel == kCrossCtaTma);
    if (kernel != kDecDefault && !dec_cross_supports(kernel, dtype, g))
      throw Unsupported(fmt("op_dec_cross_attn: kernel %d does not run dtype %d, D = %d, K = %d, Le = %d", kernel, dtype, D, K, Le));
    const int64_t nq = (int64_t)B * K * g.H, nkv = (int64_t)B * 2 * heads * Le * D;
    Scratch sc;
    int* cross_len = use_cross_len ? (int*)sc.get((size_t)B * 4) : nullptr;
    const void* q_c = q; const void* kv_c = cross_kv; void* out_c = out;
    if (dtype == kBF16) {
      q_c = sc.get(nq * 2); kv_c = sc.get(nkv * 2); out_c = sc.get(nq * 2);
      c->launches += launch_cast_f32_to(kBF16, q, (void*)q_c, nq, s);
      c->launches += launch_cast_f32_to(kBF16, cross_kv, (void*)kv_c, nkv, s);
    }
    if (cross_len) {
      c->launches += launch_cross_len(B, Le, mask, cross_len, s);
      if (out_cross_len) CUDA_CHECK(cudaMemcpyAsync(out_cross_len, cross_len, (size_t)B * 4, cudaMemcpyDeviceToDevice, s));
    }
    if (tma) c->launches += launch_dec_cross_tma(g, 0, q_c, kv_c, mask, cross_len, out_c, c->num_sms, s, kernel);
    else c->launches += launch_dec_cross_attn(dtype, g, 0, q_c, kv_c, mask, out_c, s, kernel);
    if (dtype == kBF16) c->launches += launch_cast_to_f32(kBF16, out_c, out, nq, s);
    CUDA_CHECK(cudaStreamSynchronize(s));
  });
}

int gstvd_op_anc_update(gstvd_ctx* c, int B, int K, int T, int P0, const int32_t* p0s, int step, const int32_t* beam_idx, uint8_t* anc,
                        void* stream) {
  if (!c) return GSTVD_ERR_INVALID;
  return guarded(c, [&] {
    if (B < 1 || K < 1 || K > 8 || T < 1 || T > 64 || P0 < 0 || step < 0 || P0 + step >= T)
      throw InvalidArg("op_anc_update: shape out of range (K <= 8, T <= 64, P0 + step < T)");
    if (!beam_idx || !anc) throw InvalidArg("op_anc_update: NULL buffer");
    cudaStream_t s = (cudaStream_t)stream;
    check_p0s(p0s, B, P0, s, "op_anc_update");
    DecodeGeom g;
    g.B = B; g.K = K; g.H = 0; g.heads = 0; g.D = 0; g.layers = 1; g.T = T; g.Le = 0; g.P0 = P0; g.P0s = p0s;
    Scratch sc;
    int* d_step = (int*)sc.get(4);
    CUDA_CHECK(cudaMemcpyAsync(d_step, &step, 4, cudaMemcpyHostToDevice, s));
    c->launches += launch_anc_update(g, beam_idx, d_step, anc, s);
    CUDA_CHECK(cudaStreamSynchronize(s));
  });
}

int gstvd_op_beam_begin(gstvd_ctx* c, int B, int K, int max_new, void* stream) {
  if (!c) return GSTVD_ERR_INVALID;
  return guarded(c, [&] {
    if (c->dec_layers == 0) throw StateError("beam ops need a decoder context");
    if (B < 1 || B > c->B_max || K < 1 || K > c->K_max || max_new < 1 || max_new > c->T_max) throw InvalidArg("beam_begin: shape out of range");
    c->op_B = B; c->op_K = K; c->op_T = max_new;
    c->launches += launch_beam_init(beam_buffers(c), B, K, 1, 1, max_new, 101, nullptr, 1, nullptr, (cudaStream_t)stream);
  });
}

int gstvd_op_beam_step(gstvd_ctx* c, const float* logits, int64_t ldl, int32_t* beam_idx, int32_t* next_tokens, float* next_scores,
                       void* stream) {
  if (!c || !logits) return GSTVD_ERR_INVALID;
  return guarded(c, [&] {
    if (c->op_B == 0) throw StateError("beam_step before beam_begin");
    cudaStream_t s = (cudaStream_t)stream;
    const int B = c->op_B, K = c->op_K, T = c->op_T, nsel = 2 * K;
    c->launches += launch_row_select(B * K, c->V, logits, ldl, 0, (const float*)c->beam_scores.p, 1.f, nullptr, nullptr, 0, nsel,
                                     (float*)c->sel_val.p, (int32_t*)c->sel_idx.p, nullptr, LogitsProcs(), s);
    c->launches += launch_beam_step(beam_buffers(c), B, K, 1, T, c->V, nsel, (const float*)c->sel_val.p, (const int32_t*)c->sel_idx.p, nullptr,
                                    0, nullptr, 0.f, 1.f, nullptr, 102, 1, nullptr, beam_idx, next_tokens, next_scores, s);
    c->launches += launch_step_advance((int*)c->d_step.p, s);
  });
}

int gstvd_op_beam_end(gstvd_ctx* c, int64_t* out_ids, float* out_scores, void* stream) {
  if (!c || !out_ids) return GSTVD_ERR_INVALID;
  return guarded(c, [&] {
    if (c->op_B == 0) throw StateError("beam_end before beam_begin");
    c->launches += launch_beam_finalize(beam_buffers(c), c->op_B, c->op_K, c->op_T, 102, 1, nullptr, 1, 1, out_ids, out_scores, (cudaStream_t)stream);
    c->op_B = 0;
  });
}

int gstvd_op_sample(gstvd_ctx* c, int rows, const float* logits, int64_t ldl, const gstvd_gen_params* gp, const int64_t* hist_ids,
                    const int64_t* hist_segments, int Lh, const int64_t* prefix, int prefix_len, int step, int32_t* out_tokens, void* stream) {
  if (!c || !logits || !gp || !out_tokens) return GSTVD_ERR_INVALID;
  return guarded(c, [&] {
    if (c->dec_layers == 0) throw StateError("sample op needs a decoder context");
    if (rows < 1 || rows > c->B_max) throw InvalidArg("op_sample: rows out of range");
    if (gp->top_k < 0 || gp->top_k > GSTVD_MAX_TOP_K) throw Unsupported("op_sample: top_k must be 0 (no top-k cut) or in 1..16");
    if (gp->top_k == 0 && c->V > 32768) throw Unsupported("op_sample: top_k = 0 needs a vocabulary of at most 32768 entries");
    if (!(gp->repetition_penalty > 0.f) || !std::isfinite(gp->repetition_penalty) || gp->no_repeat_ngram_size < 0 || gp->min_length < 0)
      throw InvalidArg("op_sample: repetition_penalty must be finite and > 0, no_repeat_ngram_size and min_length >= 0");
    LogitsProcs procs = logits_procs(*gp);
    cudaStream_t s = (cudaStream_t)stream;
    const int T = c->T_max;
    const bool need_prefix = gp->ngram_blocking_size > 0 || procs.active();
    if (need_prefix && (!prefix || prefix_len != step + 1 || prefix_len > std::min(T + 1, kProcMaxLen)))
      throw InvalidArg("op_sample: n-gram blocking and the logits processors need a prefix of step+1 <= min(max_new_tokens + 1, 64) tokens");
    if (gp->ngram_blocking_size > 0 && (!hist_ids || !hist_segments)) throw InvalidArg("op_sample: n-gram blocking needs the history");
    CUDA_CHECK(cudaMemcpyAsync(c->d_step.p, &step, 4, cudaMemcpyHostToDevice, s));
    CUDA_CHECK(cudaMemcpyAsync(c->d_seed.p, &gp->seed, 8, cudaMemcpyHostToDevice, s));
    CUDA_CHECK(cudaStreamSynchronize(s));
    const int32_t* bt = nullptr; const int32_t* bc = nullptr;
    if (need_prefix) {
      CUDA_CHECK(cudaMemsetAsync(c->prefix.p, 0, c->prefix.bytes, s));
      c->launches += launch_build_prefix_from_ids(rows, prefix_len, prefix, (int32_t*)c->prefix.p, T + 1, 102, s);
    }
    if (gp->ngram_blocking_size > 0) {
      c->launches += launch_ngram_ban(rows, 1, Lh, hist_ids, hist_segments, (const int32_t*)c->prefix.p, T + 1, (const int*)c->d_step.p, 1,
                                      gp->ngram_blocking_size, (int32_t*)c->ban_tokens.p, (int32_t*)c->ban_count.p, Lh, s);
      bt = (const int32_t*)c->ban_tokens.p; bc = (const int32_t*)c->ban_count.p;
    }
    // the row's decoder input is the caller's prefix ([SEP] read as [PAD]); the step comes from the device counter
    procs.keys = (const int32_t*)c->prefix.p; procs.key_stride = T + 1; procs.P = 1; procs.step = -1; procs.d_step = (const int*)c->d_step.p;
    if (gp->top_k == 0) {
      c->launches += launch_full_vocab_sample(rows, 1, c->V, logits, ldl, gp->temperature, gp->top_p, bt, bc, Lh, T, gp->seed, (uint64_t)gp->row_offset, nullptr,
                                              (const int*)c->d_step.p, 102, (int32_t*)c->seq.p, (int32_t*)c->cur_tokens.p, (int32_t*)c->prefix.p, T + 1,
                                              out_tokens, procs, s);
      return;
    }
    c->launches += launch_row_select(rows, c->V, logits, ldl, 1, nullptr, gp->temperature, bt, bc, Lh, kSelMax, (float*)c->sel_val.p,
                                     (int32_t*)c->sel_idx.p, nullptr, procs, s);
    c->launches += launch_sample_step(rows, 1, T, kSelMax, (const float*)c->sel_val.p, (const int32_t*)c->sel_idx.p, gp->top_k, gp->top_p, gp->seed, (uint64_t)gp->row_offset, nullptr,
                                      (const int*)c->d_step.p, 102, (int32_t*)c->seq.p, (int32_t*)c->cur_tokens.p, (int32_t*)c->prefix.p, T + 1,
                                      out_tokens, s);
  });
}

}  // extern "C"
