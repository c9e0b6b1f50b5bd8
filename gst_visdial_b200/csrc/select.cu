// Token selection: log-softmax + top-k per row, beam-search bookkeeping, top-k/top-p sampling, n-gram blocking,
// cross-entropy, and the dialog-history splice.  Integer / index results are bit-exact against oracle/beam.py and
// the reference's utils/decoding_utils.py; see the arithmetic contract at the top of oracle/beam.py.
//
//   row_select     : replaces torch.topk + masked fill (utils/decoding_utils.py:17-21) and, for beams, the
//                    log_softmax + top-2K of HF beam_search (absent from the reference; contract in oracle/beam.py)
//   beam_step/...  : BeamSearchScorer.process / finalize + BeamHypotheses (transformers 4.16.2 semantics)
//   beam_ngram_ban : batch_ngram_blocking (utils/decoding_utils.py:38-78) without host round trips, for the sample and the beam
//                    rows (contract in oracle/beam_ngram.py)
//   sample_step    : softmax + multinomial (models/visual_dialog_model.py:106-107), counter-based RNG
//   ce_loss        : CrossEntropyLoss(ignore_index=0, reduction='none') (models/visual_dialog_decoder.py:70-77)
//   splice         : generate.py:145-160 and :214-228
#include <cooperative_groups.h>

#include <cmath>
#include <cstdlib>
#include <stdexcept>

#include "common.cuh"
#include "kernels.h"

namespace gstvd {

namespace {

constexpr int kSelThreads = 1024;
constexpr int kSlots = 32;                 // vocab <= 32768
constexpr int kHypMaxT = 32;

struct Cand { float v; int i; };
__device__ __forceinline__ bool better(float av, int ai, float bv, int bi) { return av > bv || (av == bv && ai < bi); }

// ---- logits processors (LogitsProcs, kernels.h) ----------------------------------------------------------------------
// procs_read: the CTA of `row` reads the row's decoder input d (cur_len = pp.d.len(row, pp.step) <= 64 ids) into shared memory once
// and clears s_bw.  The kernels call it first, while few registers are live (reading d next to the row's logits makes ptxas spill).
// procs_masks, later, marks the positions whose id the n-gram rule bans, and every thread then folds d into two masks over its own
// slots: `pen` = slots whose id occurs in d (a bit mask, so an id that repeats is penalised once), `ban` = slots set to -inf (n-gram
// rule; [SEP] while cur_len < min_length).
// Bad words: the threads test the multi-id sequences whose banned id lies in [lo, hi) (the CTA's ids) against the tail of d and mark
// the matches in s_bw (one bit per sequence); every thread then folds the matches and the one-id bitmap into `ban`.
// owner(w) = the calling thread's slot of id w, or -1; slot_id(s) = the id of the calling thread's slot s, or -1 past the vocabulary.
// Every thread of the CTA must call both (procs_masks synchronises).
constexpr int kBwWords = kBadWordsMaxSeqs / 32;
__device__ __forceinline__ void procs_read(const LogitsProcs& pp, int row, int32_t* s_d, uint32_t* s_bw) {
  const int tid = threadIdx.x;
  const int L = min(pp.d.len(row, pp.step), kProcMaxLen);
  if (tid < L) s_d[tid] = pp.d.at(row, tid);
  if (tid < kBwWords) s_bw[tid] = 0u;
}
template <class Owner, class SlotId>
__device__ __forceinline__ void procs_masks(const LogitsProcs& pp, int row, int32_t* s_d, uint8_t* s_ban, uint32_t* s_bw, int lo,
                                            int hi, Owner owner, SlotId slot_id, uint32_t& pen, uint32_t& ban) {
  const int tid = threadIdx.x;
  const int L = min(pp.d.len(row, pp.step), kProcMaxLen);
  __syncthreads();
  const int n = pp.no_repeat_ngram;
  if (tid < L) {
    // position tid closes the n-gram d[tid-n+1 .. tid]: its last id is banned when the first n-1 equal the last n-1 ids of d
    bool b = n > 0 && tid >= n - 1;
    for (int q = 0; q < n - 1 && b; ++q) b = s_d[tid - n + 1 + q] == s_d[L - n + 1 + q];
    s_ban[tid] = b ? 1 : 0;
  }
  // a sequence of m + 1 ids bans its last id when m <= cur_len and the last m ids of d are its first m (4.16.2 _tokens_match)
  for (int j = tid; j < pp.bw_count; j += blockDim.x) {
    const int32_t* e = pp.bw_seq + 3 * j;
    const int m = e[1], last = e[2];
    if (last < lo || last >= hi || m > L) continue;
    const int32_t* w = pp.bw_seq + e[0];
    bool hit = true;
    for (int q = 0; q < m && hit; ++q) hit = s_d[L - m + q] == w[q];
    if (hit) atomicOr(&s_bw[j >> 5], 1u << (j & 31));
  }
  __syncthreads();
  pen = 0u; ban = 0u;
  for (int j = 0; j < L; ++j) {
    const int s = owner(s_d[j]);
    if (s >= 0) { pen |= 1u << s; if (s_ban[j]) ban |= 1u << s; }
  }
  if (L < pp.min_length) { const int s = owner(102); if (s >= 0) ban |= 1u << s; }
  for (int i = 0; i * 32 < pp.bw_count; ++i) {
    for (uint32_t m = s_bw[i]; m != 0u; m &= m - 1u) {
      const int s = owner(pp.bw_seq[3 * (i * 32 + __ffs(m) - 1) + 2]);
      if (s >= 0) ban |= 1u << s;
    }
  }
  if (pp.bw_single) {
#pragma unroll
    for (int s = 0; s < 32; ++s) {
      const int w = slot_id(s);
      if (w >= 0 && ((__ldg(pp.bw_single + (w >> 5)) >> (w & 31)) & 1u)) ban |= 1u << s;
    }
  }
}

template <int NS>
__device__ __forceinline__ void procs_apply(float (&v)[NS], float p, uint32_t pen, uint32_t ban) {
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    if (p != 1.f && ((pen >> s) & 1u)) v[s] = v[s] < 0.f ? __fmul_rn(v[s], p) : __fdiv_rn(v[s], p);
    if ((ban >> s) & 1u) v[s] = -INFINITY;
  }
}

template <bool kProcs>  // kProcs: the logits processors are on (a separate instance keeps the off path as it was)
__global__ void __launch_bounds__(kSelThreads)
row_select_kernel(int V, const float* __restrict__ logits, int64_t ldl, int mode, const float* __restrict__ row_bias,
                  float temperature, const int32_t* __restrict__ ban_tokens, const int32_t* __restrict__ ban_count,
                  int ban_stride, int nsel, float* __restrict__ sel_val, int32_t* __restrict__ sel_idx, float* __restrict__ logz,
                  const LogitsProcs procs) {
  __shared__ float s_f[32];
  __shared__ double s_d[32];
  __shared__ int s_i[32];
  __shared__ int s_bcast_i;
  __shared__ int32_t s_in[kProcMaxLen];
  __shared__ uint8_t s_ban[kProcMaxLen];
  __shared__ uint32_t s_bw[kBwWords];
  pdl_wait();
  pdl_launch_dependents();
  const int row = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (kProcs) procs_read(procs, row, s_in, s_bw);
  const float* __restrict__ x = logits + (int64_t)row * ldl;
  float v[kSlots];
#pragma unroll
  for (int s = 0; s < kSlots; ++s) {
    const int idx = tid + s * kSelThreads;
    v[s] = (idx < V) ? x[idx] : -INFINITY;
  }
  float lz = 0.f;
  if (mode == 0 || logz != nullptr) {
    float m = -INFINITY;
#pragma unroll
    for (int s = 0; s < kSlots; ++s) m = fmaxf(m, v[s]);
    m = warp_max(m);
    if (lane == 0) s_f[warp] = m;
    __syncthreads();
    m = s_f[lane];
    m = warp_max(m);
    __syncthreads();
    double acc = 0.0;
#pragma unroll
    for (int s = 0; s < kSlots; ++s)
      if (tid + s * kSelThreads < V) acc += exp((double)v[s] - (double)m);
    acc = warp_sum(acc);
    if (lane == 0) s_d[warp] = acc;
    __syncthreads();
    acc = s_d[lane];
    acc = warp_sum(acc);
    __syncthreads();
    lz = (float)((double)m + log(acc));
    if (logz != nullptr && tid == 0) logz[row] = lz;
  }
  if (mode == 0) {
    const float bias = row_bias ? row_bias[row] : 0.f;
#pragma unroll
    for (int s = 0; s < kSlots; ++s)
      if (tid + s * kSelThreads < V) v[s] = kProcs ? __fsub_rn(v[s], lz) : __fadd_rn(__fsub_rn(v[s], lz), bias);   // processors: bias below
  } else {
#pragma unroll
    for (int s = 0; s < kSlots; ++s)
      if (tid + s * kSelThreads < V) v[s] = __fdiv_rn(v[s], temperature);
  }
  if (kProcs) {
    uint32_t pen, ban;
    procs_masks(procs, row, s_in, s_ban, s_bw, 0, V,
                [&](int w) { return (w >= 0 && w < kSelThreads * kSlots && (w % kSelThreads) == tid) ? w / kSelThreads : -1; },
                [&](int s) { const int w = tid + s * kSelThreads; return w < V ? w : -1; }, pen, ban);
    procs_apply(v, procs.repetition_penalty, pen, ban);
    if (mode == 0) {
      const float bias = row_bias ? row_bias[row] : 0.f;
#pragma unroll
      for (int s = 0; s < kSlots; ++s)
        if (tid + s * kSelThreads < V) v[s] = __fadd_rn(v[s], bias);
    }
  }
  // banned tokens -> -inf after the transform: in beam mode logZ stays over the full row (log_softmax, then the n-gram
  // processor, then the beam score - the order of HF beam_search, oracle/beam_ngram.py)
  const int nb = ban_count ? ban_count[row] : 0;
  for (int j = 0; j < nb; ++j) {
    const int w = ban_tokens[(int64_t)row * ban_stride + j];
    if ((w % kSelThreads) == tid) {
      const int slot = w / kSelThreads;
#pragma unroll
      for (int s = 0; s < kSlots; ++s)
        if (s == slot) v[s] = -INFINITY;
    }
  }
  // iterative arg-max; ties resolved towards the lower index.  Each thread caches the best of its own slots and
  // only the owner of the previous winner rescans.
  float bv = -INFINITY; int bi = 0x7fffffff;
#pragma unroll
  for (int s = 0; s < kSlots; ++s) {
    const int idx = tid + s * kSelThreads;
    if (idx < V && v[s] > -INFINITY && better(v[s], idx, bv, bi)) { bv = v[s]; bi = idx; }
  }
  for (int r = 0; r < nsel; ++r) {
    float cv = bv; int ci = bi;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, cv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, ci, o);
      if (better(ov, oi, cv, ci)) { cv = ov; ci = oi; }
    }
    if (lane == 0) { s_f[warp] = cv; s_i[warp] = ci; }
    __syncthreads();
    if (warp == 0) {
      cv = s_f[lane]; ci = s_i[lane];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, cv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, ci, o);
        if (better(ov, oi, cv, ci)) { cv = ov; ci = oi; }
      }
      if (lane == 0) {
        s_bcast_i = ci;
        sel_val[(int64_t)row * nsel + r] = cv;
        sel_idx[(int64_t)row * nsel + r] = (ci == 0x7fffffff) ? 0 : ci;
      }
    }
    __syncthreads();
    const int wi = s_bcast_i;
    if (wi != 0x7fffffff && (wi % kSelThreads) == tid) {
      const int slot = wi / kSelThreads;
      bv = -INFINITY; bi = 0x7fffffff;
#pragma unroll
      for (int s = 0; s < kSlots; ++s) {
        if (s == slot) v[s] = -INFINITY;
        const int idx = tid + s * kSelThreads;
        if (idx < V && v[s] > -INFINITY && better(v[s], idx, bv, bi)) { bv = v[s]; bi = idx; }
      }
    }
    __syncthreads();
  }
}

// ---- row_select, cluster version ------------------------------------------------------------------------------------
// One thread-block CLUSTER of 4 CTAs per row: every CTA keeps 8192 consecutive vocabulary entries in registers (32 per
// thread); the per-CTA (max, sum exp) pairs and candidate lists are exchanged through distributed shared memory.
// Compared with one 1024-thread CTA per row this fills the 148 SMs evenly (1280 small CTAs instead of 320 that need three
// waves).  No warp-serial loops: the selection threshold and every ordering step are RANK computations (each element
// counts the elements that beat it), which are independent instructions instead of dependent shuffle chains.
// Arithmetic contract (oracle/beam.py): exp and the sum in fp64, logZ rounded once to fp32,
// score = fp32(fp32(x - logZ) + beam_score), order (score desc, index asc).
constexpr int kRsChunks = 4;
constexpr int kRsThreads = 256;
constexpr int kRsSlots = 32;
constexpr int kRsSpan = kRsThreads * kRsSlots;
constexpr int kRsWarps = kRsThreads / 32;
constexpr int kRsGroups = 16;         // half-warp groups whose maxima bound the nsel-th largest element (nsel <= 16)
constexpr int kRsCandCap = 128;       // candidates (elements >= tau) kept per CTA before falling back to the iterative arg-max
constexpr int kFill = 0x7fffff00;     // candidate indices >= kFill are fillers ("no candidate"), distinct so that ranks are unique
static_assert(kSelMax <= kRsGroups, "the threshold needs at least nsel groups");

// exp(d) for d <= 0 in fp64, table driven (Tang 1989): d = (32 k + j) ln2/32 + r with |r| <= ln2/64, so
// exp(d) = 2^k * 2^(j/32) * (1 + expm1(r)) with a 6-term polynomial for expm1 (truncation 3e-18) and a 32-entry table of
// 2^(j/32) kept in shared memory (indices diverge inside a warp; the constant bank would serialise them).  ~24
// instructions per value instead of libdevice's ~50, within 1.5 ulp - far inside what the fp32 rounding of logZ can see.
__constant__ double kExp2Table[32] = {1.00000000000000000e+00, 1.02189714865411663e+00, 1.04427378242741375e+00, 1.06714040067682370e+00, 1.09050773266525769e+00, 1.11438674259589243e+00, 1.13878863475669156e+00, 1.16372485877757748e+00, 1.18920711500272103e+00, 1.21524735998046896e+00, 1.24185781207348400e+00, 1.26905095719173322e+00, 1.29683955465100964e+00, 1.32523664315974132e+00, 1.35425554693689265e+00, 1.38390988196383202e+00, 1.41421356237309515e+00, 1.44518080697704665e+00, 1.47682614593949935e+00, 1.50916442759342284e+00, 1.54221082540794074e+00, 1.57598084510788650e+00, 1.61049033194925428e+00, 1.64575547815396495e+00, 1.68179283050742900e+00, 1.71861929812247793e+00, 1.75625216037329945e+00, 1.79470907500310717e+00, 1.83400808640934243e+00, 1.87416763411029996e+00, 1.91520656139714740e+00, 1.95714412417540018e+00};
__constant__ double kExpRed[3] = {46.1662413084468283841, 2.16608493865351192653e-02, 5.96317165397058656257e-12};   // 32/ln2, ln2/32 hi, lo

__device__ __forceinline__ double exp_nonpos(double d, const double* __restrict__ tbl) {
  d = fmax(d, -700.0);                               // exp(-700) ~ 1e-304: contributes nothing; keeps the result a normal number
  const double kd = rint(d * kExpRed[0]);
  double r = fma(-kd, kExpRed[1], d);
  r = fma(-kd, kExpRed[2], r);
  double q = 1.0 / 720.0;
  q = fma(q, r, 1.0 / 120.0);
  q = fma(q, r, 1.0 / 24.0);
  q = fma(q, r, 1.0 / 6.0);
  q = fma(q, r, 0.5);
  q = fma(q, r, 1.0);
  const double p = q * r;                            // expm1(r)
  const int k = (int)kd;
  const double t = tbl[k & 31];
  const double res = fma(t, p, t);                   // 2^(j/32) * exp(r), in [0.98, 2)
  return __hiloint2double(__double2hiint(res) + (k >> 5) * (1 << 20), __double2loint(res));   // * 2^floor(k/32)
}

template <bool kProcs>  // kProcs: the logits processors are on (a separate instance keeps the off path as it was)
__global__ void __cluster_dims__(kRsChunks, 1, 1) __launch_bounds__(kRsThreads, 4)
row_select_cluster_kernel(int V, const float* __restrict__ logits, int64_t ldl, int mode_in, const float* __restrict__ row_bias,
                          float temperature, const int32_t* __restrict__ ban_tokens, const int32_t* __restrict__ ban_count,
                          int ban_stride, int nsel, float* __restrict__ sel_val, int32_t* __restrict__ sel_idx, float* __restrict__ logz,
                          const LogitsProcs procs) {
  namespace cg = cooperative_groups;
  cg::cluster_group cluster = cg::this_cluster();
  int mode = mode_in;
  __shared__ float s_f[kRsWarps];
  __shared__ double s_d[kRsWarps];
  __shared__ int s_i[kRsWarps];
  __shared__ int s_bcast_i;
  __shared__ float s_lz;
  __shared__ double s_part[2];                       // this CTA's (max, sum exp(x - max)); read by the peers
  __shared__ float s_g[kRsGroups];                   // half-warp maxima
  __shared__ float s_candv[kRsCandCap];
  __shared__ int s_candi[kRsCandCap];
  __shared__ int s_cnt;
  __shared__ float s_cv[kSelMax];                    // this CTA's nsel best, best first
  __shared__ int s_ci[kSelMax];
  __shared__ double s_exp2[32];                      // 2^(j/32)
  __shared__ float s_allv[kRsChunks * kSelMax];      // rank 0: the lists of all four CTAs (written by the peers)
  __shared__ int s_alli[kRsChunks * kSelMax];
  __shared__ int32_t s_in[kProcMaxLen];              // the row's decoder input (logits processors)
  __shared__ uint8_t s_ban[kProcMaxLen];
  __shared__ uint32_t s_bw[kBwWords];                // bad-word sequences that match the row's decoder input
  pdl_wait();
  pdl_launch_dependents();
  const int chunk = (int)cluster.block_rank();
  const int row = blockIdx.x / kRsChunks, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (kProcs) procs_read(procs, row, s_in, s_bw);
  const int base = chunk * kRsSpan;
  const float* __restrict__ x = logits + (int64_t)row * ldl;
  float v[kRsSlots];
#pragma unroll
  for (int s = 0; s < kRsSlots; ++s) {
    const int idx = base + tid + s * kRsThreads;
    v[s] = (idx < V) ? x[idx] : -INFINITY;
  }
  if (tid == 0) s_cnt = 0;
  if (tid < 32) s_exp2[tid] = kExp2Table[tid];
  float lz = 0.f;
  // mode 2 = mode 0 (beam scores) with the log-sum-exp terms in fp32 (ex2.approx): the bf16 decode step, whose logits carry
  // ~1e-2 of rounding noise anyway; mode 0 keeps the fp64 terms of the bit-exact contract (oracle/beam.py, fp32 path, op tests)
  const bool fast_lse = mode == 2;
  if (fast_lse) mode = 0;
  const bool need_lz = (mode == 0 || logz != nullptr);
  if (need_lz) {
    float m = -INFINITY;
#pragma unroll
    for (int s = 0; s < kRsSlots; ++s) m = fmaxf(m, v[s]);
    m = warp_max(m);
    if (lane == 0) s_f[warp] = m;
    __syncthreads();
    m = s_f[lane & (kRsWarps - 1)];
    m = warp_max(m);
    double acc = 0.0;
    if (m > -INFINITY) {
      if (fast_lse) {
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;            // four independent chains; exp2(-inf) = 0 for the slots past the vocabulary
        const float ms = m * 1.44269504088896340736f;
#pragma unroll
        for (int s = 0; s < kRsSlots; s += 4) {
          float e0, e1, e2, e3;
          asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(fmaf(v[s], 1.44269504088896340736f, -ms)));
          asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(fmaf(v[s + 1], 1.44269504088896340736f, -ms)));
          asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e2) : "f"(fmaf(v[s + 2], 1.44269504088896340736f, -ms)));
          asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e3) : "f"(fmaf(v[s + 3], 1.44269504088896340736f, -ms)));
          a0 += e0; a1 += e1; a2 += e2; a3 += e3;
        }
        acc = (double)((a0 + a1) + (a2 + a3));
      } else {
        const double md = (double)m;
        // no bounds test per slot: slots past the vocabulary hold -inf and add exp(-700) ~ 1e-304, i.e. nothing
#pragma unroll
        for (int s = 0; s < kRsSlots; ++s) acc += exp_nonpos((double)v[s] - md, s_exp2);
      }
    }
    acc = warp_sum(acc);
    if (lane == 0) s_d[warp] = acc;
    __syncthreads();
    if (tid == 0) {
      double t = 0.0;
#pragma unroll
      for (int w = 0; w < kRsWarps; ++w) t += s_d[w];
      s_part[0] = (double)m;
      s_part[1] = t;
    }
    cluster.sync();                                  // every CTA's (max, sum) is published
    if (warp == 0) {
      double pm = -INFINITY, ps = 0.0;
      if (lane < kRsChunks) {
        const double* rp = cluster.map_shared_rank(s_part, lane);
        pm = rp[0]; ps = rp[1];
      }
      double gm = pm;
#pragma unroll
      for (int o = 2; o > 0; o >>= 1) gm = fmax(gm, __shfl_xor_sync(0xffffffffu, gm, o));
      double term = (lane < kRsChunks && pm > -INFINITY) ? ps * exp_nonpos(pm - gm, s_exp2) : 0.0;
      // fixed order 0+1, 2+3, then the pair sums: identical in all four CTAs
      term += __shfl_xor_sync(0xffffffffu, term, 1);
      term += __shfl_xor_sync(0xffffffffu, term, 2);
      if (lane == 0) s_lz = (float)(gm + log(term));
    }
    __syncthreads();
    lz = s_lz;
    if (logz != nullptr && tid == 0 && chunk == 0) logz[row] = lz;
  }
  if (mode == 0) {
    const float bias = row_bias ? row_bias[row] : 0.f;
#pragma unroll
    for (int s = 0; s < kRsSlots; ++s)
      if (base + tid + s * kRsThreads < V) v[s] = kProcs ? __fsub_rn(v[s], lz) : __fadd_rn(__fsub_rn(v[s], lz), bias);   // processors: bias below
  } else {
#pragma unroll
    for (int s = 0; s < kRsSlots; ++s)
      if (base + tid + s * kRsThreads < V) v[s] = __fdiv_rn(v[s], temperature);
  }
  // logits processors on fp32(x - logZ) (beam modes, before the beam score, as HF beam_search) or fp32(x / temperature) (sampling)
  if (kProcs) {
    uint32_t pen, ban;
    procs_masks(procs, row, s_in, s_ban, s_bw, base, base + kRsSpan,
                [&](int w) { const int o = w - base; return (o >= 0 && o < kRsSpan && (o % kRsThreads) == tid) ? o / kRsThreads : -1; },
                [&](int s) { const int w = base + tid + s * kRsThreads; return w < V ? w : -1; }, pen, ban);
    procs_apply(v, procs.repetition_penalty, pen, ban);
    if (mode == 0) {
      const float bias = row_bias ? row_bias[row] : 0.f;
#pragma unroll
      for (int s = 0; s < kRsSlots; ++s)
        if (base + tid + s * kRsThreads < V) v[s] = __fadd_rn(v[s], bias);
    }
  }
  // banned tokens -> -inf after the transform: in the beam modes logZ stays over the full row (log_softmax, then the n-gram
  // processor, then the beam score - the order of HF beam_search, oracle/beam_ngram.py)
  const int nb = ban_count ? ban_count[row] : 0;
  for (int j = 0; j < nb; ++j) {
    const int w = ban_tokens[(int64_t)row * ban_stride + j] - base;
    if (w >= 0 && w < kRsSpan && (w % kRsThreads) == tid) {
      const int slot = w / kRsThreads;
#pragma unroll
      for (int s = 0; s < kRsSlots; ++s)
        if (s == slot) v[s] = -INFINITY;
    }
  }
  // ---- this CTA's nsel best ----
  // Filter first.  The 16 half-warp maxima are 16 distinct elements, so their nsel-th largest (tau) is a lower bound of
  // the CTA's nsel-th largest element and only elements >= tau can be selected - ~16 of the 8192 on average.  They are
  // collected in shared memory and ordered by rank.  The iterative block-wide arg-max remains as the fallback when the
  // candidate list overflows (mass ties).
  float tv = -INFINITY;
#pragma unroll
  for (int s = 0; s < kRsSlots; ++s) tv = fmaxf(tv, v[s]);           // invalid / banned slots hold -inf
#pragma unroll
  for (int o = 8; o > 0; o >>= 1) tv = fmaxf(tv, __shfl_xor_sync(0xffffffffu, tv, o));
  if ((lane & 15) == 0) s_g[tid >> 4] = tv;
  __syncthreads();                                                     // (also publishes s_cnt = 0)
  float tau;
  {
    // every warp ranks the 16 maxima redundantly (lanes 16..31 mirror 0..15): no second barrier
    const float mine = s_g[lane & 15];
    int rank = 0;
#pragma unroll
    for (int j = 0; j < kRsGroups; ++j) {
      const float other = __shfl_sync(0xffffffffu, mine, j);
      rank += (other > mine || (other == mine && j < (lane & 15))) ? 1 : 0;
    }
    const unsigned pick = __ballot_sync(0xffffffffu, rank == nsel - 1);
    tau = __shfl_sync(0xffffffffu, mine, __ffs(pick) - 1);
  }
#pragma unroll
  for (int s = 0; s < kRsSlots; ++s) {
    if (v[s] >= tau && v[s] > -INFINITY) {
      const int pos = atomicAdd(&s_cnt, 1);
      if (pos < kRsCandCap) { s_candv[pos] = v[s]; s_candi[pos] = base + tid + s * kRsThreads; }
    }
  }
  __syncthreads();
  const int ncand = s_cnt;
  if (ncand <= kRsCandCap) {
    if (tid < nsel && tid >= ncand) { s_cv[tid] = -INFINITY; s_ci[tid] = kFill + tid; }
    if (tid < ncand) {
      const float mv = s_candv[tid];
      const int mi = s_candi[tid];
      int rank = 0;
      for (int j = 0; j < ncand; ++j) rank += better(s_candv[j], s_candi[j], mv, mi) ? 1 : 0;
      if (rank < nsel) { s_cv[rank] = mv; s_ci[rank] = mi; }
    }
  } else {
    // fallback: iterative block-wide arg-max (ties towards the lower index); only the previous winner's owner rescans
    float bv = -INFINITY; int bi = 0x7fffffff;
#pragma unroll
    for (int s = 0; s < kRsSlots; ++s) {
      const int idx = base + tid + s * kRsThreads;
      if (idx < V && v[s] > -INFINITY && better(v[s], idx, bv, bi)) { bv = v[s]; bi = idx; }
    }
    for (int r = 0; r < nsel; ++r) {
      float cv = bv; int ci = bi;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, cv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, ci, o);
        if (better(ov, oi, cv, ci)) { cv = ov; ci = oi; }
      }
      if (lane == 0) { s_f[warp] = cv; s_i[warp] = ci; }
      __syncthreads();
      if (warp == 0) {
        cv = s_f[lane & (kRsWarps - 1)]; ci = s_i[lane & (kRsWarps - 1)];
#pragma unroll
        for (int o = kRsWarps / 2; o > 0; o >>= 1) {
          const float ov = __shfl_xor_sync(0xffffffffu, cv, o);
          const int oi = __shfl_xor_sync(0xffffffffu, ci, o);
          if (better(ov, oi, cv, ci)) { cv = ov; ci = oi; }
        }
        if (lane == 0) { s_bcast_i = ci; s_cv[r] = cv; s_ci[r] = (ci == 0x7fffffff) ? kFill + r : ci; }
      }
      __syncthreads();
      const int wi = s_bcast_i;
      if (wi != 0x7fffffff && ((wi - base) % kRsThreads) == tid) {
        const int slot = (wi - base) / kRsThreads;
        bv = -INFINITY; bi = 0x7fffffff;
#pragma unroll
        for (int s = 0; s < kRsSlots; ++s) {
          if (s == slot) v[s] = -INFINITY;
          const int idx = base + tid + s * kRsThreads;
          if (idx < V && v[s] > -INFINITY && better(v[s], idx, bv, bi)) { bv = v[s]; bi = idx; }
        }
      }
      __syncthreads();
    }
  }
  __syncthreads();
  // push this CTA's list into rank 0's table; fillers become distinct per (chunk, position)
  if (tid < nsel) {
    const int ci = s_ci[tid];
    cluster.map_shared_rank(s_allv, 0)[chunk * nsel + tid] = s_cv[tid];
    cluster.map_shared_rank(s_alli, 0)[chunk * nsel + tid] = ci >= kFill ? kFill + chunk * kSelMax + tid : ci;
  }
  cluster.sync();                                    // the table is complete; the peers are done
  if (chunk == 0 && tid < kRsChunks * nsel) {
    const float mv = s_allv[tid];
    const int mi = s_alli[tid];
    int rank = 0;
    for (int j = 0; j < kRsChunks * nsel; ++j) rank += better(s_allv[j], s_alli[j], mv, mi) ? 1 : 0;
    if (rank < nsel) {
      sel_val[(int64_t)row * nsel + rank] = mv;
      sel_idx[(int64_t)row * nsel + rank] = mi >= kFill ? 0 : mi;
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// Length of a decoder prefix row of stride P: the column of its first negative id, or P.  A row that starts with a negative id is
// invalid input; it is read as length 1 so that every index stays in range (its output is unspecified).
__device__ __forceinline__ int prefix_len(const int64_t* __restrict__ row, int P) {
  for (int j = 1; j < P; ++j)
    if (row[j] < 0) return j;
  return P;
}

// prefix != null: int64 [B, P] decoder prefix shared by the K beams of an image; the first step's input is its last token.
// gs = beams per group: the first beam of every group starts at 0, the others at -1e9 (gs = K: one group; gs = 1: all at 0, beam
// sampling).  B = searches of K beams; N searches per image (beam sampling) share the image's prefix row b / N.
// p0s != null (needs prefix): receives every image's prefix length - 1.
__global__ void beam_init_kernel(BeamBuffers bb, int B, int K, int gs, int N, int T, int start_token, const int64_t* __restrict__ prefix, int P,
                                 int* __restrict__ p0s) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0) *bb.d_step = 0;
  if (i < B) { bb.done[i] = 0; bb.hyp_count[i] = 0; bb.hyp_worst[i] = 1e9; }
  if (p0s && i < B && i % N == 0) p0s[i / N] = prefix_len(prefix + (int64_t)(i / N) * P, P) - 1;
  if (i < B * K) {
    bb.beam_scores[i] = ((i % K) % gs == 0) ? 0.f : -1e9f;
    const int64_t* row = prefix ? prefix + (int64_t)(i / K / N) * P : nullptr;
    const int32_t w = row ? (int32_t)row[prefix_len(row, P) - 1] : start_token;
    bb.cur_tokens[i] = w < 0 ? 0 : w;                    // an invalid row's negative start is embedded as [PAD]
    bb.beam_idx[i] = i % K;
  }
  for (int j = i; j < 2 * B * K * T; j += gridDim.x * blockDim.x) bb.tokens[j] = 0;
}

// BeamHypotheses.add (transformers 4.16.2): slots are kept in insertion order, capacity K (+1 transient).  den = LenPenalty::denom of the
// hypothesis length.
__device__ void hyp_add(const BeamBuffers& bb, int b, int K, int T, const int32_t* toks, int ntok, float sum_logprobs, double den) {
  const double score = (double)sum_logprobs / den;
  const int HK = K + 1;
  double* hs = bb.hyp_score + (int64_t)b * HK;
  int32_t* hl = bb.hyp_len + (int64_t)b * HK;
  int32_t* ht = bb.hyp_tokens + (int64_t)b * HK * T;
  int cnt = bb.hyp_count[b];
  if (cnt < K || score > bb.hyp_worst[b]) {
    hs[cnt] = score; hl[cnt] = ntok;
    for (int j = 0; j < T; ++j) ht[cnt * T + j] = (j < ntok) ? toks[j] : 0;
    ++cnt;
    if (cnt > K) {
      // sorted by (score, insertion index): drop the first, worst = score of the second
      int lo = 0;
      for (int i = 1; i < cnt; ++i) if (hs[i] < hs[lo]) lo = i;
      double second = 1e300;
      for (int i = 0; i < cnt; ++i) if (i != lo && hs[i] < second) second = hs[i];
      for (int i = lo; i + 1 < cnt; ++i) {
        hs[i] = hs[i + 1]; hl[i] = hl[i + 1];
        for (int j = 0; j < T; ++j) ht[i * T + j] = ht[(i + 1) * T + j];
      }
      --cnt;
      bb.hyp_worst[b] = second;
    } else {
      bb.hyp_worst[b] = score < bb.hyp_worst[b] ? score : bb.hyp_worst[b];
    }
    bb.hyp_count[b] = cnt;
  }
}

// BeamSearchScorer.process of one group of gs beams (lane 0): walks the group's 2 gs candidates in rank order (order[rank] = index into
// val / flat, flat = beam * V + token with the beam counted from the image's / search's first beam): [SEP] at rank < gs closes a
// hypothesis of beam flat / V (history src + beam * T, t tokens), any other token becomes new beam lo + cnt, until gs beams are filled.
// Then is_done(val[order[0]], cur_len) on the heap b of capacity K; returns whether it set done[b].  den = LenPenalty::denom[cur_len];
// early = early_stopping: done as soon as the heap is full.
__device__ __forceinline__ bool beam_process(const BeamBuffers& bb, int b, int K, int T, int V, int eos, const int32_t* src, int t,
                                             double den, int early, int lo, int gs, const float* val, const int* flat, const int* order,
                                             float* nb_s, int* nb_tok, int* nb_par) {
  int cnt = 0;
  const float best_sum = val[order[0]];
  for (int rank = 0; rank < 2 * gs; ++rank) {
    const int c = order[rank];
    const float v = val[c];
    const int f = flat[c];
    const int bk = f / V, bt = f - bk * V;
    if (bt == eos) {
      if (rank >= gs) continue;
      hyp_add(bb, b, K, T, src + (int64_t)bk * T, t, v, den);
    } else {
      nb_s[lo + cnt] = v; nb_tok[lo + cnt] = bt; nb_par[lo + cnt] = bk; ++cnt;
    }
    if (cnt == gs) break;
  }
  if (bb.hyp_count[b] >= K) {
    const double cur = (double)best_sum / den;
    if (early || bb.hyp_worst[b] >= cur) { bb.done[b] = 1; return true; }
  }
  return false;
}

// One warp per image.  The K beams form G groups of gs = K / G consecutive beams (diverse beam search: HF 4.16.2
// group_beam_search with HammingDiversityLogitsProcessor, contract in oracle/beam_groups.py; G = 1 is plain beam search, contract
// in oracle/beam.py).  The groups run in order.  For group g the gs x nsel per-row candidates are loaded in parallel; a candidate
// whose token c new beams of groups 0..g-1 took at this step gets the value fp32(fp32(fp32(x - logZ) - fp32(lambda c)) +
// beam_score), recomputed from the logits and logZ of its row (-inf stays: banned tokens and fillers).  They are ranked in
// parallel by (score desc, beam * V + token asc) - all pairs are distinct, so the rank is a permutation - and lane 0 walks the
// best 2 gs exactly like BeamSearchScorer.process with group_size = gs, on the image's one hypothesis heap; `done` is tested before
// and updated after every group.  The token histories are gathered by all lanes at the end.
//
// With a repetition penalty p the re-scored value is fp32(fp32(rep(fp32(fp32(x - logZ) - fp32(lambda c)))) + beam_score), rep = the
// penalty when w occurs in the beam's decoder input (HF runs the Hamming processor first, then the repetition penalty); the other
// processors (n-gram bans, min_length, bad words) only produce -inf, which stays.
//
// Why the per-row lists suffice (nsel >= K + gs; the engine keeps nsel = 2K): row_select ranks each row's candidates by the
// processed (repetition-penalised) score WITHOUT the Hamming term.  The Hamming term only lowers a score, rep (s < 0 ? s p : s / p,
// p > 0) is monotone in s and fp32(a + b) is monotone in a, so an element outside a row's list is preceded, in the contract's order,
// by every element of that list that no earlier group took.  The earlier groups took at most K - gs distinct
// tokens, so at least nsel - (K - gs) >= 2 gs listed elements of the row keep their value, and a group takes at most 2 gs
// candidates from one row: the group's exact top 2 gs lies inside the lists.  The bans (question-history n-grams, no_repeat_ngram_size,
// min_length, bad_words_ids) only set -inf, before the lists are ranked, and the same element is -inf with or without the Hamming term:
// they leave the argument as it is.
//
// Hypothesis scores and is_done use the LenPenalty denominators (length_penalty, early_stopping).
constexpr int kBeamWarps = 4;
// Register budget of the two beam-step kernels: 65536 / (7 * 128 threads) = 72 registers per thread.  Left to its default, ptxas
// keeps them near 48 - 64 registers and spills the values that stay live across the calls into the fp64 / fp32 division subroutines
// of the hypothesis walk (20 bytes in each kernel); with this budget neither spills (-Xptxas -v: beam_step_kernel 68 registers,
// beam_sample_step_kernel 70).  The budget still lets 7 blocks share an SM; the grids have B / 4 and B * N / 4 blocks.
constexpr int kBeamMinBlocks = 7;
__global__ void __launch_bounds__(kBeamWarps * 32, kBeamMinBlocks)
beam_step_kernel(BeamBuffers bb, int B, int K, int G, int T, int V, int nsel, const float* __restrict__ sel_val,
                 const int32_t* __restrict__ sel_idx, const float* __restrict__ logits, int64_t ldl, const float* __restrict__ logz,
                 float penalty, float rep_penalty, const DecInput d, int eos, const LenPenalty lp, int32_t* out_beam_idx,
                 int32_t* out_tokens, float* out_scores) {
  __shared__ float s_val[kBeamWarps][128];
  __shared__ int s_flat[kBeamWarps][128];
  __shared__ int s_order[kBeamWarps][16];
  __shared__ float nb_s[kBeamWarps][8];
  __shared__ int nb_tok[kBeamWarps][8], nb_par[kBeamWarps][8];
  pdl_wait();
  pdl_launch_dependents();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * kBeamWarps + warp;
  if (b >= B) return;
  const int t = *bb.d_step;
  const int cur_len = d.len(b * K, t);         // HF input_ids.shape[-1]: the image's decoder prefix + t generated
  const int32_t* src = bb.tokens + (int64_t)(t & 1) * B * K * T + (int64_t)b * K * T;
  int32_t* dst = bb.tokens + (int64_t)((t + 1) & 1) * B * K * T + (int64_t)b * K * T;
  const int gs = K / G;
  const int n = gs * nsel;                     // candidates of one group, <= 8 * 16 = 128
  // padded beams (image done): score 0, token PAD, parent = the first beam of their group
  if (lane < 8) { nb_s[warp][lane] = 0.f; nb_tok[warp][lane] = 0; nb_par[warp][lane] = (lane / gs) * gs; }
  __syncwarp();
  bool done = bb.done[b];
  for (int g = 0; g < G && !done; ++g) {
    const int lo = g * gs;
    const int64_t c0 = ((int64_t)b * K + lo) * nsel;
    for (int c = lane; c < n; c += 32) {
      const int beam = lo + c / nsel;
      float v = sel_val[c0 + c];
      const int w = sel_idx[c0 + c];
      if (g > 0 && v > -INFINITY) {
        int cnt = 0;
        for (int j = 0; j < lo; ++j) cnt += nb_tok[warp][j] == w ? 1 : 0;
        if (cnt > 0) {
          const int64_t row = (int64_t)b * K + beam;
          float s = __fsub_rn(__fsub_rn(logits[row * ldl + w], logz[row]), __fmul_rn(penalty, (float)cnt));
          if (rep_penalty != 1.f) {
            // HF order: the Hamming term, then the repetition penalty when w occurs in the beam's decoder input
            bool seen = false;
            for (int j = 0; j < cur_len && !seen; ++j) seen = d.at((int)row, j) == w;
            if (seen) s = s < 0.f ? __fmul_rn(s, rep_penalty) : __fdiv_rn(s, rep_penalty);
          }
          v = __fadd_rn(s, bb.beam_scores[row]);
        }
      }
      s_val[warp][c] = v;
      s_flat[warp][c] = beam * V + w;
    }
    __syncwarp();
    for (int c = lane; c < n; c += 32) {
      const float v = s_val[warp][c]; const int f = s_flat[warp][c];
      int rank = 0;
      for (int o = 0; o < n; ++o) {
        const float ov = s_val[warp][o]; const int of = s_flat[warp][o];
        rank += (ov > v || (ov == v && of < f)) ? 1 : 0;
      }
      if (rank < 2 * gs) s_order[warp][rank] = c;
    }
    __syncwarp();
    int fin = 0;
    if (lane == 0)
      fin = beam_process(bb, b, K, T, V, eos, src, t, lp.denom[cur_len], lp.early_stopping, lo, gs, s_val[warp], s_flat[warp], s_order[warp],
                         nb_s[warp], nb_tok[warp], nb_par[warp]) ? 1 : 0;
    __syncwarp();
    done = __shfl_sync(0xffffffffu, fin, 0) != 0;
  }
  for (int i = lane; i < K * T; i += 32) {
    const int k = i / T, j = i - k * T;
    dst[i] = (j == t) ? nb_tok[warp][k] : src[nb_par[warp][k] * T + j];
  }
  if (lane < K) {
    const int k = lane;
    bb.beam_scores[b * K + k] = nb_s[warp][k];
    bb.cur_tokens[b * K + k] = nb_tok[warp][k];
    bb.beam_idx[b * K + k] = nb_par[warp][k];
    if (out_beam_idx) out_beam_idx[b * K + k] = nb_par[warp][k];
    if (out_tokens) out_tokens[b * K + k] = nb_tok[warp][k];
    if (out_scores) out_scores[b * K + k] = nb_s[warp][k];
  }
}

// BeamSearchScorer.finalize: a stable ascending sort of the image's hypotheses (kept in insertion order by hyp_add), then N pops.
// Output n of image b is the hypothesis of rank n by (score desc, insertion index desc); N = 1 is the last of the best scores.
__global__ void beam_finalize_kernel(BeamBuffers bb, int B, int K, int T, int eos, int len0, const int* __restrict__ p0s, int per_image, int N,
                                     const LenPenalty lp, int64_t* out_ids, float* out_scores) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int t = *bb.d_step;                     // steps executed
  const int HK = K + 1;
  if (!bb.done[b]) {
    const int len_b = p0s ? p0s[b / per_image] + 1 : len0;
    const int32_t* cur = bb.tokens + (int64_t)(t & 1) * B * K * T + (int64_t)b * K * T;
    const double den = lp.denom[t + len_b];
    for (int k = 0; k < K; ++k) hyp_add(bb, b, K, T, cur + (int64_t)k * T, t, bb.beam_scores[b * K + k], den);
  }
  const double* hs = bb.hyp_score + (int64_t)b * HK;
  const int cnt = bb.hyp_count[b];
  for (int i = 0; i < cnt; ++i) {
    int rank = 0;
    for (int j = 0; j < cnt; ++j) rank += (hs[j] > hs[i] || (hs[j] == hs[i] && j > i)) ? 1 : 0;
    if (rank >= N) continue;
    const int len = bb.hyp_len[(int64_t)b * HK + i];
    const int32_t* ht = bb.hyp_tokens + ((int64_t)b * HK + i) * T;
    const int64_t o = (int64_t)b * N + rank;
    for (int j = 0; j < T; ++j) out_ids[o * T + j] = (j < len) ? ht[j] : (j == len ? eos : 0);
    if (out_scores) out_scores[o] = (float)hs[i];
  }
}

// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool is_special(int64_t t) { return t == 0 || (t >= 100 && t <= 103); }

// One CTA per image scans its question history once and tests every n-gram against the keys of the image's rows: the key of row r
// at step t is the last n-1 ids of its decoder input d (DecInput).  A key longer than the decoder input bans nothing, as a key that
// holds a special id does (the [CLS] start): n-grams with a special id are never banned.  Ban lists are per row.
constexpr int kBanMaxK = 8;
__global__ void __launch_bounds__(256)
beam_ngram_ban_kernel(int Lh, const int64_t* __restrict__ hist_ids, const int64_t* __restrict__ hist_seg, const DecInput d, int step,
                      int n, int32_t* __restrict__ ban_tokens, int32_t* __restrict__ ban_count, int ban_stride) {
  __shared__ int32_t s_key[kBanMaxK][kProcMaxLen];
  __shared__ int s_cnt[kBanMaxK];
  pdl_wait();
  pdl_launch_dependents();
  const int b = blockIdx.x, K = d.rows_per_image, klen = n - 1;
  const int first = d.len(b * K, step) - klen;           // first key position in the decoder input
  if (first < 0) {                                       // a decoder input shorter than n - 1 bans nothing
    if (threadIdx.x < K) ban_count[b * K + threadIdx.x] = 0;
    return;
  }
  for (int i = threadIdx.x; i < K * klen; i += blockDim.x) {
    const int k = i / klen, j = i - k * klen;
    s_key[k][j] = d.at(b * K + k, first + j);
  }
  if (threadIdx.x < K) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  const int64_t* ids = hist_ids + (int64_t)b * Lh;
  const int64_t* seg = hist_seg + (int64_t)b * Lh;
  for (int p = threadIdx.x; p + n <= Lh; p += blockDim.x) {
    bool ok = true;                                      // question history = ids * (segments == 0); no special id inside
    for (int j = 0; j < n && ok; ++j) ok = seg[p + j] == 0 && !is_special(ids[p + j]);
    if (!ok) continue;
    const int32_t w = (int32_t)ids[p + n - 1];
    for (int k = 0; k < K; ++k) {
      bool match = true;
      for (int j = 0; j < klen && match; ++j) match = ids[p + j] == (int64_t)s_key[k][j];
      if (match) {
        const int slot = atomicAdd(&s_cnt[k], 1);
        if (slot < ban_stride) ban_tokens[((int64_t)b * K + k) * ban_stride + slot] = w;
      }
    }
  }
  __syncthreads();
  if (threadIdx.x < K) ban_count[b * K + threadIdx.x] = s_cnt[threadIdx.x] < ban_stride ? s_cnt[threadIdx.x] : ban_stride;
}

__device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

// Sampling seed of candidate n of an image (gstvd_gen_params.num_return_sequences): candidate n draws what a single-sample call seeded
// candidate_seed(seed, n) draws, and candidate 0 is that call itself.  Mirrored by models/visual_dialog_model.candidate_seed.
__device__ __forceinline__ uint64_t candidate_seed(uint64_t seed, int n) {
  return n == 0 ? seed : splitmix64(seed ^ splitmix64((uint64_t)n * 0xD1B54A32D192ED03ull));
}

// Beam sampling (HF 4.16.2 beam_sample + BeamSearchScorer; contract in oracle/beam_sample.py).  One warp per search s of K beams; N
// searches per image (search n of image b is s = b N + n, its beams are decode rows s K + k).  Each row's list (row_select mode 0 / 2
// with the beam scores as row bias, nsel = 16, bans applied) holds s = fp32(fp32(x - logZ) + beam_score) by (s desc, token asc).  Per row:
//   w = fp32(s / temperature); top-k keeps w >= the k'-th listed w, k' = max(top_k, 2) (a prefix of the list: w is monotone in s);
//   top-p (> 0) inside it drops rank r >= 2 when the probability mass before r exceeds top_p (sample_step_kernel's rule).
// The survivors of the K rows (<= 128) get the Gumbel key fp64(w) - log(-log u), u from the counter-based RNG keyed by
// (candidate_seed(seed, n), row_offset + b, t, k * V + token); the 2K largest keys are a draw of 2K entries without replacement from
// softmax(w) over the search's K V warped scores (Gumbel-top-k).  The drawn entries are ordered by (w desc, k V + token asc) and
// walked by beam_process, exactly as in beam_step_kernel.  Parents are written image-local (n K + parent) for the cache reorder.
__device__ __forceinline__ double gumbel_u(uint64_t sd, uint64_t grow, int t, int flat) {
  const uint64_t h = splitmix64(splitmix64(sd ^ splitmix64((grow << 20) ^ (uint64_t)t)) ^ (uint64_t)flat);
  return ((double)(h >> 11) + 0.5) * 0x1p-53;
}

__global__ void __launch_bounds__(kBeamWarps * 32, kBeamMinBlocks)
beam_sample_step_kernel(BeamBuffers bb, int S, int N, int K, int T, int V, const float* __restrict__ sel_val, const int32_t* __restrict__ sel_idx,
                        int top_k, float temperature, float top_p, const uint64_t* __restrict__ d_seed, int eos, int len0,
                        const int* __restrict__ p0s, const LenPenalty lp) {
  constexpr int nsel = kSelMax;
  __shared__ double s_key[kBeamWarps][8 * nsel];
  __shared__ float s_val[kBeamWarps][8 * nsel];
  __shared__ int s_flat[kBeamWarps][8 * nsel];
  __shared__ int s_kept[kBeamWarps][8];
  __shared__ int s_draw[kBeamWarps][2 * 8], s_order[kBeamWarps][2 * 8];
  __shared__ float nb_s[kBeamWarps][8];
  __shared__ int nb_tok[kBeamWarps][8], nb_par[kBeamWarps][8];
  pdl_wait();
  pdl_launch_dependents();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int s = blockIdx.x * kBeamWarps + warp;
  if (s >= S) return;
  const int t = *bb.d_step;
  const int cur_len = t + (p0s ? p0s[s / N] + 1 : len0);   // the image's decoder prefix + t generated
  const int32_t* src = bb.tokens + (int64_t)(t & 1) * S * K * T + (int64_t)s * K * T;
  int32_t* dst = bb.tokens + (int64_t)((t + 1) & 1) * S * K * T + (int64_t)s * K * T;
  const int n = K * nsel;
  if (lane < 8) { nb_s[warp][lane] = 0.f; nb_tok[warp][lane] = 0; nb_par[warp][lane] = 0; }
  if (!bb.done[s]) {
    const int64_t c0 = (int64_t)s * K * nsel;
    for (int c = lane; c < n; c += 32) {
      s_val[warp][c] = __fdiv_rn(sel_val[c0 + c], temperature);
      s_flat[warp][c] = (c / nsel) * V + sel_idx[c0 + c];
    }
    __syncwarp();
    if (lane < K) {
      const float* w = s_val[warp] + lane * nsel;
      const float thr = w[(top_k > 2 ? top_k : 2) - 1];
      int kept = 0;
      while (kept < nsel && w[kept] >= thr && w[kept] > -INFINITY) ++kept;
      if (top_p > 0.f && kept > 2) {
        float sum = 0.f;
        for (int r = 0; r < kept; ++r) sum += expf(w[r] - w[0]);
        float cum = 0.f;
        for (int r = 0; r < kept; ++r) {
          if (r >= 2 && cum > top_p) { kept = r; break; }
          cum += expf(w[r] - w[0]) / sum;
        }
      }
      s_kept[warp][lane] = kept;
    }
    __syncwarp();
    const uint64_t sd = candidate_seed(d_seed[0], s % N);
    const uint64_t grow = (uint64_t)(s / N) + d_seed[1];
    for (int c = lane; c < n; c += 32) {
      double key = -INFINITY;
      if (c % nsel < s_kept[warp][c / nsel]) key = (double)s_val[warp][c] - log(-log(gumbel_u(sd, grow, t, s_flat[warp][c])));
      s_key[warp][c] = key;
    }
    __syncwarp();
    // the 2K largest keys (ties: list position asc), then those 2K by (w desc, flat asc, list position asc)
    for (int c = lane; c < n; c += 32) {
      const double kv = s_key[warp][c];
      int rank = 0;
      for (int o = 0; o < n; ++o) {
        const double ok = s_key[warp][o];
        rank += (ok > kv || (ok == kv && o < c)) ? 1 : 0;
      }
      if (rank < 2 * K) s_draw[warp][rank] = c;
    }
    __syncwarp();
    if (lane < 2 * K) {
      const int c = s_draw[warp][lane];
      const float v = s_val[warp][c]; const int f = s_flat[warp][c];
      int rank = 0;
      for (int o = 0; o < 2 * K; ++o) {
        const int oc = s_draw[warp][o];
        const float ov = s_val[warp][oc]; const int of = s_flat[warp][oc];
        rank += (ov > v || (ov == v && (of < f || (of == f && oc < c)))) ? 1 : 0;
      }
      s_order[warp][rank] = c;
    }
    __syncwarp();
    if (lane == 0)
      beam_process(bb, s, K, T, V, eos, src, t, lp.denom[cur_len], lp.early_stopping, 0, K, s_val[warp], s_flat[warp], s_order[warp], nb_s[warp],
                   nb_tok[warp], nb_par[warp]);
  }
  __syncwarp();
  for (int i = lane; i < K * T; i += 32) {
    const int k = i / T, j = i - k * T;
    dst[i] = (j == t) ? nb_tok[warp][k] : src[nb_par[warp][k] * T + j];
  }
  if (lane < K) {
    const int64_t r = (int64_t)s * K + lane;
    bb.beam_scores[r] = nb_s[warp][lane];
    bb.cur_tokens[r] = nb_tok[warp][lane];
    bb.beam_idx[r] = (s % N) * K + nb_par[warp][lane];
  }
}

// dec_prefix != null: int64 [rows / N, P] decoder prefix of the row's image, Pb = prefix_len tokens.  p0s != null: receives Pb - 1
// per image.
__global__ void sample_init_kernel(int rows, int N, int T, int start_token, int32_t* seq, int32_t* cur_tokens, int* d_step,
                                   const int64_t* __restrict__ dec_prefix, int P, int* __restrict__ p0s) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0) *d_step = 0;
  if (i < rows) {
    const int64_t img = i / N;
    const int64_t* row = dec_prefix ? dec_prefix + img * P : nullptr;
    const int Pb = row ? prefix_len(row, P) : 1;
    if (p0s && i % N == 0) p0s[img] = Pb - 1;
    const int32_t w0 = row ? (int32_t)row[Pb - 1] : start_token;
    cur_tokens[i] = w0 < 0 ? 0 : w0;                     // an invalid row's negative start is embedded as [PAD]
    for (int j = 0; j < T; ++j) seq[(int64_t)i * T + j] = 0;
  }
}

__global__ void sample_step_kernel(int rows, int N, int T, int nsel, const float* __restrict__ sel_val, const int32_t* __restrict__ sel_idx,
                                   int top_k, float top_p, uint64_t seed, uint64_t row_offset, const uint64_t* __restrict__ d_seed,
                                   const int* __restrict__ d_step, int32_t* seq, int32_t* cur_tokens, int32_t* out_tokens) {
  pdl_wait();
  pdl_launch_dependents();
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= rows) return;
  const int step = *d_step;
  const float* v = sel_val + (int64_t)row * nsel;
  const int32_t* ix = sel_idx + (int64_t)row * nsel;
  // keep everything >= the k-th largest (ties survive as far as the candidate list reaches)
  const float thr = v[top_k - 1];
  int kept = 0;
  while (kept < nsel && v[kept] >= thr && v[kept] > -INFINITY) ++kept;
  if (kept == 0) kept = 1;
  float pr[kSelMax];
  float sum = 0.f;
  for (int r = 0; r < kept; ++r) { pr[r] = expf(v[r] - v[0]); sum += pr[r]; }
  if (top_p > 0.f) {
    // nucleus inside the kept set: drop entry r when the cumulative probability BEFORE it already exceeds top_p
    float cum = 0.f; int keep2 = kept;
    for (int r = 0; r < kept; ++r) {
      if (r > 0 && cum > top_p) { keep2 = r; break; }
      cum += pr[r] / sum;
    }
    kept = keep2;
    sum = 0.f;
    for (int r = 0; r < kept; ++r) sum += pr[r];
  }
  int choice = 0;
  if (kept > 1 && top_k > 1) {     // top_k == 1 is the deterministic greedy path (lowest index among exact ties)
    // keyed by the GLOBAL image (d_seed[1] = row offset of this batch): the draws of an image are the same whichever batch / rank
    // holds it; candidate row % N of the image draws with its own seed
    const uint64_t sd = candidate_seed(d_seed ? d_seed[0] : seed, row % N);
    const uint64_t grow = (uint64_t)(row / N) + (d_seed ? d_seed[1] : row_offset);
    const uint64_t h = splitmix64(sd ^ splitmix64((grow << 20) ^ (uint64_t)step));
    const float u = (float)(h >> 40) * (1.0f / 16777216.0f) * sum;
    float c = 0.f;
    choice = kept - 1;
    for (int r = 0; r < kept; ++r) { c += pr[r]; if (u < c) { choice = r; break; } }
  }
  const int tok = ix[choice];
  if (step < T) seq[(int64_t)row * T + step] = tok;
  cur_tokens[row] = tok;
  if (out_tokens) out_tokens[row] = tok;
}

// ---- top_k = 0: unrestricted / pure-nucleus multinomial over the whole vocabulary (utils/decoding_utils.py:17-35 with top_k == 0,
// then softmax + torch.multinomial, models/visual_dialog_model.py:100-105) ---------------------------------------------------------
// One CTA per row; thread t owns the 32 consecutive tokens [32 t, 32 t + 32) in registers (V <= 32768).
//   x = logit / temperature, then the logits processors, banned tokens -> -inf;  p = exp(x - max);  Z = sum p
//   nucleus (top_p > 0): the reference sorts descending and removes position r when the cumulative probability of positions 0..r-1
//     exceeds top_p, i.e. a token survives iff  S(x) = sum of p over tokens with a strictly larger logit  <=  top_p Z.  S is monotone
//     in x, so the survivors are {x >= x*}; x* is found by a 32-step bit-wise search over the order-preserving integer image of the
//     float (no sort).  Tokens with bit-identical logits survive or fall together (torch.sort leaves their order undefined).
//   draw: u Z_kept located by a block-wide exclusive scan of the per-thread sums in token order (the distribution does not depend on
//     the order in which the survivors are laid out).  All reductions run in a fixed order: deterministic for a given seed.
constexpr int kFvThreads = 1024, kFvPer = 32;
__device__ __forceinline__ uint32_t float_order_key(float f) {
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float fv_block_sum(float v, float* s_red) {      // every thread gets the total; fixed order
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) s_red[warp] = v;
  __syncthreads();
  float t = s_red[lane];
  t = warp_sum(t);
  return t;
}
template <bool kProcs>  // kProcs: the logits processors are on (a separate instance keeps the off path as it was)
__global__ void __launch_bounds__(kFvThreads)
full_vocab_sample_kernel(int N, int V, const float* __restrict__ logits, int64_t ldl, float temperature, float top_p,
                         const int32_t* __restrict__ ban_tokens, const int32_t* __restrict__ ban_count, int ban_stride,
                         int T, uint64_t seed, uint64_t row_offset, const uint64_t* __restrict__ d_seed, const int* __restrict__ d_step,
                         int32_t* seq, int32_t* cur_tokens, int32_t* out_tokens, const LogitsProcs procs) {
  extern __shared__ float s_p[];                   // [kFvPer][kFvThreads]: p of token 32 t + j at s_p[j * 1024 + t] (conflict free)
  __shared__ float s_red[32];
  __shared__ float s_scan[32];
  __shared__ int s_choice;
  __shared__ int32_t s_in[kProcMaxLen];
  __shared__ uint8_t s_ban[kProcMaxLen];
  __shared__ uint32_t s_bw[kBwWords];
  pdl_wait();
  pdl_launch_dependents();
  const int row = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (kProcs) procs_read(procs, row, s_in, s_bw);
  const float* x = logits + (int64_t)row * ldl;
  const int base = tid * kFvPer;
  float v[kFvPer];
#pragma unroll
  for (int j = 0; j < kFvPer; ++j) v[j] = (base + j < V) ? __fdiv_rn(x[base + j], temperature) : -INFINITY;
  if (kProcs) {
    uint32_t pen, ban;
    procs_masks(procs, row, s_in, s_ban, s_bw, 0, V, [&](int w) { return (w >= base && w < base + kFvPer) ? w - base : -1; },
                [&](int s) { return base + s < V ? base + s : -1; }, pen, ban);
    procs_apply(v, procs.repetition_penalty, pen, ban);
  }
  if (ban_tokens != nullptr) {
    const int nb = ban_count[row];
    for (int i = 0; i < nb; ++i) {
      const int tk = ban_tokens[(int64_t)row * ban_stride + i];
      if (tk >= base && tk < base + kFvPer) {
#pragma unroll
        for (int j = 0; j < kFvPer; ++j) if (base + j == tk) v[j] = -INFINITY;
      }
    }
  }
  float m = -INFINITY;
#pragma unroll
  for (int j = 0; j < kFvPer; ++j) m = fmaxf(m, v[j]);
  m = warp_max(m);
  if (lane == 0) s_red[warp] = m;
  __syncthreads();
  m = warp_max(s_red[lane]);
  float local = 0.f;
#pragma unroll
  for (int j = 0; j < kFvPer; ++j) { const float pj = (v[j] > -INFINITY) ? expf(v[j] - m) : 0.f; s_p[j * kFvThreads + tid] = pj; local += pj; }
  float total = fv_block_sum(local, s_red);
  if (top_p > 0.f) {
    const float budget = top_p * total;
    // largest r with S(r) > budget (S(0) > budget unless the whole mass sits on the smallest key); survivors: key >= r + 1
    uint32_t r = 0;
    bool any_false;
    {
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < kFvPer; ++j) s += float_order_key(v[j]) > 0u ? s_p[j * kFvThreads + tid] : 0.f;
      any_false = fv_block_sum(s, s_red) > budget;
    }
    if (any_false) {                               // block-uniform: every thread holds the same total
      for (int bit = 31; bit >= 0; --bit) {
        const uint32_t c = r | (1u << bit);
        float s = 0.f;
#pragma unroll
        for (int j = 0; j < kFvPer; ++j) s += float_order_key(v[j]) > c ? s_p[j * kFvThreads + tid] : 0.f;
        if (fv_block_sum(s, s_red) > budget) r = c;
      }
      const uint32_t kmin = r + 1u;
      local = 0.f;
#pragma unroll
      for (int j = 0; j < kFvPer; ++j) {
        if (float_order_key(v[j]) < kmin) s_p[j * kFvThreads + tid] = 0.f;
        local += s_p[j * kFvThreads + tid];
      }
      total = fv_block_sum(local, s_red);
    }
  }
  // draw: first token (in index order) whose inclusive prefix sum exceeds u * total
  const int step = *d_step;
  const uint64_t sd = candidate_seed(d_seed ? d_seed[0] : seed, row % N);
  const uint64_t grow = (uint64_t)(row / N) + (d_seed ? d_seed[1] : row_offset);
  const uint64_t h = splitmix64(sd ^ splitmix64((grow << 20) ^ (uint64_t)step));
  const float target = (float)(h >> 40) * (1.0f / 16777216.0f) * total;
  float incl = local;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const float n = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += n; }
  __syncthreads();
  if (lane == 31) s_scan[warp] = incl;
  if (tid == 0) s_choice = -1;
  __syncthreads();
  float woff = 0.f;
  for (int w = 0; w < warp; ++w) woff += s_scan[w];                 // fixed order
  const float excl = woff + incl - local;
  if (local > 0.f && target >= excl && target < excl + local) {
    float c = excl; int pick = -1, last = -1;
#pragma unroll
    for (int j = 0; j < kFvPer; ++j) {
      const float pj = s_p[j * kFvThreads + tid];
      if (pj > 0.f) { c += pj; last = base + j; if (pick < 0 && target < c) pick = base + j; }
    }
    atomicMax(&s_choice, pick < 0 ? last : pick);                    // rounding at the end of the range: last survivor of this thread
  }
  __syncthreads();
  const int found = s_choice;
  __syncthreads();
  if (found < 0) {                                                   // rounding pushed the target past every range: last survivor overall
    int last = -1;
#pragma unroll
    for (int j = 0; j < kFvPer; ++j) if (s_p[j * kFvThreads + tid] > 0.f) last = base + j;
    if (last >= 0) atomicMax(&s_choice, last);
    __syncthreads();
  }
  if (tid == 0) {
    const int tok = s_choice < 0 ? 0 : s_choice;
    if (step < T) seq[(int64_t)row * T + step] = tok;
    cur_tokens[row] = tok;
    if (out_tokens) out_tokens[row] = tok;
  }
}

__global__ void sample_finalize_kernel(int rows, int T, int eos, const int32_t* __restrict__ seq, int64_t* __restrict__ out_ids) {
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= rows) return;
  bool ended = false;
  for (int j = 0; j < T; ++j) {
    const int tk = seq[(int64_t)row * T + j];
    out_ids[(int64_t)row * T + j] = ended ? 0 : tk;
    if (tk == eos) ended = true;
  }
}

__global__ void set_u64_kernel(uint64_t* dst, uint64_t v, uint64_t v1) { if (threadIdx.x == 0 && blockIdx.x == 0) { dst[0] = v; dst[1] = v1; } }

__global__ void step_advance_kernel(int* d_step) {
  pdl_wait();
  if (threadIdx.x == 0 && blockIdx.x == 0) *d_step += 1;
}

__global__ void shift_labels_kernel(int L, int64_t* __restrict__ ids, int64_t* __restrict__ labels, int eos) {
  const int b = blockIdx.x;
  int64_t* row = ids + (int64_t)b * L;
  for (int i = threadIdx.x; i < L; i += blockDim.x) labels[(int64_t)b * L + i] = (i + 1 < L) ? row[i + 1] : 0;
  __syncthreads();
  for (int i = threadIdx.x; i < L; i += blockDim.x) if (row[i] == eos) row[i] = 0;
}

__global__ void __launch_bounds__(256)
ce_loss_kernel(int V, const float* __restrict__ logits, int64_t ldl, const int64_t* __restrict__ labels, float* __restrict__ loss) {
  __shared__ float s_f[8];
  __shared__ double s_d[8];
  const int row = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t label = labels[row];
  if (label == 0) { if (tid == 0) loss[row] = 0.f; return; }     // ignore_index = pad
  const float* x = logits + (int64_t)row * ldl;
  float m = -INFINITY;
  for (int i = tid; i < V; i += 256) m = fmaxf(m, x[i]);
  m = warp_max(m);
  if (lane == 0) s_f[warp] = m;
  __syncthreads();
  m = s_f[lane & 7];
  m = warp_max(m);
  double acc = 0.0;
  for (int i = tid; i < V; i += 256) acc += (double)expf(x[i] - m);
  acc = warp_sum(acc);
  if (lane == 0) s_d[warp] = acc;
  __syncthreads();
  if (tid == 0) {
    double tot = 0.0;
    for (int w = 0; w < 8; ++w) tot += s_d[w];
    loss[row] = (m + logf((float)tot)) - x[label];
  }
}

__global__ void splice_kernel(int B, int Lt, int Lu, int64_t* ids, int64_t* seg, float* mask, int32_t* enc_len,
                              const int64_t* __restrict__ utt, int segment_value, int strip_sep, int32_t* abnormal, int sep) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  int64_t* row = ids + (int64_t)b * Lt;
  const int64_t* u = utt + (int64_t)b * Lu;
  int n = 0;
  for (int j = 0; j < Lu; ++j) {
    const int64_t tk = (strip_sep && u[j] == sep) ? 0 : u[j];
    if (tk != 0) ++n;
  }
  const int start = enc_len[b];
  int end = start + n;
  if (end <= Lt) {
    for (int j = 0; j < n; ++j) row[start + j] = (strip_sep && u[j] == sep) ? 0 : u[j];
  } else {
    if (start < Lt) row[start] = sep;
    n = 1; end = start + 1;
    if (abnormal) abnormal[b] = 1;
  }
  if (segment_value >= 0 && seg != nullptr)
    for (int j = start; j < end && j < Lt; ++j) seg[(int64_t)b * Lt + j] = segment_value;
  enc_len[b] = start + n;
  if (mask != nullptr)
    for (int j = 0; j < Lt; ++j) mask[(int64_t)b * Lt + j] = row[j] != 0 ? 1.f : 0.f;
}

void check_dec_input(const DecInput& d, int step, const char* who) {
  if (d.P < 1 || (d.P > 1 && !d.prefix) || d.rows_per_image < 1 || step < 0 || d.P + step > kProcMaxLen || (step > 0 && !d.tokens))
    throw std::runtime_error(std::string(who) + ": the rows' decoder input needs 1 <= P <= P + step <= 64, the prefix when P > 1 and "
                             "the tokens when step > 0");
}

void check_procs(const LogitsProcs& p, const char* who) {
  if (!p.active()) return;
  if (!(p.repetition_penalty > 0.f) || !std::isfinite(p.repetition_penalty) || p.no_repeat_ngram < 0 || p.min_length < 0)
    throw std::runtime_error(std::string(who) + ": logits processor parameters out of range");
  check_dec_input(p.d, p.step, who);
  if (p.bw_count < 0 || p.bw_count > kBadWordsMaxSeqs || (p.bw_count > 0 && !p.bw_seq))
    throw std::runtime_error(std::string(who) + ": bad-word sequences out of range");
}

}  // namespace

int launch_row_select(int rows, int V, const float* logits, int64_t ldl, int mode, const float* row_bias, float temperature,
                      const int32_t* ban_tokens, const int32_t* ban_count, int ban_stride, int nsel,
                      float* sel_val, int32_t* sel_idx, float* logz, const LogitsProcs& procs, cudaStream_t stream) {
  if (rows <= 0) return 0;
  if (V > kSelThreads * kSlots) throw std::runtime_error("row_select: vocab > 32768");
  if (nsel > kSelMax || nsel < 1) throw std::runtime_error("row_select: nsel out of range");
  check_procs(procs, "row_select");
  static const bool v1 = getenv("GSTVD_ROW_SELECT_V1") != nullptr;      // A/B aid: the single-CTA-per-row kernel
  if (v1)
    launch_k(procs.active() ? row_select_kernel<true> : row_select_kernel<false>, dim3(rows), dim3(kSelThreads), 0, stream, V, logits, ldl, mode == 2 ? 0 : mode, row_bias, temperature, ban_tokens, ban_count,
             ban_stride, nsel, sel_val, sel_idx, logz, procs);
  else
    launch_k(procs.active() ? row_select_cluster_kernel<true> : row_select_cluster_kernel<false>, dim3(rows * kRsChunks), dim3(kRsThreads), 0, stream, V, logits, ldl, mode, row_bias, temperature,
             ban_tokens, ban_count, ban_stride, nsel, sel_val, sel_idx, logz, procs);
  return 1;
}

int launch_beam_init(const BeamBuffers& bb, int B, int K, int G, int N, int T, int start_token, const int64_t* prefix, int P, int* p0s,
                     cudaStream_t stream) {
  if (G < 1 || K % G != 0) throw std::runtime_error("beam_init: the beam groups must divide the beams");
  if (N < 1 || B % N != 0) throw std::runtime_error("beam_init: the searches must be a multiple of N >= 1");
  if (p0s && !prefix) throw std::runtime_error("beam_init: per-image prefix lengths need a prefix");
  const int n = B * K;
  beam_init_kernel<<<(n + 255) / 256, 256, 0, stream>>>(bb, B, K, K / G, N, T, start_token, prefix, P, p0s);
  return 1;
}
LenPenalty len_penalty(float length_penalty, int early_stopping) {
  LenPenalty lp;
  for (int len = 0; len <= kMaxHypLen; ++len)
    lp.denom[len] = length_penalty == 1.f ? (double)len : std::pow((double)len, (double)length_penalty);
  lp.early_stopping = early_stopping ? 1 : 0;
  return lp;
}

int launch_beam_sample_step(const BeamBuffers& bb, int S, int N, int K, int T, int V, const float* sel_val, const int32_t* sel_idx, int top_k,
                            float temperature, float top_p, const uint64_t* d_seed, int eos, int len0, const int* p0s, const LenPenalty& lp,
                            cudaStream_t stream) {
  if (K < 2 || 2 * K > kSelMax || T > kHypMaxT) throw std::runtime_error("beam_sample_step: 2 <= K <= 8 and T <= 32");
  if (len0 - 1 + T > kMaxHypLen - 1) throw std::runtime_error("beam_sample_step: prefix + new tokens exceed the length table");
  if (N < 1 || S % N != 0) throw std::runtime_error("beam_sample_step: the searches must be a multiple of N >= 1");
  if (top_k < 1 || top_k > kSelMax) throw std::runtime_error("beam_sample_step: top_k out of range");
  launch_k(beam_sample_step_kernel, dim3((S + kBeamWarps - 1) / kBeamWarps), dim3(kBeamWarps * 32), 0, stream, bb, S, N, K, T, V, sel_val,
           sel_idx, top_k, temperature, top_p, d_seed, eos, len0, p0s, lp);
  return 1;
}
int launch_beam_step(const BeamBuffers& bb, int B, int K, int G, int T, int V, int nsel, const float* sel_val,
                     const int32_t* sel_idx, const float* logits, int64_t ldl, const float* logz, float penalty, float rep_penalty,
                     const DecInput& d, int eos, const LenPenalty& lp, int32_t* out_beam_idx, int32_t* out_tokens, float* out_scores,
                     cudaStream_t stream) {
  if (K > 8 || T > kHypMaxT) throw std::runtime_error("beam_step: K <= 8 and T <= 32");
  if (d.P - 1 + T > kMaxHypLen - 1) throw std::runtime_error("beam_step: prefix + new tokens exceed the length table");
  if (G < 1 || K % G != 0) throw std::runtime_error("beam_step: the beam groups must divide the beams");
  if (G > 1 && (!logits || !logz || nsel < K + K / G))
    throw std::runtime_error("beam_step: beam groups need the logits, logZ and nsel >= K + K / G per-row candidates");
  if (!(rep_penalty > 0.f) || !std::isfinite(rep_penalty) || (d.P > 1 && !d.prefix))
    throw std::runtime_error("beam_step: repetition penalty must be finite and > 0, prefix given when P > 1");
  launch_k(beam_step_kernel, dim3((B + kBeamWarps - 1) / kBeamWarps), dim3(kBeamWarps * 32), 0, stream, bb, B, K, G, T, V, nsel, sel_val, sel_idx,
           logits, ldl, logz, penalty, rep_penalty, d, eos, lp, out_beam_idx, out_tokens, out_scores);
  return 1;
}
int launch_beam_finalize(const BeamBuffers& bb, int B, int K, int T, int eos, int len0, const int* p0s, int per_image, int N,
                         const LenPenalty& lp, int64_t* out_ids, float* out_scores, cudaStream_t stream) {
  if (N < 1 || N > K) throw std::runtime_error("beam_finalize: 1 <= N <= K");
  if (len0 + T > kMaxHypLen) throw std::runtime_error("beam_finalize: prefix + new tokens exceed the length table");
  if (per_image < 1 || B % per_image != 0) throw std::runtime_error("beam_finalize: the searches must be a multiple of per_image >= 1");
  beam_finalize_kernel<<<(B + 31) / 32, 32, 0, stream>>>(bb, B, K, T, eos, len0, p0s, per_image, N, lp, out_ids, out_scores);
  return 1;
}
int launch_beam_ngram_ban(int B, int Lh, const int64_t* hist_ids, const int64_t* hist_seg, const DecInput& d, int step, int n,
                          int32_t* ban_tokens, int32_t* ban_count, int ban_stride, cudaStream_t stream) {
  if (B <= 0) return 0;
  if (d.rows_per_image > kBanMaxK || n < 1) throw std::runtime_error("beam_ngram_ban: at most 8 rows per image, n >= 1");
  check_dec_input(d, step, "beam_ngram_ban");
  launch_k(beam_ngram_ban_kernel, dim3(B), dim3(256), 0, stream, Lh, hist_ids, hist_seg, d, step, n, ban_tokens, ban_count, ban_stride);
  return 1;
}
int launch_sample_step(int rows, int N, int T, int nsel, const float* sel_val, const int32_t* sel_idx, int top_k, float top_p,
                       uint64_t seed, uint64_t row_offset, const uint64_t* d_seed, const int* d_step, int32_t* seq, int32_t* cur_tokens,
                       int32_t* out_tokens, cudaStream_t stream) {
  if (top_k < 1 || top_k > nsel) throw std::runtime_error("sample_step: top_k out of range");
  if (N < 1 || rows % N != 0) throw std::runtime_error("sample_step: rows must be a multiple of N >= 1");
  launch_k(sample_step_kernel, dim3((rows + 63) / 64), dim3(64), 0, stream, rows, N, T, nsel, sel_val, sel_idx, top_k, top_p, seed, row_offset, d_seed, d_step, seq,
                                                          cur_tokens, out_tokens);
  return 1;
}
int launch_full_vocab_sample(int rows, int N, int V, const float* logits, int64_t ldl, float temperature, float top_p, const int32_t* ban_tokens,
                             const int32_t* ban_count, int ban_stride, int T, uint64_t seed, uint64_t row_offset, const uint64_t* d_seed,
                             const int* d_step, int32_t* seq, int32_t* cur_tokens, int32_t* out_tokens, const LogitsProcs& procs,
                             cudaStream_t stream) {
  if (rows <= 0) return 0;
  if (N < 1 || rows % N != 0) throw std::runtime_error("full_vocab_sample: rows must be a multiple of N >= 1");
  if (V > kFvThreads * kFvPer) throw std::runtime_error("full_vocab_sample: vocab > 32768");
  check_procs(procs, "full_vocab_sample");
  constexpr size_t smem = (size_t)kFvThreads * kFvPer * sizeof(float);
  static bool attr_set = false;
  if (!attr_set) {
    for (auto k : {full_vocab_sample_kernel<false>, full_vocab_sample_kernel<true>}) {
      cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) throw std::runtime_error(std::string("full_vocab_sample: cudaFuncSetAttribute: ") + cudaGetErrorString(e));
    }
    attr_set = true;
  }
  launch_k(procs.active() ? full_vocab_sample_kernel<true> : full_vocab_sample_kernel<false>, dim3(rows), dim3(kFvThreads), smem, stream, N, V, logits, ldl, temperature, top_p, ban_tokens, ban_count, ban_stride,
           T, seed, row_offset, d_seed, d_step, seq, cur_tokens, out_tokens, procs);
  return 1;
}
int launch_sample_init(int rows, int N, int T, int start_token, int32_t* seq, int32_t* cur_tokens, int* d_step, const int64_t* dec_prefix,
                       int P, int* p0s, cudaStream_t stream) {
  if (P < 1 || (P > 1 && !dec_prefix)) throw std::runtime_error("sample_init: P >= 1, prefix given when P > 1");
  if (N < 1 || rows % N != 0) throw std::runtime_error("sample_init: rows must be a multiple of N >= 1");
  if (p0s && !dec_prefix) throw std::runtime_error("sample_init: per-image prefix lengths need a prefix");
  sample_init_kernel<<<(rows + 63) / 64, 64, 0, stream>>>(rows, N, T, start_token, seq, cur_tokens, d_step, dec_prefix, P, p0s);
  return 1;
}
int launch_sample_finalize(int rows, int T, int eos, const int32_t* seq, int64_t* out_ids, cudaStream_t stream) {
  sample_finalize_kernel<<<(rows + 63) / 64, 64, 0, stream>>>(rows, T, eos, seq, out_ids);
  return 1;
}
int launch_set_u64(uint64_t* dst, uint64_t v, uint64_t v1, cudaStream_t stream) {
  set_u64_kernel<<<1, 32, 0, stream>>>(dst, v, v1);
  return 1;
}
int launch_step_advance(int* d_step, cudaStream_t stream) {
  launch_k(step_advance_kernel, dim3(1), dim3(32), 0, stream, d_step);
  return 1;
}
int launch_shift_labels(int B, int L, int64_t* dec_ids, int64_t* labels, int eos, cudaStream_t stream) {
  shift_labels_kernel<<<B, 128, 0, stream>>>(L, dec_ids, labels, eos);
  return 1;
}
int launch_ce_loss(int rows, int V, const float* logits, int64_t ldl, const int64_t* labels, float* loss, cudaStream_t stream) {
  if (rows <= 0) return 0;
  ce_loss_kernel<<<rows, 256, 0, stream>>>(V, logits, ldl, labels, loss);
  return 1;
}
int launch_splice(int B, int Lt, int Lu, int64_t* ids, int64_t* seg, float* mask, int32_t* enc_len, const int64_t* utt,
                  int segment_value, int strip_sep, int32_t* abnormal, int sep, cudaStream_t stream) {
  splice_kernel<<<(B + 63) / 64, 64, 0, stream>>>(B, Lt, Lu, ids, seg, mask, enc_len, utt, segment_value, strip_sep, abnormal, sep);
  return 1;
}

}  // namespace gstvd
