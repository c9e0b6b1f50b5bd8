// Decode-step kernels over the persistent KV cache (HBM-bound).
//
// The reference has no KV cache: it re-runs the whole decoder over the whole prefix and re-projects the
// cross-attention K/V on every step (use_cache=False hard-wired, models/visual_dialog_decoder.py:64; loop at
// models/visual_dialog_model.py:86-110).  Here each step processes ONE new position per beam row:
//   dec_self_attn  : appends the new K/V at position g.p0(b) + *d_step and attends over positions 0..g.p0(b) + *d_step
//                    (g.p0(b) = image b's decoder prefix length - 1; positions below it were stored by prefix_kv_store)
//   dec_cross_attn : every beam row of an image attends over that image's cross K/V (stored once per image)
//   reorder_cache  : in-place beam gather, the semantic of _reorder_cache / index_select(0, beam_idx)
//                    (models/visual_dialog_decoder.py:29-31,177-181)
// Layouts:  self cache  [layer][k|v][image][position][beam][hidden]   (a beam gather touches contiguous rows)
//           cross cache [layer][image][k|v, head][position][head_dim]  (one contiguous block per (image, head))
#include <algorithm>
#include <cstdlib>
#include <stdexcept>

#include "common.cuh"
#include "kernels.h"

namespace gstvd {

namespace {

constexpr int kMaxSteps = 32;     // one score per lane / one ancestry row of today's decode calls
constexpr int kMaxPos = 64;       // cached positions of a prefixed call (prefix up to max_dec_len + new tokens): two scores per lane
constexpr int kMaxBeams = 8;

template <typename T> struct Raw16 {};
template <> struct Raw16<bf16> {
  static __device__ __forceinline__ void unpack(const uint4& r, float (&o)[8]) {
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&r);
#pragma unroll
    for (int i = 0; i < 4; ++i) { float2 f = __bfloat1622float2(h[i]); o[2 * i] = f.x; o[2 * i + 1] = f.y; }
  }
};
template <> struct Raw16<float> {
  static __device__ __forceinline__ void unpack(const uint4& r, float (&o)[4]) {
    o[0] = __uint_as_float(r.x); o[1] = __uint_as_float(r.y); o[2] = __uint_as_float(r.z); o[3] = __uint_as_float(r.w);
  }
};

// Self-attention of one new position per (beam row, head) over the persistent cache (one warp per (row, head)).
// Scores: lane t owns cached positions t and, with NS = 2 (more than 32 positions), t + 32 and reads its whole key row (16-byte loads, all issued back to back) against the
// query held in shared memory - no serial chain of load + warp-reduction per position; the new position's score is one
// warp reduction.  P*V: lanes split the head dimension; the value rows of the first 16 positions are requested BEFORE the
// scores are computed (they do not depend on them), so key and value loads share one memory round trip.
template <typename T, int ND, int NS>
__global__ void __launch_bounds__(128)
dec_self_attn_kernel(DecodeGeom g, int layer, const T* __restrict__ qkv, T* __restrict__ cache, const int* __restrict__ d_step,
                     T* __restrict__ out) {
  constexpr int EPL = 16 / sizeof(T);
  __shared__ __align__(16) float qs[4][128];
  pdl_wait();
  pdl_launch_dependents();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row = blockIdx.x;
  const int h = blockIdx.y * 4 + warp;
  if (h >= g.heads) return;
  const int b = row / g.K, kb = row - b * g.K;
  const int step = g.p0(b) + *d_step;          // cache position of the new token
  const int H = g.H, D = g.D;
  constexpr int nd = ND;                       // dims per lane (2 for D=64, 4 for D=128)
  const T* qrow = qkv + (int64_t)row * 3 * H + h * D;
  float q[4], kn[4], vn[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    if (u < nd) {
      const int d = lane + 32 * u;
      q[u] = to_f32(qrow[d]); kn[u] = to_f32(qrow[H + d]); vn[u] = to_f32(qrow[2 * H + d]);
      qs[warp][d] = q[u];
    } else { q[u] = kn[u] = vn[u] = 0.f; }
  }
  // cache row of (kv, position t) for this beam/head
  auto cache_ptr = [&](int kv, int t) -> T* {
    return cache + (((((int64_t)layer * 2 + kv) * g.B + b) * g.T + t) * g.K + kb) * H + h * D;
  };
  {
    T* kc = cache_ptr(0, step); T* vc = cache_ptr(1, step);
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (u < nd) { kc[lane + 32 * u] = from_f32<T>(kn[u]); vc[lane + 32 * u] = from_f32<T>(vn[u]); }
  }
  __syncwarp();
  constexpr int VB = 16;                       // value rows in flight per batch
  float vv[VB][ND];
  auto load_v = [&](int t0) {
#pragma unroll
    for (int i = 0; i < VB; ++i) {
      const int t = t0 + i;
      const T* vc = cache_ptr(1, t < step ? t : 0);
#pragma unroll
      for (int u = 0; u < ND; ++u) vv[i][u] = (t < step) ? to_f32(vc[lane + 32 * u]) : 0.f;
    }
  };
  load_v(0);
  const float scale_div = sqrtf((float)D);
  // score of the new position: one reduction over the lanes' dims
  float part = 0.f;
#pragma unroll
  for (int u = 0; u < 4; ++u) part = fmaf(q[u], kn[u], part);
  const float s_new = warp_sum(part) / scale_div;
  // scores of the cached positions: lane t reads key rows t (+ 32)
  float my_score[NS];
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    const int t = lane + 32 * s;
    my_score[s] = -INFINITY;
    if (t < step) {
      const T* kc = cache_ptr(0, t);
      float dot = 0.f;
      for (int c = 0; c < D / EPL; ++c) {
        float kr[EPL];
        const uint4 raw = *reinterpret_cast<const uint4*>(kc + c * EPL);
        Raw16<T>::unpack(raw, kr);
#pragma unroll
        for (int e4 = 0; e4 < EPL; e4 += 4) {
          const float4 qv = *reinterpret_cast<const float4*>(&qs[warp][c * EPL + e4]);
          dot = fmaf(qv.x, kr[e4], dot); dot = fmaf(qv.y, kr[e4 + 1], dot);
          dot = fmaf(qv.z, kr[e4 + 2], dot); dot = fmaf(qv.w, kr[e4 + 3], dot);
        }
      }
      my_score[s] = dot / scale_div;
    } else if (t == step) {
      my_score[s] = s_new;
    }
  }
  float mx = my_score[0];
#pragma unroll
  for (int s = 1; s < NS; ++s) mx = fmaxf(mx, my_score[s]);
  mx = warp_max(mx);
  float e[NS], esum = 0.f;
#pragma unroll
  for (int s = 0; s < NS; ++s) { e[s] = (lane + 32 * s <= step) ? expf(my_score[s] - mx) : 0.f; esum += e[s]; }
  const float sum = warp_sum(esum);
  float pr[NS];
#pragma unroll
  for (int s = 0; s < NS; ++s) pr[s] = e[s] / sum;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  for (int t0 = 0; t0 < step; t0 += VB) {
    if (t0 > 0) load_v(t0);
    const float prs = (NS == 1 || t0 < 32) ? pr[0] : pr[NS - 1];   // VB divides 32: one score register per batch
#pragma unroll
    for (int i = 0; i < VB; ++i) {
      const float pt = __shfl_sync(0xffffffffu, prs, (t0 + i) & 31);
      if (t0 + i < step) {
#pragma unroll
        for (int u = 0; u < ND; ++u) acc[u] = fmaf(pt, vv[i][u], acc[u]);
      }
    }
  }
  {
    const float pt = __shfl_sync(0xffffffffu, (NS == 1 || step < 32) ? pr[0] : pr[NS - 1], step & 31);
    // in bf16 mode later steps read the ROUNDED new value from the cache; use the same value now
#pragma unroll
    for (int u = 0; u < 4; ++u) acc[u] = fmaf(pt, to_f32(from_f32<T>(vn[u])), acc[u]);
  }
  T* o = out + (int64_t)row * H + h * D;
#pragma unroll
  for (int u = 0; u < 4; ++u)
    if (u < nd) o[lane + 32 * u] = from_f32<T>(acc[u]);
}

// bf16, D = 64 variant with a third of the instructions (the kernel above is issue-bound: ~1100 warp instructions per (row, head),
// 56 % issue-slot utilisation in ncu).  One warp per (row, head); a cached key / value row is 128 bytes = eight 16-byte chunks, so
// eight lanes own one position and the warp covers four positions per load instruction: lane = 8 * (position % 4) + chunk.
//   * every load of the kernel - q / k / v of the new position, *d_step, the K and V rows of ALL g.T cache positions - is issued
//     in one batch right after the PDL wait (rows past *d_step are allocated; their scores are masked afterwards), so the kernel
//     pays ONE memory round trip instead of three dependent ones;
//   * scores: 8 FMAs per lane + a 3-step butterfly inside the 8-lane group; softmax statistics: 2-step butterflies across groups;
//   * P * V: each lane accumulates its 8 dims over its positions, one 2-step butterfly per dim merges the four groups and lanes 0-7
//     store the 128-byte output row.
// The new position's k / v are taken from qkv (rounded to bf16, i.e. exactly what later steps will read back from the cache).
// NIT = 16 covers the 64 positions of a prefixed call; its ancestry rows are 64 entries wide (kAncRow).
template <int NIT> struct AncRow { static constexpr int value = NIT * 4 > kMaxSteps ? kMaxPos : kMaxSteps; };
template <int NIT>
__global__ void __launch_bounds__(128)
dec_self_attn_v2_kernel(DecodeGeom g, int layer, const bf16* __restrict__ qkv, bf16* __restrict__ cache, const int* __restrict__ d_step,
                        int step_host, const uint8_t* __restrict__ anc, bf16* __restrict__ out) {
  pdl_wait();
  pdl_launch_dependents();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row = blockIdx.x;
  const int h = blockIdx.y * 4 + warp;
  if (h >= g.heads) return;
  const int b = row / g.K, kb = row - b * g.K;
  const int H = g.H;
  const int chunk = lane & 7, grp = lane >> 3;
  const bf16* qrow = qkv + (int64_t)row * 3 * H + h * 64 + chunk * 8;
  const uint4 q_raw = *reinterpret_cast<const uint4*>(qrow);
  const uint4 kn_raw = *reinterpret_cast<const uint4*>(qrow + H);
  const uint4 vn_raw = *reinterpret_cast<const uint4*>(qrow + 2 * H);
  // step_host >= 0: the launch knows the step (eager loops and the all-steps graph unroll them), so the loads below are bounded by
  // it - on average half of the g.T cache rows - without waiting for *d_step; otherwise every row is requested and masked afterwards
  // cache position of the new token; g.P0s is read after the PDL wait (the init kernel that wrote it may precede this launch)
  const int step = g.p0(b) + (step_host >= 0 ? step_host : *d_step);
  const int bound = step_host >= 0 ? step : g.T;                     // cache positions < bound are requested (per row)
  // element offset of (kv, position t) for this beam / head / chunk
  const int64_t pos_stride = (int64_t)g.K * H;
  const int64_t k_base = ((((int64_t)layer * 2 + 0) * g.B + b) * g.T) * pos_stride + h * 64 + chunk * 8;   // slot 0 of position 0
  const int64_t v_base = k_base + (int64_t)g.B * g.T * pos_stride;
  // Beam search without moving the cache (anc != null): position t of this beam's history lives in the slot of the beam that
  // wrote it, anc[(b*K + kb)*W + t] (anc_update_kernel permutes the W-byte rows after every selection); the new position is
  // always written to the beam's own slot.  Entries at or past the new position are stale but always < 8; they are clamped and
  // masked.  Prefix positions (below g.p0(b)) hold the same K / V in every slot, so whatever their entries say is correct.
  constexpr int W = AncRow<NIT>::value;
  int slot[NIT];
#pragma unroll
  for (int it = 0; it < NIT; ++it) {
    const int t = it * 4 + grp;
    slot[it] = (anc != nullptr && t < bound) ? min((int)anc[((int64_t)b * g.K + kb) * W + (t & (W - 1))], g.K - 1) : kb;
  }
  uint4 k_raw[NIT], v_raw[NIT];
#pragma unroll
  for (int it = 0; it < NIT; ++it) {
    const int t = it * 4 + grp;
    if (t < bound && t < g.T) {                      // rows at or past the bound are never used (t == step comes from qkv, t > step is masked)
      k_raw[it] = *reinterpret_cast<const uint4*>(cache + k_base + t * pos_stride + (int64_t)slot[it] * H);
      v_raw[it] = *reinterpret_cast<const uint4*>(cache + v_base + t * pos_stride + (int64_t)slot[it] * H);
    } else {
      k_raw[it] = make_uint4(0, 0, 0, 0);
      v_raw[it] = make_uint4(0, 0, 0, 0);
    }
  }
  // append the new position (lanes 0-7: key chunks, lanes 8-15: value chunks)
  if (grp == 0) *reinterpret_cast<uint4*>(cache + k_base + step * pos_stride + (int64_t)kb * H) = kn_raw;
  else if (grp == 1) *reinterpret_cast<uint4*>(cache + v_base + step * pos_stride + (int64_t)kb * H) = vn_raw;

  float q[8];
  Raw16<bf16>::unpack(q_raw, q);
  float sc[NIT];
  float mx = -INFINITY;
#pragma unroll
  for (int it = 0; it < NIT; ++it) {
    const int t = it * 4 + grp;
    if (t == step) { k_raw[it] = kn_raw; v_raw[it] = vn_raw; }
    float kr[8];
    Raw16<bf16>::unpack(k_raw[it], kr);
    float dot = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) dot = fmaf(q[j], kr[j], dot);
    dot += __shfl_xor_sync(0xffffffffu, dot, 1);
    dot += __shfl_xor_sync(0xffffffffu, dot, 2);
    dot += __shfl_xor_sync(0xffffffffu, dot, 4);
    sc[it] = t <= step ? dot * 0.125f : -INFINITY;   // 1 / sqrt(64), exact
    mx = fmaxf(mx, sc[it]);
  }
  mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 8));
  mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 16));
  float sum = 0.f;
#pragma unroll
  for (int it = 0; it < NIT; ++it) { sc[it] = expf(sc[it] - mx); sum += sc[it]; }   // exp(-inf) = 0 for the masked slots
  sum += __shfl_xor_sync(0xffffffffu, sum, 8);
  sum += __shfl_xor_sync(0xffffffffu, sum, 16);
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int it = 0; it < NIT; ++it) {
    const float pr = sc[it] / sum;
    float vr[8];
    Raw16<bf16>::unpack(v_raw[it], vr);
    if (it * 4 + grp <= step) {                      // stale rows may hold anything (NaN bit patterns included): skip, do not scale by 0
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] = fmaf(pr, vr[j], acc[j]);
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], 8);
    acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], 16);
  }
  if (grp == 0) Vec8<bf16>::store(out + (int64_t)row * H + h * 64 + chunk * 8, acc);
}

constexpr int kCrossThreads = 320;            // 10 warps: one thread per key in the score phase (Le = 293 in the real model)

template <typename T, int KB, int D>
__global__ void __launch_bounds__(kCrossThreads, 2)
dec_cross_attn_kernel(DecodeGeom g, const T* __restrict__ q, const T* __restrict__ kv_layer, const float* __restrict__ enc_mask,
                      T* __restrict__ out) {
  constexpr int EPL = 16 / sizeof(T);          // elements per 16-byte load
  constexpr int CPR = D / EPL;                 // 16-byte chunks per key row (8 for bf16, 16 for fp32)
  constexpr int LPR = CPR;                     // phase 2: lanes per key row
  constexpr int RPI = 32 / LPR;                // phase 2: key rows per warp-wide load
  constexpr int kWarps = kCrossThreads / 32;
  constexpr int NIT = 8;                       // phase 2: V loads in flight per lane (10 warps x RPI x 8 keys per pass)
  constexpr int kPass = kWarps * RPI * NIT;
  extern __shared__ float smem[];
  const int Le = g.Le;
  float* S = smem;                             // [KB][Le] scores, then probabilities
  float* part = smem + ((KB * Le + 3) & ~3);   // [kWarps][KB][D] partial outputs
  float* qs = part + kWarps * KB * D;          // [KB][D] queries (fp32), 16-byte aligned
  pdl_launch_dependents();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int h = blockIdx.x, b = blockIdx.y;
  const T* Kp = kv_layer + ((int64_t)b * 2 * g.heads + h) * Le * D;
  const T* Vp = kv_layer + ((int64_t)b * 2 * g.heads + g.heads + h) * Le * D;
  const float* mrow = enc_mask ? enc_mask + (int64_t)b * Le : nullptr;
  const uint4 zero4 = make_uint4(0, 0, 0, 0);

  // ---- phase 1: scores, one thread per key.  The whole key row (D elements) is loaded with CPR independent 16-byte
  // loads issued back to back (in flight together), the queries are broadcast from shared memory; no shuffles. ----
  const int j1 = threadIdx.x;
  uint4 kreg[CPR];
  float madd = 0.f;
  if (j1 < Le) {
#pragma unroll
    for (int c = 0; c < CPR; ++c) kreg[c] = *reinterpret_cast<const uint4*>(Kp + (int64_t)j1 * D + c * EPL);
    madd = (1.0f - (mrow ? mrow[j1] : 1.f)) * -1e9f;
  } else {
#pragma unroll
    for (int c = 0; c < CPR; ++c) kreg[c] = zero4;
  }
  pdl_wait();                                 // the K rows above were written at prefill time; q comes from the previous kernel
  for (int i = threadIdx.x; i < KB * D; i += blockDim.x) {
    const int k = i / D, d = i - k * D;
    qs[i] = (k < g.K) ? to_f32(q[((int64_t)(b * g.K + k)) * g.H + h * D + d]) : 0.f;
  }
  __syncthreads();
  const float scale_div = sqrtf((float)D);
  for (int j = j1; j < Le; j += blockDim.x) {
    if (j != j1) {                             // only when Le > blockDim.x
#pragma unroll
      for (int c = 0; c < CPR; ++c) kreg[c] = *reinterpret_cast<const uint4*>(Kp + (int64_t)j * D + c * EPL);
      madd = (1.0f - (mrow ? mrow[j] : 1.f)) * -1e9f;
    }
    float dot[KB];
#pragma unroll
    for (int k = 0; k < KB; ++k) dot[k] = 0.f;
#pragma unroll
    for (int c = 0; c < CPR; ++c) {
      float kr[EPL];
      Raw16<T>::unpack(kreg[c], kr);
#pragma unroll
      for (int k = 0; k < KB; ++k) {
#pragma unroll
        for (int e4 = 0; e4 < EPL; e4 += 4) {
          const float4 qv = *reinterpret_cast<const float4*>(qs + k * D + c * EPL + e4);   // warp-wide broadcast
          dot[k] = fmaf(qv.x, kr[e4], dot[k]); dot[k] = fmaf(qv.y, kr[e4 + 1], dot[k]);
          dot[k] = fmaf(qv.z, kr[e4 + 2], dot[k]); dot[k] = fmaf(qv.w, kr[e4 + 3], dot[k]);
        }
      }
    }
#pragma unroll
    for (int k = 0; k < KB; ++k)
      if (k < g.K) S[k * Le + j] = dot[k] / scale_div + madd;
  }
  // V loads of the first pass: in flight while the softmax runs
  const int sub = lane / LPR, chunk = lane % LPR;
  uint4 vreg[NIT];
#pragma unroll
  for (int it = 0; it < NIT; ++it) {
    const int j = (it * kWarps + warp) * RPI + sub;
    vreg[it] = (j < Le) ? *reinterpret_cast<const uint4*>(Vp + (int64_t)j * D + chunk * EPL) : zero4;
  }
  __syncthreads();
  // ---- softmax: one warp per beam ----
  for (int k = warp; k < g.K; k += kWarps) {
    float mx = -INFINITY;
    for (int j = lane; j < Le; j += 32) mx = fmaxf(mx, S[k * Le + j]);
    mx = warp_max(mx);
    float sum = 0.f;
    for (int j = lane; j < Le; j += 32) { const float e = expf(S[k * Le + j] - mx); S[k * Le + j] = e; sum += e; }
    sum = warp_sum(sum);
    for (int j = lane; j < Le; j += 32) S[k * Le + j] = S[k * Le + j] / sum;
  }
  __syncthreads();
  // ---- phase 2: P * V (lanes split the head dimension; every V byte is read once, coalesced) ----
  float acc[KB][EPL];
#pragma unroll
  for (int k = 0; k < KB; ++k)
#pragma unroll
    for (int e = 0; e < EPL; ++e) acc[k][e] = 0.f;
  for (int base = 0; base < Le; base += kPass) {
    if (base > 0) {
#pragma unroll
      for (int it = 0; it < NIT; ++it) {
        const int j = base + (it * kWarps + warp) * RPI + sub;
        vreg[it] = (j < Le) ? *reinterpret_cast<const uint4*>(Vp + (int64_t)j * D + chunk * EPL) : zero4;
      }
    }
#pragma unroll
    for (int it = 0; it < NIT; ++it) {
      const int j = base + (it * kWarps + warp) * RPI + sub;
      if (j < Le) {
        float vr[EPL];
        Raw16<T>::unpack(vreg[it], vr);
#pragma unroll
        for (int k = 0; k < KB; ++k) {
          const float p = (k < g.K) ? S[k * Le + j] : 0.f;
#pragma unroll
          for (int e = 0; e < EPL; ++e) acc[k][e] = fmaf(p, vr[e], acc[k][e]);
        }
      }
    }
  }
  // reduce over the RPI key sub-rows held by different lane groups, then over warps through shared memory
#pragma unroll
  for (int k = 0; k < KB; ++k)
#pragma unroll
    for (int e = 0; e < EPL; ++e) {
      float v = acc[k][e];
#pragma unroll
      for (int o = LPR; o < 32; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      acc[k][e] = v;
    }
  if (sub == 0) {
#pragma unroll
    for (int k = 0; k < KB; ++k)
#pragma unroll
      for (int e = 0; e < EPL; ++e) part[(warp * KB + k) * D + chunk * EPL + e] = acc[k][e];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < g.K * D; i += blockDim.x) {
    const int k = i / D, d = i - k * D;
    float v = 0.f;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) v += part[(w * KB + k) * D + d];
    out[((int64_t)(b * g.K + k)) * g.H + h * D + d] = from_f32<T>(v);
  }
}

// ---- tensor-core decode cross-attention (bf16, head_dim 64, <= 8 beams, Le <= 320) ----------------------------------
// One CTA of 4 warps per (image, head).  Every K / V byte is loaded from global exactly once, as a 16-byte load, straight
// into mma.sync fragments - no shared-memory staging of K or V:
//   scores  S = Q K^T : the 8 keys of a tile are the N dimension, the beams the (zero padded) M rows.  The reduction index
//            (head dim) may be permuted freely as long as A and B agree, so the natural 16-byte chunk a lane loads from a key
//            row (8 consecutive dims) is used as the lane's two k-slot pairs of two k-steps; Q is loaded the same way.
//   context O = P V   : V rows are loaded the same way and transposed in registers with movmatrix (8x8 b16), which yields
//            B fragments whose N index is a permutation of the head dim; the permutation is chosen so that each lane ends up
//            with 8 CONSECUTIVE output dims.
// Softmax is the exact two-pass softmax over all keys (scores in shared memory), like the reference.
__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], uint32_t a0, uint32_t a2, uint32_t b0, uint32_t b1) {
  const uint32_t z = 0u;   // rows 8..15 of the A tile (beams that do not exist) are zero
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(z), "r"(a2), "r"(z), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t movmatrix_trans(uint32_t a) {
  uint32_t d;
  asm volatile("movmatrix.sync.aligned.m8n8.trans.b16 %0, %1;" : "=r"(d) : "r"(a));
  return d;
}

constexpr int kXMaxTiles = 10;   // key tiles (8 keys) per warp: 4 warps x 10 x 8 = 320 keys
constexpr int kXMaxGroups = 5;   // 16-key groups per warp

__global__ void __launch_bounds__(128, 6)
dec_cross_mma_kernel(DecodeGeom g, const bf16* __restrict__ q, const bf16* __restrict__ kv_layer, const float* __restrict__ enc_mask,
                     bf16* __restrict__ out) {
  constexpr int D = 64;
  extern __shared__ __align__(16) uint8_t xsm[];
  const int Le = g.Le, LeP = (Le + 15) & ~15;
  float* S = reinterpret_cast<float*>(xsm);                       // [8][LeP]
  float* madd = S + 8 * LeP;                                      // [LeP]
  float* part = madd + LeP;                                       // [4][8][64]
  bf16* P = reinterpret_cast<bf16*>(part + 4 * 8 * D);            // [8][LeP]
  pdl_launch_dependents();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int h = blockIdx.x, b = blockIdx.y;
  const int beam = lane >> 2, p4 = lane & 3;
  const bf16* Kp = kv_layer + ((int64_t)b * 2 * g.heads + h) * Le * D;
  const bf16* Vp = kv_layer + ((int64_t)b * 2 * g.heads + g.heads + h) * Le * D;
  const uint4 zero4 = make_uint4(0, 0, 0, 0);
  const int ntiles = (Le + 7) >> 3, ngroups = LeP >> 4;

  // K fragments of this warp's first key tiles: independent of the previous kernel (written at prefill), issued before the
  // PDL wait.  Tiles are processed in two batches of 5 to keep the register count low enough for 6 CTAs per SM (one wave).
  constexpr int kKB = kXMaxTiles / 2;
  uint4 kreg[kKB][2];
  auto load_k = [&](int i0) {
#pragma unroll
    for (int i = 0; i < kKB; ++i) {
      const int t = warp + 4 * (i0 + i);
      const int key = t * 8 + beam;                               // lane / 4 = key inside the tile
      if (t < ntiles && key < Le) {
        const bf16* kp = Kp + (int64_t)key * D + p4 * 8;
        kreg[i][0] = *reinterpret_cast<const uint4*>(kp);
        kreg[i][1] = *reinterpret_cast<const uint4*>(kp + 32);
      } else { kreg[i][0] = zero4; kreg[i][1] = zero4; }
    }
  };
  load_k(0);
  for (int j = threadIdx.x; j < LeP; j += blockDim.x)
    madd[j] = (j < Le) ? (1.0f - (enc_mask ? enc_mask[(int64_t)b * Le + j] : 1.f)) * -1e9f : 0.f;
  pdl_wait();
  uint4 qlo = zero4, qhi = zero4;
  if (beam < g.K) {
    const bf16* qp = q + ((int64_t)(b * g.K + beam)) * g.H + h * D + p4 * 8;
    qlo = *reinterpret_cast<const uint4*>(qp);
    qhi = *reinterpret_cast<const uint4*>(qp + 32);
  }
  __syncthreads();                                                // madd visible
  // ---- scores ----
#pragma unroll
  for (int i0 = 0; i0 < kXMaxTiles; i0 += kKB) {
    if (i0 > 0) load_k(i0);
#pragma unroll
    for (int i = 0; i < kKB; ++i) {
      const int t = warp + 4 * (i0 + i);
      if (t < ntiles) {
        float c[4] = {0.f, 0.f, 0.f, 0.f};
        mma_bf16_16816(c, qlo.x, qlo.y, kreg[i][0].x, kreg[i][0].y);
        mma_bf16_16816(c, qlo.z, qlo.w, kreg[i][0].z, kreg[i][0].w);
        mma_bf16_16816(c, qhi.x, qhi.y, kreg[i][1].x, kreg[i][1].y);
        mma_bf16_16816(c, qhi.z, qhi.w, kreg[i][1].z, kreg[i][1].w);
        const int key0 = t * 8 + p4 * 2;                          // C fragment: row = lane/4 (beam), cols = (lane%4)*2 + {0,1}
        if (beam < g.K) {
          if (key0 < Le) S[beam * LeP + key0] = c[0] / 8.0f + madd[key0];
          if (key0 + 1 < Le) S[beam * LeP + key0 + 1] = c[1] / 8.0f + madd[key0 + 1];
        }
      }
    }
  }
  // V rows of this warp's first 16-key groups: in flight while the softmax runs
  constexpr int kVB = 3;
  uint4 vreg[kVB][2][2];                                          // [group][8-key half][dim half]
  auto load_v = [&](int i0) {
#pragma unroll
    for (int i = 0; i < kVB; ++i) {
#pragma unroll
      for (int kh = 0; kh < 2; ++kh) {
        const int G = warp + 4 * (i0 + i);
        const int key = G * 16 + kh * 8 + beam;
        if (i0 + i < kXMaxGroups && G < ngroups && key < Le) {
          const bf16* vp = Vp + (int64_t)key * D + p4 * 8;
          vreg[i][kh][0] = *reinterpret_cast<const uint4*>(vp);
          vreg[i][kh][1] = *reinterpret_cast<const uint4*>(vp + 32);
        } else { vreg[i][kh][0] = zero4; vreg[i][kh][1] = zero4; }
      }
    }
  };
  load_v(0);
  __syncthreads();
  // ---- exact softmax, one warp per beam; probabilities stored as bf16 (zero past Le) ----
  for (int k = warp; k < 8; k += 4) {
    float* Sr = S + k * LeP;
    bf16* Pr = P + k * LeP;
    if (k < g.K) {
      float mx = -INFINITY;
      for (int j = lane; j < Le; j += 32) mx = fmaxf(mx, Sr[j]);
      mx = warp_max(mx);
      float sum = 0.f;
      for (int j = lane; j < Le; j += 32) { const float e = expf(Sr[j] - mx); Sr[j] = e; sum += e; }
      sum = warp_sum(sum);
      for (int j = lane; j < LeP; j += 32) Pr[j] = __float2bfloat16_rn(j < Le ? Sr[j] / sum : 0.f);
    } else {
      for (int j = lane; j < LeP; j += 32) Pr[j] = __float2bfloat16_rn(0.f);
    }
  }
  __syncthreads();
  // ---- context ----
  float o[8][4];
#pragma unroll
  for (int n = 0; n < 8; ++n) { o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f; }
#pragma unroll
  for (int i0 = 0; i0 < kXMaxGroups; i0 += kVB) {
    if (i0 > 0) load_v(i0);
#pragma unroll
    for (int i = 0; i < kVB; ++i) {
      const int G = warp + 4 * (i0 + i);
      if (i0 + i < kXMaxGroups && G < ngroups) {
        const uint32_t* prow = reinterpret_cast<const uint32_t*>(P + beam * LeP + G * 16);
        const uint32_t a0 = prow[p4], a2 = prow[4 + p4];          // keys 16G + (lane%4)*2 + {0,1} and + 8
#pragma unroll
        for (int dh = 0; dh < 2; ++dh) {
          const uint4 v0 = vreg[i][0][dh], v1 = vreg[i][1][dh];
          const uint32_t w0[4] = {v0.x, v0.y, v0.z, v0.w}, w1[4] = {v1.x, v1.y, v1.z, v1.w};
#pragma unroll
          for (int j = 0; j < 4; ++j)
            mma_bf16_16816(o[dh * 4 + j], a0, a2, movmatrix_trans(w0[j]), movmatrix_trans(w1[j]));
        }
      }
    }
  }
  // lane holds O[beam = lane/4][dims dh*32 + (lane%4)*8 + 2j + {0,1}] summed over this warp's keys; reduce over warps
#pragma unroll
  for (int dh = 0; dh < 2; ++dh)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float* pp = part + ((warp * 8 + beam) * D) + dh * 32 + p4 * 8 + 2 * j;
      pp[0] = o[dh * 4 + j][0];
      pp[1] = o[dh * 4 + j][1];
    }
  __syncthreads();
  for (int i = threadIdx.x; i < g.K * D; i += blockDim.x) {
    const int k = i / D, d = i - k * D;
    const float v = (part[(0 * 8 + k) * D + d] + part[(1 * 8 + k) * D + d]) + (part[(2 * 8 + k) * D + d] + part[(3 * 8 + k) * D + d]);
    out[((int64_t)(b * g.K + k)) * g.H + h * D + d] = __float2bfloat16_rn(v);
  }
}

template <typename T, int KB>
void launch_cross_kb(const DecodeGeom& g, const T* q, const T* kv_layer, const float* enc_mask, T* out, cudaStream_t stream) {
  const size_t s_elems = ((size_t)KB * g.Le + 3) & ~size_t(3);          // keeps the query tile 16-byte aligned
  const size_t smem = (s_elems + (size_t)(kCrossThreads / 32) * KB * 64 + (size_t)KB * 64) * sizeof(float);
  dim3 grid(g.heads, g.B);
  launch_k(dec_cross_attn_kernel<T, KB, 64>, grid, dim3(kCrossThreads), smem, stream, g, q, kv_layer, enc_mask, out);
}
template <typename T>
void launch_cross_t(const DecodeGeom& g, const void* q, const void* kv_layer, const float* enc_mask, void* out, cudaStream_t stream) {
  const T* qq = (const T*)q; const T* kv = (const T*)kv_layer; T* o = (T*)out;
  if (g.K == 1) launch_cross_kb<T, 1>(g, qq, kv, enc_mask, o, stream);
  else if (g.K == 2) launch_cross_kb<T, 2>(g, qq, kv, enc_mask, o, stream);
  else if (g.K <= 4) launch_cross_kb<T, 4>(g, qq, kv, enc_mask, o, stream);
  else if (g.K == 5) launch_cross_kb<T, 5>(g, qq, kv, enc_mask, o, stream);
  else launch_cross_kb<T, 8>(g, qq, kv, enc_mask, o, stream);
}

// Beam reorder without moving the cache: new beam k continues old beam parent = beam_idx[b][k]; its history row becomes the
// parent's row and the position just written (t = *d_step) is found in the parent's slot.  One CTA per image; every entry is
// read before any is written (parents may repeat).  Replaces reorder_cache_kernel (up to 2 x 100 MB of HBM traffic per step at
// B = 64, K = 5) when the self-attention kernel reads through the table (dec_self_attn_v2_kernel).  W = row width (positions);
// the position just written is p0 + *d_step, p0 = p0s[b] (per-image decoder prefixes) or the uniform p0.
template <int W>
__global__ void __launch_bounds__(kMaxBeams * W)
anc_update_kernel(int B, int K, int p0, const int* __restrict__ p0s, const int32_t* __restrict__ beam_idx, const int* __restrict__ d_step,
                  uint8_t* __restrict__ anc) {
  pdl_wait();
  pdl_launch_dependents();
  const int b = blockIdx.x, k = threadIdx.x / W, t = threadIdx.x % W;
  const int step = (p0s ? p0s[b] : p0) + *d_step;
  int val = 0;
  const bool live = k < K && t <= step;
  if (live) {
    const int parent = beam_idx[b * K + k];
    val = (t == step) ? parent : anc[((int64_t)b * K + parent) * W + t];
  }
  __syncthreads();
  if (live) anc[((int64_t)b * K + k) * W + t] = (uint8_t)val;
}

// Decoder prefix prefill: K / V of the first P-1 prefix positions of every image, computed by a teacher-forced pass (qkv rows
// [B * P0][3H], row = b * P0 + p), copied into EVERY beam slot of that image's cache rows 0..P0-1 - all beams share the prefix, so the
// gather (reorder_cache) and the ancestry path both read correct data there whatever their tables say.  16-byte chunks.
template <typename T>
__global__ void __launch_bounds__(256)
prefix_kv_store_kernel(DecodeGeom g, int layer, const T* __restrict__ qkv, T* __restrict__ cache) {
  constexpr int EPL = 16 / sizeof(T);
  const int chunks = g.H / EPL;
  const int64_t n = (int64_t)g.B * g.P0 * 2 * chunks;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % chunks);
    const int64_t r2 = i / chunks;
    const int kv = (int)(r2 & 1);
    const int64_t row = r2 >> 1;
    const int b = (int)(row / g.P0), p = (int)(row - (int64_t)b * g.P0);
    const uint4 v = *reinterpret_cast<const uint4*>(qkv + row * 3 * g.H + (1 + kv) * g.H + c * EPL);
    T* dst = cache + ((((int64_t)layer * 2 + kv) * g.B + b) * g.T + p) * g.K * g.H + c * EPL;
    for (int k = 0; k < g.K; ++k) *reinterpret_cast<uint4*>(dst + (int64_t)k * g.H) = v;
  }
}

// One CTA per (image, layer*2+kv).  Thread-local dependency only: every thread loads the K source values of its
// column chunk before it stores any of them, so duplicated parents (beam_idx is not a permutation) are safe in place.
template <typename T>
__global__ void __launch_bounds__(256)
reorder_cache_kernel(DecodeGeom g, T* __restrict__ cache, const int32_t* __restrict__ beam_idx, const int* __restrict__ d_len,
                     int len_host, const uint8_t* __restrict__ d_skip) {
  pdl_wait();
  pdl_launch_dependents();
  const int b = blockIdx.x, lk = blockIdx.y;
  if (d_skip && d_skip[b]) return;
  const int len = d_len ? (*d_len + 1) : len_host;   // positions after the image's prefix rows (identical in every slot, never moved)
  int parent[kMaxBeams];
  bool moved = false;
#pragma unroll
  for (int k = 0; k < kMaxBeams; ++k) {
    parent[k] = (k < g.K) ? beam_idx[b * g.K + k] : k;
    moved |= (parent[k] != k);
  }
  if (!moved) return;
  const int chunks = g.H / 8;
  T* base = cache + (((int64_t)lk * g.B + b) * g.T + g.p0(b)) * g.K * g.H;
  for (int i = threadIdx.x; i < len * chunks; i += blockDim.x) {
    const int t = i / chunks, c = (i - t * chunks) * 8;
    T* p = base + (int64_t)t * g.K * g.H + c;
    float vals[kMaxBeams][8];
#pragma unroll
    for (int k = 0; k < kMaxBeams; ++k)
      if (k < g.K && parent[k] != k) Vec8<T>::load(p + (int64_t)parent[k] * g.H, vals[k]);
#pragma unroll
    for (int k = 0; k < kMaxBeams; ++k)
      if (k < g.K && parent[k] != k) Vec8<T>::store(p + (int64_t)k * g.H, vals[k]);
  }
}

}  // namespace

template <int NS>
static void launch_self_generic(int dtype, const DecodeGeom& g, dim3 grid, int layer, const void* qkv, void* self_cache, const int* d_step, void* out,
                         cudaStream_t stream) {
  if (g.D == 64) {
    if (dtype == kF32) launch_k(dec_self_attn_kernel<float, 2, NS>, grid, dim3(128), 0, stream, g, layer, (const float*)qkv, (float*)self_cache, d_step, (float*)out);
    else launch_k(dec_self_attn_kernel<bf16, 2, NS>, grid, dim3(128), 0, stream, g, layer, (const bf16*)qkv, (bf16*)self_cache, d_step, (bf16*)out);
  } else {
    if (dtype == kF32) launch_k(dec_self_attn_kernel<float, 4, NS>, grid, dim3(128), 0, stream, g, layer, (const float*)qkv, (float*)self_cache, d_step, (float*)out);
    else launch_k(dec_self_attn_kernel<bf16, 4, NS>, grid, dim3(128), 0, stream, g, layer, (const bf16*)qkv, (bf16*)self_cache, d_step, (bf16*)out);
  }
}

static bool self_v2_fits(int dtype, const DecodeGeom& g, const void* qkv, const void* self_cache, const void* out) {
  return dtype == kBF16 && g.D == 64 && g.H % 8 == 0 && g.T <= kMaxPos && g.K <= kMaxBeams &&
         (reinterpret_cast<uintptr_t>(qkv) & 15) == 0 && (reinterpret_cast<uintptr_t>(self_cache) & 15) == 0 &&
         (reinterpret_cast<uintptr_t>(out) & 15) == 0;
}

bool dec_self_attn_v2_active(int dtype, const DecodeGeom& g, const void* qkv, const void* self_cache, const void* out) {
  const char* v2_env = getenv("GSTVD_SELF_V2");            // read per call (captured graphs keep what was set at capture time)
  const bool v2 = v2_env == nullptr || atoi(v2_env) != 0;  // default on; GSTVD_SELF_V2=0 selects the first kernel
  return v2 && self_v2_fits(dtype, g, qkv, self_cache, out);
}

bool dec_self_attn_supports(int kernel, int dtype, const DecodeGeom& g, const void* qkv, const void* self_cache, const void* out,
                            const uint8_t* anc) {
  if (g.T > kMaxPos || g.H != g.heads * g.D) return false;
  if (kernel == kSelfV2) return self_v2_fits(dtype, g, qkv, self_cache, out);
  if (kernel == kSelfFirst) return anc == nullptr && (g.D == 64 || g.D == 128);
  return false;
}

bool dec_cross_supports(int kernel, int dtype, const DecodeGeom& g) {
  if (g.H != g.heads * g.D) return false;
  switch (kernel) {
    case kCrossWarpTma: case kCrossCtaTma: return dec_cross_tma_fits(dtype, g);
    case kCrossMma: return dtype == kBF16 && g.D == 64 && g.K <= 8 && g.Le <= 4 * kXMaxTiles * 8;
    // 512 = the encoder length limit of a context: the shared score tile of 8 rows x 1024 keys would not fit 48 KB
    case kCrossSimt: return g.D == 64 && g.K <= 8 && g.Le <= 512;
    case kCrossGeneric: return g.D <= 128 && g.D % 8 == 0 && g.Le <= 512;
    default: return false;
  }
}

int launch_anc_update(const DecodeGeom& g, const int32_t* beam_idx, const int* d_step, uint8_t* anc, cudaStream_t stream) {
  if (g.K > kMaxBeams || g.T > kMaxPos) throw std::runtime_error("anc_update: at most 8 beams and 64 positions");
  if (g.T <= kMaxSteps) launch_k(anc_update_kernel<kMaxSteps>, dim3(g.B), dim3(kMaxBeams * kMaxSteps), 0, stream, g.B, g.K, g.P0, g.P0s, beam_idx, d_step, anc);
  else launch_k(anc_update_kernel<kMaxPos>, dim3(g.B), dim3(kMaxBeams * kMaxPos), 0, stream, g.B, g.K, g.P0, g.P0s, beam_idx, d_step, anc);
  return 1;
}

int launch_prefix_kv_store(int dtype, const DecodeGeom& g, int layer, const void* qkv, void* self_cache, cudaStream_t stream) {
  if (g.P0 < 1) return 0;
  if (g.H % 8) throw std::runtime_error("prefix_kv_store: hidden % 8 != 0");
  const int64_t n = (int64_t)g.B * g.P0 * 2 * (g.H / (dtype == kF32 ? 4 : 8));
  const int blocks = (int)std::min<int64_t>((n + 255) / 256, 1024);
  if (dtype == kF32) prefix_kv_store_kernel<float><<<blocks, 256, 0, stream>>>(g, layer, (const float*)qkv, (float*)self_cache);
  else prefix_kv_store_kernel<bf16><<<blocks, 256, 0, stream>>>(g, layer, (const bf16*)qkv, (bf16*)self_cache);
  return 1;
}

int launch_dec_self_attn(int dtype, const DecodeGeom& g, int layer, const void* qkv, void* self_cache, const int* d_step, int step_host,
                         const uint8_t* anc, void* out, cudaStream_t stream, int force) {
  if (g.D != 64 && g.D != 128) throw std::runtime_error("dec_self_attn: head_dim must be 64 or 128");
  if (g.T > kMaxPos) throw std::runtime_error("dec_self_attn: at most 64 cached positions");
  if (force != kDecDefault && !dec_self_attn_supports(force, dtype, g, qkv, self_cache, out, anc))
    throw std::runtime_error("dec_self_attn: the forced kernel does not support these arguments");
  dim3 grid(g.B * g.K, (g.heads + 3) / 4);
  // lean variant: bf16, 64-dim heads, 16-byte aligned rows
  if (force == kDecDefault ? dec_self_attn_v2_active(dtype, g, qkv, self_cache, out) : force == kSelfV2) {
    if (g.T <= 20) launch_k(dec_self_attn_v2_kernel<5>, grid, dim3(128), 0, stream, g, layer, (const bf16*)qkv, (bf16*)self_cache, d_step, step_host, anc, (bf16*)out);
    else if (g.T <= kMaxSteps) launch_k(dec_self_attn_v2_kernel<8>, grid, dim3(128), 0, stream, g, layer, (const bf16*)qkv, (bf16*)self_cache, d_step, step_host, anc, (bf16*)out);
    else launch_k(dec_self_attn_v2_kernel<16>, grid, dim3(128), 0, stream, g, layer, (const bf16*)qkv, (bf16*)self_cache, d_step, step_host, anc, (bf16*)out);
    return 1;
  }
  if (anc != nullptr) throw std::runtime_error("dec_self_attn: the ancestry table is only read by the bf16 / 64-dim kernel");
  if (g.T <= kMaxSteps) launch_self_generic<1>(dtype, g, grid, layer, qkv, self_cache, d_step, out, stream);
  else launch_self_generic<2>(dtype, g, grid, layer, qkv, self_cache, d_step, out, stream);
  return 1;
}

int launch_dec_cross_attn(int dtype, const DecodeGeom& g, int layer, const void* q, const void* cross_cache,
                          const float* enc_mask, void* out, cudaStream_t stream, int force) {
  if (force != kDecDefault && (force < kCrossMma || !dec_cross_supports(force, dtype, g)))
    throw std::runtime_error("dec_cross_attn: the forced kernel does not support this geometry");
  const int64_t esz = dtype == kF32 ? 4 : 2;
  const int64_t per_image = (int64_t)2 * g.heads * g.Le * g.D;
  const char* kbase = (const char*)cross_cache + ((int64_t)layer * g.B) * per_image * esz;
  const bool mma = force == kDecDefault
                       ? dtype == kBF16 && g.D == 64 && g.K <= 8 && g.Le <= 4 * kXMaxTiles * 8 && getenv("GSTVD_CROSS_SIMT") == nullptr
                       : force == kCrossMma;
  if (mma) {
    const int LeP = (g.Le + 15) & ~15;
    const size_t smem = (size_t)(8 * LeP + LeP + 4 * 8 * 64) * sizeof(float) + (size_t)8 * LeP * sizeof(bf16);
    launch_k(dec_cross_mma_kernel, dim3(g.heads, g.B), dim3(128), smem, stream, g, (const bf16*)q, (const bf16*)kbase, enc_mask, (bf16*)out);
    return 1;
  }
  if (force == kDecDefault ? g.D == 64 && g.K <= 8 && g.Le <= 1024 : force == kCrossSimt) {
    if (dtype == kF32) launch_cross_t<float>(g, q, kbase, enc_mask, out, stream);
    else launch_cross_t<bf16>(g, q, kbase, enc_mask, out, stream);
    return 1;
  }
  AttnArgs a;
  a.q = q; a.q_bs = g.H; a.q_hs = g.D; a.q_rs = 0;
  a.k = kbase; a.k_bs = per_image; a.k_hs = (int64_t)g.Le * g.D; a.k_rs = g.D;
  a.v = kbase + (int64_t)g.heads * g.Le * g.D * esz; a.v_bs = per_image; a.v_hs = a.k_hs; a.v_rs = g.D;
  a.o = out; a.o_bs = g.H; a.o_hs = g.D; a.o_rs = 0;
  a.kmask = enc_mask; a.kmask_bs = g.Le; a.neg = -1e9f; a.causal = 0;
  a.B = g.B * g.K; a.H = g.heads; a.Lq = 1; a.Lk = g.Le; a.D = g.D; a.kv_batch_div = g.K;
  return launch_attention_generic(a, dtype, stream);
}

int launch_reorder_cache(int dtype, const DecodeGeom& g, void* self_cache, const int32_t* beam_idx, const int* d_len,
                         int len_host, const uint8_t* d_skip, cudaStream_t stream) {
  if (g.K > kMaxBeams) throw std::runtime_error("reorder_cache: at most 8 beams");
  if (g.H % 8) throw std::runtime_error("reorder_cache: hidden % 8 != 0");
  dim3 grid(g.B, g.layers * 2);
  if (dtype == kF32) launch_k(reorder_cache_kernel<float>, grid, dim3(256), 0, stream, g, (float*)self_cache, beam_idx, d_len, len_host, d_skip);
  else launch_k(reorder_cache_kernel<bf16>, grid, dim3(256), 0, stream, g, (bf16*)self_cache, beam_idx, d_len, len_host, d_skip);
  return 1;
}

}  // namespace gstvd
