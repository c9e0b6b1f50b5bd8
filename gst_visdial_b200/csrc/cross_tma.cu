// Decode-step cross-attention, TMA-streamed (bf16, head_dim 64, <= 8 beams, Le <= 304).
//
// The K beams of an image attend over that image's encoder states (HF BertSelfAttention in cross mode, call site
// models/visual_dialog_decoder.py:300-311; mask (1-m)*-1e9, :285).  Per layer the step reads every cached cross K / V
// byte once - 10.8 MB per image, the dominant HBM stream of decoding (SURVEY.md 8d) - so the kernel is organised around
// keeping bulk copies in flight, not around the (tiny) math:
//   * K and V of an (image, head) item arrive through TMA (cp.async.bulk.tensor, 64-row boxes, 128-byte swizzle) and complete on
//     mbarriers; the default kernel (dec_cross_warp_kernel, below) gives every item to ONE warp with a private FIFO of boxes,
//     the earlier one (dec_cross_tma2_kernel) loops 8-warp CTAs over the items;
//   * the first boxes are requested before the programmatic-dependent-launch wait: the cross cache is written at prefill, so the
//     stream overlaps the tail of the preceding query-projection GEMM;
//   * only the boxes up to the image's last unmasked key are fetched (cross_len, computed at prefill): the fused mask is
//     [37 image regions | 256 history tokens] and the padded tail of the history has weight exp(-1e9) = 0 exactly.
// Math: mma.sync m16n8k16 with the beams as the (zero padded) M rows, ldmatrix from the swizzled tiles, exact softmax over all
// fetched keys (scores in registers, true maximum) in the log2 domain.
#include <cuda.h>

#include <cstdio>
#include <cstdlib>
#include <stdexcept>

#include "kernels.h"
#include "tma.cuh"

namespace gstvd {

namespace {

using namespace dev;

constexpr int kXtRows = 64;                                // key rows per TMA box
constexpr int kXtMaxBoxes = 5;
constexpr int kXtLeP = 304;                                // row stride of the score / probability tiles (19 groups of 16 keys)
constexpr int kXtBoxBytes = kXtRows * 128;                 // 64 rows x 64 bf16
constexpr int kXtBufBytes = kXtMaxBoxes * kXtBoxBytes;     // 40 KB
constexpr float kLog2e = 1.44269504088896340736f;

// ---- CTA-per-item kernel (rounds 1 and 2 until the warp-per-item kernel below; kept as GSTVD_CROSS_TMA=2 for A/B and as the
// second opinion of test_cross_attention_kernels_agree): 8 warps share an item, scores and probabilities never leave the registers ----
// A warp owns at most three 16-key groups; the m16n8k16 accumulator layout of its scores IS the A-operand layout of the
// probabilities, so after one block-wide max exchange (8 floats per warp) it exponentiates in registers and multiplies by its V
// rows directly; partial contexts and partial sums meet in shared memory once per item.
// Template: kX2Warps warps, kStages (K, V) buffer pairs, kX2Groups key groups per warp; <8, 1, 3> fits two CTAs per SM with single
// buffers (K re-armed after the scores, V after the context product).
template <int kX2Warps, int kStages, int kX2Groups>
struct X2Cfg {
  static constexpr int kThreads = kX2Warps * 32;
  static constexpr int kSmem = 2 * kStages * kXtBufBytes + 2 * kXtLeP * 4 + kX2Warps * 8 * 64 * 4 + 2 * kX2Warps * 8 * 4 + 64 + 1024;
  static_assert(kX2Warps * kX2Groups * 16 >= kXtLeP, "every key group needs an owner");
};

template <int kX2Warps, int kStages, int kX2Groups>
__global__ void __launch_bounds__(kX2Warps * 32, kStages == 1 ? 2 : 1)
dec_cross_tma2_kernel(const __grid_constant__ CUtensorMap tm, DecodeGeom g, int layer, const bf16* __restrict__ q,
                      const float* __restrict__ enc_mask, const int* __restrict__ cross_len, bf16* __restrict__ out,
                      unsigned long long* __restrict__ stamps_all) {
  extern __shared__ uint8_t xt_raw[];
  // measurement aid (env GSTVD_CROSS_TIMES): 16 globaltimer stamps per CTA - start, dependency resolved, then per item
  // K arrived / scores done / V arrived / item stored
  unsigned long long* stamps = (stamps_all != nullptr && threadIdx.x == 0) ? stamps_all + (size_t)blockIdx.x * 16 : nullptr;
  auto stamp = [&](int i) { if (stamps != nullptr && i < 16) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); stamps[i] = t; } };
  stamp(0);
  const uint32_t raw = smem_u32(xt_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;             // swizzled boxes need 1024-byte alignment
  uint8_t* gen = xt_raw + (base - raw);
  // stage s: K at base + s * 80 KB, V 40 KB behind it
  constexpr int kX2Threads = kX2Warps * 32;
  float* madd = reinterpret_cast<float*>(gen + 2 * kStages * kXtBufBytes);         // [2][304] additive mask rows (log2 domain)
  float* part = madd + 2 * kXtLeP;                                       // [16][8][64] partial contexts
  float* wmax = part + kX2Warps * 8 * 64;                                // [16][8] per-warp score maxima
  float* wsum = wmax + kX2Warps * 8;                                     // [16][8] per-warp sums of exp
  const uint32_t bar0 = smem_u32(wsum + kX2Warps * 8);                   // K0, V0, K1, V1
  auto k_buf = [&](int s) { return base + (uint32_t)s * 2u * kXtBufBytes; };
  auto v_buf = [&](int s) { return base + (uint32_t)s * 2u * kXtBufBytes + kXtBufBytes; };
  auto bar_k = [&](int s) { return bar0 + 16u * s; };
  auto bar_v = [&](int s) { return bar0 + 16u * s + 8u; };

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int beam = lane >> 2, p4 = lane & 3, mi = lane >> 3;
  const int items = g.B * g.heads;
  if (tid == 0) {
    tma_prefetch_desc(&tm);
    for (int i = 0; i < 2 * kStages; ++i) mbar_init(bar0 + 8u * i, 1);
    fence_barrier_init();
  }
  __syncthreads();
  pdl_launch_dependents();

  auto keys_of = [&](int b) { const int n = cross_len ? cross_len[b] : g.Le; return n < 1 ? 1 : (n > g.Le ? g.Le : n); };
  // warp 0: request K and V of `item` into stage s; lanes 0..nb-1 fetch the K boxes, lanes 8..8+nb-1 the V boxes
  auto issue = [&](int item, int kv, int s, int nk_item) {
    const int b = item / g.heads, h = item - b * g.heads;
    const int nb = (nk_item + kXtRows - 1) / kXtRows;
    const uint32_t bar = kv ? bar_v(s) : bar_k(s), buf = kv ? v_buf(s) : k_buf(s);
    if (lane == 0) mbar_arrive_expect_tx(bar, (uint32_t)(nb * kXtBoxBytes));
    __syncwarp();
    const int z = ((layer * g.B + b) * 2 + kv) * g.heads + h;
    if (lane < nb) tma_load_3d(buf + lane * kXtBoxBytes, &tm, 0, lane * kXtRows, z, bar);
  };
  // mask entries of this thread (kMaskPer x threads >= 304): the RAW values are loaded early and only converted when they
  // are stored, so the load latency is not on the critical path
  constexpr int kMaskPer = (kXtLeP + kX2Threads - 1) / kX2Threads;
  float mraw[kMaskPer];
  auto load_mask = [&](int b) {
#pragma unroll
    for (int i = 0; i < kMaskPer; ++i) {
      const int j = tid + i * kX2Threads;
      mraw[i] = (enc_mask && j < g.Le) ? enc_mask[(int64_t)b * g.Le + j] : 1.f;
    }
  };
  auto store_mask = [&](float* dst) {
#pragma unroll
    for (int i = 0; i < kMaskPer; ++i) {
      const int j = tid + i * kX2Threads;
      if (j < kXtLeP) dst[j] = (j < g.Le) ? (1.0f - mraw[i]) * (-1e9f * kLog2e) : -INFINITY;
    }
  };
  uint32_t qa0[4], qa2[4];
  auto load_q = [&](int item) {
    const int b = item / g.heads, h = item - b * g.heads;
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) { qa0[kk] = 0u; qa2[kk] = 0u; }
    if (beam < g.K) {
      const bf16* qp = q + ((int64_t)(b * g.K + beam)) * g.H + h * 64 + p4 * 2;
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        qa0[kk] = *reinterpret_cast<const uint32_t*>(qp + kk * 16);
        qa2[kk] = *reinterpret_cast<const uint32_t*>(qp + kk * 16 + 8);
      }
    }
  };
  const int first = blockIdx.x, stride = gridDim.x;
  if (first >= items) return;
  // key counts of this item and the next two, fetched one item ahead of their use (a global load each)
  int nk0 = keys_of(first / g.heads);
  int nk1 = first + stride < items ? keys_of((first + stride) / g.heads) : 1;
  int nk2 = first + 2 * stride < items ? keys_of((first + 2 * stride) / g.heads) : 1;
  if (warp == 0) {
    issue(first, 0, 0, nk0);                                // cross K/V, cross_len and the mask date from the prefill: safe before the wait
    issue(first, 1, 0, nk0);
    if (kStages > 1 && first + stride < items) { issue(first + stride, 0, 1, nk1); issue(first + stride, 1, 1, nk1); }
  }
  load_mask(first / g.heads);
  store_mask(madd);
  pdl_wait();                                               // the query projection of this step is complete
  stamp(1);
  load_q(first);

  const float sc = kLog2e / 8.0f;                           // scores / sqrt(64), log2 domain
  int it = 0;
  for (int item = first; item < items; item += stride, ++it) {
    const int s = it % kStages, mb = it & 1;               // buffer stage; mask-row buffer
    const uint32_t phase = (uint32_t)(it / kStages) & 1u;
    const int ahead = item + kStages * stride;               // the item that will reuse this stage
    const int nk_ahead = kStages == 1 ? nk1 : nk2;
    const int b = item / g.heads, h = item - b * g.heads;
    const int nk = nk0;
    const int ngroups = (nk + 15) >> 4;
    const int nw = ngroups < kX2Warps ? ngroups : kX2Warps;  // warps that own at least one key group
    const int next = item + stride;
    const int nk3 = item + 3 * stride < items ? keys_of((item + 3 * stride) / g.heads) : 1;   // used two iterations from now
    const float* md = madd + mb * kXtLeP;
    const uint32_t kb_s = k_buf(s), vb_s = v_buf(s);
    uint32_t a_q0[4], a_q2[4];
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) { a_q0[kk] = qa0[kk]; a_q2[kk] = qa2[kk]; }
    if (next < items) load_mask(next / g.heads);
    __syncthreads();                                        // (1) mask row visible; the previous item's shared results have been read
    mbar_wait(bar_k(s), phase);
    stamp(2 + 4 * it);
    // ---- scores of this warp's key groups: s[gi][0..1] keys 16G + p4*2 + {0,1}, s[gi][2..3] the same + 8; row = beam ----
    float sv[kX2Groups][4];
    float mloc = -INFINITY;
#pragma unroll
    for (int gi = 0; gi < kX2Groups; ++gi) {
      const int G = warp + gi * kX2Warps;
      sv[gi][0] = sv[gi][1] = sv[gi][2] = sv[gi][3] = -INFINITY;
      if (G < ngroups) {
        float c0[4] = {0.f, 0.f, 0.f, 0.f}, c1[4] = {0.f, 0.f, 0.f, 0.f};
        const int row = G * 16 + (mi >> 1) * 8 + (lane & 7);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          uint32_t kb[4];
          const int chunk = kk * 2 + (mi & 1);
          ldmatrix_x4(kb, kb_s + row * 128 + ((chunk ^ (row & 7)) << 4));
          mma_bf16_m8(c0, a_q0[kk], a_q2[kk], kb[0], kb[1]);
          mma_bf16_m8(c1, a_q0[kk], a_q2[kk], kb[2], kb[3]);
        }
        const int key = G * 16 + p4 * 2;
        const float2 m0 = *reinterpret_cast<const float2*>(md + key), m1 = *reinterpret_cast<const float2*>(md + key + 8);
        sv[gi][0] = fmaf(c0[0], sc, m0.x); sv[gi][1] = fmaf(c0[1], sc, m0.y);
        sv[gi][2] = fmaf(c1[0], sc, m1.x); sv[gi][3] = fmaf(c1[1], sc, m1.y);
        mloc = fmaxf(fmaxf(mloc, fmaxf(sv[gi][0], sv[gi][1])), fmaxf(sv[gi][2], sv[gi][3]));
      }
    }
    mloc = fmaxf(mloc, __shfl_xor_sync(0xffffffffu, mloc, 1));
    mloc = fmaxf(mloc, __shfl_xor_sync(0xffffffffu, mloc, 2));
    if (p4 == 0) wmax[warp * 8 + beam] = mloc;
    __syncthreads();                                        // (2) per-warp maxima visible
    stamp(3 + 4 * it);
    if (warp == 0 && ahead < items) issue(ahead, 0, s, nk_ahead);   // every warp is past its scores: the K buffer is free
    if (next < items) {
      load_q(next);                                         // in flight during the rest of this item
      store_mask(madd + (mb ^ 1) * kXtLeP);
    }
    float gm = -INFINITY;
#pragma unroll
    for (int w = 0; w < kX2Warps; ++w) gm = fmaxf(gm, w < nw ? wmax[w * 8 + beam] : -INFINITY);   // independent loads
    // ---- probabilities (un-normalised, <= 1) as the A operand of the context product ----
    uint32_t pa0[kX2Groups], pa2[kX2Groups];
    float sloc = 0.f;
#pragma unroll
    for (int gi = 0; gi < kX2Groups; ++gi) {
      const float e0 = ex2_approx(sv[gi][0] - gm), e1 = ex2_approx(sv[gi][1] - gm);
      const float e2 = ex2_approx(sv[gi][2] - gm), e3 = ex2_approx(sv[gi][3] - gm);   // 2^(-inf) = 0: groups not owned, keys past Le
      sloc += (e0 + e1) + (e2 + e3);
      __nv_bfloat162 lo = __floats2bfloat162_rn(e0, e1), hi = __floats2bfloat162_rn(e2, e3);
      pa0[gi] = *reinterpret_cast<uint32_t*>(&lo);
      pa2[gi] = *reinterpret_cast<uint32_t*>(&hi);
    }
    sloc += __shfl_xor_sync(0xffffffffu, sloc, 1);
    sloc += __shfl_xor_sync(0xffffffffu, sloc, 2);
    if (p4 == 0) wsum[warp * 8 + beam] = sloc;
    mbar_wait(bar_v(s), phase);
    stamp(4 + 4 * it);
    // ---- context: O[beam][d] += P[beam][keys of the group] V[keys][d] ----
    float o[8][4];
#pragma unroll
    for (int n = 0; n < 8; ++n) { o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f; }
#pragma unroll
    for (int gi = 0; gi < kX2Groups; ++gi) {
      const int G = warp + gi * kX2Warps;
      if (G < ngroups) {
        const int row = G * 16 + (mi & 1) * 8 + (lane & 7);
#pragma unroll
        for (int dt = 0; dt < 8; dt += 2) {
          uint32_t vb[4];
          const int chunk = dt + (mi >> 1);
          ldmatrix_x4_trans(vb, vb_s + row * 128 + ((chunk ^ (row & 7)) << 4));
          mma_bf16_m8(o[dt], pa0[gi], pa2[gi], vb[0], vb[1]);
          mma_bf16_m8(o[dt + 1], pa0[gi], pa2[gi], vb[2], vb[3]);
        }
      }
    }
    if (warp < nw) {
      float* pp = part + (warp * 8 + beam) * 64 + p4 * 2;
#pragma unroll
      for (int dt = 0; dt < 8; ++dt) *reinterpret_cast<float2*>(pp + dt * 8) = make_float2(o[dt][0], o[dt][1]);
    }
    __syncthreads();                                        // (3) partial contexts / sums complete; stage s is free
    if (warp == 0 && ahead < items) issue(ahead, 1, s, nk_ahead);
    for (int i = tid; i < g.K * 64; i += kX2Threads) {
      const int k = i >> 6, d = i & 63;
      float v = 0.f, t = 0.f;
#pragma unroll
      for (int w = 0; w < kX2Warps; ++w) {
        if (w < nw) { v += part[(w * 8 + k) * 64 + d]; t += wsum[w * 8 + k]; }
      }
      out[((int64_t)(b * g.K + k)) * g.H + h * 64 + d] = __float2bfloat16_rn(v / t);
    }
    stamp(5 + 4 * it);
    nk0 = nk1; nk1 = nk2; nk2 = nk3;
  }
}

// ---- third version: one WARP per (image, head) item, no block-wide synchronisation ------------------------------------
// The 8-warp kernel above spends most of an item in its three block barriers, the cross-warp reduction of partial contexts
// and the K -> scores -> V -> context chain of ONE item per CTA (profiles/r2_cross_phases.txt: ~1.5 us of math + ~1.5 us of
// waiting per item, 2.6 items per CTA in sequence).  Here every warp owns a whole item: its K boxes and then its V boxes
// (64 keys x 64 dims, 8 KB) stream through a private FIFO of kBufs buffers with one mbarrier each; the warp keeps ALL scores
// of the item in registers (<= 19 key groups x 4 values per lane), takes the exact maximum, exponentiates in registers and
// accumulates the context product in its own MMA accumulators - no shared-memory score tiles, no partial sums, no
// __syncthreads.  Two 3-warp CTAs per SM (888 warp slots for the 768 items of a B = 64, 12-head step: one wave) keep
// 6 x 24 KB of boxes in flight per SM; everything that does not depend on the query projection (barrier set-up, key count,
// mask row, the first kBufs boxes) is done before the programmatic dependency is awaited.
// Arithmetic: identical formulation to the kernel above (log2 domain, un-normalised bf16 probabilities <= 1, fp32
// accumulation, one division at the end); the sums are taken in key order by one warp instead of per-warp partials.
template <int kWarps, int kBufs>
struct XwCfg {
  static constexpr int kThreads = kWarps * 32;
  static constexpr int kMaskFloats = kXtMaxBoxes * kXtRows;                       // 320: every fetched key has an entry
  static constexpr int kWarpBytes = kBufs * kXtBoxBytes;
  static constexpr int kSmem = kWarps * kWarpBytes + kWarps * kMaskFloats * 4 + kWarps * kBufs * 8 + 1024;
};

template <int kWarps, int kBufs>
__global__ void __launch_bounds__(kWarps * 32, 2)
dec_cross_warp_kernel(const __grid_constant__ CUtensorMap tm, DecodeGeom g, int layer, const bf16* __restrict__ q,
                      const float* __restrict__ enc_mask, const int* __restrict__ cross_len, bf16* __restrict__ out) {
  using Cfg = XwCfg<kWarps, kBufs>;
  extern __shared__ uint8_t xw_raw[];
  const uint32_t raw = smem_u32(xw_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* gen = xw_raw + (base - raw);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int beam = lane >> 2, p4 = lane & 3, mi = lane >> 3;
  const uint32_t buf0 = base + (uint32_t)warp * Cfg::kWarpBytes;
  float* madd = reinterpret_cast<float*>(gen + kWarps * Cfg::kWarpBytes) + warp * Cfg::kMaskFloats;
  const uint32_t bar0 = smem_u32(gen + kWarps * Cfg::kWarpBytes + kWarps * Cfg::kMaskFloats * 4) + (uint32_t)warp * kBufs * 8u;
  const int items = g.B * g.heads;
  if (lane == 0) {
    if (warp == 0) tma_prefetch_desc(&tm);
    for (int i = 0; i < kBufs; ++i) mbar_init(bar0 + 8u * i, 1);
    fence_barrier_init();
  }
  __syncwarp();
  pdl_launch_dependents();
  const int nslots = gridDim.x * kWarps;
  int item = warp * gridDim.x + blockIdx.x;                 // warp-major: the CTAs of one SM get equally many items
  if (item >= items) return;

  uint32_t seq = 0;                                          // FIFO element counter of this warp (buffer = seq % kBufs)
  bool first = true;
  const float sc = kLog2e / 8.0f;                            // scores / sqrt(64), log2 domain
  for (; item < items; item += nslots) {
    const int b = item / g.heads, h = item - b * g.heads;
    int nk = cross_len ? cross_len[b] : g.Le;
    nk = nk < 1 ? 1 : (nk > g.Le ? g.Le : nk);
    const int nb = (nk + kXtRows - 1) / kXtRows;            // boxes of K (and of V)
    const int ngroups = (nk + 15) >> 4;
    const int nel = 2 * nb;                                  // FIFO elements of this item: K boxes, then V boxes
    const int zk = ((layer * g.B + b) * 2 + 0) * g.heads + h, zv = zk + g.heads;
    auto issue = [&](int el) {                               // lane 0
      const uint32_t sl = (seq + (uint32_t)el) % kBufs;
      const int kv = el >= nb, box = kv ? el - nb : el;
      mbar_arrive_expect_tx(bar0 + 8u * sl, (uint32_t)kXtBoxBytes);
      tma_load_3d(buf0 + sl * kXtBoxBytes, &tm, 0, box * kXtRows, kv ? zv : zk, bar0 + 8u * sl);
    };
    // cross K / V, cross_len and the mask date from the prefill: safe before the programmatic dependency resolves
    if (lane == 0) {
      const int pre = nel < kBufs ? nel : kBufs;
      for (int el = 0; el < pre; ++el) issue(el);
    }
    for (int j = lane; j < Cfg::kMaskFloats; j += 32) {
      const float m = (enc_mask && j < g.Le) ? enc_mask[(int64_t)b * g.Le + j] : 1.f;
      madd[j] = (j < g.Le) ? (1.0f - m) * (-1e9f * kLog2e) : -INFINITY;
    }
    if (first) { pdl_wait(); first = false; }                // the query projection of this step is complete
    uint32_t qa0[4], qa2[4];
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) { qa0[kk] = 0u; qa2[kk] = 0u; }
    if (beam < g.K) {
      const bf16* qp = q + ((int64_t)(b * g.K + beam)) * g.H + h * 64 + p4 * 2;
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        qa0[kk] = *reinterpret_cast<const uint32_t*>(qp + kk * 16);
        qa2[kk] = *reinterpret_cast<const uint32_t*>(qp + kk * 16 + 8);
      }
    }
    __syncwarp();                                            // mask row visible to the whole warp

    // ---- phase A: scores of every key group, kept in registers: sv[G][0..1] keys 16G + p4*2 + {0,1}, sv[G][2..3] the same + 8 ----
    float sv[kXtMaxBoxes * 4][4];
    float mloc = -INFINITY;
#pragma unroll
    for (int j = 0; j < kXtMaxBoxes; ++j) {
      if (j < nb) {
        const uint32_t el = seq + (uint32_t)j;
        mbar_wait(bar0 + 8u * (el % kBufs), (el / kBufs) & 1u);
        const uint32_t kb_s = buf0 + (el % kBufs) * kXtBoxBytes;
#pragma unroll
        for (int gl = 0; gl < 4; ++gl) {
          const int G = j * 4 + gl;
          sv[G][0] = sv[G][1] = sv[G][2] = sv[G][3] = -INFINITY;
          if (G < ngroups) {
            float c0[4] = {0.f, 0.f, 0.f, 0.f}, c1[4] = {0.f, 0.f, 0.f, 0.f};
            const int row = gl * 16 + (mi >> 1) * 8 + (lane & 7);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
              uint32_t kb[4];
              const int chunk = kk * 2 + (mi & 1);
              ldmatrix_x4(kb, kb_s + row * 128 + ((chunk ^ (row & 7)) << 4));
              mma_bf16_m8(c0, qa0[kk], qa2[kk], kb[0], kb[1]);
              mma_bf16_m8(c1, qa0[kk], qa2[kk], kb[2], kb[3]);
            }
            const int key = G * 16 + p4 * 2;
            const float2 m0 = *reinterpret_cast<const float2*>(madd + key), m1 = *reinterpret_cast<const float2*>(madd + key + 8);
            sv[G][0] = fmaf(c0[0], sc, m0.x); sv[G][1] = fmaf(c0[1], sc, m0.y);
            sv[G][2] = fmaf(c1[0], sc, m1.x); sv[G][3] = fmaf(c1[1], sc, m1.y);
            mloc = fmaxf(fmaxf(mloc, fmaxf(sv[G][0], sv[G][1])), fmaxf(sv[G][2], sv[G][3]));
          }
        }
        __syncwarp();                                        // every lane has read this box: the buffer may be refilled
        if (lane == 0 && j + kBufs < nel) issue(j + kBufs);
      } else {
#pragma unroll
        for (int gl = 0; gl < 4; ++gl) { const int G = j * 4 + gl; sv[G][0] = sv[G][1] = sv[G][2] = sv[G][3] = -INFINITY; }
      }
    }
    mloc = fmaxf(mloc, __shfl_xor_sync(0xffffffffu, mloc, 1));
    mloc = fmaxf(mloc, __shfl_xor_sync(0xffffffffu, mloc, 2));
    // ---- probabilities (un-normalised, <= 1) as the A operand of the context product ----
    uint32_t pa0[kXtMaxBoxes * 4], pa2[kXtMaxBoxes * 4];
    float sloc = 0.f;
#pragma unroll
    for (int G = 0; G < kXtMaxBoxes * 4; ++G) {
      const float e0 = ex2_approx(sv[G][0] - mloc), e1 = ex2_approx(sv[G][1] - mloc);
      const float e2 = ex2_approx(sv[G][2] - mloc), e3 = ex2_approx(sv[G][3] - mloc);   // 2^(-inf) = 0: groups past the last key
      sloc += (e0 + e1) + (e2 + e3);
      __nv_bfloat162 lo = __floats2bfloat162_rn(e0, e1), hi = __floats2bfloat162_rn(e2, e3);
      pa0[G] = *reinterpret_cast<uint32_t*>(&lo);
      pa2[G] = *reinterpret_cast<uint32_t*>(&hi);
    }
    sloc += __shfl_xor_sync(0xffffffffu, sloc, 1);
    sloc += __shfl_xor_sync(0xffffffffu, sloc, 2);
    // ---- phase B: context O[beam][d] += P[beam][keys] V[keys][d] ----
    float o[8][4];
#pragma unroll
    for (int n = 0; n < 8; ++n) { o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f; }
#pragma unroll
    for (int j = 0; j < kXtMaxBoxes; ++j) {
      if (j < nb) {
        const uint32_t el = seq + (uint32_t)(nb + j);
        mbar_wait(bar0 + 8u * (el % kBufs), (el / kBufs) & 1u);
        const uint32_t vb_s = buf0 + (el % kBufs) * kXtBoxBytes;
#pragma unroll
        for (int gl = 0; gl < 4; ++gl) {
          const int G = j * 4 + gl;
          if (G < ngroups) {
            const int row = gl * 16 + (mi & 1) * 8 + (lane & 7);
#pragma unroll
            for (int dt = 0; dt < 8; dt += 2) {
              uint32_t vb[4];
              const int chunk = dt + (mi >> 1);
              ldmatrix_x4_trans(vb, vb_s + row * 128 + ((chunk ^ (row & 7)) << 4));
              mma_bf16_m8(o[dt], pa0[G], pa2[G], vb[0], vb[1]);
              mma_bf16_m8(o[dt + 1], pa0[G], pa2[G], vb[2], vb[3]);
            }
          }
        }
        __syncwarp();
        if (lane == 0 && nb + j + kBufs < nel) issue(nb + j + kBufs);
      }
    }
    if (beam < g.K) {
      bf16* op = out + ((int64_t)(b * g.K + beam)) * g.H + h * 64 + p4 * 2;
#pragma unroll
      for (int dt = 0; dt < 8; ++dt) *reinterpret_cast<__nv_bfloat162*>(op + dt * 8) = __floats2bfloat162_rn(o[dt][0] / sloc, o[dt][1] / sloc);
    }
    seq += (uint32_t)nel;
    __syncwarp();                                            // the mask row is rewritten by the next item
  }
}

// cross_len[b] = 1 + index of the last key whose mask is non-zero (Le when the whole row is masked: the reference then
// spreads uniform weight over every key, which needs them all).
__global__ void cross_len_kernel(int B, int Le, const float* __restrict__ mask, int* __restrict__ out) {
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= B) return;
  int last = -1;
  for (int j = lane; j < Le; j += 32)
    if (mask[(int64_t)b * Le + j] != 0.f) last = j;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) last = max(last, __shfl_xor_sync(0xffffffffu, last, o));
  if (lane == 0) out[b] = last < 0 ? Le : last + 1;
}

}  // namespace

unsigned long long* g_cross_stamps = nullptr;

// Prints the stamps of the most recent dec_cross_tma2 launch (after a device synchronisation); measurement aid.
void dec_cross_print_times() {
  if (g_cross_stamps == nullptr) return;
  cudaDeviceSynchronize();
  static unsigned long long h[1024 * 16];
  cudaMemcpy(h, g_cross_stamps, sizeof h, cudaMemcpyDeviceToHost);
  unsigned long long t0 = ~0ull; int ctas = 0;
  for (int i = 0; i < 1024; ++i) if (h[i * 16]) { if (h[i * 16] < t0) t0 = h[i * 16]; ++ctas; }
  const char* names[14] = {"start", "dep", "i0 K", "i0 scores", "i0 V", "i0 done", "i1 K", "i1 scores", "i1 V", "i1 done", "i2 K", "i2 scores", "i2 V", "i2 done"};
  fprintf(stderr, "[cross times, %d CTAs] ns since the first CTA started, mean / max over the CTAs that reached the stamp (count):\n", ctas);
  for (int j = 0; j < 14; ++j) {
    double sum = 0, mx = 0; int n = 0;
    for (int i = 0; i < 1024; ++i) if (h[i * 16] && h[i * 16 + j] >= h[i * 16]) { const double v = (double)(h[i * 16 + j] - t0); sum += v; if (v > mx) mx = v; ++n; }
    if (n) fprintf(stderr, "  %-10s %8.0f / %8.0f  (%d)\n", names[j], sum / n, mx, n);
  }
}

bool dec_cross_tma_fits(int dtype, const DecodeGeom& g) {
  return dtype == kBF16 && g.D == 64 && g.K <= 8 && g.Le <= kXtLeP && g.H == g.heads * 64;
}

bool dec_cross_tma_supported(int dtype, const DecodeGeom& g) {
  static const bool off = getenv("GSTVD_CROSS_NO_TMA") != nullptr;
  return !off && dec_cross_tma_fits(dtype, g);
}

int launch_dec_cross_tma(const DecodeGeom& g, int layer, const void* q, const void* cross_cache, const float* enc_mask,
                         const int* cross_len, void* out, int num_sms, cudaStream_t stream, int force) {
  if (force != kDecDefault && force != kCrossWarpTma && force != kCrossCtaTma) throw std::runtime_error("dec_cross_tma: not a TMA kernel");
  if (!dec_cross_tma_fits(kBF16, g)) throw std::runtime_error("dec_cross_tma: needs head_dim 64, at most 8 beams and 304 keys");
  // GSTVD_CROSS_TMA=2: the CTA-per-item kernel; anything else / unset: one warp per item.  Read at every launch (a captured graph keeps
  // what it was captured with), so that a test can compare the two in one process.  A forced kernel ignores the variable.
  const char* venv = getenv("GSTVD_CROSS_TMA");
  const int variant = force == kCrossCtaTma ? 2 : force == kCrossWarpTma ? 4 : (venv && atoi(venv) == 2) ? 2 : 4;
  using Cfg2 = X2Cfg<8, 1, 3>;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(dec_cross_tma2_kernel<8, 1, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg2::kSmem);
    if (e != cudaSuccess) throw std::runtime_error(std::string("dec_cross_tma: ") + cudaGetErrorString(e));
    configured = true;
  }
  const CUtensorMap* tm = reinterpret_cast<const CUtensorMap*>(
      tma_map_rows3(cross_cache, 64, g.Le, (int64_t)g.layers * g.B * 2 * g.heads, kXtRows));
  const int items = g.B * g.heads;
  if (variant == 4) {                                     // one warp per item (default)
    // three boxes in flight per warp measured best (profiles/r2_cross_warp_ab.txt): 2 starve the warp, 4 leave no room on the SM for the
    // look-ahead CTA of the following GEMM and take HBM bandwidth from its weight prefetch
    using CfgW = XwCfg<3, 3>;
    static bool configured_w = false;
    if (!configured_w) {
      cudaError_t e = cudaFuncSetAttribute(dec_cross_warp_kernel<3, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, CfgW::kSmem);
      if (e != cudaSuccess) throw std::runtime_error(std::string("dec_cross_warp: ") + cudaGetErrorString(e));
      configured_w = true;
    }
    const int ctas = (items + 2) / 3;
    const int grid_w = ctas < 2 * num_sms ? ctas : 2 * num_sms;
    launch_k(dec_cross_warp_kernel<3, 3>, dim3(grid_w), dim3(CfgW::kThreads), (size_t)CfgW::kSmem, stream, *tm, g, layer, (const bf16*)q, enc_mask,
             cross_len, (bf16*)out);
    return 1;
  }
  const int slots = 2 * num_sms;
  const int grid = items < slots ? items : slots;
  static unsigned long long* d_stamps = nullptr;          // measurement aid: GSTVD_CROSS_TIMES=1, read back by dec_cross_print_times()
  static const bool want_times = getenv("GSTVD_CROSS_TIMES") != nullptr;
  if (want_times && d_stamps == nullptr) { cudaMalloc(&d_stamps, 1024 * 16 * 8); cudaMemset(d_stamps, 0, 1024 * 16 * 8); g_cross_stamps = d_stamps; }
  launch_k(dec_cross_tma2_kernel<8, 1, 3>, dim3(grid), dim3(Cfg2::kThreads), (size_t)Cfg2::kSmem, stream, *tm, g, layer, (const bf16*)q,
           enc_mask, cross_len, (bf16*)out, d_stamps);
  return 1;
}

int launch_cross_len(int B, int Le, const float* mask, int* out, cudaStream_t stream) {
  cross_len_kernel<<<(B + 3) / 4, 128, 0, stream>>>(B, Le, mask, out);
  return 1;
}

}  // namespace gstvd
