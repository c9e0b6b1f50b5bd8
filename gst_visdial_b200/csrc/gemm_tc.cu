// tcgen05 / TMEM / TMA GEMM for sm_100a:  C[M,N] = act(A[M,K] * W[N,K]^T + bias), bf16 operands, fp32 accumulate.
//
// Replaces every nn.Linear on the hot path when the compute dtype is bf16: the q/k/v, output and FFN projections of
// the text / image / connection layers (models/vilbert_dialog.py:366-368,412,437,454,493-495,539,564,581,624-633,
// 718,725,753-757), the image embedding (:1415), VLFusion (models/visual_dialog_model.py:127-128), the decoder
// layers and the LM head (models/visual_dialog_decoder.py:300-311,329-339).
//
// Design (persistent over output tiles, warp specialised; one CTA per SM, two in the shared-SM decode configuration):
//   warp 0      : TMA producer  - cp.async.bulk.tensor loads of the A (128 rows) and W (BN rows) k-blocks into a shared-
//                 memory ring (128-byte swizzle), completion on mbarriers.  Wide tiles move one 64-element k-chunk per
//                 2-D box; the narrow decode tiles move several chunks per 3-D box (one thread issues a TMA operation
//                 every ~0.13 us).  The weights of the first ring are requested before griddepcontrol.wait (PDL).
//   warp 1      : MMA issuer    - one lane issues tcgen05.mma.cta_group::1.kind::f16 (M=128, N=BN, K=16) x4 per k-chunk
//                 into one of two TMEM accumulator stages; tcgen05.commit releases ring slots / signals the epilogue
//   warps 2..   : epilogue      - 16 warps (4 per TMEM lane quadrant; 4 in the shared-SM configuration): tcgen05.ld
//                 (32 lanes x 32 columns), + bias, GELU, convert, then either a swizzled shared-memory tile + TMA store
//                 (throughput problems), direct 16-byte row stores (skinny decode problems) or the generic
//                 transpose-through-shared-memory path (outputs a tensor map cannot describe).
//                 Two accumulator stages let the epilogue of tile i overlap the main loop of tile i+1.
// Both operands are K-major ("TN"), which is the layout of activations [rows, features] and nn.Linear weights
// [out, in], so no transposes are ever materialised.  TMA zero-fills out-of-range rows / k, so M, N, K need not be
// multiples of the tile (K % 8 == 0 for the 16-byte stride rule).
// Sibling built on the same helpers (gemm_tc.cuh): gemm_tc2.cu (CTA-pair tiles, cta_group::2, for the large-M problems).  This file
// also owns the tensor-map cache they share.
#include <cuda.h>

#include <algorithm>
#include <cstdlib>
#include <mutex>
#include <stdexcept>
#include <string>
#include <unordered_map>

#include "gemm_tc.cuh"

namespace gstvd {

using namespace tc;

namespace {

template <int BN, int EW> struct TileCfg {
  static constexpr bool kSkinny = EW == kEpiWarpsSkinny;
  static constexpr int kThreads = (2 + EW) * 32;
  // Rows per tile = UMMA M.  The skinny (decode, M = 320) configuration uses M = 64: five exact row tiles instead of three
  // 128-row tiles with 17 % padding, 40 % fewer bytes through the L2->SM port per CTA ((64+BN) instead of (128+BN) rows per
  // k-step) on more SMs, and a CTA small enough for two per SM.  The M = 64 accumulator occupies lanes 0-15 of every
  // 32-lane TMEM quadrant: row r lives in lane (r / 16) * 32 + r % 16 (tools/probes/umma_m64_layout.cu).
  static constexpr int kBM = kSkinny ? 64 : BM;
  // k-chunks (64 elements each) per pipeline stage.  The narrow tiles serve the M <= 512 decode GEMMs, whose main loop is
  // bound by the RATE of TMA operations issued by one thread (~0.13 us each), not by bytes: one 3-D box
  // {64, rows, chunks} moves several k-blocks per operation.
  static constexpr int kCK = kSkinny ? (BN <= 32 ? 4 : 2) : (BN <= 64 ? 4 : 1);
  static constexpr int kStages = kSkinny ? (BN <= 32 ? 2 : (BN <= 64 ? 3 : 2)) : (BN == 256 ? 4 : (BN == 128 ? 6 : 2));
  static constexpr int kAChunk = kBM * BK * 2;                 // one kBM-row x 64-element SW128 tile
  static constexpr int kBChunk = BN * BK * 2;
  static constexpr int kABytes = kAChunk * kCK;
  static constexpr int kBBytes = kBChunk * kCK;
  static constexpr int kTmemCols = 2 * BN < 32 ? 32 : 2 * BN;   // power of two for BN in {16,32,64,128,256}
  static constexpr int kBarBytes = 256;
  static constexpr int kStageWords = 32 * 33;                   // per epilogue warp: 32 rows x 32 words, padded rows
  // wide: 33 KB = 4 x 8 KB (bf16) / 2 x 16 KB (fp32) TMA-store tiles, or 8 generic tiles; skinny: none (direct row stores only)
  static constexpr int kStagingBytes = kSkinny ? 0 : 8 * kStageWords * 4;
  // deferred-LayerNorm epilogue: per warp, four 32-float column vectors - inside the (then unused) staging tiles of the wide
  // configurations, appended to the allocation of the skinny one (LN instantiations only)
  static constexpr int kLnVecBytes = EW * 4 * 32 * 4;
  static constexpr int kLnVecExtra = kSkinny ? kLnVecBytes : 0;
  static_assert(kSkinny || kLnVecBytes <= 8 * 32 * 33 * 4, "column vectors must fit the staging area");
  static constexpr int kSmemBytes = kStages * (kABytes + kBBytes) + kBarBytes + kStagingBytes + 1024;   // +1024: alignment slack; LN kernels add kLnVecBytes
  static_assert(!kSkinny || 2 * (kSmemBytes + kLnVecExtra + 1024) <= 233472, "skinny configuration must fit two CTAs per SM");
};

// Epilogue of one W-column block of this warp's 32 accumulator rows: TMEM -> registers (thread = row) -> + bias,
// activation, convert -> transpose through a warp-private padded shared-memory tile -> global stores in which the 32
// lanes of one instruction cover CONTIGUOUS bytes of one (or two) output rows (128 B segments), instead of 32 different
// rows.  The uncoalesced variant (one 16-byte store per row per instruction) was L2-transaction bound: 3x slower.
template <typename OutT, int W>
__device__ __forceinline__ void epilogue_block(const GemmArgs& p, uint32_t taddr, uint32_t* stage, int row0, int col0, int lane) {
  constexpr bool kBf16 = sizeof(OutT) == 2;
  constexpr int kWords = kBf16 ? W / 2 : W;       // 32-bit words per output row in this block
  static_assert(kWords <= 32, "block too wide for the staging tile");
  const bool full = (col0 + W <= p.N);
  const bool bias_vec = p.bias != nullptr && full && ((reinterpret_cast<uintptr_t>(p.bias + col0) & 15) == 0);
#pragma unroll
  for (int part = 0; part < W / 32; ++part) {
    uint32_t acc[32];
    tmem_ld32(taddr + part * 32, acc);
#pragma unroll
    for (int g8 = 0; g8 < 4; ++g8) {
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = __uint_as_float(acc[g8 * 8 + j]);
      const int cb = col0 + part * 32 + g8 * 8;
      if (p.bias) {
        if (bias_vec) {
          const float4 b0 = __ldg(reinterpret_cast<const float4*>(p.bias + cb));
          const float4 b1 = __ldg(reinterpret_cast<const float4*>(p.bias + cb + 4));
          v[0] += b0.x; v[1] += b0.y; v[2] += b0.z; v[3] += b0.w; v[4] += b1.x; v[5] += b1.y; v[6] += b1.z; v[7] += b1.w;
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j)
            if (cb + j < p.N) v[j] += __ldg(p.bias + cb + j);
        }
      }
      if (p.act == 1) {
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = gelu_fast(v[j]);
      }
      if constexpr (kBf16) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
          stage[lane * 33 + part * 16 + g8 * 4 + j] = *reinterpret_cast<uint32_t*>(&h);
        }
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) stage[lane * 33 + part * 32 + g8 * 8 + j] = __float_as_uint(v[j]);
      }
    }
  }
  __syncwarp();
  constexpr int kRowsPerInstr = 32 / kWords;
  constexpr int kColsPerWord = kBf16 ? 2 : 1;
  const int w = lane % kWords, rsub = lane / kWords;
  const int col = col0 + w * kColsPerWord;
  const bool ld_even = kBf16 ? ((p.hm_D > 0) || ((p.ldc & 1) == 0)) : true;
#pragma unroll 4
  for (int i0 = 0; i0 < 32; i0 += kRowsPerInstr) {
    const int r = i0 + rsub;
    const int row = row0 + r;
    const uint32_t word = stage[r * 33 + w];
    if (row < p.M && col < p.N && p.dbg != 1) {
      OutT* dst = reinterpret_cast<OutT*>(p.C) + out_index(p, row, col);
      if constexpr (kBf16) {
        if (col + 1 < p.N && ld_even) {
          *reinterpret_cast<uint32_t*>(dst) = word;
        } else {
          const __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(&word);
          dst[0] = h.x;
          if (col + 1 < p.N) dst[1] = h.y;
        }
      } else {
        *reinterpret_cast<uint32_t*>(dst) = word;
      }
    }
  }
  __syncwarp();
}

// Epilogue of one 32-column block straight from registers: thread = accumulator row, 64 (bf16) or 128 (fp32) contiguous
// bytes per row as 16-byte stores.  Uncoalesced across the warp, which costs L2 transactions on big outputs (that is why
// the throughput configurations stage through shared memory + TMA), but for the skinny decode GEMMs the whole tile is 8 KB
// and what matters is latency: no staging tile, no proxy fence, no group barrier, no wait for the TMA engine at the end.
template <typename OutT>
__device__ __forceinline__ void epilogue_direct_block(const GemmArgs& p, uint32_t taddr, int row, int col0, const float* bpre) {
  constexpr int kWords = 32 * (int)sizeof(OutT) / 4;
  uint32_t acc[32];
  tmem_ld32(taddr, acc);
  uint32_t packed[kWords];
  const bool full = (col0 + 32 <= p.N);
  const bool bias_vec = p.bias != nullptr && full && ((reinterpret_cast<uintptr_t>(p.bias + col0) & 15) == 0);
#pragma unroll
  for (int g8 = 0; g8 < 4; ++g8) {
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = __uint_as_float(acc[g8 * 8 + j]);
    const int cb = col0 + g8 * 8;
    if (bpre != nullptr) {                               // bias values fetched while the main loop was running
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] += bpre[g8 * 8 + j];
    } else if (p.bias) {
      if (bias_vec) {
        const float4 b0 = __ldg(reinterpret_cast<const float4*>(p.bias + cb));
        const float4 b1 = __ldg(reinterpret_cast<const float4*>(p.bias + cb + 4));
        v[0] += b0.x; v[1] += b0.y; v[2] += b0.z; v[3] += b0.w; v[4] += b1.x; v[5] += b1.y; v[6] += b1.z; v[7] += b1.w;
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (cb + j < p.N) v[j] += __ldg(p.bias + cb + j);
      }
    }
    if (p.act == 1) {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = gelu_fast(v[j]);
    }
    if constexpr (sizeof(OutT) == 2) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
        packed[g8 * 4 + j] = *reinterpret_cast<uint32_t*>(&h);
      }
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) packed[g8 * 8 + j] = __float_as_uint(v[j]);
    }
  }
  if (row >= p.M || p.dbg == 1) return;
  OutT* dst = reinterpret_cast<OutT*>(p.C) + (int64_t)row * p.ldc + col0;
  if (full) {                                            // launch_cfg guarantees 16-byte aligned rows in this mode
#pragma unroll
    for (int c = 0; c < kWords / 4; ++c)
      *reinterpret_cast<uint4*>(reinterpret_cast<uint32_t*>(dst) + 4 * c) = make_uint4(packed[4 * c], packed[4 * c + 1], packed[4 * c + 2], packed[4 * c + 3]);
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      if (col0 + j < p.N) {
        if constexpr (sizeof(OutT) == 2) {
          const __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(&packed[j >> 1]);
          dst[j] = (j & 1) ? h.y : h.x;
        } else {
          dst[j] = __uint_as_float(packed[j]);
        }
      }
    }
  }
}

// ---- deferred LayerNorm (GemmArgs::fold_stats / res / stats_out; decode step) ------------------------------------------------
// Row statistics from the per-32-column partials (mean_i, M2_i) a producing GEMM stored, layout [part][row] (ld rows per part) so
// that the lanes of a warp - consecutive rows - read consecutive addresses.  Equal counts: mean = avg(mean_i),
// M2 = sum M2_i + 32 sum (mean_i - mean)^2 (Chan et al.); the second sum is taken in one pass over d_i = mean_i - mean_0
// (sum d^2 - (sum d)^2 / P: the shift keeps the subtraction benign), so no partial has to be kept and every load of the fully
// unrolled loop is independent - one memory round trip.  Fixed evaluation order -> deterministic.
// Returns (mean, 1 / sqrt(var + eps)) with the biased variance of models/vilbert_dialog.py:292-296 / nn.LayerNorm(eps=1e-12).
__device__ __forceinline__ float2 ln_merge_stats(const float2* __restrict__ st, int64_t ld, int parts) {
  float2 v[kLnStatStride];
#pragma unroll
  for (int i = 0; i < kLnStatStride; ++i) v[i] = i < parts ? st[i * ld] : make_float2(0.f, 0.f);
  const float m0 = v[0].x;
  float sd = 0.f, sd2 = 0.f, m2 = 0.f;
#pragma unroll
  for (int i = 0; i < kLnStatStride; ++i) {
    if (i < parts) {
      const float d = v[i].x - m0;
      sd += d; sd2 = fmaf(d, d, sd2); m2 += v[i].y;
    }
  }
  const float inv_p = 1.0f / (float)parts;
  const float mean = fmaf(sd, inv_p, m0);
  const float dev = fmaxf(fmaf(-sd * inv_p, sd, sd2), 0.f);
  const float var = fmaf(32.f, dev, m2) * inv_p * (1.0f / 32.0f);
  return make_float2(mean, 1.0f / sqrtf(var + kLnEpsDeferred));
}

// Direct-store epilogue of one 32-column block with the deferred-LayerNorm extras (thread = accumulator row, bf16 output):
//   v = acc;  fold: v = rstd_a (v - mean_a c_n);  v += bias_n;  residual: v += res (raw: (res - mean_r) rstd_r gamma_n + beta_n);
//   activation;  round to bf16;  stats_out: (mean, M2) of the 32 ROUNDED values (what the consumers will read back).
// sv = this warp's shared-memory copy of the block's column vectors: [0] bias / d, [1] c, [2] gamma, [3] beta (32 floats each),
// fetched before the accumulator is ready so that nothing after the TMEM load waits for global memory.
__device__ __forceinline__ void epilogue_direct_block_ln(const GemmArgs& p, uint32_t taddr, int row, int col0, float2 fstat, float2 rstat,
                                                         const uint4* rpre, const float* __restrict__ sv) {
  uint32_t acc[32];
  tmem_ld32(taddr, acc);
  const bool valid = row < p.M && p.dbg != 1;
  uint4 rres[4];
  if (p.res != nullptr) {
    if (rpre != nullptr) {
#pragma unroll
      for (int c = 0; c < 4; ++c) rres[c] = rpre[c];
    } else if (valid) {
      const uint4* rp = reinterpret_cast<const uint4*>(reinterpret_cast<const bf16*>(p.res) + (int64_t)row * p.ldr + col0);
#pragma unroll
      for (int c = 0; c < 4; ++c) rres[c] = rp[c];
    } else {
#pragma unroll
      for (int c = 0; c < 4; ++c) rres[c] = make_uint4(0, 0, 0, 0);
    }
  }
  // statistics of the 32 rounded values in one pass, shifted by the first one: d_j = v_j - v_0, mean = v_0 + sum d / 32,
  // M2 = sum d^2 - (sum d)^2 / 32 (the shift keeps the subtraction benign whatever the common offset of the block)
  float shift = 0.f, s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int g8 = 0; g8 < 4; ++g8) {
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = __uint_as_float(acc[g8 * 8 + j]);
    const int cb = col0 + g8 * 8;
    (void)cb;
    if (p.fold_stats != nullptr) {
      const float4 c0 = *reinterpret_cast<const float4*>(sv + 32 + g8 * 8), c1 = *reinterpret_cast<const float4*>(sv + 32 + g8 * 8 + 4);
      const float cc[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = fstat.y * fmaf(-fstat.x, cc[j], v[j]);
    }
    if (p.bias != nullptr) {
      const float4 b0 = *reinterpret_cast<const float4*>(sv + g8 * 8), b1 = *reinterpret_cast<const float4*>(sv + g8 * 8 + 4);
      v[0] += b0.x; v[1] += b0.y; v[2] += b0.z; v[3] += b0.w; v[4] += b1.x; v[5] += b1.y; v[6] += b1.z; v[7] += b1.w;
    }
    if (p.res != nullptr) {
      float r[8];
      Vec8<bf16>::load(reinterpret_cast<const bf16*>(&rres[g8]), r);
      if (p.res_stats != nullptr) {
        const float4 g0 = *reinterpret_cast<const float4*>(sv + 64 + g8 * 8), g1 = *reinterpret_cast<const float4*>(sv + 64 + g8 * 8 + 4);
        const float4 e0 = *reinterpret_cast<const float4*>(sv + 96 + g8 * 8), e1 = *reinterpret_cast<const float4*>(sv + 96 + g8 * 8 + 4);
        const float gg[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w}, ee[8] = {e0.x, e0.y, e0.z, e0.w, e1.x, e1.y, e1.z, e1.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] = fmaf((r[j] - rstat.x) * rstat.y, gg[j], ee[j]);
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] += r[j];
    }
    if (p.act == 1) {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = gelu_fast(v[j]);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
      acc[g8 * 4 + j] = *reinterpret_cast<const uint32_t*>(&h);
      const float2 back = __bfloat1622float2(h);
      if (g8 == 0 && j == 0) shift = back.x;
      const float d0 = back.x - shift, d1 = back.y - shift;
      s1 += d0 + d1; s2 = fmaf(d0, d0, s2); s2 = fmaf(d1, d1, s2);
    }
  }
  if (!valid) return;
  if (p.stats_out != nullptr)
    p.stats_out[(int64_t)(col0 >> 5) * p.stats_ld + row] = make_float2(fmaf(s1, 1.0f / 32.0f, shift), fmaxf(fmaf(-s1 * (1.0f / 32.0f), s1, s2), 0.f));
  bf16* dst = reinterpret_cast<bf16*>(p.C) + (int64_t)row * p.ldc + col0;
#pragma unroll
  for (int c = 0; c < 4; ++c)
    *reinterpret_cast<uint4*>(reinterpret_cast<uint32_t*>(dst) + 4 * c) = make_uint4(acc[4 * c], acc[4 * c + 1], acc[4 * c + 2], acc[4 * c + 3]);
}

template <int BN, int EW, bool LN = false>
__global__ void __launch_bounds__((2 + EW) * 32, EW == kEpiWarpsSkinny ? 2 : 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
               const __grid_constant__ CUtensorMap tm_c, const GemmArgs p) {
  using Cfg = TileCfg<BN, EW>;
  constexpr int kStages = Cfg::kStages;
  constexpr int kGroups = EW / 4;                               // epilogue groups of 4 warps (one warp per TMEM lane quadrant)
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;                 // 128B-swizzle atoms need 1024-byte alignment
  const uint32_t a_base = base;
  const uint32_t b_base = base + kStages * Cfg::kABytes;
  const uint32_t stage_base = b_base + kStages * Cfg::kBBytes;   // epilogue staging (1024-byte aligned: TMA-store source)
  const uint32_t bar_base = stage_base + Cfg::kStagingBytes;
  const uint32_t lnvec_base = Cfg::kSkinny ? bar_base + Cfg::kBarBytes : stage_base;   // deferred-LayerNorm column vectors (LN kernels only)
  // barrier layout: full[kStages] | empty[kStages] | tmem_full[2] | tmem_empty[2] | tmem base address (u32)
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kStages + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * kStages + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * kStages + 2 + s); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * kStages + 4);
  uint8_t* smem_gen = smem_raw + (base - raw);
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - base));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned long long* stamps = p.dbg_times ? p.dbg_times + (size_t)blockIdx.x * 8 : nullptr;
  if (stamps && threadIdx.x == 0) stamps[0] = global_ns();
  const int tiles_n = (p.N + BN - 1) / BN;
  constexpr int kBM = Cfg::kBM;
  const int tiles_m = p.hm_tpi > 0 ? p.hm_B * p.hm_tpi : (p.M + kBM - 1) / kBM;
  const int num_tiles = tiles_m * tiles_n;
  constexpr int kCK = Cfg::kCK;
  const int num_kb = (p.K + BK * kCK - 1) / (BK * kCK);      // pipeline stages per tile

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_a);
    tma_prefetch_desc(&tm_b);
    if (p.tma_store == 1) tma_prefetch_desc(&tm_c);
    for (int s = 0; s < kStages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(tfull_bar(s), 1); mbar_init(tempty_bar(s), EW * 32); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<Cfg::kTmemCols>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  if (stamps && threadIdx.x == 0) stamps[1] = global_ns();

  if (warp == 0) {
    // ---------------- TMA producer ----------------
    if (lane == 0) {
      pdl_launch_dependents();                       // the next kernel may start its prologue / weight prefetch
      int stage = 0; uint32_t phase = 0;
      bool first = true;
      auto load_b = [&](int st, int kb, int n_blk) {
        if constexpr (kCK > 1) tma_load_3d(b_base + st * Cfg::kBBytes, &tm_b, 0, n_blk * BN, kb * kCK, full_bar(st));
        else tma_load_2d(b_base + st * Cfg::kBBytes, &tm_b, kb * BK, n_blk * BN, full_bar(st));
      };
      auto load_a = [&](int st, int kb, int m_blk) {
        if constexpr (kCK > 1) {
          tma_load_3d(a_base + st * Cfg::kABytes, &tm_a, 0, m_blk * kBM, kb * kCK, full_bar(st));
        } else if (p.hm_tpi > 0) {
          const int img = m_blk / p.hm_tpi;
          tma_load_3d(a_base + st * Cfg::kABytes, &tm_a, kb * BK, (m_blk - img * p.hm_tpi) * BM, img, full_bar(st));
        } else {
          tma_load_2d(a_base + st * Cfg::kABytes, &tm_a, kb * BK, m_blk * BM, full_bar(st));
        }
      };
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int m_blk = tile / tiles_n, n_blk = tile - m_blk * tiles_n;
        int kb0 = 0;
        if (first) {
          // Programmatic dependent launch: the weights (B) never depend on the previous kernel, so the first ring of
          // B tiles is requested before waiting for it; the activations (A) are requested after the wait.
          first = false;
          const int pre = num_kb < kStages ? num_kb : kStages;
          for (int st = 0; st < pre; ++st) {
            mbar_arrive_expect_tx(full_bar(st), Cfg::kABytes + Cfg::kBBytes);
            load_b(st, st, n_blk);
          }
          pdl_wait();
          if (stamps) stamps[2] = global_ns();
          for (int st = 0; st < pre; ++st) load_a(st, st, m_blk);
          kb0 = pre;
          if (pre == kStages) { stage = 0; phase = 1u; } else { stage = pre; }
        }
        for (int kb = kb0; kb < num_kb; ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1u);
          mbar_arrive_expect_tx(full_bar(stage), Cfg::kABytes + Cfg::kBBytes);
          load_a(stage, kb, m_blk);
          load_b(stage, kb, n_blk);
          if (++stage == kStages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ---------------- MMA issuer ----------------
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc(kBM, BN);
      int stage = 0; uint32_t phase = 0; int iter = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++iter) {
        const int as = iter & 1; const uint32_t aphase = (iter >> 1) & 1;
        mbar_wait(tempty_bar(as), aphase ^ 1u);      // epilogue has drained this accumulator stage
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(full_bar(stage), phase);         // TMA bytes have landed
          tc_fence_after();
          if (stamps && iter == 0 && kb == 0 && !LN) stamps[3] = global_ns();
#pragma unroll
          for (int ck = 0; ck < kCK; ++ck) {
            const uint64_t a_desc = make_smem_desc(a_base + stage * Cfg::kABytes + ck * Cfg::kAChunk);
            const uint64_t b_desc = make_smem_desc(b_base + stage * Cfg::kBBytes + ck * Cfg::kBChunk);
#pragma unroll
            for (int k = 0; k < BK / UMMA_K; ++k) {
              // advance 16 elements (32 bytes) along K inside the 128-byte swizzle row: +2 in the (addr >> 4) field
              if (p.dbg != 3) umma_f16(d_tmem, a_desc + 2u * k, b_desc + 2u * k, idesc, (kb | ck | k) != 0 ? 1u : 0u);
            }
          }
          umma_commit(empty_bar(stage));             // frees the smem slot when these MMAs retire
          if (kb == num_kb - 1) { umma_commit(tfull_bar(as)); if (stamps) stamps[4] = global_ns(); }
          if (++stage == kStages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else {
    // ---------------- epilogue ----------------
    const int e = warp - 2;
    const int quad = warp & 3;                        // TMEM lane quadrant this warp may access
    const int grp = e >> 2;                           // 4 groups of 4 warps (one warp per quadrant = 128 accumulator rows)
    const int half = grp;                             // the generic (non-TMA) path only uses groups 0 and 1
    constexpr bool kSplit = BN >= 64 && kGroups >= 2;       // generic path: two groups share the columns of a wide tile
    constexpr int kColsPerHalf = kSplit ? BN / 2 : BN;
    const int c_begin = kSplit ? half * kColsPerHalf : 0;
    const int c_end = (grp >= 2) ? 0 : (kSplit ? c_begin + kColsPerHalf : (half == 0 ? BN : 0));
    uint32_t* stage = reinterpret_cast<uint32_t*>(smem_gen + (stage_base - base)) + (e & 7) * Cfg::kStageWords;
    int iter = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++iter) {
      const int m_blk = tile / tiles_n, n_blk = tile - m_blk * tiles_n;
      const int as = iter & 1; const uint32_t aphase = (iter >> 1) & 1;
      if constexpr (LN) {
        // Deferred LayerNorm (a separate instantiation: no register cost elsewhere).  Each warp owns at most one 32-column block
        // (BN / 32 <= epilogue groups).  Everything that does not need the accumulator is fetched while the main loop runs:
        //   - the block's column vectors (weights: requested BEFORE the programmatic dependency is awaited) into shared memory,
        //   - after the wait - row statistics and residual are outputs of preceding kernels, and these warps read them themselves,
        //     so they wait for the dependency themselves - the merged statistics of this thread's row and its residual values.
        static_assert(BN / 32 <= kGroups, "one column block per epilogue warp");
        const int cfirst = n_blk * BN + grp * 32;
        const bool active = grp < BN / 32 && cfirst < p.N;
        float* sv = reinterpret_cast<float*>(smem_gen + (lnvec_base - base)) + e * 128;
        if (active) {
          sv[lane] = p.bias != nullptr ? __ldg(p.bias + cfirst + lane) : 0.f;
          sv[32 + lane] = p.fold_c != nullptr ? __ldg(p.fold_c + cfirst + lane) : 0.f;
          sv[64 + lane] = p.res_gamma != nullptr ? __ldg(p.res_gamma + cfirst + lane) : 0.f;
          sv[96 + lane] = p.res_beta != nullptr ? __ldg(p.res_beta + cfirst + lane) : 0.f;
        }
        if (iter == 0) pdl_wait();
        const int row = kBM == 128 ? m_blk * BM + quad * 32 + lane : (lane < 16 ? m_blk * kBM + quad * 16 + lane : p.M);
        const bool rv = active && row < p.M;
        float2 fstat = make_float2(0.f, 1.f), rstat = make_float2(0.f, 1.f);
        if (p.fold_stats != nullptr && rv) fstat = ln_merge_stats(p.fold_stats + row, p.stats_ld, p.fold_parts);
        if (p.res_stats != nullptr && rv) rstat = ln_merge_stats(p.res_stats + row, p.stats_ld, p.res_parts);
        uint4 rpre[4];
        const bool have_rpre = p.res != nullptr && active;
        if (have_rpre) {
          if (rv) {
            const uint4* rp = reinterpret_cast<const uint4*>(reinterpret_cast<const bf16*>(p.res) + (int64_t)row * p.ldr + cfirst);
#pragma unroll
            for (int c = 0; c < 4; ++c) rpre[c] = rp[c];
          } else {
#pragma unroll
            for (int c = 0; c < 4; ++c) rpre[c] = make_uint4(0, 0, 0, 0);
          }
        }
        __syncwarp();                                             // sv complete
        if (stamps && e == 0 && lane == 0) stamps[3] = global_ns() + (unsigned long long)(__float_as_uint(fstat.x + rstat.x) & 1u);   // statistics merged
        mbar_wait(tfull_bar(as), aphase);
        tc_fence_after();
        if (stamps && e == 0 && lane == 0) stamps[5] = global_ns();
        const uint32_t tq = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + as * BN;
        if (active) epilogue_direct_block_ln(p, tq + grp * 32, row, cfirst, fstat, rstat, have_rpre ? rpre : nullptr, sv);
        tc_fence_before();
        mbar_arrive(tempty_bar(as));
        continue;
      }
      if (p.bias != nullptr && lane == 0) {              // pull this tile's bias segment into L1 while the main loop runs
        const int c0 = n_blk * BN + (e & 7) * (BN / 8);
        if (c0 < p.N) asm volatile("prefetch.global.L1 [%0];" ::"l"(p.bias + c0));
      }
      // direct-store (decode) mode: the bias of this warp's first column block is fetched now, under the main loop
      float bpre[32];
      bool have_bpre = false;
      if (p.tma_store == 2 && p.bias != nullptr && grp < BN / 32) {
        const int c0 = n_blk * BN + grp * 32;
        if (c0 + 32 <= p.N && (reinterpret_cast<uintptr_t>(p.bias + c0) & 15) == 0) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias + c0) + j);
            bpre[4 * j] = b4.x; bpre[4 * j + 1] = b4.y; bpre[4 * j + 2] = b4.z; bpre[4 * j + 3] = b4.w;
          }
          have_bpre = true;
        }
      }
      mbar_wait(tfull_bar(as), aphase);
      tc_fence_after();
      if (stamps && e == 0 && lane == 0) stamps[5] = global_ns();
      const int row0 = m_blk * BM + quad * 32;
      if (p.dbg == 2) { tc_fence_before(); mbar_arrive(tempty_bar(as)); continue; }
      constexpr int kWb = (BN >= 128) ? 64 : 32;           // block width of the generic (non-TMA) bf16 path
      if (p.tma_store == 2) {
        const uint32_t tq = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + as * BN;
        for (int j = grp; j < BN / 32; j += kGroups) {
          const int col0 = n_blk * BN + j * 32;
          if (col0 >= p.N) break;
          const float* bp = (have_bpre && j == grp) ? bpre : nullptr;
          // M = 128: TMEM lane == tile row.  M = 64: lanes 0-15 of each quadrant hold rows quad * 16 + lane, the rest nothing.
          const int row = kBM == 128 ? row0 + lane : (lane < 16 ? m_blk * kBM + quad * 16 + lane : p.M);
          if (p.out_f32) epilogue_direct_block<float>(p, tq + j * 32, row, col0, bp);
          else epilogue_direct_block<bf16>(p, tq + j * 32, row, col0, bp);
        }
      } else if (p.tma_store) {
        const int r = quad * 32 + lane;                     // accumulator row == TMEM lane == staging row
        const bool issuer = (e & 3) == 0 && lane == 0;
        const uint32_t tq = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + as * BN;
        if (p.out_f32) {
          // fp32 rows of 32 columns are 128 bytes: two 16 KB staging tiles, groups 0 and 1 only
          constexpr int kFGroups = kGroups < 2 ? kGroups : 2;
          if (grp < kFGroups) {
            const uint32_t stg = stage_base + grp * 16384;
            for (int j = grp; j < BN / 32; j += kFGroups) {
              const int col0 = n_blk * BN + j * 32;
              if (col0 >= p.N) break;                       // uniform across the group
              epilogue_tma_block<float, 32>(p, &tm_c, tq + j * 32, stg, m_blk * BM, col0, r, grp, issuer);
            }
          }
        } else {
          // bf16 rows of 32 columns are 64 bytes: four 8 KB staging tiles, one per group
          const uint32_t stg = stage_base + grp * 8192;
          for (int j = grp; j < BN / 32; j += kGroups) {
            const int col0 = n_blk * BN + j * 32;
            if (col0 >= p.N) break;
            epilogue_tma_block<bf16, 32>(p, &tm_c, tq + j * 32, stg, m_blk * BM, col0, r, grp, issuer);
          }
        }
      } else if (p.out_f32) {
        for (int c = c_begin; c < c_end; c += 32) {
          const int col0 = n_blk * BN + c;
          if (col0 >= p.N) break;                           // warp-uniform
          epilogue_block<float, 32>(p, tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + as * BN + c, stage, row0, col0, lane);
        }
      } else {
        for (int c = c_begin; c < c_end; c += kWb) {
          const int col0 = n_blk * BN + c;
          if (col0 >= p.N) break;
          epilogue_block<bf16, kWb>(p, tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + as * BN + c, stage, row0, col0, lane);
        }
      }
      tc_fence_before();
      mbar_arrive(tempty_bar(as));
    }
    // the staging tiles must have been read before the CTA's shared memory goes away; the global writes themselves are
    // complete (and visible to the next kernel) at grid end like any other store
    if (p.tma_store == 1 && (e & 3) == 0 && lane == 0) bulk_wait_read0();
    if (stamps && e == 0 && lane == 0) stamps[6] = global_ns();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc<Cfg::kTmemCols>(tmem_base);
  if (stamps && threadIdx.x == 32) stamps[7] = global_ns();
}

// ------------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode = nullptr;
std::once_flag g_once;

struct MapKey {
  const void* ptr; int64_t rows, cols, ld; int box_rows, box_cols, esz, kind; int64_t d2, d3;
  bool operator==(const MapKey& o) const {
    return ptr == o.ptr && rows == o.rows && cols == o.cols && ld == o.ld && box_rows == o.box_rows && box_cols == o.box_cols &&
           esz == o.esz && kind == o.kind && d2 == o.d2 && d3 == o.d3;
  }
};
struct MapKeyHash {
  size_t operator()(const MapKey& k) const {
    size_t h = reinterpret_cast<size_t>(k.ptr);
    for (int64_t v : {k.rows, k.cols, k.ld, (int64_t)k.box_rows, (int64_t)k.box_cols, (int64_t)k.esz, (int64_t)k.kind, k.d2, k.d3})
      h = h * 1000003u ^ static_cast<size_t>(v);
    return h;
  }
};
std::mutex g_map_mu;
std::unordered_map<MapKey, CUtensorMap, MapKeyHash> g_maps;

const CUtensorMap& cached_map(const MapKey& key, CUtensorMapDataType dt, int rank, const cuuint64_t* gdim, const cuuint64_t* gstride,
                              const cuuint32_t* box, CUtensorMapSwizzle swz) {
  std::lock_guard<std::mutex> lk(g_map_mu);
  auto it = g_maps.find(key);
  if (it != g_maps.end()) return it->second;
  CUtensorMap m;
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = g_encode(&m, dt, rank, const_cast<void*>(key.ptr), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) throw std::runtime_error("cuTensorMapEncodeTiled failed with code " + std::to_string((int)r));
  if (g_maps.size() > 4096) g_maps.clear();
  return g_maps.emplace(key, m).first->second;
}

}  // namespace

namespace tc {

// 2-D bf16 operand [rows, cols] with row stride ld (elements); box = 64 columns x box_rows rows, 128-byte swizzle.
const CUtensorMap& get_map(const void* ptr, int64_t rows, int64_t cols, int64_t ld, int box_rows) {
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) != 0 || (ld * 2) % 16 != 0)
    throw std::runtime_error("gemm_tc: operand must be 16-byte aligned with a row stride that is a multiple of 8 elements");
  MapKey key{ptr, rows, cols, ld, box_rows, BK, 2, 0, 0, 0};
  cuuint64_t gdim[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t gstride[1] = {static_cast<cuuint64_t>(ld * 2)};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(BK), static_cast<cuuint32_t>(box_rows)};
  return cached_map(key, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, gdim, gstride, box, CU_TENSOR_MAP_SWIZZLE_128B);
}

// Operand viewed as [K/64 chunks][rows][64]: one box = 64 elements x box_rows rows x `chunks` consecutive k-chunks, each chunk
// landing as its own 128-byte-swizzled tile (row stride 128 B) - the layout the UMMA descriptors expect.
const CUtensorMap& get_map_k3(const void* ptr, int64_t rows, int64_t cols, int64_t ld, int box_rows, int chunks) {
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) != 0 || (ld * 2) % 16 != 0 || cols % BK != 0)
    throw std::runtime_error("gemm_tc: chunked operand needs 16-byte alignment, ld % 8 == 0 and K % 64 == 0");
  MapKey key{ptr, rows, cols, ld, box_rows, BK, 2, 5, chunks, 0};
  cuuint64_t gdim[3] = {(cuuint64_t)BK, (cuuint64_t)rows, (cuuint64_t)(cols / BK)};
  cuuint64_t gstride[2] = {(cuuint64_t)ld * 2, (cuuint64_t)BK * 2};
  cuuint32_t box[3] = {(cuuint32_t)BK, (cuuint32_t)box_rows, (cuuint32_t)chunks};
  return cached_map(key, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, gdim, gstride, box, CU_TENSOR_MAP_SWIZZLE_128B);
}

// Output map for the TMA-store epilogue: [M, N] row-major with box = box_cols x 128 rows.
const CUtensorMap& get_map_c(const void* ptr, int64_t rows, int64_t cols, int64_t ld, int esz, int box_cols) {
  MapKey key{ptr, rows, cols, ld, BM, box_cols, esz, 1, 0, 0};
  cuuint64_t gdim[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t gstride[1] = {static_cast<cuuint64_t>(ld * esz)};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(box_cols), static_cast<cuuint32_t>(BM)};
  return cached_map(key, esz == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, gdim, gstride, box,
                    box_cols * esz == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B);
}


// Head-major cross-KV output [layers*B][G][L][D] bf16 (GemmArgs::hm_*): box = D x 128 positions of one (layer-image, group).
// Activations of the head-major mode viewed as [B][L][K]: box = 64 k x 128 positions of one image (rows past L are zero-filled).
const CUtensorMap& get_map_a3(const void* ptr, int64_t K, int L, int B, int64_t ld) {
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) != 0 || (ld * 2) % 16 != 0)
    throw std::runtime_error("gemm_tc: operand must be 16-byte aligned with a row stride that is a multiple of 8 elements");
  MapKey key{ptr, L, K, ld, BM, BK, 2, 4, B, 0};
  cuuint64_t gdim[3] = {(cuuint64_t)K, (cuuint64_t)L, (cuuint64_t)B};
  cuuint64_t gstride[2] = {(cuuint64_t)ld * 2, (cuuint64_t)L * ld * 2};
  cuuint32_t box[3] = {(cuuint32_t)BK, (cuuint32_t)BM, 1};
  return cached_map(key, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, gdim, gstride, box, CU_TENSOR_MAP_SWIZZLE_128B);
}
const CUtensorMap& get_map_hm3(const void* ptr, int D, int L, int64_t LBG, int box_cols) {
  MapKey key{ptr, L, D, D, BM, box_cols, 2, 3, LBG, 0};
  cuuint64_t gdim[3] = {(cuuint64_t)D, (cuuint64_t)L, (cuuint64_t)LBG};
  cuuint64_t gstride[2] = {(cuuint64_t)D * 2, (cuuint64_t)L * D * 2};
  cuuint32_t box[3] = {(cuuint32_t)box_cols, (cuuint32_t)BM, 1};
  return cached_map(key, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, gdim, gstride, box,
                    box_cols * 2 == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B);
}

}  // namespace tc

namespace {

const CUtensorMap& get_map_hm(const void* ptr, int D, int L, int G, int64_t LB) {
  MapKey key{ptr, L, D, D, BM, D, 2, 2, G, LB};
  cuuint64_t gdim[4] = {(cuuint64_t)D, (cuuint64_t)L, (cuuint64_t)G, (cuuint64_t)LB};
  cuuint64_t gstride[3] = {(cuuint64_t)D * 2, (cuuint64_t)L * D * 2, (cuuint64_t)G * L * D * 2};
  cuuint32_t box[4] = {(cuuint32_t)D, (cuuint32_t)BM, 1, 1};
  return cached_map(key, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, gdim, gstride, box, CU_TENSOR_MAP_SWIZZLE_128B);
}

template <int BN, int EW = kEpiWarpsWide, bool LN = false>
void launch_cfg(const GemmArgs& a_in, int num_sms, cudaStream_t stream) {
  using Cfg = TileCfg<BN, EW>;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(gemm_tc_kernel<BN, EW, LN>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes + (LN ? Cfg::kLnVecExtra : 0));
    if (e != cudaSuccess) throw std::runtime_error(std::string("gemm_tc: cudaFuncSetAttribute: ") + cudaGetErrorString(e));
    attr_set = true;
  }
  const bool ln_args = a_in.fold_stats != nullptr || a_in.res != nullptr || a_in.stats_out != nullptr;
  if (ln_args != LN) throw std::runtime_error("gemm_tc: deferred-LayerNorm arguments reached a kernel configuration without that epilogue");
  // a.tma_store = the store gemm_tc_variant chose and checked: TMA store when the output is expressible as a tensor map, direct row
  // stores, or the generic register/shared path
  GemmArgs a = a_in;
  const CUtensorMap* ma_ptr = Cfg::kCK > 1 ? &get_map_k3(a.A, a.M, a.K, a.lda, Cfg::kBM, Cfg::kCK) : &get_map(a.A, a.M, a.K, a.lda, Cfg::kBM);
  const CUtensorMap& mb = Cfg::kCK > 1 ? get_map_k3(a.W, a.N, a.K, a.ldw, BN, Cfg::kCK) : get_map(a.W, a.N, a.K, a.ldw, BN);
  const int esz = a.out_f32 ? 4 : 2;
  const int cw = 32;                                  // columns per TMA-store box (bf16: 64-byte rows, fp32: 128-byte rows)
  const CUtensorMap* mc = ma_ptr;
  if (a.tma_store == kStoreTma) {
    if (a.hm_D > 0) {
      const int64_t LB = (int64_t)(a.N / (a.hm_D * a.hm_G)) * a.hm_B;
      mc = &get_map_hm3(a.C, a.hm_D, a.hm_L, LB * a.hm_G, cw);
      a.hm_tpi = (a.hm_L + BM - 1) / BM;
      ma_ptr = &get_map_a3(a.A, a.K, a.hm_L, a.hm_B, a.lda);
    } else {
      a.tma_cols = tma_store_cols(a.N, esz);
      mc = &get_map_c(a.C, a.M, a.tma_cols, a.ldc, esz, cw);
    }
  }
  const int tiles_m = a.hm_tpi > 0 ? a.hm_B * a.hm_tpi : (a.M + Cfg::kBM - 1) / Cfg::kBM;
  const int tiles = tiles_m * ((a.N + BN - 1) / BN);
  if (a.fold_stats != nullptr || a.res != nullptr || a.stats_out != nullptr) {
    auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
    if ((a.bias && !al16(a.bias)) || (a.fold_stats && (!a.fold_c || !al16(a.fold_c) || a.fold_parts < 1 || a.fold_parts > kLnStatStride)) ||
        ((a.fold_stats || a.res_stats || a.stats_out) && a.stats_ld < a.M) ||
        (a.res && (!al16(a.res) || a.ldr % 8 != 0)) ||
        (a.res_stats && (!a.res || !a.res_gamma || !a.res_beta || !al16(a.res_gamma) || !al16(a.res_beta) || a.res_parts != a.N / 32)) ||
        (a.stats_out && a.N / 32 > kLnStatStride))
      throw std::runtime_error("gemm_tc: malformed deferred-LayerNorm arguments");
  }
  const int slots = Cfg::kSkinny ? 2 * num_sms : num_sms;      // resident CTAs: the kernel is persistent over the remaining tiles
  const int grid = tiles < slots ? tiles : slots;
  launch_k(gemm_tc_kernel<BN, EW, LN>, dim3(grid), dim3(Cfg::kThreads), (size_t)(Cfg::kSmemBytes + (LN ? Cfg::kLnVecExtra : 0)), stream, *ma_ptr, mb, *mc, a);
}

}  // namespace

void gemm_tc_init() {
  std::call_once(g_once, [] {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || fn == nullptr)
      throw std::runtime_error("gemm_tc: cannot resolve cuTensorMapEncodeTiled");
    g_encode = reinterpret_cast<EncodeTiledFn>(fn);
  });
}

// [groups][L][D] bf16 rows (the decoder's cross K/V cache) as a 3-D map: box = D x box_rows rows of one group, 128-byte swizzle.
const void* tma_map_rows3(const void* ptr, int D, int L, int64_t groups, int box_rows) {
  gemm_tc_init();
  if (D * 2 != 128 || (reinterpret_cast<uintptr_t>(ptr) & 15) != 0) throw std::runtime_error("tma_map_rows3: rows must be 128 bytes, base 16-byte aligned");
  MapKey key{ptr, L, D, D, box_rows, D, 2, 6, groups, 0};
  cuuint64_t gdim[3] = {(cuuint64_t)D, (cuuint64_t)L, (cuuint64_t)groups};
  cuuint64_t gstride[2] = {(cuuint64_t)D * 2, (cuuint64_t)L * D * 2};
  cuuint32_t box[3] = {(cuuint32_t)D, (cuuint32_t)box_rows, 1};
  return &cached_map(key, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, gdim, gstride, box, CU_TENSOR_MAP_SWIZZLE_128B);
}

namespace {

// The selection rule (engine call sites: force_kernel = force_store = -1).  Environment switches are A/B aids and act here only.
int rule_kernel(const GemmArgs& a, int num_sms) {
  static const int bn_env = [] { const char* e = getenv("GSTVD_GEMM_BN"); return e ? atoi(e) : 0; }();
  if (a.fold_stats != nullptr || a.res != nullptr || a.stats_out != nullptr) {
    // deferred-LayerNorm epilogue (decode step): the M = 64 two-per-SM configuration with 32-column tiles while they fit the
    // resident slots (the N = H projections, the only ones that write statistics), 64-column tiles of 128 rows for the wide ones
    return ((a.M + 63) / 64) * ((a.N + 31) / 32) <= 2 * num_sms ? kGemmLn32 : kGemmLn64;
  }
  const int pair_bn = pick_pair_bn(a);   // CTA-pair tiles (cta_group::2) where they measured faster: large M
  if (pair_bn) return pair_bn == 256 ? kGemmPair256 : kGemmPair128;
  const int tiles_m = (a.M + BM - 1) / BM;
  int bn = 32;
  const int cand[4] = {256, 128, 64, 32};
  if (tiles_m <= 4) {
    // skinny (decode) problems are latency-bound: prefer ONE wave - the narrowest tile whose tile count still fits the SMs
    bn = 256;
    for (int i = 3; i >= 0; --i) {
      if (tiles_m * ((a.N + cand[i] - 1) / cand[i]) <= num_sms) { bn = cand[i]; break; }
    }
  } else {
    // Throughput problems: the tile width that maximises (wave efficiency) x (per-tile efficiency of that width).  Wide tiles
    // run the tensor pipe best, but a persistent grid of 148 CTAs wastes the last wave: e.g. M = 2048, N = 3072 is 192 tiles
    // of 256 columns (two waves, 65 % full) or 384 tiles of 128 columns (three waves, 86 % full).
    const double tile_eff[4] = {1.0, 0.88, 0.6, 0.35};
    double best = -1.0;
    for (int i = 0; i < 4; ++i) {
      const int64_t tiles = (int64_t)tiles_m * ((a.N + cand[i] - 1) / cand[i]);
      const int64_t waves = (tiles + num_sms - 1) / num_sms;
      const double used = (double)a.N / ((double)((a.N + cand[i] - 1) / cand[i]) * cand[i]);     // columns of the last tile that exist
      const double eff = (double)tiles / (double)(waves * num_sms) * tile_eff[i] * used;
      if (eff > best + 1e-9) { best = eff; bn = cand[i]; }
    }
  }
  if (bn_env) bn = bn_env;
  if (bn <= 64 && a.K % BK != 0) bn = 128;               // the chunked (3-D box) operand view needs whole 64-element chunks
  // Skinny (decode) problems whose output qualifies for direct row stores run the M = 64 configuration (two CTAs per SM):
  // 32-column tiles when they all fit the 2 x SMs resident slots, else 64-column tiles.
  static const int skinny_env = [] { const char* e = getenv("GSTVD_GEMM_SKINNY"); return e ? atoi(e) : -1; }();   // A/B aid: force 0 / 1
  const bool skinny = skinny_env >= 0 ? skinny_env != 0 : true;
  {
    const int esz = a.out_f32 ? 4 : 2;
    const bool direct_ok = a.hm_D == 0 && (reinterpret_cast<uintptr_t>(a.C) & 15) == 0 && (a.ldc * esz) % 16 == 0 && a.M <= 4 * BM &&
                           (int64_t)a.M * a.N * esz <= (4 << 20) && getenv("GSTVD_GEMM_NO_DIRECT") == nullptr &&
                           getenv("GSTVD_GEMM_NO_TMA_STORE") == nullptr;
    if (skinny && direct_ok && a.K % BK == 0 && !bn_env) {
      const int tm64 = (a.M + 63) / 64;
      static const int multi = [] { const char* e = getenv("GSTVD_GEMM_SKINNY_WAVES"); return e ? atoi(e) : 1; }();   // A/B aid
      if (tm64 * ((a.N + 31) / 32) <= 2 * num_sms * multi) return kGemmSkinny32;
      // wider outputs (N = 2304 / 3072 at M = 320) measured faster in the 128-row configuration with 16 epilogue warps
      // (5.5 / 5.7 us vs 5.9 / 6.2 us): 64-column tiles make each of the four epilogue warps handle two column blocks
      static const bool wide64 = getenv("GSTVD_GEMM_SKINNY64") != nullptr;
      if (wide64 && tm64 * ((a.N + 63) / 64) <= 2 * num_sms) return kGemmSkinny64;
    }
  }
  switch (bn) {
    case 256: return kGemmTc256;
    case 128: return kGemmTc128;
    case 64: return kGemmTc64;
    default: return kGemmTc32;
  }
}

// The store the rule picks for `kernel`: TMA store when the output is expressible as a tensor map (head-major: 128-row tiles of
// whole k-blocks only), direct row stores for small outputs, else the generic register/shared path.
int rule_store(const GemmArgs& a, int kernel) {
  if (kernel == kGemmSimt) return kStoreGeneric;
  if (kernel == kGemmPair128 || kernel == kGemmPair256) return kStoreTma;
  static const bool no_tma_store = getenv("GSTVD_GEMM_NO_TMA_STORE") != nullptr;
  static const bool no_tma_hm = getenv("GSTVD_GEMM_NO_TMA_HM") != nullptr;
  static const bool no_direct = getenv("GSTVD_GEMM_NO_DIRECT") != nullptr;     // A/B aid
  const int esz = a.out_f32 ? 4 : 2;
  if (no_tma_store || (reinterpret_cast<uintptr_t>(a.C) & 15) != 0) return kStoreGeneric;
  if (a.hm_D > 0) {
    const bool whole_kblocks = kernel == kGemmTc128 || kernel == kGemmTc256;
    return !no_tma_hm && whole_kblocks && !a.out_f32 && a.hm_D % 32 == 0 && a.M == a.hm_B * a.hm_L ? kStoreTma : kStoreGeneric;
  }
  if ((a.ldc * esz) % 16 != 0) return kStoreGeneric;
  // skinny (decode) problems: latency matters, the tile is tiny
  if (a.M <= 4 * BM && (int64_t)a.M * a.N * esz <= (4 << 20) && !no_direct) return kStoreDirect;
  return tma_store_cols(a.N, esz) > 0 ? kStoreTma : kStoreGeneric;
}

const char* const kKernelNames[kGemmKernels] = {"simt", "tc32", "tc64", "tc128", "tc256", "skinny32", "skinny64", "pair128", "pair256", "ln32", "ln64"};
const char* const kStoreNames[kGemmStores] = {"generic", "TMA", "direct"};

// What (kernel, store) cannot run, or "".  Only kernel limits are checked here, never the rule's preferences.
std::string variant_unsupported(const GemmArgs& a, int kernel, int store) {
  if (kernel < 0 || kernel >= kGemmKernels) return "unknown GEMM kernel id " + std::to_string(kernel);
  if (store < 0 || store >= kGemmStores) return "unknown GEMM store id " + std::to_string(store);
  const std::string what = std::string(kKernelNames[kernel]) + " with the " + kStoreNames[store] + " store: ";
  const bool ln_args = a.fold_stats != nullptr || a.res != nullptr || a.stats_out != nullptr;
  const bool ln = kernel == kGemmLn32 || kernel == kGemmLn64;
  const bool skinny = kernel == kGemmSkinny32 || kernel == kGemmSkinny64;
  const bool pair = kernel == kGemmPair128 || kernel == kGemmPair256;
  const bool chunked = kernel == kGemmTc32 || kernel == kGemmTc64 || skinny || ln;    // 3-D boxes of several 64-element k-chunks
  const int esz = a.out_f32 ? 4 : 2;
  const bool c16 = (reinterpret_cast<uintptr_t>(a.C) & 15) == 0;
  if (kernel == kGemmSimt) {
    if (store != kStoreGeneric) return what + "the SIMT kernel stores element by element (generic store only)";
    if (ln_args) return what + "the SIMT kernel has no deferred-LayerNorm epilogue";
    return "";
  }
  if (ln_args != ln) return what + (ln ? "the deferred-LayerNorm kernels need a deferred-LayerNorm argument"
                                       : "deferred-LayerNorm arguments need the ln32 / ln64 kernels");
  if (a.K % 8 != 0) return what + "K must be a multiple of 8 (16-byte TMA strides)";
  if (chunked && a.K % BK != 0) return what + "this configuration loads whole 64-element k-chunks: K % 64 == 0";
  if (a.hm_D > 0 && a.hm_D % 32 != 0) return what + "the head-major scatter needs head_dim % 32 == 0";
  if (skinny && store != kStoreDirect) return what + "the 64-row configurations only have the direct-store epilogue";
  if (ln && store != kStoreDirect) return what + "the deferred-LayerNorm epilogue stores directly";
  if (ln && (a.out_f32 || a.N % 32 != 0 || (a.ldc * 2) % 16 != 0)) return what + "the deferred-LayerNorm epilogue needs bf16 output, N % 32 == 0, ldc % 8 == 0";
  if (pair && store != kStoreTma) return what + "the CTA-pair kernel only has the TMA-store epilogue";
  switch (store) {
    case kStoreTma:
      if (!c16) return what + "the output must be 16-byte aligned";
      if (a.hm_D > 0) {
        if (!(kernel == kGemmTc128 || kernel == kGemmTc256 || pair)) return what + "head-major TMA tiles need whole 64-element k-blocks per stage (tc128 / tc256 / pairs)";
        if (a.out_f32) return what + "the head-major TMA store writes bf16";
        if (a.M != a.hm_B * a.hm_L || a.N % (a.hm_D * a.hm_G) != 0) return what + "the head-major TMA store needs M = B * L and N % (D * G) == 0";
      } else if ((a.ldc * esz) % 16 != 0 || tma_store_cols(a.N, esz) == 0) {
        return what + "output rows must be 16-byte aligned (ldc * element size % 16 == 0) and at least 16 bytes long";
      }
      break;
    case kStoreDirect:
      if (a.hm_D > 0) return what + "direct stores write row-major rows, not the head-major layout";
      if (!c16 || (a.ldc * esz) % 16 != 0) return what + "direct stores need a 16-byte aligned output and rows (ldc * element size % 16 == 0)";
      break;
    default:
      if (skinny || ln || pair) return what + "no generic epilogue in this configuration";
      break;
  }
  return "";
}

}  // namespace

std::string gemm_tc_variant(const GemmArgs& a, int num_sms, GemmVariant* v) {
  const int kernel = a.force_kernel >= 0 ? a.force_kernel : rule_kernel(a, num_sms);
  const int store = a.force_store >= 0 ? a.force_store : rule_store(a, kernel);
  std::string why = variant_unsupported(a, kernel, store);
  if (why.empty() && v) { v->kernel = kernel; v->store = store; }
  return why;
}

int launch_gemm_tc(const GemmArgs& a_in, int num_sms, cudaStream_t stream, GemmVariant* ran) {
  if (a_in.M <= 0 || a_in.N <= 0) return 0;
  static const int dbg_env = [] { const char* e = getenv("GSTVD_GEMM_DBG"); return e ? atoi(e) : 0; }();
  GemmArgs a = a_in;
  a.dbg = dbg_env;
  GemmVariant v;
  const std::string why = gemm_tc_variant(a, num_sms, &v);
  if (!why.empty()) throw std::runtime_error("gemm_tc: " + why);
  gemm_tc_init();
  a.tma_store = v.store;
  switch (v.kernel) {
    case kGemmTc32: launch_cfg<32>(a, num_sms, stream); break;
    case kGemmTc64: launch_cfg<64>(a, num_sms, stream); break;
    case kGemmTc128: launch_cfg<128>(a, num_sms, stream); break;
    case kGemmTc256: launch_cfg<256>(a, num_sms, stream); break;
    case kGemmSkinny32: launch_cfg<32, kEpiWarpsSkinny>(a, num_sms, stream); break;
    case kGemmSkinny64: launch_cfg<64, kEpiWarpsSkinny>(a, num_sms, stream); break;
    case kGemmPair128: launch_gemm_tc2(a, 128, num_sms, stream); break;
    case kGemmPair256: launch_gemm_tc2(a, 256, num_sms, stream); break;
    case kGemmLn32: launch_cfg<32, kEpiWarpsSkinny, true>(a, num_sms, stream); break;
    case kGemmLn64: launch_cfg<64, kEpiWarpsWide, true>(a, num_sms, stream); break;
    default: throw std::runtime_error("gemm_tc: the SIMT kernel is launched by launch_gemm_simt");
  }
  if (ran) *ran = v;
  return 1;
}

}  // namespace gstvd
