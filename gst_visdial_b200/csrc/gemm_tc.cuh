// Device helpers shared by the tcgen05 GEMM family (gemm_tc.cu: single-CTA tiles, gemm_tc2.cu: CTA pairs): mbarrier / TMA / tcgen05 / cluster PTX wrappers, the UMMA descriptors, the TMA-store epilogue block, and
// the interface of the host-side tensor-map cache.  sm_100a only.
#pragma once
#include <cuda.h>

#include <cstdint>

#include "common.cuh"
#include "kernels.h"

namespace gstvd {
namespace tc {

constexpr int BM = 128;          // rows per tile  (UMMA M)
constexpr int BK = 64;           // k per stage: 64 bf16 = 128 bytes = one swizzle row
constexpr int UMMA_K = 16;
// Epilogue warps: 16 (4 per TMEM lane quadrant) for the throughput configurations - the epilogue is ALU/latency bound and
// needs the warps; 4 (one per quadrant) for the "skinny" decode configuration (64-row tiles, see TileCfg), whose 6-warp CTA
// with ~100 KB of shared memory lets TWO CTAs share an SM: decode GEMMs (M = 320) are latency bound, so a co-resident CTA -
// the next GEMM of the same stream under PDL, or another stream's - fills the SM time this one spends waiting.
constexpr int kEpiWarpsWide = 16;
constexpr int kEpiWarpsSkinny = 4;
constexpr unsigned long long kWaitTimeoutNs = 4000000000ull;   // 4 s: far beyond any legitimate wait

__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok = 0, spins = 0;
  unsigned long long t0 = 0;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    if (!ok && (++spins & 1023u) == 0) {         // a protocol bug must fail the launch, never hang the GPU
      unsigned long long now = global_ns();
      if (t0 == 0) t0 = now;
      else if (now - t0 > kWaitTimeoutNs) __trap();
    }
  } while (!ok);
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(c2), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(map)), "r"(src), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(map)), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(map)), "r"(src), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

template <int COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "n"(COLS) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(COLS) : "memory");
}

// K-major operand tile in shared memory, 128-byte swizzle: rows of 64 bf16 (128 B); 8-row groups are 1024 B apart.
// Descriptor fields (PTX ISA "tcgen05 shared memory descriptor"): start address >> 4 [0,14), leading byte offset >> 4
// [16,30) (unused for swizzled K-major, set to 1), stride byte offset >> 4 [32,46) = 1024 >> 4, version 1 at [46,48),
// layout type SWIZZLE_128B = 2 at [61,64).
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// Instruction descriptor for kind::f16: D fp32 (bits 4-5 = 1), A/B bf16 (bits 7-9 / 10-12 = 1), both K-major
// (bits 15, 16 = 0), N >> 3 at [17,23), M >> 4 at [24,29).
__host__ __device__ constexpr uint32_t make_idesc(int m, int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// 32 lanes x 32 consecutive 32-bit columns: thread i of the warp receives lane (base_lane + i), columns c..c+31
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// GELU(x) = 0.5 x (1 + erf(x / sqrt 2)).  The epilogue of the FFN1 GEMMs is bound by issue slots (profiles/r2_pair_gemm_ncu_summary.txt:
// ~6 100 warp instructions per scheduler and 128 x 256 tile against 6 144 tensor-pipe cycles), so what counts is instructions per element:
//   default : erf(z) = tanh(z (a + b z^2 + c z^4)) with a minimax fit over z in [0, 5] (|error| <= 3.7e-5, tools/fit_erf_tanh.py) and the
//             single-instruction MUFU tanh (relative error 2^-11): 8 instructions, |GELU error| <= 2.5e-4 |x| - an eighth of a bf16 ulp of
//             the result for |x| >= 1/4 and below 2e-4 absolutely everywhere, i.e. far inside the rounding of the bf16 output it feeds;
//   GSTVD_GELU_AS (compile-time, -DGSTVD_GELU_AS) : Abramowitz-Stegun 7.1.25 with MUFU reciprocal / exp2 (|error| <= 2.5e-5, ~15 instructions).
// The fp32 parity path uses the exact erff (gemm_simt.cu).
__device__ __forceinline__ float gelu_fast(float x) {
#ifdef GSTVD_GELU_AS
  const float z = fabsf(x) * 0.70710678118654752440f;
  float t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.47047f, z, 1.0f)));
  float poly = fmaf(t, 0.7478556f, -0.0958798f);
  poly = fmaf(t, poly, 0.3480242f);
  poly *= t;
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-1.44269504088896340736f * z * z));
  const float erf_abs = fmaf(-poly, e, 1.0f);
  const float erf = copysignf(erf_abs, x);
  return 0.5f * x * (1.0f + erf);
#else
  // z = x / sqrt 2;  u = z (a + b z^2 + c z^4) written in x:  a / sqrt2, b / sqrt2^3, c / sqrt2^5
  const float x2 = fminf(x * x, 50.0f);                 // the fit covers |x| <= 7.07; beyond it tanh has saturated (and the quartic would turn over)
  float q = fmaf(x2, -0.00031580700f, 0.036798256f);
  q = fmaf(x2, q, 0.79771782f);
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(x * q));
  const float hx = 0.5f * x;
  return fmaf(hx, t, hx);
#endif
}

__device__ __forceinline__ int64_t out_index(const GemmArgs& p, int row, int col) {
  if (p.hm_D > 0) {
    const int b = row / p.hm_L, pos = row - b * p.hm_L;
    const int g = col / p.hm_D, d = col - g * p.hm_D;
    const int layer = g / p.hm_G, r = g - layer * p.hm_G;
    return ((((int64_t)layer * p.hm_B + b) * p.hm_G + r) * p.hm_L + pos) * p.hm_D + d;
  }
  return (int64_t)row * p.ldc + col;
}

// Epilogue of one CW-column block for the 128 rows of a tile, through a TMA store.  The 4 warps of a half-group (128
// threads, thread = accumulator row) convert their row to the output type, write it into a 128-row staging tile in the
// TMA swizzle pattern (16-byte chunk index XOR row bits -> conflict-free st.shared.v4), and one thread issues
// cp.async.bulk.tensor (global <- shared), which clips at the M / N edges.  ~2 instructions per output element instead of
// ~28 for the register/shared transpose with per-row address arithmetic, so 8 epilogue warps keep up with the MMA.
template <typename OutT, int CW>
__device__ __forceinline__ void epilogue_tma_block(const GemmArgs& p, const CUtensorMap* tm_c, uint32_t taddr, uint32_t stage_addr,
                                                   int tile_row0, int col0, int r, int grp, bool issuer) {
  constexpr int kRowBytes = CW * (int)sizeof(OutT);     // 64 or 128
  constexpr int kChunks = kRowBytes / 16;
  constexpr int kWordsRow = kRowBytes / 4;
  if (issuer) bulk_wait_read0();                        // the previous store out of this staging tile has been read
  named_bar_sync(1 + grp, 128);
  uint32_t packed[kWordsRow];
  const bool full = (col0 + CW <= p.N);
  const bool bias_vec = p.bias != nullptr && full && ((reinterpret_cast<uintptr_t>(p.bias + col0) & 15) == 0);
#pragma unroll
  for (int part = 0; part < CW / 32; ++part) {
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
      if constexpr (sizeof(OutT) == 2) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
          packed[part * 16 + g8 * 4 + j] = *reinterpret_cast<uint32_t*>(&h);
        }
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) packed[part * 32 + g8 * 8 + j] = __float_as_uint(v[j]);
      }
    }
  }
  if (p.hm_D == 0 && col0 + CW > p.tma_cols && p.dbg != 1 && p.dbg != 5) {
    // the row's last partial 16-byte chunk: past the map's columns (a TMA store would write the whole chunk, beyond N)
    const int row = tile_row0 + r;
    if (row < p.M) {
      OutT* dst = reinterpret_cast<OutT*>(p.C) + (int64_t)row * p.ldc + col0;
#pragma unroll
      for (int j = 0; j < CW; ++j) {
        if (col0 + j >= p.tma_cols && col0 + j < p.N) {
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
  const int sw = (kRowBytes == 128) ? (r & 7) : ((r >> 1) & 3);
  const uint32_t row_addr = stage_addr + r * kRowBytes;
  if (p.dbg == 5) {                                     // measurement: keep the math alive without touching shared memory
    uint32_t x = 0;
#pragma unroll
    for (int c = 0; c < kWordsRow; ++c) x ^= packed[c];
    if (x == 0x12345678u) st_shared_v4(row_addr, x, x, x, x);
  } else {
#pragma unroll
    for (int c = 0; c < kChunks; ++c)
      st_shared_v4(row_addr + ((c ^ sw) << 4), packed[4 * c], packed[4 * c + 1], packed[4 * c + 2], packed[4 * c + 3]);
  }
  if (p.dbg != 5) fence_proxy_async();                  // generic-proxy writes -> visible to the async (TMA) proxy
  named_bar_sync(1 + grp, 128);
  if (issuer && p.dbg != 1 && p.dbg != 5) {
    if (p.hm_D > 0) {
      // head-major scatter: column block = one (layer, k|v, head); the M tiles of this mode never straddle two images
      // (hm_tpi tiles per image, rows past hm_L are clipped by the store - TMA stores reject negative coordinates)
      const int g = col0 / p.hm_D, layer = g / p.hm_G, rr = g - layer * p.hm_G;
      const int m_blk = tile_row0 / BM;
      const int b = m_blk / p.hm_tpi, pos0 = (m_blk - b * p.hm_tpi) * BM;
      tma_store_3d(tm_c, stage_addr, col0 - g * p.hm_D, pos0, (layer * p.hm_B + b) * p.hm_G + rr);
    } else {
      tma_store_2d(tm_c, stage_addr, col0, tile_row0);
    }
    bulk_commit();
  }
}

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_arrive_release() { asm volatile("barrier.cluster.arrive.release;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait_acquire() { asm volatile("barrier.cluster.wait.acquire;" ::: "memory"); }
__device__ __forceinline__ uint32_t map_to_cta(uint32_t local_saddr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_saddr), "r"(rank));
  return r;
}
__device__ __forceinline__ void st_cluster_f32x2(uint32_t addr, float a, float b) {
  asm volatile("st.shared::cluster.v2.f32 [%0], {%1, %2};" ::"r"(addr), "f"(a), "f"(b) : "memory");
}
// 32 lanes x 16 consecutive 32-bit columns, no wait (several loads are issued back to back, then one tcgen05.wait::ld)
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }


// ---- host side: cached CUtensorMap descriptors (defined in gemm_tc.cu; gemm_tc_init() must have run) ------------------------
// 2-D bf16 operand [rows, cols] with row stride ld (elements); box = 64 columns x box_rows rows, 128-byte swizzle.
const CUtensorMap& get_map(const void* ptr, int64_t rows, int64_t cols, int64_t ld, int box_rows);
// Operand viewed as [K/64 chunks][rows][64]: one box = 64 elements x box_rows rows x `chunks` consecutive k-chunks.
const CUtensorMap& get_map_k3(const void* ptr, int64_t rows, int64_t cols, int64_t ld, int box_rows, int chunks);
// Output map for the TMA-store epilogue: [M, N] row-major with box = box_cols x 128 rows (N: GemmArgs::tma_cols).
const CUtensorMap& get_map_c(const void* ptr, int64_t rows, int64_t cols, int64_t ld, int esz, int box_cols);

// Head-major mode (cross-attention K/V prefill, GemmArgs::hm_*): activations viewed as [B][L][K] (box = 64 k x 128 positions of one
// image, rows past L zero-filled) and the output [layers*B*G][L][D] (box = box_cols x 128 positions of one (layer-image, group)).
const CUtensorMap& get_map_a3(const void* ptr, int64_t K, int L, int B, int64_t ld);
const CUtensorMap& get_map_hm3(const void* ptr, int D, int L, int64_t LBG, int box_cols);
// GemmArgs::tma_cols: N rounded down to whole 16-byte chunks of esz-byte elements.
inline int tma_store_cols(int N, int esz) { return N - N % (16 / esz); }

// CTA-pair kernel (gemm_tc2.cu).  pick_pair_bn: the pair tile width the selection rule picks for this problem, or 0 (large M, see its
// definition; env GSTVD_GEMM_2CTA=0 disables it, =128 / =256 force a width wherever the kernel applies).  launch_gemm_tc2 launches the
// bn-column pair kernel with the TMA-store epilogue on arguments gemm_tc_variant has accepted.
int pick_pair_bn(const GemmArgs& a);
void launch_gemm_tc2(const GemmArgs& a, int bn, int num_sms, cudaStream_t stream);

}  // namespace tc
}  // namespace gstvd
