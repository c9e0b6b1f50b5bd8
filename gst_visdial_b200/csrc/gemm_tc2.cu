// CTA-pair tcgen05 GEMM (cta_group::2): 256 x BN tiles computed by two SMs of one TPC.  Default for the large-M throughput problems
// (pick_pair_bn below); parity: tests/test_gpu_ops.py::test_linear_pair_bf16 and the model-level pair-GEMM tests.
#include <algorithm>
#include <cstdlib>
#include <stdexcept>
#include <string>

#include "gemm_tc.cuh"

namespace gstvd {

using namespace tc;

namespace {

// ------------------------------------------------------------------------------------------------------------
// CTA-pair GEMM (tcgen05 cta_group::2) for the throughput problems (encoder / prefill / teacher-forced passes, M >= 1024).
//
// Why: with one CTA per 128 x 256 tile every SM pulls 48 KB of operands per 64-wide k-block (512 tensor-pipe cycles): 96 B / cycle
// against the ~45-64 B / cycle one SM ingests (the decode GEMMs' main loops run at 86 GB/s per CTA whatever the grid size,
// profiles/r2_gemm_phases.txt).  A CTA pair (two SMs of one TPC, cluster of 2) computes a 256 x BN tile with ONE tcgen05.mma.cta_group::2
// per k-step issued by the leader: each CTA stages its own 128 rows of A and only HALF of the W tile (BN/2 rows) - the tensor
// cores read the other half from the peer's shared memory - so the per-SM operand traffic drops to 32 KB per k-block (-33 %)
// for the same math.
//
// Protocol (follows the published CUTLASS sm100 2-SM pipeline):
//   * both CTAs run a TMA producer (warp 0): cp.async.bulk.tensor ... .cta_group::2 with the mbarrier address' peer bit cleared,
//     so the bytes of BOTH CTAs complete on the LEADER's full barrier; only the leader's producer arms it (expect_tx = 2 x stage);
//   * the leader's warp 1 issues the MMAs; tcgen05.commit ... multicast::cluster (mask 0b11) releases the ring slot in both CTAs
//     and, after the last k-block, signals both CTAs' accumulator-full barriers;
//   * each CTA's 16 epilogue warps drain their own 128 accumulator rows (bias / GELU / convert / TMA store, shared with the
//     single-CTA kernel) and arrive on the leader's accumulator-empty barrier (remote mbarrier.arrive for the follower);
//   * TMEM is allocated / freed with the cta_group::2 forms by warp 1 of both CTAs.
// Measured (profiles/r2_gemm_pair_vs_single.txt): +2 ... +8 % over the single-CTA kernel from M = 12 288 on, slower below.
template <int BN> struct Tile2Cfg {
  static constexpr int kBMc = BM;                               // rows per CTA; the pair tile has 2 * BM rows
  static constexpr int kBH = BN / 2;                            // W rows staged by each CTA
  static constexpr int kStages = BN == 256 ? 6 : 8;
  static constexpr int kABytes = kBMc * BK * 2;
  static constexpr int kBBytes = kBH * BK * 2;
  static constexpr int kTmemCols = 2 * BN;                      // two accumulator stages
  static constexpr int kBarBytes = 256;
  static constexpr int kStageWords = 32 * 33;
  static constexpr int kStagingBytes = 8 * kStageWords * 4;
  static constexpr int kSmemBytes = kStages * (kABytes + kBBytes) + kBarBytes + kStagingBytes + 1024;
  static constexpr int kThreads = (2 + kEpiWarpsWide) * 32;
  static_assert(BN == 128 || BN == 256, "pair tile width");
  static_assert(kSmemBytes <= 232448, "shared memory budget");
  static_assert(8 * (2 * kStages + 4) + 4 <= kBarBytes, "barrier block");
};

constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;                  // shared::cluster address of the same offset in the even CTA of a pair

__device__ __forceinline__ void tma2_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t leader_bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(leader_bar)
      : "memory");
}
__device__ __forceinline__ void tma2_load_3d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, uint32_t leader_bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(c2), "r"(leader_bar)
      : "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_alloc2(uint32_t smem_dst) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "n"(COLS) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(COLS) : "memory");
}
__device__ __forceinline__ void umma2_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
  const uint32_t z = 0u;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc), "r"(z)
      : "memory");
}
__device__ __forceinline__ void umma2_commit_mc(uint32_t bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"(cta_mask) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cta(uint32_t bar, uint32_t cta_rank) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}"
      ::"r"(bar), "r"(cta_rank) : "memory");
}

template <int BN>
__global__ void __launch_bounds__((2 + kEpiWarpsWide) * 32, 1)
gemm_tc2_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
                const __grid_constant__ CUtensorMap tm_c, const GemmArgs p) {
  using Cfg = Tile2Cfg<BN>;
  constexpr int kStages = Cfg::kStages;
  constexpr int EW = kEpiWarpsWide;
  constexpr int kGroups = EW / 4;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  const uint32_t a_base = base;
  const uint32_t b_base = base + kStages * Cfg::kABytes;
  const uint32_t stage_base = b_base + kStages * Cfg::kBBytes;
  const uint32_t bar_base = stage_base + Cfg::kStagingBytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kStages + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * kStages + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * kStages + 2 + s); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * kStages + 4);
  uint8_t* smem_gen = smem_raw + (base - raw);
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - base));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();              // 0 = leader (issues the MMAs), 1 = follower
  const bool leader = rank == 0;
  const int pair = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;
  const int tiles_n = (p.N + BN - 1) / BN;
  // 128-row units: CTA `rank` of pair tile m_blk works on unit 2 * m_blk + rank.  In the head-major (prefill) mode a unit never
  // straddles two images (hm_tpi units per image, the rows past hm_L are zero-filled on load and clipped on store).
  const int units = p.hm_tpi > 0 ? p.hm_B * p.hm_tpi : (p.M + BM - 1) / BM;
  const int tiles_m = (units + 1) / 2;
  const int num_tiles = tiles_m * tiles_n;
  const int num_kb = (p.K + BK - 1) / BK;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_a);
    tma_prefetch_desc(&tm_b);
    tma_prefetch_desc(&tm_c);
    for (int s = 0; s < kStages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(tfull_bar(s), 1); mbar_init(tempty_bar(s), 2 * EW * 32); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc2<Cfg::kTmemCols>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  // the barriers of both CTAs are initialised (and both halves of the TMEM allocation exist) before either CTA signals the other
  cluster_arrive_release();
  cluster_wait_acquire();

  if (warp == 0) {
    // ---------------- TMA producer (both CTAs) ----------------
    if (lane == 0) {
      pdl_launch_dependents();
      int stage = 0; uint32_t phase = 0;
      bool first = true;
      constexpr uint32_t kPairStageBytes = 2u * (Cfg::kABytes + Cfg::kBBytes);
      auto load_b = [&](int st, int kb, int n_blk) {
        tma2_load_2d(b_base + st * Cfg::kBBytes, &tm_b, kb * BK, n_blk * BN + (int)rank * Cfg::kBH, full_bar(st) & kPeerBitMask);
      };
      auto load_a = [&](int st, int kb, int m_blk) {
        const int u = m_blk * 2 + (int)rank;
        if (p.hm_tpi > 0) {
          const int img = u / p.hm_tpi;                   // a unit past the last image is out of bounds in the third coordinate: zeros
          tma2_load_3d(a_base + st * Cfg::kABytes, &tm_a, kb * BK, (u - img * p.hm_tpi) * BM, img, full_bar(st) & kPeerBitMask);
        } else {
          tma2_load_2d(a_base + st * Cfg::kABytes, &tm_a, kb * BK, u * BM, full_bar(st) & kPeerBitMask);
        }
      };
      for (int tile = pair; tile < num_tiles; tile += num_pairs) {
        const int m_blk = tile / tiles_n, n_blk = tile - m_blk * tiles_n;
        int kb0 = 0;
        if (first) {
          first = false;
          const int pre = num_kb < kStages ? num_kb : kStages;
          for (int st = 0; st < pre; ++st) {
            if (leader) mbar_arrive_expect_tx(full_bar(st), kPairStageBytes);
            load_b(st, st, n_blk);
          }
          pdl_wait();
          for (int st = 0; st < pre; ++st) load_a(st, st, m_blk);
          kb0 = pre;
          if (pre == kStages) { stage = 0; phase = 1u; } else { stage = pre; }
        }
        for (int kb = kb0; kb < num_kb; ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1u);      // own ring slot released (multicast commit of the leader's MMAs)
          if (leader) mbar_arrive_expect_tx(full_bar(stage), kPairStageBytes);
          load_a(stage, kb, m_blk);
          load_b(stage, kb, n_blk);
          if (++stage == kStages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ---------------- MMA issuer (leader CTA only) ----------------
    if (lane == 0 && leader) {
      constexpr uint32_t idesc = make_idesc(2 * BM, BN);
      int stage = 0; uint32_t phase = 0; int iter = 0;
      for (int tile = pair; tile < num_tiles; tile += num_pairs, ++iter) {
        const int as = iter & 1; const uint32_t aphase = (iter >> 1) & 1;
        mbar_wait(tempty_bar(as), aphase ^ 1u);         // both CTAs' epilogues have drained this accumulator stage
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(full_bar(stage), phase);            // the bytes of BOTH CTAs have landed
          tc_fence_after();
          const uint64_t a_desc = make_smem_desc(a_base + stage * Cfg::kABytes);
          const uint64_t b_desc = make_smem_desc(b_base + stage * Cfg::kBBytes);
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) umma2_f16(d_tmem, a_desc + 2u * k, b_desc + 2u * k, idesc, (kb | k) != 0 ? 1u : 0u);
          umma2_commit_mc(empty_bar(stage), 3);         // frees the slot in both CTAs when these MMAs retire
          if (kb == num_kb - 1) umma2_commit_mc(tfull_bar(as), 3);
          if (++stage == kStages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else {
    // ---------------- epilogue (both CTAs: own 128 rows of the pair tile) ----------------
    const int e = warp - 2;
    const int quad = warp & 3;
    const int grp = e >> 2;
    int iter = 0;
    for (int tile = pair; tile < num_tiles; tile += num_pairs, ++iter) {
      const int m_blk = tile / tiles_n, n_blk = tile - m_blk * tiles_n;
      const int as = iter & 1; const uint32_t aphase = (iter >> 1) & 1;
      if (p.bias != nullptr && lane == 0) {
        const int c0 = n_blk * BN + (e & 7) * (BN / 8);
        if (c0 < p.N) asm volatile("prefetch.global.L1 [%0];" ::"l"(p.bias + c0));
      }
      mbar_wait(tfull_bar(as), aphase);
      tc_fence_after();
      const int unit = m_blk * 2 + (int)rank;
      const int tile_row0 = unit * BM;
      const int r = quad * 32 + lane;
      const bool issuer = (e & 3) == 0 && lane == 0;
      const uint32_t tq = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + as * BN;
      if (p.hm_tpi > 0 ? unit < units : tile_row0 < p.M) {   // block-uniform: the second half of the last pair tile may not exist
        if (p.out_f32) {
          if (grp < 2) {
            const uint32_t stg = stage_base + grp * 16384;
            for (int j = grp; j < BN / 32; j += 2) {
              const int col0 = n_blk * BN + j * 32;
              if (col0 >= p.N) break;
              epilogue_tma_block<float, 32>(p, &tm_c, tq + j * 32, stg, tile_row0, col0, r, grp, issuer);
            }
          }
        } else {
          const uint32_t stg = stage_base + grp * 8192;
          for (int j = grp; j < BN / 32; j += kGroups) {
            const int col0 = n_blk * BN + j * 32;
            if (col0 >= p.N) break;
            epilogue_tma_block<bf16, 32>(p, &tm_c, tq + j * 32, stg, tile_row0, col0, r, grp, issuer);
          }
        }
      }
      tc_fence_before();
      mbar_arrive_cta(tempty_bar(as), 0u);              // on the leader's barrier (remote arrive for the follower)
    }
    if ((e & 3) == 0 && lane == 0) bulk_wait_read0();
  }
  tc_fence_before();
  __syncthreads();
  // neither CTA may leave while the other can still signal its barriers or read its shared memory
  cluster_arrive_release();
  cluster_wait_acquire();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc2<Cfg::kTmemCols>(tmem_base);
  }
}

template <int BN>
void launch_cfg2(const GemmArgs& a_in, int num_sms, cudaStream_t stream) {
  using Cfg = Tile2Cfg<BN>;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(gemm_tc2_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes);
    if (e != cudaSuccess) throw std::runtime_error(std::string("gemm_tc2: cudaFuncSetAttribute: ") + cudaGetErrorString(e));
    attr_set = true;
  }
  GemmArgs a = a_in;
  const int esz = a.out_f32 ? 4 : 2;
  const bool hm = a.hm_D > 0;                                 // head-major prefill mode (pick_pair_bn has checked its preconditions)
  a.tma_store = 1;
  a.hm_tpi = hm ? (a.hm_L + BM - 1) / BM : 0;
  a.tma_cols = hm ? a.N : tma_store_cols(a.N, esz);
  const CUtensorMap& ma = hm ? get_map_a3(a.A, a.K, a.hm_L, a.hm_B, a.lda) : get_map(a.A, a.M, a.K, a.lda, BM);
  const CUtensorMap& mb = get_map(a.W, a.N, a.K, a.ldw, Cfg::kBH);
  const CUtensorMap& mc = hm ? get_map_hm3(a.C, a.hm_D, a.hm_L, (int64_t)(a.N / (a.hm_D * a.hm_G)) * a.hm_B * a.hm_G, 32)
                             : get_map_c(a.C, a.M, a.tma_cols, a.ldc, esz, 32);
  const int units = hm ? a.hm_B * a.hm_tpi : (a.M + BM - 1) / BM;
  const int tiles = ((units + 1) / 2) * ((a.N + BN - 1) / BN);
  const int pairs = std::min(tiles, num_sms / 2);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * pairs); cfg.blockDim = dim3(Cfg::kThreads); cfg.dynamicSmemBytes = Cfg::kSmemBytes; cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = pdl_flag() ? 2 : 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, gemm_tc2_kernel<BN>, ma, mb, mc, a);
  if (e != cudaSuccess) throw std::runtime_error(std::string("gemm_tc2: launch failed: ") + cudaGetErrorString(e));
}

}  // namespace

namespace tc {

// CTA-pair configuration the rule picks for this problem, or 0.  Needs the plain [M, N] (or head-major) TMA-store epilogue and enough
// rows to fill pair tiles.  Selection rule from a same-box sweep over the encoder shapes (profiles/r2_gemm_pair_vs_single.txt): the
// 256-column pair tile is 2-8 % faster than the single-CTA 128 x 256 tile from M = 12 288 on (and from M = 8 192 for the wide / deep
// problems), slower below (fewer, larger tiles quantise worse); the 128-column pair tile never wins.  M >= 8 BM and N >= 128 are
// policy: the kernel itself runs any M and N (a half-empty pair tile's second CTA stores nothing, TMA zero-fills missing rows).
// env GSTVD_GEMM_2CTA: 0 = never, 128 / 256 = force that pair width wherever the kernel applies (tests), unset / 1 = the rule.
int pick_pair_bn(const GemmArgs& a) {
  const char* env = getenv("GSTVD_GEMM_2CTA");
  const int forced = env ? atoi(env) : 1;
  if (forced == 0) return 0;
  const int esz = a.out_f32 ? 4 : 2;
  if (a.M < 8 * BM || a.N < 128 || a.K % 8 != 0 || (reinterpret_cast<uintptr_t>(a.C) & 15) != 0 || getenv("GSTVD_GEMM_NO_TMA_STORE") != nullptr)
    return 0;
  if (a.fold_stats != nullptr || a.res != nullptr || a.stats_out != nullptr) return 0;   // deferred-LayerNorm epilogue: gemm_tc.cu only
  if (a.hm_D != 0) {
    if (a.out_f32 || a.hm_D % 32 != 0 || a.M != a.hm_B * a.hm_L || a.N % (a.hm_D * a.hm_G) != 0 || getenv("GSTVD_GEMM_NO_TMA_HM") != nullptr)
      return 0;
  } else if ((a.ldc * esz) % 16 != 0) {
    return 0;
  }
  if (forced == 128 || forced == 256) return forced;
  if (a.M >= 12288) return 256;
  if (a.M >= 8192 && (a.N >= 2304 || a.K >= 2048)) return 256;
  return 0;
}

void launch_gemm_tc2(const GemmArgs& a, int bn, int num_sms, cudaStream_t stream) {
  if (bn == 256) launch_cfg2<256>(a, num_sms, stream); else launch_cfg2<128>(a, num_sms, stream);
}

}  // namespace tc

}  // namespace gstvd
