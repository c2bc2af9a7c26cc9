// CTA-pair flavour of the tcgen05 GEMM (bf16 operands, TMA epilogue): two CTAs on the two SMs of one TPC form a
// cluster and compute a 256 x BN output tile with tcgen05.mma.cta_group::2.
//
//   CTA r of the pair   loads its own 128 rows of A and HALF of the W tile (rows n0 + r*BN/2 ..) -- the tensor core
//                       reads the other half out of the peer's shared memory, so every W byte crosses L2->SM once
//                       per pair and each SM's shared memory serves 8 KB instead of 12 KB per K=16 MMA step;
//   leader (rank 0)     warp 9 issues the MMAs (M = 256: accumulator rows 0..127 land in its own TMEM, rows 128..255
//                       in the peer's), commits multicast to both CTAs' `empty` / `tfull` barriers;
//   both CTAs           warp 8 = TMA producer (completion bytes are credited to the LEADER's `full` barrier),
//                       warps 0-7 = epilogue of their own 128 rows (same code as the 1-CTA kernel), arriving on the
//                       leader's `tempty` barrier when an accumulator stage has been drained.
//
// Used for the large-M encoder GEMMs; small problems stay on the 1-CTA kernel (more, smaller tiles).
#include <stdio.h>
#include <stdlib.h>

#include "gemm_common.cuh"
#include "ops.h"

namespace evt {
namespace {

using namespace gemm_detail;

// EW = epilogue warps per CTA (8, or 16 = 4 per TMEM lane quadrant with one 64-column chunk each); launch_pair chooses.
template <int BN, int EW>
struct Cfg2 {
  static constexpr int kABytes = BM * kStageRowBytes;
  static constexpr int kBBytes = (BN / 2) * kStageRowBytes;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kStagingBytes = EW * kStgBytes;
  static constexpr int kMaxStages = (232448 - 1024 - kStagingBytes - 256) / kStageBytes;
  static constexpr int kStages = kMaxStages < (BN == 128 ? 8 : 6) ? kMaxStages : (BN == 128 ? 8 : 6);
  static constexpr int kTmemCols = BN == 128 ? 256 : 512;
  static constexpr int kProducer = EW, kMma = EW + 1, kThreadsCta = 32 * (EW + 2);
  static constexpr int kBarBytes = (2 * kStages + 4) * 8 + 16;
  static constexpr int kSmemBytes = 1024 /*align slack*/ + kStages * kStageBytes + kStagingBytes + kBarBytes;
  static_assert(kSmemBytes <= 232448, "exceeds the 227 KB of shared memory a CTA can opt in to");
};

template <int BN, bool OUT_F32, int ACT, int EW>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(32 * (EW + 2), 1)
gemm_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW,
                 const __grid_constant__ CUtensorMap tmO, const GemmParams p) {
  using C = Cfg2<BN, EW>;
  constexpr int kProducerWarp = C::kProducer, kMmaWarp = C::kMma, kEpiWarps = EW;
  extern __shared__ uint8_t smem_raw[];
  // The dynamic shared window starts at the same offset in both CTAs, so the aligned carve-up below is identical in
  // the two CTAs -- required: the MMA and the multicast commits address the peer by shared-memory OFFSET.
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* stage_base = smem;
  uint8_t* staging = smem + C::kStages * C::kStageBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::kStages * C::kStageBytes + C::kStagingBytes);
  uint64_t* full = bars;                     // used in the leader only: its producer's arrive + BOTH CTAs' bytes
  uint64_t* empty = bars + C::kStages;       // per CTA: multicast commit from the leader's MMA thread
  uint64_t* tfull = bars + 2 * C::kStages;   // per CTA: multicast commit
  uint64_t* tempty = tfull + 2;              // used in the leader only: 2 x kEpiWarps arrivals
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tempty + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = ptx::cluster_ctarank();
  const int pair = blockIdx.x >> 1;
  const int num_pairs = gridDim.x >> 1;
  const int num_tiles = p.tiles_m * p.tiles_n;  // tiles_m counts 256-row blocks here

  if (warp == kProducerWarp && lane == 0) {
    ptx::prefetch_tmap(&tmA);
    ptx::prefetch_tmap(&tmW);
    ptx::prefetch_tmap(&tmO);
    for (int s = 0; s < C::kStages; ++s) {
      ptx::mbar_init(&full[s], 1);
      ptx::mbar_init(&empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&tfull[s], 1);
      ptx::mbar_init(&tempty[s], 2 * kEpiWarps);
    }
    ptx::fence_mbar_init();
  }
  if (warp == kMmaWarp) ptx::tmem_alloc_pair<C::kTmemCols>(tmem_ptr);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();  // the peer's barriers are initialised and its TMEM is allocated before anyone touches them
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  ptx::grid_dep_launch();  // the next kernel may begin its own prologue
  // Model-owned weights do not depend on the previous kernel: request the W half-tiles of the first pipeline stages before
  // the dependency wait (see gemm.cu; matters when programmatic dependent launch is on, i.e. for launches under ~100 us).
  int w_pre = 0;
  if (p.w_static && warp == kProducerWarp && pair < num_tiles) {
    const int n0 = (pair % p.tiles_n) * BN + static_cast<int>(rank) * (BN / 2);
    w_pre = min(C::kStages, p.num_kb);  // warp-uniform; consumed by the elected producer thread below
    if (ptx::elect_one()) {
      for (int i = 0; i < w_pre; ++i) {
        if (rank == 0) ptx::mbar_arrive_expect_tx(&full[i], 2 * C::kStageBytes);
        ptx::tma_load_2d_pair(stage_base + i * C::kStageBytes + C::kABytes, &tmW, ptx::mapa(&full[i], 0), i * p.k_step, n0, ptx::kEvictLast);
      }
    }
  }
  ptx::grid_dep_wait();    // operands / outputs of the previous kernel are complete from here on

  if (warp == kProducerWarp) {
    // ------------------------------------------------------------ TMA producer (both CTAs)
    // elect.sync, not `lane == 0`: ptxas keeps the single-threaded region on the uniform datapath (see gemm.cu)
    if (ptx::elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = pair; tile < num_tiles; tile += num_pairs) {
        const int m0 = (tile / p.tiles_n) * (2 * BM) + static_cast<int>(rank) * BM;
        const int n0 = (tile % p.tiles_n) * BN + static_cast<int>(rank) * (BN / 2);
        for (int kb = 0; kb < p.num_kb; ++kb) {
          uint8_t* sa = stage_base + stage * C::kStageBytes;
          uint8_t* sb = sa + C::kABytes;
          const uint32_t lead_full = ptx::mapa(&full[stage], 0);
          if (w_pre > 0) {  // first stages of the first tile: barrier armed and W already in flight
            --w_pre;
            ptx::tma_load_2d_pair(sa, &tmA, lead_full, kb * p.k_step, m0, ptx::kEvictNormal);
          } else {
            ptx::mbar_wait(&empty[stage], phase ^ 1);
            // The leader expects the bytes of both CTAs; the peer's bytes may land first (the transaction count goes
            // transiently negative, the phase cannot complete before the leader's arrive) -- no remote arrive needed.
            if (rank == 0) ptx::mbar_arrive_expect_tx(&full[stage], 2 * C::kStageBytes);
            ptx::tma_load_2d_pair(sa, &tmA, lead_full, kb * p.k_step, m0, ptx::kEvictNormal);
            ptx::tma_load_2d_pair(sb, &tmW, lead_full, kb * p.k_step, n0, ptx::kEvictLast);
          }
          if (++stage == C::kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == kMmaWarp) {
    // ------------------------------------------------------------ MMA issuer (leader CTA only)
    if (rank == 0 && ptx::elect_one()) {
      constexpr uint32_t idesc = ptx::make_idesc(2 * BM, BN, 1, 0, 0);
      int stage = 0;
      uint32_t phase = 0;
      int as = 0;
      uint32_t aphase = 0;
      for (int tile = pair; tile < num_tiles; tile += num_pairs) {
        ptx::mbar_wait(&tempty[as], aphase ^ 1);
        ptx::tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN;
        for (int kb = 0; kb < p.num_kb; ++kb) {
          ptx::mbar_wait(&full[stage], phase);
          ptx::tc_fence_after();
          const uint32_t sa = ptx::smem_u32(stage_base + stage * C::kStageBytes);
          const uint64_t adesc = ptx::smem_desc_sw128(sa);
          const uint64_t bdesc = ptx::smem_desc_sw128(sa + C::kABytes);
#pragma unroll
          for (int k = 0; k < 4; ++k)  // 4 x 32 bytes of K per stage row
            ptx::mma_f16_ss_pair(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
          ptx::mma_commit_pair(&empty[stage], 3);  // frees the slot in BOTH CTAs once these MMAs have read it
          if (++stage == C::kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
        ptx::mma_commit_pair(&tfull[as], 3);  // accumulator complete (both halves)
        if (++as == 2) {
          as = 0;
          aphase ^= 1;
        }
      }
    }
  } else {
    // ------------------------------------------------------------ epilogue warps 0..7 (both CTAs, own 128 rows)
    const int quad = warp & 3;
    uint8_t* stg = staging + warp * kStgBytes;
    int as = 0;
    uint32_t aphase = 0;
    // With a group count that does not divide the chunk count (BN = 192, bf16 out: 3 chunks of 64 columns for 2 or 4 groups)
    // the group assignment rotates from tile to tile, so every warp gets the same share of chunks over 2 (or 4) tiles.
    constexpr int kGroups = EW / 4;
    constexpr bool kRotate = ((BN / (OUT_F32 ? 32 : 64)) % kGroups) != 0;
    const int grp0 = warp >> 2;
    int rot = 0;
    for (int tile = pair; tile < num_tiles; tile += num_pairs) {
      const int m0 = (tile / p.tiles_n) * (2 * BM) + static_cast<int>(rank) * BM + quad * 32;
      const int nt0 = (tile % p.tiles_n) * BN;
      int grp = grp0;
      if (kRotate) {
        grp = grp0 + rot;
        if (grp >= kGroups) grp -= kGroups;
        if (++rot == kGroups) rot = 0;
      }
      prefetch_bias<BN, OUT_F32, EW / 4>(p, grp, lane, nt0);
      ptx::mbar_wait(&tfull[as], aphase);
      ptx::tc_fence_after();
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + as * BN;
      epilogue_tile<BN, false, OUT_F32, ACT, true, EW / 4>(p, &tmO, stg, grp, lane, m0, nt0, t_row);
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive_cluster(ptx::mapa(&tempty[as], 0));
      if (++as == 2) {
        as = 0;
        aphase ^= 1;
      }
    }
    if (ptx::elect_one()) ptx::bulk_wait<0>();
  }

  // Neither CTA may leave while the other can still reach into its shared memory / TMEM or signal its barriers.
  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();
  if (warp == kMmaWarp) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc_pair<C::kTmemCols>(tmem_base);
  }
}

template <int BN, bool OUT_F32, int ACT, int EW>
int launch_pair_ew(const void* W, int64_t ldw, const CUtensorMap& tmA, const CUtensorMap& tmO, GemmParams p, cudaStream_t stream) {
  using C = Cfg2<BN, EW>;
  constexpr int kThreads = C::kThreadsCta;
  constexpr auto kern = gemm_pair_kernel<BN, OUT_F32, ACT, EW>;
  EVT_TRY(opt_in_smem<kern>(C::kSmemBytes));
  static int pairs_dev = -1;
  static int max_pairs = 0;
  int dev = 0;
  EVT_CUDA(cudaGetDevice(&dev));
  if (pairs_dev != dev) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(num_sms() & ~1, 1, 1);
    cfg.blockDim = dim3(kThreads, 1, 1);
    cfg.dynamicSmemBytes = C::kSmemBytes;
    int n = 0;
    EVT_CUDA(cudaOccupancyMaxActiveClusters(&n, kern, &cfg));
    if (n <= 0) return fail(EVT_ERR_CUDA, "gemm: no CTA pair of this configuration fits on the device");
    max_pairs = n;
    if (getenv("EVT_DEBUG")) fprintf(stderr, "evt: gemm_pair_kernel<%d> max active clusters %d, smem %d\n", BN, n, C::kSmemBytes);
    pairs_dev = dev;
  }
  CUtensorMap tmW;
  int rc = make_tmap_2d(&tmW, W, 2, static_cast<uint64_t>(p.N), static_cast<uint64_t>(p.K), static_cast<uint64_t>(ldw), BN / 2,
                        p.k_step);
  if (rc != EVT_OK) return rc;
  p.tiles_m = (p.M + 2 * BM - 1) / (2 * BM);
  const int num_tiles = p.tiles_m * p.tiles_n;
  const int pairs = num_tiles < max_pairs ? num_tiles : max_pairs;
  EVT_CUDA(launch_pdl(kern, dim3(2 * pairs), dim3(kThreads), C::kSmemBytes, stream, pdl_for_gemm(p.M, p.N, p.K), tmA, tmW, tmO, p));
  EVT_LAUNCH_CHECK("gemm_pair_kernel");
  return EVT_OK;
}

// Epilogue warps per CTA.  With a fused activation and a SHORT K loop (K <= 384: DeiT-Tiny / -Small / T2T FC1, three to six
// k-blocks per tile) the tile time is the epilogue's, and sixteen warps (four per TMEM lane quadrant, one 64-column chunk each)
// finish it sooner: FC1 74.6 -> 68.9 us at D = 384 (batch 256), 49.1 -> 45.2 us for the pruned Tiny (batch 1024), same box.  With
// a long K loop the MMAs bound the tile and sixteen warps LOSE (DeiT-Base FC1 0.944 vs 0.912 ms in the step, 1101 vs 1248
// TFLOP/s alone: 576 threads leave 96 registers per thread, the unrolled GELU loses its interleaving, and the extra staging
// costs a pipeline stage), so eight stay there; twelve (three groups, rotating) measured equal to eight within noise.  Without
// an activation sixteen warps lose as well (QKV at D = 384: 55 vs 49 us): the plain bf16 epilogue is bound by its TMA stores,
// not by instruction latency.
template <int BN, bool OUT_F32, int ACT>
int launch_pair(const void* W, int64_t ldw, const CUtensorMap& tmA, const CUtensorMap& tmO, const GemmParams& p, cudaStream_t stream) {
  if constexpr (ACT != EVT_ACT_NONE && !OUT_F32) {
    if (p.K <= 384) return launch_pair_ew<BN, OUT_F32, ACT, 16>(W, ldw, tmA, tmO, p, stream);
    return launch_pair_ew<BN, OUT_F32, ACT, 8>(W, ldw, tmA, tmO, p, stream);
  } else {
    return launch_pair_ew<BN, OUT_F32, ACT, 8>(W, ldw, tmA, tmO, p, stream);
  }
}

template <int BN>
int dispatch_pair(const void* W, int64_t ldw, const CUtensorMap& a, const CUtensorMap& o, const GemmParams& p, bool out_f32,
                  int act, cudaStream_t s) {
  if (out_f32) {
    switch (act) {
      case EVT_ACT_NONE: return launch_pair<BN, true, EVT_ACT_NONE>(W, ldw, a, o, p, s);
      case EVT_ACT_GELU_ERF: return launch_pair<BN, true, EVT_ACT_GELU_ERF>(W, ldw, a, o, p, s);
      default: return launch_pair<BN, true, EVT_ACT_GELU_TANH>(W, ldw, a, o, p, s);
    }
  }
  switch (act) {
    case EVT_ACT_NONE: return launch_pair<BN, false, EVT_ACT_NONE>(W, ldw, a, o, p, s);
    case EVT_ACT_GELU_ERF: return launch_pair<BN, false, EVT_ACT_GELU_ERF>(W, ldw, a, o, p, s);
    default: return launch_pair<BN, false, EVT_ACT_GELU_TANH>(W, ldw, a, o, p, s);
  }
}

}  // namespace

namespace gemm_detail {

bool pair_supported(int bn) { return bn == 256 || bn == 192 || bn == 128; }

int gemm_pair_launch(int bn, const void* W, int64_t ldw, const CUtensorMap& tmA, const CUtensorMap& tmO, const GemmParams& p,
                     bool out_f32, int act, cudaStream_t stream) {
  switch (bn) {
    case 256: return dispatch_pair<256>(W, ldw, tmA, tmO, p, out_f32, act, stream);
    case 192: return dispatch_pair<192>(W, ldw, tmA, tmO, p, out_f32, act, stream);
    case 128: return dispatch_pair<128>(W, ldw, tmA, tmO, p, out_f32, act, stream);
  }
  return fail(EVT_ERR_INVALID, "gemm: no CTA-pair tile configuration");
}

}  // namespace gemm_detail
}  // namespace evt
