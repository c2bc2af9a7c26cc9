// Residual projection with the FOLLOWING LayerNorm in its epilogue, for residual streams narrow enough that a CTA pair
// keeps whole rows in tensor memory (D = 192 or 384: DeiT-Tiny / -Small, T2T-ViT; bf16 operands, tcgen05 cta_group::2):
//
//     x[M,D]  <-  x + A[M,K] . W[D,K]^T + bias          (f32 residual stream, in place)
//     xn[M,D] <-  LayerNorm(x) * gamma + beta           (bf16: the A operand of the following QKV / FC1 projection)
//
// replaces  ViTSelfOutput.dense + residual + layernorm_after  and  ViTOutput.dense + residual + the next layer's
// layernorm_before  (SITE/models/vit/modeling_vit.py:265-268, 308-312, 333-340).  `copy_ln` is the reference's TF dialect
// (modeling/models/vit.py: the skip connection carries the normalised rows): the residual stream then receives the
// unrounded f32 LayerNorm output instead of x.
//
// Why a second attempt after the first GEMM + LayerNorm epilogue fusion (removed, DESIGN.md, negative results): that kernel
// walked the N tiles of a row block one after the other and had to re-read the new residual from L2 for the normalisation pass.  Here the full row block (256 rows x D
// columns of f32) stays in TMEM (192-column accumulator slots, two of them), the old residual comes in through a TMA ring
// that a dedicated thread keeps full across row blocks, and the three epilogue passes (x' and row sums; centred squares;
// normalise) read tensor memory only.  HBM traffic per row: K*2 (A) + 4D (x in) + 4D (x out) + 2D (xn) bytes -- the LayerNorm
// kernel's 4D read is gone and the f32 add no longer round-trips through L2 atomics.
//
//   warp 0-7   epilogue: thread == row (TMEM lane), warp w%4 = lane quadrant, w/4 = which 32-column chunks (even / odd);
//              the two threads of a row combine their partial sums through shared memory + a 64-thread named barrier
//   warp 8     TMA producer of the A / W pipeline stages (both CTAs, bytes credited to the leader's barrier)
//   warp 9     MMA issuer (leader CTA): M = 256, N = 192 per accumulator slot
//   warp 10    TMA producer of the residual ring: 128 rows x 32 columns of f32 per entry; the epilogue warps update the
//              entry in place and TMA-store it back from the same shared memory
#include <stdio.h>
#include <stdlib.h>

#include "gemm_common.cuh"
#include "ops.h"

namespace evt {
namespace {

using namespace gemm_detail;

constexpr int kSlotCols = 192;             // accumulator slot = one UMMA N
constexpr int kChunksPerSlot = kSlotCols / 32;
constexpr int kResBytes = BM * 128;        // ring entry: 128 rows x 32 f32
constexpr int kXnStgBytes = 32 * 64;       // bf16 staging tile of one epilogue warp: 32 rows x 32 bf16, 64B-swizzled
constexpr int kMaxD = 384;
constexpr int kSmemLimit = 232448;

struct RowLnParams {
  const float* bias;   // [D] or null
  const float* gamma;  // [D]
  const float* beta;   // [D]
  int M, D, K;
  int num_kb, row_blocks;
  float eps, d_f;
};

// EW epilogue warps = G column groups x 4 TMEM lane quadrants.  Built with EW = 8: twelve warps (three groups, 128 registers)
// measured the same within noise at D = 192 (out-proj 75.1 vs 75.7 us, FC2 92.1 vs 91.9) and at D = 384 -- the kernel runs at
// 5.2-5.5 TB/s there, the epilogue chain is not what bounds it; sixteen leave one ring entry per group, which the deferred
// release of the in-place stores cannot work with.
template <int NT, bool COPY, int EW>
struct CfgR {
  static constexpr int G = EW / 4;
  static constexpr int kChunks = NT * kChunksPerSlot;  // 32-column chunks per row
  static_assert(EW % 4 == 0 && kChunks % G == 0, "every column group takes the same number of chunks");
  static constexpr int kABytes = BM * kStageRowBytes;
  static constexpr int kBBytes = (kSlotCols / 2) * kStageRowBytes;  // this CTA's half of one slot's W tile
  static constexpr int kStageBytes = kABytes + kBBytes;
  // NT == 1: two accumulator slots double-buffer the row blocks, the K loop is short and hidden -> two stages are enough.
  // NT == 2: one K loop per slot (the A tile is re-read from L2), so that pass 1 of slot 0 runs under the MMAs of slot 1.  A
  // single K loop feeding both slots (A read once, 40 KB stages) measured slower: out-proj 66 vs 56 us at D = 384, and so did
  // four stages with a 4-deep residual ring (57 -> 65 us).
  static constexpr int kStages = NT == 1 ? 2 : 3;
  static constexpr int kCopyBytes = COPY ? EW * kStgBytes : 0;  // f32 staging of the normalised rows (TF dialect)
  static constexpr int kVecBytes = 3 * kMaxD * 4;               // bias, gamma, beta
  static constexpr int kStatBytes = 2 * G * BM * 4;             // [sum | squares][column group][row]
  static constexpr int kFixed = 1024 + kStages * kStageBytes + kCopyBytes + kVecBytes + kStatBytes + 512 /*barriers*/;
  // Residual ring entries: chunk i lives in entry i % depth and belongs to column group i % G, so the depth must be a
  // multiple of G -- then an entry is only ever consumed by ONE group, and a consumer has seen round k-1 of an entry before
  // it waits for round k.  (A depth of 5 with two groups deadlocked: a group waiting for round 1 of an entry whose round 0 --
  // the other group's chunk -- had not landed yet passed its parity wait on the untouched barrier.)
  static constexpr int kDepthWant = G == 4 ? 8 : 6;
  static constexpr int kDepthMin = G == 3 ? 3 : 4;
  static constexpr int kResDepth = (kFixed + EW * kXnStgBytes + kDepthWant * kResBytes <= kSmemLimit) ? kDepthWant : kDepthMin;
  // (the TF-dialect variant stores the f32 rows from a single staging tile in the same bulk group: one tile there too)
  static constexpr int kXnBufs = (!COPY && kFixed + kResDepth * kResBytes + 2 * EW * kXnStgBytes <= kSmemLimit) ? 2 : 1;
  static constexpr int kXnBytes = EW * kXnStgBytes * kXnBufs;
  static_assert(kResDepth % G == 0, "ring entries must not alternate between column groups");
  static_assert(COPY || kResDepth / G >= 2, "the deferred release of an in-place store needs a second entry per group");
  static constexpr int kRingBytes = kResDepth * kResBytes;
  static constexpr int kSmemBytes = kFixed + kRingBytes + kXnBytes;
  static constexpr int kThreads = 32 * (EW + 3);
  static_assert((2 * kStages + 4 + 2 * kResDepth) * 8 + 16 <= 512, "barrier area");
  static_assert(kSmemBytes <= kSmemLimit, "exceeds the 227 KB of shared memory a CTA can opt in to");
};

__device__ __forceinline__ void tmem_st_x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
      "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),
      "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]),
      "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}

template <int NT, bool COPY, int EW>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(32 * (EW + 3), 1)
gemm_rowln_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW,
                  const __grid_constant__ CUtensorMap tmRin,   // residual, box 128 rows x 32 f32 (ring loads)
                  const __grid_constant__ CUtensorMap tmRout,  // residual, box 32 rows x 32 f32 (per-warp stores)
                  const __grid_constant__ CUtensorMap tmXn,    // xn, box 32 rows x 32 bf16, 64B swizzle
                  const RowLnParams p) {
  using C = CfgR<NT, COPY, EW>;
  constexpr int G = C::G;
  constexpr int kResDepth = C::kResDepth;
  constexpr int kProdWarp = EW, kIssueWarp = EW + 1, kResWarp = EW + 2;
  constexpr int kChunks = C::kChunks;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* stage_base = smem;
  uint8_t* ring = stage_base + C::kStages * C::kStageBytes;
  uint8_t* xn_stg = ring + C::kRingBytes;
  uint8_t* copy_stg = xn_stg + C::kXnBytes;
  float* vec = reinterpret_cast<float*>(copy_stg + C::kCopyBytes);  // bias | gamma | beta, kMaxD each
  float* stat = vec + 3 * kMaxD;
  uint64_t* bars = reinterpret_cast<uint64_t*>(stat + 2 * G * BM);
  uint64_t* full = bars;                    // leader only
  uint64_t* empty = bars + C::kStages;      // per CTA (multicast commit)
  uint64_t* tfull = bars + 2 * C::kStages;  // per CTA (multicast commit), one per accumulator slot
  uint64_t* tempty = tfull + 2;             // leader only: 2 x EW arrivals
  uint64_t* rfull = tempty + 2;             // per CTA: residual ring
  uint64_t* rempty = rfull + kResDepth;     // per CTA: 4 arrivals (the warps of the owning column group)
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(rempty + kResDepth);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = ptx::cluster_ctarank();
  const int pair = blockIdx.x >> 1;
  const int num_pairs = gridDim.x >> 1;

  if (warp == kProdWarp && lane == 0) {
    ptx::prefetch_tmap(&tmA);
    ptx::prefetch_tmap(&tmW);
    ptx::prefetch_tmap(&tmRin);
    ptx::prefetch_tmap(&tmRout);
    ptx::prefetch_tmap(&tmXn);
    for (int s = 0; s < C::kStages; ++s) {
      ptx::mbar_init(&full[s], 1);
      ptx::mbar_init(&empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&tfull[s], 1);
      ptx::mbar_init(&tempty[s], 2 * EW);
    }
    for (int s = 0; s < kResDepth; ++s) {
      ptx::mbar_init(&rfull[s], 1);
      ptx::mbar_init(&rempty[s], 4);
    }
    ptx::fence_mbar_init();
  }
  if (warp == kIssueWarp) ptx::tmem_alloc_pair<512>(tmem_ptr);
  // bias / gamma / beta are model parameters, not outputs of the previous kernel: staged before the dependency wait
  for (int i = threadIdx.x; i < p.D; i += blockDim.x) {
    vec[i] = p.bias != nullptr ? __ldg(p.bias + i) : 0.f;
    vec[kMaxD + i] = __ldg(p.gamma + i);
    vec[2 * kMaxD + i] = __ldg(p.beta + i);
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();

  if (warp == kProdWarp) {
    // ------------------------------------------------------------ A / W pipeline stages (both CTAs)
    if (ptx::elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int rb = pair; rb < p.row_blocks; rb += num_pairs) {
        const int m0 = rb * (2 * BM) + static_cast<int>(rank) * BM;
        for (int j = 0; j < NT; ++j) {
          const int n0 = j * kSlotCols + static_cast<int>(rank) * (kSlotCols / 2);
          for (int kb = 0; kb < p.num_kb; ++kb) {
            uint8_t* sa = stage_base + stage * C::kStageBytes;
            const uint32_t lead_full = ptx::mapa(&full[stage], 0);
            ptx::mbar_wait(&empty[stage], phase ^ 1);
            if (rank == 0) ptx::mbar_arrive_expect_tx(&full[stage], 2 * C::kStageBytes);
            ptx::tma_load_2d_pair(sa, &tmA, lead_full, kb * 64, m0, ptx::kEvictNormal);
            ptx::tma_load_2d_pair(sa + C::kABytes, &tmW, lead_full, kb * 64, n0, ptx::kEvictLast);
            if (++stage == C::kStages) {
              stage = 0;
              phase ^= 1;
            }
          }
        }
      }
    }
  } else if (warp == kIssueWarp) {
    // ------------------------------------------------------------ MMA issuer (leader CTA)
    if (rank == 0 && ptx::elect_one()) {
      constexpr uint32_t idesc = ptx::make_idesc(2 * BM, kSlotCols, 1, 0, 0);
      int stage = 0;
      uint32_t phase = 0;
      uint32_t sphase = 0;  // bit per accumulator slot: parity of its next `tempty` wait
      int it = 0;
      for (int rb = pair; rb < p.row_blocks; rb += num_pairs, ++it) {
        for (int j = 0; j < NT; ++j) {
          const int slot = NT == 1 ? (it & 1) : j;
          ptx::mbar_wait(&tempty[slot], ((sphase >> slot) & 1) ^ 1);
          sphase ^= 1u << slot;
          ptx::tc_fence_after();
          const uint32_t d_tmem = tmem_base + slot * kSlotCols;
          for (int kb = 0; kb < p.num_kb; ++kb) {
            ptx::mbar_wait(&full[stage], phase);
            ptx::tc_fence_after();
            const uint32_t sa = ptx::smem_u32(stage_base + stage * C::kStageBytes);
            const uint64_t adesc = ptx::smem_desc_sw128(sa);
            const uint64_t bdesc = ptx::smem_desc_sw128(sa + C::kABytes);
#pragma unroll
            for (int k = 0; k < 4; ++k)
              ptx::mma_f16_ss_pair(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
            ptx::mma_commit_pair(&empty[stage], 3);
            if (++stage == C::kStages) {
              stage = 0;
              phase ^= 1;
            }
          }
          ptx::mma_commit_pair(&tfull[slot], 3);
        }
      }
    }
  } else if (warp == kResWarp) {
    // ------------------------------------------------------------ residual ring producer (each CTA its own 128 rows)
    if (ptx::elect_one()) {
      int e = 0;
      uint32_t par = 0;
      for (int rb = pair; rb < p.row_blocks; rb += num_pairs) {
        const int m0 = rb * (2 * BM) + static_cast<int>(rank) * BM;
        for (int q = 0; q < kChunks; ++q) {
          ptx::mbar_wait(&rempty[e], par ^ 1);
          ptx::mbar_arrive_expect_tx(&rfull[e], kResBytes);
          ptx::tma_load_2d_hint(ring + e * kResBytes, &tmRin, &rfull[e], q * 32, m0, ptx::kEvictFirst);
          if (++e == kResDepth) {
            e = 0;
            par ^= 1;
          }
        }
      }
    }
  } else {
    // ------------------------------------------------------------ epilogue warps 0 .. EW-1
    const int quad = warp & 3;
    const int grp = warp >> 2;
    const int row = quad * 32 + lane;  // row of this CTA's 128 == TMEM lane
    const int sw = lane & 7;
    uint8_t* my_xn = xn_stg + warp * kXnStgBytes * C::kXnBufs;
    uint8_t* my_copy = copy_stg + warp * kStgBytes;
    int xn_sel = 0;
    // ring position of this warp's next chunk: its column group owns every G-th entry of the stream of chunks
    int re = grp;
    uint32_t rpar = 0;
    // 32-bit shared addresses: every access below is an explicit LDS / STS (see ptx.cuh)
    const uint32_t ring_a = ptx::smem_u32(ring) + row * 128;
    const uint32_t bias_a = ptx::smem_u32(vec), gamma_a = bias_a + kMaxD * 4, beta_a = bias_a + 2 * kMaxD * 4;
    const uint32_t sum_a = ptx::smem_u32(stat) + row * 4, sq_a = sum_a + G * BM * 4;
    uint32_t sphase = 0;  // bit per slot: parity of its next `tfull` wait
    int pending = -1;     // ring entry whose in-place store may still be reading shared memory
    int it = 0;
    for (int rb = pair; rb < p.row_blocks; rb += num_pairs, ++it) {
      const int m0 = rb * (2 * BM) + static_cast<int>(rank) * BM + quad * 32;  // first global row of this warp
      const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
      // ---- pass 1: x' = x + (acc + bias) -> TMEM (and, HF dialect, back to the residual stream); row sums
      float sum = 0.f;
      uint32_t seen = 0;  // slots whose accumulator this warp has already waited for in this row block
#pragma unroll 1
      for (int q = grp; q < kChunks; q += G) {
        const int slot = NT == 1 ? (it & 1) : q / kChunksPerSlot;
        if (!((seen >> slot) & 1)) {
          ptx::mbar_wait(&tfull[slot], (sphase >> slot) & 1);
          sphase ^= 1u << slot;
          seen |= 1u << slot;
          ptx::tc_fence_after();
        }
        const uint32_t taddr = t_lane + slot * kSlotCols + (q % kChunksPerSlot) * 32;
        uint32_t r[32];
        ptx::tmem_ld_x32(taddr, r);
        const int e = re;
        ptx::mbar_wait(&rfull[e], rpar);
        re += G;
        if (re >= kResDepth) {
          re -= kResDepth;
          rpar ^= 1;
        }
        const uint32_t ent = ring_a + e * kResBytes;
        float4 x[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) x[i] = ptx::lds_f4(ent + ((i ^ sw) << 4));  // all eight pieces in flight together
        ptx::tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 b = ptx::lds_f4(bias_a + (q * 8 + i) * 16);
          float4 v;
          v.x = x[i].x + (__uint_as_float(r[4 * i]) + b.x);
          v.y = x[i].y + (__uint_as_float(r[4 * i + 1]) + b.y);
          v.z = x[i].z + (__uint_as_float(r[4 * i + 2]) + b.z);
          v.w = x[i].w + (__uint_as_float(r[4 * i + 3]) + b.w);
          sum += (v.x + v.y) + (v.z + v.w);
          r[4 * i] = __float_as_uint(v.x);
          r[4 * i + 1] = __float_as_uint(v.y);
          r[4 * i + 2] = __float_as_uint(v.z);
          r[4 * i + 3] = __float_as_uint(v.w);
          if (!COPY) ptx::sts_f4(ent + ((i ^ sw) << 4), v.x, v.y, v.z, v.w);
        }
        tmem_st_x32(taddr, r);
        if (!COPY) {
          ptx::fence_proxy_async_smem();
          __syncwarp();
          if (ptx::elect_one()) {
            if (pending >= 0) {  // the previous in-place store has had a whole chunk's time to read its entry
              ptx::bulk_wait_read<0>();
              ptx::mbar_arrive(&rempty[pending]);
            }
            ptx::tma_store_2d(&tmRout, ring + e * kResBytes + quad * 32 * 128, q * 32, m0);
            ptx::bulk_commit();
          }
          pending = e;
        } else {
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&rempty[e]);
        }
      }
      ptx::tmem_st_wait();
      ptx::sts_f1(sum_a + grp * BM * 4, sum);
      named_bar_sync(1 + quad, 32 * G);
      float tot = 0.f;
#pragma unroll
      for (int g = 0; g < G; ++g) tot += ptx::lds_f1(sum_a + g * BM * 4);  // same order in every warp: identical means
      const float mean = tot / p.d_f;  // true division: exact for constant rows
      // ---- pass 2: centred squares
      float sq = 0.f;
#pragma unroll 1
      for (int q = grp; q < kChunks; q += G) {
        const int slot = NT == 1 ? (it & 1) : q / kChunksPerSlot;
        uint32_t r[32];
        ptx::tmem_ld_x32(t_lane + slot * kSlotCols + (q % kChunksPerSlot) * 32, r);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; i += 4) {
          const float a0 = __uint_as_float(r[i]) - mean, a1 = __uint_as_float(r[i + 1]) - mean;
          const float a2 = __uint_as_float(r[i + 2]) - mean, a3 = __uint_as_float(r[i + 3]) - mean;
          sq += (a0 * a0 + a1 * a1) + (a2 * a2 + a3 * a3);
        }
      }
      ptx::sts_f1(sq_a + grp * BM * 4, sq);
      if (!COPY) {
        if (pending >= 0 && ptx::elect_one()) {  // last in-place store of pass 1: its entry goes back to the ring
          ptx::bulk_wait_read<0>();
          ptx::mbar_arrive(&rempty[pending]);
        }
        pending = -1;
      }
      named_bar_sync(1 + quad, 32 * G);
      float tsq = 0.f;
#pragma unroll
      for (int g = 0; g < G; ++g) tsq += ptx::lds_f1(sq_a + g * BM * 4);
      const float rstd = rsqrtf(tsq / p.d_f + p.eps);
      // ---- pass 3: normalise -> bf16 xn (and, TF dialect, the f32 rows into the residual stream)
#pragma unroll 1
      for (int q = grp; q < kChunks; q += G) {
        const int slot = NT == 1 ? (it & 1) : q / kChunksPerSlot;
        uint32_t r[32];
        ptx::tmem_ld_x32(t_lane + slot * kSlotCols + (q % kChunksPerSlot) * 32, r);
        ptx::tmem_ld_wait();
        // last read of a slot by this warp: its accumulator columns are free for the MMAs of the next row block
        if (NT == 1 ? (q + G >= kChunks) : (q + G >= kChunks || (q + G) / kChunksPerSlot != slot)) {
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive_cluster(ptx::mapa(&tempty[slot], 0));
        }
        float y[32];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 g = ptx::lds_f4(gamma_a + (q * 8 + i) * 16);
          const float4 b = ptx::lds_f4(beta_a + (q * 8 + i) * 16);
          y[4 * i] = (__uint_as_float(r[4 * i]) - mean) * rstd * g.x + b.x;
          y[4 * i + 1] = (__uint_as_float(r[4 * i + 1]) - mean) * rstd * g.y + b.y;
          y[4 * i + 2] = (__uint_as_float(r[4 * i + 2]) - mean) * rstd * g.z + b.z;
          y[4 * i + 3] = (__uint_as_float(r[4 * i + 3]) - mean) * rstd * g.w + b.w;
        }
        // the store that last used this staging tile has finished reading it
        if (ptx::elect_one()) ptx::bulk_wait_read<C::kXnBufs - 1>();
        __syncwarp();
        // bf16: 64-byte rows, 16-byte pieces XOR-swizzled by (row >> 1) & 3 (SWIZZLE_64B)
        uint8_t* xb = my_xn + xn_sel * kXnStgBytes;
        if (++xn_sel == C::kXnBufs) xn_sel = 0;
        const uint32_t sb = ptx::smem_u32(xb) + lane * 64;
        const int sw64 = (lane >> 1) & 3;
#pragma unroll
        for (int i = 0; i < 4; ++i)
          ptx::sts_u4(sb + ((i ^ sw64) << 4), pack_bf16x2(y[8 * i], y[8 * i + 1]), pack_bf16x2(y[8 * i + 2], y[8 * i + 3]),
                      pack_bf16x2(y[8 * i + 4], y[8 * i + 5]), pack_bf16x2(y[8 * i + 6], y[8 * i + 7]));
        if (COPY) {
          const uint32_t sc = ptx::smem_u32(my_copy) + lane * 128;
#pragma unroll
          for (int i = 0; i < 8; ++i) ptx::sts_f4(sc + ((i ^ sw) << 4), y[4 * i], y[4 * i + 1], y[4 * i + 2], y[4 * i + 3]);
        }
        ptx::fence_proxy_async_smem();
        __syncwarp();
        if (ptx::elect_one()) {
          ptx::tma_store_2d(&tmXn, xb, q * 32, m0);
          if (COPY) ptx::tma_store_2d(&tmRout, my_copy, q * 32, m0);
          ptx::bulk_commit();
        }
      }
    }
    if (ptx::elect_one()) ptx::bulk_wait<0>();
  }

  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();
  if (warp == kIssueWarp) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc_pair<512>(tmem_base);
  }
}

template <int NT, bool COPY, int EW>
int launch_rowln(const CUtensorMap& tmA, const CUtensorMap& tmW, const CUtensorMap& tmRin, const CUtensorMap& tmRout,
                 const CUtensorMap& tmXn, const RowLnParams& p, cudaStream_t stream) {
  using C = CfgR<NT, COPY, EW>;
  constexpr auto kern = gemm_rowln_kernel<NT, COPY, EW>;
  EVT_TRY(opt_in_smem<kern>(C::kSmemBytes));
  static int pairs_dev = -1;
  static int max_pairs = 0;
  int dev = 0;
  EVT_CUDA(cudaGetDevice(&dev));
  if (pairs_dev != dev) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(num_sms() & ~1, 1, 1);
    cfg.blockDim = dim3(C::kThreads, 1, 1);
    cfg.dynamicSmemBytes = C::kSmemBytes;
    int n = 0;
    EVT_CUDA(cudaOccupancyMaxActiveClusters(&n, kern, &cfg));
    if (n <= 0) return fail(EVT_ERR_CUDA, "gemm+layernorm: no CTA pair of this configuration fits on the device");
    max_pairs = n;
    if (getenv("EVT_DEBUG"))
      fprintf(stderr, "evt: gemm_rowln_kernel<%d,%d,%d> smem %d ring %d xn bufs %d\n", NT, (int)COPY, EW, C::kSmemBytes, C::kResDepth, C::kXnBufs);
    pairs_dev = dev;
  }
  const int pairs = p.row_blocks < max_pairs ? p.row_blocks : max_pairs;
  EVT_CUDA(launch_pdl(kern, dim3(2 * pairs), dim3(C::kThreads), C::kSmemBytes, stream, pdl_for_gemm(p.M, p.D, p.K), tmA, tmW, tmRin,
                      tmRout, tmXn, p));
  EVT_LAUNCH_CHECK("gemm_rowln_kernel");
  return EVT_OK;
}

}  // namespace

bool gemm_rowln_supported(int64_t M, int N, int K, bool copy_ln) {
  // whole rows in two 192-column accumulator slots; enough 256-row blocks to give every CTA pair one
  (void)copy_ln;
  return (N == kSlotCols || N == 2 * kSlotCols) && K >= 1 && M < (1ll << 31) - 256 &&
         (M + 2 * BM - 1) / (2 * BM) >= num_sms() / 2;
}

// Whether the model runtime should take the fused kernel for this projection (the op-level entry point always does when the
// shape allows).  D = 384 holds a row block in BOTH accumulator slots, so the MMAs of the next block cannot run under the
// epilogue: with a long K loop (HF DeiT-Small FC2, K = 1536: 104 us against 72 + 25 for the two kernels) the fusion loses; it
// wins for the out-projection (56 against 41 + 25) and in the TF dialect, whose LayerNorm kernel also writes the f32 rows back.
bool gemm_rowln_pays(int N, int K, bool copy_ln) {
  return N == kSlotCols || copy_ln || K <= 2 * kSlotCols;
}

int gemm_rowln_launch(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias, float* resid, int64_t ldr,
                      const float* gamma, const float* beta, float eps, bool copy_ln, void* xn, int64_t ldxn, int64_t M, int N,
                      int K, cudaStream_t stream) {
  EVT_CHECK_ARG(A && W && resid && gamma && beta && xn, "gemm+layernorm: null pointer");
  EVT_CHECK_ARG(N == kSlotCols || N == 2 * kSlotCols, "gemm+layernorm: the row length must be 192 or 384");
  EVT_CHECK_ARG(M > 0 && K > 0 && M < (1ll << 31) - 256, "gemm+layernorm: bad M or K");
  EVT_CHECK_ARG(lda >= K && ldw >= K && ldr >= N && ldxn >= N, "gemm+layernorm: leading dimension smaller than the row length");
  CUtensorMap tmA, tmW, tmRin, tmRout, tmXn;
  int rc = make_tmap_2d(&tmA, A, 2, static_cast<uint64_t>(M), static_cast<uint64_t>(K), static_cast<uint64_t>(lda), BM, 64);
  if (rc != EVT_OK) return rc;
  rc = make_tmap_2d(&tmW, W, 2, static_cast<uint64_t>(N), static_cast<uint64_t>(K), static_cast<uint64_t>(ldw), kSlotCols / 2, 64);
  if (rc != EVT_OK) return rc;
  rc = make_tmap_2d(&tmRin, resid, 4, static_cast<uint64_t>(M), static_cast<uint64_t>(N), static_cast<uint64_t>(ldr), BM, 32);
  if (rc != EVT_OK) return rc;
  rc = make_tmap_2d(&tmRout, resid, 4, static_cast<uint64_t>(M), static_cast<uint64_t>(N), static_cast<uint64_t>(ldr), 32, 32);
  if (rc != EVT_OK) return rc;
  rc = make_tmap_2d_sw(&tmXn, xn, 2, static_cast<uint64_t>(M), static_cast<uint64_t>(N), static_cast<uint64_t>(ldxn), 32, 32, 64);
  if (rc != EVT_OK) return rc;
  RowLnParams p;
  p.bias = bias;
  p.gamma = gamma;
  p.beta = beta;
  p.M = static_cast<int>(M);
  p.D = N;
  p.K = K;
  p.num_kb = (K + 63) / 64;
  p.row_blocks = static_cast<int>((M + 2 * BM - 1) / (2 * BM));
  p.eps = eps;
  p.d_f = static_cast<float>(N);
  const int nt = N / kSlotCols;
#define EVT_ROWLN_CASE(NTV, COPYV) \
  if (nt == NTV && copy_ln == COPYV) return launch_rowln<NTV, COPYV, 8>(tmA, tmW, tmRin, tmRout, tmXn, p, stream);
  EVT_ROWLN_CASE(1, false) EVT_ROWLN_CASE(2, false) EVT_ROWLN_CASE(1, true) EVT_ROWLN_CASE(2, true)
#undef EVT_ROWLN_CASE
  return fail(EVT_ERR_INVALID, "gemm+layernorm: no kernel configuration");
}

}  // namespace evt
