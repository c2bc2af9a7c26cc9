// Fused short-sequence attention for sm_100a: softmax(Q K^T * scale) V with all keys of one head
// resident on chip (S <= 256 tokens, head size 64).  Persistent, warp-specialised, one CTA per SM:
//
//   work unit          (image b, head h): a CTA walks the (b, h) pairs blockIdx.x, +gridDim.x, .. and both 128-row
//                      query tiles of each pair (items); small batches split the tiles of a pair across CTAs instead.
//   warp 8 (1 thread)  TMA producer: K [SKx64] and V [SKx64] once per pair into a ring of 2-4 stages, each query tile as
//                      four 32-row boxes into a 2-deep Q ring (bf16, 128B swizzle) straight out of the packed QKV matrix.
//   warp 9 (1 thread)  S = Q K^T issuer (tcgen05.mma M=128, N=SK, 4 x K=16) into one of two TMEM slots.
//   warp 10 (1 thread) O = P V issuer (A operand = P read from TMEM, B = V as an MN-major smem operand, SK/16 MMAs) --
//                      no transposes anywhere, no score tensor in HBM.
//   warps 0-3 / 4-7    softmax group 0 / 1, one per TMEM slot (items alternate between the slots, so one group's
//                      exponentials overlap the other's MMAs, O read-out and stores).  One thread per query row:
//                      row max (FMNMX3), exp2 on packed f32x2 pairs, bf16 P written back over the consumed S columns
//                      (tcgen05.st), row sum; then O * 1/sum -> bf16 context through a swizzled staging tile and a
//                      3-D TMA store.
//
// Sq <= S: only the first Sq query rows of every image are computed and stored (context [B, Sq, heads*64]); K and V are
// still all S rows, so those rows come out exactly as in the full run (Sq = 1: the cls row of the last encoder layer).
// SK = S rounded up to 16; key columns >= S are masked to probability 0, so the extra K/V rows the TMA box
// picks up (next image's tokens, or zero fill past the end of the matrix) never contribute.
// TMEM: 2 slots x 256 columns (S at [0,SK), P overlaid at [0,SK/2), O overlaid at [128,192)).
#include <cuda_bf16.h>

#include <math_constants.h>

#include "common.h"
#include "ptx.cuh"

namespace evt {
namespace {

constexpr int kHD = 64;
constexpr int kQRows = 128;
constexpr int kAttnThreads = 160;   // tf32 kernel below
constexpr int kSoftmaxWarps = 8;
constexpr int kProdWarp = 8;
constexpr int kSlotCols = 256;
constexpr int kOCol = 128;
// Of every 4 pairs of exponentials, how many run on the FMA pipe (0..4).  Measured at B = 1024, S = 197, 12 heads on one box:
// 0 -> 0.319 ms, 1 -> 0.309, 2 -> 0.318, 3 -> 0.342 (0.330 before the division-free item bookkeeping).
constexpr int kPolyPairs = 1;

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float max3(float a, float b, float c) {
  float d;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}
__device__ __forceinline__ uint64_t pk2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void upk2(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}

// 2^t for t <= 0 on the FMA / ALU pipes (no MUFU): t = n + f with n = round(t) taken from the low mantissa bits of
// t + 1.5 * 2^23 and f in [-0.5, 0.5]; 2^f by a degree-3 minimax polynomial (relative error 7.5e-5, far below the bf16
// rounding of P) and n added into the exponent field.  Used for one element pair in four: the exponential phase of the
// two softmax groups is MUFU-bound whenever they overlap (ncu: mio-throttle stalls on MUFU.EX2), the FMA pipe is idle.
__device__ __forceinline__ void ex2_poly_pair(float t0, float t1, float& p0, float& p1) {
  const uint64_t tt = pk2(fmaxf(t0, -126.f), fmaxf(t1, -126.f));
  const uint64_t r = add2(tt, pk2(12582912.f, 12582912.f));
  const uint64_t f = add2(tt, fma2(r, pk2(-1.f, -1.f), pk2(12582912.f, 12582912.f)));  // t - n
  uint64_t q = fma2(f, pk2(0.0551716685f, 0.0551716685f), pk2(0.2426111251f, 0.2426111251f));
  q = fma2(q, f, pk2(0.6932609677f, 0.6932609677f));
  q = fma2(q, f, pk2(0.9999280572f, 0.9999280572f));
  float q0, q1, r0, r1;
  upk2(q, q0, q1);
  upk2(r, r0, r1);
  p0 = __int_as_float(__float_as_int(q0) + (__float_as_int(r0) << 23));
  p1 = __int_as_float(__float_as_int(q1) + (__float_as_int(r1) << 23));
}

// Row max over W score columns held in r (columns >= nvalid ignored when MASKED).
template <int W, bool MASKED>
__device__ __forceinline__ void chunk_max(const uint32_t (&r)[W], int nvalid, float (&m)[4]) {
  if (!MASKED) {
#pragma unroll
    for (int j = 0; j < W; j += 8) {
      m[0] = max3(m[0], __uint_as_float(r[j]), __uint_as_float(r[j + 1]));
      m[1] = max3(m[1], __uint_as_float(r[j + 2]), __uint_as_float(r[j + 3]));
      m[2] = max3(m[2], __uint_as_float(r[j + 4]), __uint_as_float(r[j + 5]));
      m[3] = max3(m[3], __uint_as_float(r[j + 6]), __uint_as_float(r[j + 7]));
    }
  } else {
#pragma unroll
    for (int j = 0; j < W; ++j)
      if (j < nvalid) m[j & 3] = fmaxf(m[j & 3], __uint_as_float(r[j]));
  }
}
// p = 2^(s*scale - m*scale) for W columns -> bf16 pairs in pk[W/2], f32 sums accumulated in sum2[2] (packed pairs).
template <int W, bool MASKED>
__device__ __forceinline__ void chunk_exp(const uint32_t (&r)[W], int nvalid, uint64_t scale2, uint64_t negm2,
                                          uint64_t (&sum2)[2], uint32_t (&pk)[W / 2]) {
#pragma unroll
  for (int j = 0; j < W; j += 2) {
    float t0, t1;
    upk2(fma2(pk2(__uint_as_float(r[j]), __uint_as_float(r[j + 1])), scale2, negm2), t0, t1);
    float p0, p1;
    if (((j >> 1) & 3) >= 4 - kPolyPairs) {
      ex2_poly_pair(t0, t1, p0, p1);
    } else {
      p0 = ex2_approx(t0);
      p1 = ex2_approx(t1);
    }
    if (MASKED) {
      if (j >= nvalid) p0 = 0.f;
      if (j + 1 >= nvalid) p1 = 0.f;
    }
    sum2[(j >> 1) & 1] = add2(sum2[(j >> 1) & 1], pk2(p0, p1));
    __nv_bfloat162 hb = __floats2bfloat162_rn(p0, p1);
    pk[j >> 1] = *reinterpret_cast<uint32_t*>(&hb);
  }
}

// One query row per thread: row maximum, exponentials, bf16 P written over the consumed S columns of the slot at t_row,
// f32 row sum returned (the caller issues tcgen05.wait::st).  n16 = score chunks of 16 columns, last_valid = valid columns
// in the last one.
__device__ __forceinline__ float softmax_row(uint32_t t_row, int n16, int last_valid, float scale_log2e) {
  const uint64_t scale2 = pk2(scale_log2e, scale_log2e);
  float sum;
  {
    // Both passes walk the row in 16-column chunks, double-buffered: the next tcgen05.ld is in flight while the
    // current chunk is reduced / exponentiated.
    uint32_t ra[16], rb[16];
    // pass 1: row max
    float m[4] = {-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F};
    {
      ptx::tmem_ld_x16(t_row, ra);
      int c = 0;
#pragma unroll 1
      for (; c + 2 <= n16 - 1; c += 2) {
        ptx::tmem_ld_wait();
        ptx::tmem_ld_x16(t_row + (c + 1) * 16, rb);
        chunk_max<16, false>(ra, 16, m);
        ptx::tmem_ld_wait();
        ptx::tmem_ld_x16(t_row + (c + 2) * 16, ra);
        chunk_max<16, false>(rb, 16, m);
      }
      if (c + 1 < n16) {
        ptx::tmem_ld_wait();
        ptx::tmem_ld_x16(t_row + (c + 1) * 16, rb);
        chunk_max<16, false>(ra, 16, m);
        ptx::tmem_ld_wait();
        chunk_max<16, true>(rb, last_valid, m);
      } else {
        ptx::tmem_ld_wait();
        chunk_max<16, true>(ra, last_valid, m);
      }
    }
    const float mx = fmaxf(fmaxf(m[0], m[1]), fmaxf(m[2], m[3]));
    const float nm = -mx * scale_log2e;
    const uint64_t negm2 = pk2(nm, nm);
    // pass 2: probabilities (bf16) written over the S columns already consumed; fp32 row sum
    uint64_t sum2[2] = {0ull, 0ull};
    {
      uint32_t pk[8];
      ptx::tmem_ld_x16(t_row, ra);
      int c = 0;
#pragma unroll 1
      for (; c + 2 <= n16 - 1; c += 2) {
        ptx::tmem_ld_wait();
        ptx::tmem_ld_x16(t_row + (c + 1) * 16, rb);
        chunk_exp<16, false>(ra, 16, scale2, negm2, sum2, pk);
        ptx::tmem_st_x8(t_row + c * 8, pk);
        ptx::tmem_ld_wait();
        ptx::tmem_ld_x16(t_row + (c + 2) * 16, ra);
        chunk_exp<16, false>(rb, 16, scale2, negm2, sum2, pk);
        ptx::tmem_st_x8(t_row + (c + 1) * 8, pk);
      }
      if (c + 1 < n16) {
        ptx::tmem_ld_wait();
        ptx::tmem_ld_x16(t_row + (c + 1) * 16, rb);
        chunk_exp<16, false>(ra, 16, scale2, negm2, sum2, pk);
        ptx::tmem_st_x8(t_row + c * 8, pk);
        ptx::tmem_ld_wait();
        chunk_exp<16, true>(rb, last_valid, scale2, negm2, sum2, pk);
        ptx::tmem_st_x8(t_row + (c + 1) * 8, pk);
      } else {
        ptx::tmem_ld_wait();
        chunk_exp<16, true>(ra, last_valid, scale2, negm2, sum2, pk);
        ptx::tmem_st_x8(t_row + c * 8, pk);
      }
    }
    float s0, s1, s2, s3;
    upk2(sum2[0], s0, s1);
    upk2(sum2[1], s2, s3);
    sum = (s0 + s1) + (s2 + s3);
  }
  return sum;
}

// ------------------------------------------------------------------------------------------------------------
// Why the kernel is organised this way (a warp-sample profile of the first, single-issuer version: 56 % of the softmax
// warps' time was spent WAITING, 31 % for O = P V alone, although the tensor pipe was 25 % busy):
//   * a single issuer thread was the bottleneck: written under `lane == 0`, every tcgen05.mma was wrapped by ptxas in an
//     ELECT / R2UR.BROADCAST / BRA.U.ANY loop and the descriptor arithmetic ran on per-thread registers (~110 cycles per MMA
//     issued, 3650 per item).  The roles are chosen with elect.sync (uniform datapath, MMAs issue back to back), and
//     S = Q K^T and O = P V are issued by TWO warps, so a P that is ready never queues behind the other group's slot wait.
//   * K and V of an (image, head) pair are loaded ONCE for both query tiles (ring of n_kv pair stages, Q tiles in their
//     own 2-deep ring -- one per softmax group): 138 -> 85 KB of L2 -> SM traffic per pair.
//   * the context tile leaves through a 128B-swizzled staging tile and a 3-D TMA store (box = 32 rows of one image, rows
//     past the sequence end clipped by the tensor map) instead of 32 scattered 16-byte stores per instruction, whose
//     source registers held the warp for 13 % of its time.
//   * a query tile is assembled from four 32-row TMA boxes, one per TMEM lane quadrant, and the assignment of an image's
//     32-row blocks to quadrants ROTATES from unit to unit (quadrant q of tile t holds block 4t + ((q - r) & 3), r = unit
//     & 3).  S = 197 is 6 full blocks + one 5-row block + one empty slot: unrotated, the softmax warps of quadrants 0 and 1
//     (= SM sub-partitions 0 and 1) always had two full blocks per (image, head) while quadrant 3 had one; rotated, every
//     sub-partition gets 7 blocks per 4 units.
constexpr int kQKWarp = 9;
constexpr int kPVWarp = 10;
constexpr int kThreads2 = 32 * (kSoftmaxWarps + 3);
constexpr int kQTileBytes = kQRows * 128;
constexpr int kStgWarpBytes = 32 * 128;
constexpr int kMaxKV = 4;

struct Attn2Params {
  const float* head_mask;
  int S, SK, heads, B;
  int Sq;        // query rows per image (S, or fewer: only rows < Sq are computed and stored)
  int n_mt;      // query tiles per work unit (q_tiles, or 1 when the tiles of a pair are split across CTAs)
  int q_tiles;   // query tiles per (image, head)
  int n_kv;      // K/V ring depth
  float scale_log2e;
};

struct Unit {
  int b, h, mt0;  // mt0: the tile of a split-mode unit (else 0)
};
__device__ __forceinline__ Unit unit_of(const Attn2Params& p, int ql) {
  const int unit = blockIdx.x + ql * gridDim.x;
  Unit u;
  int pair = unit;
  u.mt0 = 0;
  if (p.n_mt != p.q_tiles) {
    pair = unit / p.q_tiles;
    u.mt0 = unit - pair * p.q_tiles;
  }
  u.b = pair / p.heads;
  u.h = pair - u.b * p.heads;
  return u;
}
// query tile of item s (0 .. n_mt-1) of unit ql: the order flips on every other unit so that both softmax groups see
// full and ragged tiles
// 32-row block of the image held by TMEM lane quadrant `quad` of query tile `mt` in unit ql (see the header comment)
__device__ __forceinline__ int block_of(int mt, int quad, int rot) { return 4 * mt + ((quad - rot) & 3); }
__device__ __forceinline__ int tile_of(const Attn2Params& p, const Unit& u, int ql, int s) {
  if (p.n_mt != p.q_tiles) return u.mt0;
  return p.n_mt == 2 ? (s ^ (ql & 1)) : s;
}

__global__ void __launch_bounds__(kThreads2, 1)
attention2_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmKV,
                  const __grid_constant__ CUtensorMap tmO, const Attn2Params p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int kv_bytes = p.SK * 128;
  uint8_t* kv_ring = smem;                                   // n_kv x (K | V)
  uint8_t* q_ring = smem + p.n_kv * 2 * kv_bytes;            // 2 x Q tile, one per softmax group
  uint8_t* staging = q_ring + 2 * kQTileBytes;               // 8 x 4 KB context staging
  uint64_t* bars = reinterpret_cast<uint64_t*>(staging + kSoftmaxWarps * kStgWarpBytes);
  uint64_t* kv_full = bars;                   // [kMaxKV] producer -> issuers
  uint64_t* kv_empty = bars + kMaxKV;         // [kMaxKV] PV issuer (n_mt commits) -> producer
  uint64_t* q_full = bars + 2 * kMaxKV;       // [2] producer -> QK issuer
  uint64_t* q_empty = q_full + 2;             // [2] QK issuer (commit) -> producer
  uint64_t* s_ready = q_empty + 2;            // [2] QK issuer (commit) -> softmax group
  uint64_t* p_ready = s_ready + 2;            // [2] softmax group (4 warps) -> PV issuer
  uint64_t* o_ready = p_ready + 2;            // [2] PV issuer (commit) -> softmax group
  uint64_t* slot_free = o_ready + 2;          // [2] softmax group (4 warps) -> QK issuer
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(slot_free + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int a = p.heads * kHD;
  const int total_units = p.B * p.heads * (p.q_tiles / p.n_mt);
  const int my_units = (total_units - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);
  const int n_items = my_units * p.n_mt;

  if (warp == kProdWarp && ptx::elect_one()) {
    ptx::prefetch_tmap(&tmQ);
    ptx::prefetch_tmap(&tmKV);
    ptx::prefetch_tmap(&tmO);
    for (int s = 0; s < kMaxKV; ++s) {
      ptx::mbar_init(&kv_full[s], 1);
      ptx::mbar_init(&kv_empty[s], p.n_mt);
    }
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&q_full[s], 1);
      ptx::mbar_init(&q_empty[s], 1);
      ptx::mbar_init(&s_ready[s], 1);
      ptx::mbar_init(&p_ready[s], 4);
      ptx::mbar_init(&o_ready[s], 1);
      ptx::mbar_init(&slot_free[s], 4);
    }
    ptx::fence_mbar_init();
  }
  if (warp == kQKWarp) ptx::tmem_alloc<512>(tmem_ptr);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();  // qkv (previous kernel's output) is complete from here on

  if (warp == kProdWarp) {
    // ------------------------------------------------------------ TMA producer
    if (ptx::elect_one()) {
      int kst = 0;
      uint32_t kph = 0;
      int j = 0;
      for (int ql = 0; ql < my_units; ++ql) {
        const Unit u = unit_of(p, ql);
        const int row0 = u.b * p.S;
        ptx::mbar_wait(&kv_empty[kst], kph ^ 1);
        uint8_t* sK = kv_ring + kst * 2 * kv_bytes;
        ptx::mbar_arrive_expect_tx(&kv_full[kst], 2 * kv_bytes);
        ptx::tma_load_2d(sK, &tmKV, &kv_full[kst], a + u.h * kHD, row0);
        ptx::tma_load_2d(sK + kv_bytes, &tmKV, &kv_full[kst], 2 * a + u.h * kHD, row0);
        for (int s = 0; s < p.n_mt; ++s, ++j) {
          const int g = j & 1;
          ptx::mbar_wait(&q_empty[g], ((j >> 1) & 1) ^ 1);
          ptx::mbar_arrive_expect_tx(&q_full[g], kQTileBytes);
          const int mt = tile_of(p, u, ql, s);
#pragma unroll
          for (int q = 0; q < 4; ++q)  // rows past the end of the image (and whole empty blocks) arrive as zeros
            ptx::tma_load_3d(q_ring + g * kQTileBytes + q * kStgWarpBytes, &tmQ, &q_full[g], u.h * kHD, 32 * block_of(mt, q, ql & 3), u.b);
        }
        if (++kst == p.n_kv) {
          kst = 0;
          kph ^= 1;
        }
      }
    }
  } else if (warp == kQKWarp) {
    // ------------------------------------------------------------ S = Q K^T issuer
    if (ptx::elect_one()) {
      const uint32_t idesc_qk = ptx::make_idesc(kQRows, p.SK, 1, 0, 0);
      int kst = 0;
      uint32_t kph = 0;
      int j = 0;
      for (int ql = 0; ql < my_units; ++ql) {
        ptx::mbar_wait(&kv_full[kst], kph);
        const uint64_t kd = ptx::smem_desc_sw128(ptx::smem_u32(kv_ring + kst * 2 * kv_bytes));
        for (int s = 0; s < p.n_mt; ++s, ++j) {
          const int g = j & 1;
          const uint32_t ph = (j >> 1) & 1;
          ptx::mbar_wait(&q_full[g], ph);
          ptx::mbar_wait(&slot_free[g], ph ^ 1);
          ptx::tc_fence_after();
          const uint64_t qd = ptx::smem_desc_sw128(ptx::smem_u32(q_ring + g * kQTileBytes));
          const uint32_t slot = tmem_base + g * kSlotCols;
#pragma unroll
          for (int k = 0; k < kHD / 16; ++k) ptx::mma_f16_ss(slot, qd + 2 * k, kd + 2 * k, idesc_qk, k != 0 ? 1u : 0u);
          ptx::mma_commit(&s_ready[g]);
          ptx::mma_commit(&q_empty[g]);  // the Q tile can be replaced as soon as these MMAs have read it
        }
        if (++kst == p.n_kv) {
          kst = 0;
          kph ^= 1;
        }
      }
    }
  } else if (warp == kPVWarp) {
    // ------------------------------------------------------------ O = P V issuer
    if (ptx::elect_one()) {
      const uint32_t idesc_pv = ptx::make_idesc(kQRows, kHD, 1, 0, 1);
      const int nk = p.SK / 16;
      int kst = 0;
      uint32_t kph = 0;
      int j = 0;
      for (int ql = 0; ql < my_units; ++ql) {
        ptx::mbar_wait(&kv_full[kst], kph);  // complete long ago (S of this unit exists); taken for the memory ordering
        const uint64_t vd = ptx::smem_desc_sw128(ptx::smem_u32(kv_ring + kst * 2 * kv_bytes + kv_bytes));
        for (int s = 0; s < p.n_mt; ++s, ++j) {
          const int g = j & 1;
          ptx::mbar_wait(&p_ready[g], (j >> 1) & 1);
          ptx::tc_fence_after();
          const uint32_t slot = tmem_base + g * kSlotCols;
          // P from TMEM (8 columns per K = 16), V MN-major (2048 B per step)
          for (int k = 0; k < nk; ++k)
            ptx::mma_f16_ts(slot + kOCol, slot + 8 * k, vd + static_cast<uint64_t>(128 * k), idesc_pv, k != 0 ? 1u : 0u);
          ptx::mma_commit(&o_ready[g]);
          ptx::mma_commit(&kv_empty[kst]);  // n_mt arrivals release K and V of the unit
        }
        if (++kst == p.n_kv) {
          kst = 0;
          kph ^= 1;
        }
      }
    }
  } else {
    // ------------------------------------------------------------ softmax groups
    const int grp = warp >> 2;
    const int quad = warp & 3;
    const uint32_t t_row = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + grp * kSlotCols;
    const int n16 = p.SK / 16;                    // 16-column score chunks; only the last one can hold masked keys
    const int last_valid = p.S - (n16 - 1) * 16;  // valid columns in it (1..16)
    uint8_t* stg = staging + warp * kStgWarpBytes;
    uint8_t* stg_row = stg + lane * 128;
    const int sw = lane & 7;
    // This group's items are j = grp, grp + 2, ...: unit ql = j / n_mt advances by dql per iteration.  (b, h) follow
    // incrementally -- two integer divisions per item were 11 % of the softmax warps' instructions in the first version.
    const int dql = p.n_mt == 2 ? 1 : 2;
    const int step_pairs = dql * static_cast<int>(gridDim.x);
    const int db = step_pairs / p.heads, dh = step_pairs - db * p.heads;
    const bool split = p.n_mt != p.q_tiles;
    int ql = p.n_mt == 2 ? 0 : grp;
    Unit u = unit_of(p, ql);
#pragma unroll 1
    for (int j = grp; j < n_items; j += 2, ql += dql) {
      const uint32_t ph = (j >> 1) & 1;
      if (j != grp) {
        if (split) {
          u = unit_of(p, ql);
        } else {
          u.h += dh;
          u.b += db;
          if (u.h >= p.heads) {
            u.h -= p.heads;
            ++u.b;
          }
        }
      }
      const int mt = tile_of(p, u, ql, p.n_mt == 2 ? grp : 0);
      const int qrow0 = 32 * block_of(mt, quad, ql & 3);
      const bool warp_live = qrow0 < p.Sq;  // block 7 (rows 224..255) when S = 197, or a block past Sq: nothing to do
      float hm = 1.f;
      if (p.head_mask != nullptr) hm = p.head_mask[u.h];
      ptx::mbar_wait(&s_ready[grp], ph);
      ptx::tc_fence_after();
      float sum = 1.f;
      if (warp_live) {
        sum = softmax_row(t_row, n16, last_valid, p.scale_log2e);
        ptx::tmem_st_wait();
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&p_ready[grp]);
      float inv;
      asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(inv) : "f"(sum));  // sum >= 1 (the max contributes 2^0)
      inv *= hm;
      if (warp_live && ptx::elect_one()) ptx::bulk_wait_read<0>();  // the previous context tile has left the staging buffer
      ptx::mbar_wait(&o_ready[grp], ph);
      ptx::tc_fence_after();
      uint32_t o0[32], o1[32];
      if (warp_live) {
        ptx::tmem_ld_x32(t_row + kOCol, o0);
        ptx::tmem_ld_x32(t_row + kOCol + 32, o1);
        ptx::tmem_ld_wait();
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&slot_free[grp]);  // the slot can take the next S while we convert and store
      if (warp_live) {
        // O / sum -> bf16, row per thread into the 128B-swizzled staging tile (16-byte piece i of row r at piece i ^ (r & 7))
#pragma unroll
        for (int half = 0; half < 2; ++half) {
#pragma unroll
          for (int jj = 0; jj < 32; jj += 8) {
            const uint32_t* r = half == 0 ? &o0[jj] : &o1[jj];
            uint4 o;
            __nv_bfloat162 t0 = __floats2bfloat162_rn(__uint_as_float(r[0]) * inv, __uint_as_float(r[1]) * inv);
            __nv_bfloat162 t1 = __floats2bfloat162_rn(__uint_as_float(r[2]) * inv, __uint_as_float(r[3]) * inv);
            __nv_bfloat162 t2 = __floats2bfloat162_rn(__uint_as_float(r[4]) * inv, __uint_as_float(r[5]) * inv);
            __nv_bfloat162 t3 = __floats2bfloat162_rn(__uint_as_float(r[6]) * inv, __uint_as_float(r[7]) * inv);
            o.x = *reinterpret_cast<uint32_t*>(&t0);
            o.y = *reinterpret_cast<uint32_t*>(&t1);
            o.z = *reinterpret_cast<uint32_t*>(&t2);
            o.w = *reinterpret_cast<uint32_t*>(&t3);
            const int piece = half * 4 + (jj >> 3);
            ptx::sts_u4(ptx::smem_u32(stg_row) + ((piece ^ sw) << 4), o.x, o.y, o.z, o.w);  // explicit STS (a C++ store here is generic)
          }
        }
        ptx::fence_proxy_async_smem();
        __syncwarp();
        if (ptx::elect_one()) {
          ptx::tma_store_3d(&tmO, stg, u.h * kHD, qrow0, u.b);  // rows >= S of the image are clipped by the tensor map
          ptx::bulk_commit();
        }
      }
    }
    if (ptx::elect_one()) ptx::bulk_wait<0>();
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == kQKWarp) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<512>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------------------------------
// tf32 accuracy mode: Q, K, V and the context are fp32 in HBM; the tensor core reads them as tf32 (kind::tf32,
// K = 8 per MMA) and accumulates in fp32.  A 64-float head row is two 128-byte swizzle atoms, so Q and K are
// loaded as two TMA boxes of 32 columns each.  V is needed as the B operand of O = P V with the KEY index
// contiguous; instead of an MN-major 32-bit descriptor the softmax warps transpose V from global memory into
// K-major 128B-swizzled atoms (64 rows of d x 32 keys) while the TMA / S = Q K^T pipeline is in flight.
// P stays fp32 and overwrites S column for column; O has its own 64 TMEM columns (512 allocated -> one CTA
// per SM; this mode serves the small-batch / 1e-3 tolerance path).  SK is S rounded up to 32 here.
constexpr int kTmemColsTf32 = 512;
constexpr int kOColTf32 = 256;

struct AttnParamsTf32 {
  const float* qkv;
  float* ctx;
  const float* head_mask;
  long long ldq, ldc;
  long long total_rows;
  int S, SK, heads;
  float scale_log2e;
};

__global__ void __launch_bounds__(kAttnThreads, 1)
attention_tf32_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                      const AttnParamsTf32 p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int k_atom = p.SK * 128;   // one 32-column atom of K
  const int n_vt = p.SK / 32;      // V^T atoms: 64 rows (d) x 32 keys, 8 KB each
  uint8_t* sQ = smem;              // 2 atoms x 128 rows x 128 B
  uint8_t* sK = sQ + 2 * kQRows * 128;
  uint8_t* sVT = sK + 2 * k_atom;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sVT + n_vt * 8192);
  uint64_t* bar_load = bars;
  uint64_t* bar_s = bars + 1;
  uint64_t* bar_p = bars + 2;
  uint64_t* bar_o = bars + 3;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int mt = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int a = p.heads * kHD;

  if (warp == 4) {
    if (lane == 0) {
      ptx::prefetch_tmap(&tmQ);
      ptx::prefetch_tmap(&tmK);
      ptx::mbar_init(bar_load, 1);
      ptx::mbar_init(bar_s, 1);
      ptx::mbar_init(bar_p, 128);
      ptx::mbar_init(bar_o, 1);
      ptx::fence_mbar_init();
    }
    __syncwarp();
    ptx::tmem_alloc<kTmemColsTf32>(tmem_ptr);
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();  // qkv (previous kernel's output) is complete from here on

  if (warp == 4) {
    if (ptx::elect_one()) {
      const int row0 = b * p.S;
      ptx::mbar_arrive_expect_tx(bar_load, 2 * kQRows * 128 + 2 * k_atom);
      for (int t = 0; t < 2; ++t) {
        ptx::tma_load_2d(sQ + t * kQRows * 128, &tmQ, bar_load, h * kHD + t * 32, row0 + mt * kQRows);
        ptx::tma_load_2d(sK + t * k_atom, &tmK, bar_load, a + h * kHD + t * 32, row0);
      }
      ptx::mbar_wait(bar_load, 0);
      ptx::tc_fence_after();
      {  // S = Q K^T : 2 atoms x 4 MMAs of K = 8
        const uint32_t idesc = ptx::make_idesc(kQRows, p.SK, 2, 0, 0);
        for (int t = 0; t < 2; ++t) {
          const uint64_t qd = ptx::smem_desc_sw128(ptx::smem_u32(sQ + t * kQRows * 128));
          const uint64_t kd = ptx::smem_desc_sw128(ptx::smem_u32(sK + t * k_atom));
#pragma unroll
          for (int k = 0; k < 4; ++k) ptx::mma_tf32_ss(tmem_base, qd + 2 * k, kd + 2 * k, idesc, (t | k) != 0 ? 1u : 0u);
        }
        ptx::mma_commit(bar_s);
      }
      ptx::mbar_wait(bar_p, 0);
      ptx::tc_fence_after();
      {  // O = P V : P (fp32 read as tf32) from TMEM, 8 columns per MMA; V^T K-major atoms of 32 keys
        const uint32_t idesc = ptx::make_idesc(kQRows, kHD, 2, 0, 0);
        for (int j = 0; j < n_vt; ++j) {
          const uint64_t vd = ptx::smem_desc_sw128(ptx::smem_u32(sVT + j * 8192));
#pragma unroll
          for (int k = 0; k < 4; ++k)
            ptx::mma_tf32_ts(tmem_base + kOColTf32, tmem_base + j * 32 + k * 8, vd + 2 * k, idesc, (j | k) != 0 ? 1u : 0u);
        }
        ptx::mma_commit(bar_o);
      }
    }
  } else {
    // ---- transpose V (keys x 64) from global into K-major swizzled atoms: thread == key
    {
      const int tid = threadIdx.x;  // 0..127
      for (int key = tid; key < p.SK; key += 128) {
        const long long grow = static_cast<long long>(b) * p.S + key;
        const bool ok = grow < p.total_rows;  // rows past the sequence end are multiplied by P = 0; just keep them finite
        const float* src = p.qkv + grow * p.ldq + 2 * a + h * kHD;
        uint8_t* atom = sVT + (key >> 5) * 8192;
        const int kc = (key & 31) >> 2, ke = (key & 3) * 4;
#pragma unroll
        for (int d4 = 0; d4 < 16; ++d4) {
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (ok) v = *reinterpret_cast<const float4*>(src + d4 * 4);
          const float e[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int d = d4 * 4 + q;
            *reinterpret_cast<float*>(atom + d * 128 + ((kc ^ (d & 7)) << 4) + ke) = ptx::round_tf32(e[q]);
          }
        }
      }
    }
    const int qrow = mt * kQRows + warp * 32 + lane;
    const uint32_t t_row = tmem_base + (static_cast<uint32_t>(warp * 32) << 16);
    const int nchunk = p.SK / 16;
    ptx::mbar_wait(bar_s, 0);
    ptx::tc_fence_after();
    float m = -CUDART_INF_F;
    for (int c = 0; c < nchunk; ++c) {
      uint32_t r[16];
      ptx::tmem_ld_x16(t_row + c * 16, r);
      ptx::tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 16; ++j)
        if (c * 16 + j < p.S) m = fmaxf(m, __uint_as_float(r[j]));
    }
    const float msl = m * p.scale_log2e;
    float sum = 0.f;
    for (int c = 0; c < nchunk; ++c) {
      uint32_t r[16];
      ptx::tmem_ld_x16(t_row + c * 16, r);
      ptx::tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        // exp2f (not the approx intrinsic): this mode is the accuracy path
        float pv = c * 16 + j < p.S ? exp2f(fmaf(__uint_as_float(r[j]), p.scale_log2e, -msl)) : 0.f;
        pv = ptx::round_tf32(pv);  // the value the tensor core will actually use (it would truncate otherwise)
        sum += pv;
        r[j] = __float_as_uint(pv);
      }
      ptx::tmem_st_x16(t_row + c * 16, r);
    }
    ptx::tmem_st_wait();
    ptx::fence_proxy_async_smem();  // V^T written with ordinary stores, read by the tensor core
    ptx::tc_fence_before();
    ptx::mbar_arrive(bar_p);
    ptx::mbar_wait(bar_o, 0);
    ptx::tc_fence_after();
    float inv = 1.0f / sum;
    if (p.head_mask != nullptr) inv *= p.head_mask[h];
    const bool valid = qrow < p.S;
    float* dst = p.ctx + (static_cast<long long>(b) * p.S + qrow) * p.ldc + h * kHD;
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      uint32_t r[32];
      ptx::tmem_ld_x32(t_row + kOColTf32 + half * 32, r);
      ptx::tmem_ld_wait();
      if (valid) {
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          *reinterpret_cast<float4*>(dst + half * 32 + j) =
              make_float4(ptx::round_tf32(__uint_as_float(r[j]) * inv), ptx::round_tf32(__uint_as_float(r[j + 1]) * inv),
                          ptx::round_tf32(__uint_as_float(r[j + 2]) * inv), ptx::round_tf32(__uint_as_float(r[j + 3]) * inv));
      }
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 4) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<kTmemColsTf32>(tmem_base);
  }
}

}  // namespace

int attention_launch(const void* qkv, int64_t ldq, void* ctx, int64_t ldc, const float* head_mask, int B, int S, int Sq,
                     int heads, int head_size, float scale, cudaStream_t stream) {
  EVT_CHECK_ARG(qkv && ctx, "attention: null pointer");
  EVT_CHECK_ARG(B > 0 && S > 0 && heads > 0, "attention: B, S, heads must be positive");
  EVT_CHECK_ARG(Sq > 0 && Sq <= S, "attention: query rows must be in 1..S");
  if (head_size != kHD) return fail(EVT_ERR_UNSUPPORTED, "attention: only head size 64 is implemented");
  if (S > 256) return fail(EVT_ERR_UNSUPPORTED, "attention: sequence length above 256 is not implemented");
  EVT_CHECK_ARG(ldq >= 3ll * heads * kHD && ldc >= static_cast<int64_t>(heads) * kHD, "attention: leading dimension too small");
  EVT_CHECK_ARG(ldc % 8 == 0 && reinterpret_cast<uintptr_t>(ctx) % 16 == 0, "attention: ctx must be 16-byte aligned rows");
  EVT_CHECK_ARG(static_cast<int64_t>(B) * S < (1ll << 31) - 512, "attention: B*S too large");
  const int SK = (S + 15) / 16 * 16;
  const uint64_t rows = static_cast<uint64_t>(B) * S;
  const int q_tiles = (Sq + kQRows - 1) / kQRows;
  const long long n_pairs = static_cast<long long>(B) * heads;
  const int n_mt = (q_tiles > 1 && n_pairs * q_tiles <= num_sms()) ? 1 : q_tiles;  // split the tiles across CTAs at small batch
  const float scale_log2e = scale * 1.4426950408889634f;
  const int max_smem = 232448;
  const long long units = n_pairs * (q_tiles / n_mt);
  const int grid = units < num_sms() ? static_cast<int>(units) : num_sms();
  const bool pdl = pdl_for_work(static_cast<long long>(B) * S, static_cast<long long>(heads) * kHD);
  CUtensorMap tmKV;
  int rc = make_tmap_2d(&tmKV, qkv, 2, rows, 3ull * heads * kHD, static_cast<uint64_t>(ldq), SK, kHD);
  if (rc != EVT_OK) return rc;
  CUtensorMap tmO, tmQ;
  // Q: the first Sq rows of every image (rows past them arrive as zeros); context: Sq rows per image, packed
  rc = make_tmap_3d_rows(&tmQ, qkv, 2, 3ull * heads * kHD, static_cast<uint64_t>(Sq), static_cast<uint64_t>(B),
                         static_cast<uint64_t>(ldq), 32, kHD, static_cast<uint64_t>(S));
  if (rc != EVT_OK) return rc;
  rc = make_tmap_3d_rows(&tmO, ctx, 2, static_cast<uint64_t>(heads) * kHD, static_cast<uint64_t>(Sq), static_cast<uint64_t>(B),
                         static_cast<uint64_t>(ldc), 32, kHD);
  if (rc != EVT_OK) return rc;
  Attn2Params q;
  q.head_mask = head_mask;
  q.S = S;
  q.Sq = Sq;
  q.SK = SK;
  q.heads = heads;
  q.B = B;
  q.n_mt = n_mt;
  q.q_tiles = q_tiles;
  q.scale_log2e = scale_log2e;
  const int fixed = 1024 + 2 * kQTileBytes + kSoftmaxWarps * kStgWarpBytes + (2 * kMaxKV + 12) * 8 + 16;
  int n_kv = (max_smem - fixed) / (2 * SK * 128);
  if (n_kv > kMaxKV) n_kv = kMaxKV;
  if (n_kv < 2) return fail(EVT_ERR_UNSUPPORTED, "attention: sequence too long for two K/V stages");
  q.n_kv = n_kv;
  const int smem2 = fixed + n_kv * 2 * SK * 128;
  EVT_TRY(opt_in_smem<attention2_kernel>(max_smem));
  EVT_CUDA(launch_pdl(attention2_kernel, dim3(grid), dim3(kThreads2), smem2, stream, pdl, tmQ, tmKV, tmO, q));
  EVT_LAUNCH_CHECK("attention2_kernel");
  return EVT_OK;
}

int attention_tf32_launch(const float* qkv, int64_t ldq, float* ctx, int64_t ldc, const float* head_mask, int B, int S,
                          int heads, int head_size, float scale, cudaStream_t stream) {
  EVT_CHECK_ARG(qkv && ctx, "attention_tf32: null pointer");
  EVT_CHECK_ARG(B > 0 && S > 0 && heads > 0, "attention_tf32: B, S, heads must be positive");
  if (head_size != kHD) return fail(EVT_ERR_UNSUPPORTED, "attention_tf32: only head size 64 is implemented");
  if (S > 256) return fail(EVT_ERR_UNSUPPORTED, "attention_tf32: sequence length above 256 is not implemented");
  EVT_CHECK_ARG(ldq >= 3ll * heads * kHD && ldc >= static_cast<int64_t>(heads) * kHD, "attention_tf32: leading dimension too small");
  EVT_CHECK_ARG(ldc % 4 == 0 && reinterpret_cast<uintptr_t>(ctx) % 16 == 0, "attention_tf32: ctx must be 16-byte aligned rows");
  EVT_CHECK_ARG(ldq % 4 == 0 && reinterpret_cast<uintptr_t>(qkv) % 16 == 0, "attention_tf32: qkv must be 16-byte aligned rows");
  const int SK = (S + 31) / 32 * 32;
  CUtensorMap tmQ, tmKV;
  const uint64_t rows = static_cast<uint64_t>(B) * S;
  int rc = make_tmap_2d(&tmQ, qkv, 4, rows, 3ull * heads * kHD, static_cast<uint64_t>(ldq), kQRows, 32);
  if (rc != EVT_OK) return rc;
  rc = make_tmap_2d(&tmKV, qkv, 4, rows, 3ull * heads * kHD, static_cast<uint64_t>(ldq), SK, 32);
  if (rc != EVT_OK) return rc;
  AttnParamsTf32 p;
  p.qkv = qkv;
  p.ldq = ldq;
  p.total_rows = static_cast<long long>(rows);
  p.ctx = ctx;
  p.head_mask = head_mask;
  p.ldc = ldc;
  p.S = S;
  p.SK = SK;
  p.heads = heads;
  p.scale_log2e = scale * 1.4426950408889634f;
  const int smem = 1024 + 2 * kQRows * 128 + 2 * SK * 128 + (SK / 32) * 8192 + 64;
  EVT_TRY(opt_in_smem<attention_tf32_kernel>(1024 + 2 * kQRows * 128 + 2 * 256 * 128 + 8 * 8192 + 64));
  dim3 grid((S + kQRows - 1) / kQRows, heads, B);
  EVT_CUDA(launch_pdl(attention_tf32_kernel, grid, dim3(kAttnThreads), smem, stream, pdl_for_work(static_cast<long long>(B) * S, static_cast<long long>(heads) * kHD), tmQ, tmKV, p));
  EVT_LAUNCH_CHECK("attention_tf32_kernel");
  return EVT_OK;
}

}  // namespace evt

extern "C" int evt_attention_fwd(const void* qkv, int64_t ldq, void* ctx, int64_t ldc, const float* head_mask, int B,
                                 int S, int heads, int head_size, float scale, evt_stream stream) {
  int rc = evt_device_check();
  if (rc != EVT_OK) return rc;
  return evt::attention_launch(qkv, ldq, ctx, ldc, head_mask, B, S, S, heads, head_size, scale,
                               static_cast<cudaStream_t>(stream));
}

// Only the first Sq query rows of every image (all S keys): ctx is [B*Sq, ldc].
extern "C" int evt_attention_query_rows_fwd(const void* qkv, int64_t ldq, void* ctx, int64_t ldc, const float* head_mask,
                                            int B, int S, int Sq, int heads, int head_size, float scale, evt_stream stream) {
  int rc = evt_device_check();
  if (rc != EVT_OK) return rc;
  return evt::attention_launch(qkv, ldq, ctx, ldc, head_mask, B, S, Sq, heads, head_size, scale,
                               static_cast<cudaStream_t>(stream));
}

// tf32 accuracy mode: qkv and ctx are f32.
extern "C" int evt_attention_fwd_tf32(const float* qkv, int64_t ldq, float* ctx, int64_t ldc, const float* head_mask,
                                      int B, int S, int heads, int head_size, float scale, evt_stream stream) {
  int rc = evt_device_check();
  if (rc != EVT_OK) return rc;
  return evt::attention_tf32_launch(qkv, ldq, ctx, ldc, head_mask, B, S, heads, head_size, scale,
                                    static_cast<cudaStream_t>(stream));
}
