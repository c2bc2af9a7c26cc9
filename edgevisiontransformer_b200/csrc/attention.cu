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
// Longer sequences (257 .. EVT_ATTN_MAX_TOKENS) run attention_long_kernel below; attention_launch picks by S.  Head size 80
// runs attention_long_kernel<80> at every S.
#include <cuda_bf16.h>

#include <math_constants.h>

#include "common.h"
#include "ops.h"
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

__device__ __forceinline__ float max3(float a, float b, float c) {
  float d;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}

// 2^t for t <= 0 on the FMA / ALU pipes (no MUFU): t = n + f with n = round(t) taken from the low mantissa bits of
// t + 1.5 * 2^23 and f in [-0.5, 0.5]; 2^f by a degree-3 minimax polynomial (relative error 7.5e-5, far below the bf16
// rounding of P) and n added into the exponent field.  Used for one element pair in four: the exponential phase of the
// two softmax groups is MUFU-bound whenever they overlap (ncu: mio-throttle stalls on MUFU.EX2), the FMA pipe is idle.
__device__ __forceinline__ void ex2_poly_pair(float t0, float t1, float& p0, float& p1) {
  const uint64_t tt = ptx::pk2(fmaxf(t0, -126.f), fmaxf(t1, -126.f));
  const uint64_t r = ptx::add2(tt, ptx::pk2(12582912.f, 12582912.f));
  const uint64_t f = ptx::add2(tt, ptx::fma2(r, ptx::pk2(-1.f, -1.f), ptx::pk2(12582912.f, 12582912.f)));  // t - n
  uint64_t q = ptx::fma2(f, ptx::pk2(0.0551716685f, 0.0551716685f), ptx::pk2(0.2426111251f, 0.2426111251f));
  q = ptx::fma2(q, f, ptx::pk2(0.6932609677f, 0.6932609677f));
  q = ptx::fma2(q, f, ptx::pk2(0.9999280572f, 0.9999280572f));
  float q0, q1, r0, r1;
  ptx::upk2(q, q0, q1);
  ptx::upk2(r, r0, r1);
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
    ptx::upk2(ptx::fma2(ptx::pk2(__uint_as_float(r[j]), __uint_as_float(r[j + 1])), scale2, negm2), t0, t1);
    float p0, p1;
    if (((j >> 1) & 3) >= 4 - kPolyPairs) {
      ex2_poly_pair(t0, t1, p0, p1);
    } else {
      p0 = ptx::ex2_approx(t0);
      p1 = ptx::ex2_approx(t1);
    }
    if (MASKED) {
      if (j >= nvalid) p0 = 0.f;
      if (j + 1 >= nvalid) p1 = 0.f;
    }
    sum2[(j >> 1) & 1] = ptx::add2(sum2[(j >> 1) & 1], ptx::pk2(p0, p1));
    pk[j >> 1] = ptx::pack_bf16x2(p0, p1);
  }
}

// One query row per thread: row maximum, exponentials, bf16 P written over the consumed S columns of the slot at t_row,
// f32 row sum returned (the caller issues tcgen05.wait::st).  n16 = score chunks of 16 columns, last_valid = valid columns
// in the last one.
__device__ __forceinline__ float softmax_row(uint32_t t_row, int n16, int last_valid, float scale_log2e) {
  const uint64_t scale2 = ptx::pk2(scale_log2e, scale_log2e);
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
    const uint64_t negm2 = ptx::pk2(nm, nm);
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
    ptx::upk2(sum2[0], s0, s1);
    ptx::upk2(sum2[1], s2, s3);
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

// ------------------------------------------------------------------------------------------------------------
// The skeleton attention2_kernel and attention_long_kernel share: shared memory, prologue, context epilogue, teardown.

// Shared memory: the K/V ring, 2 Q tiles (one per softmax group), 8 context staging tiles, 2 x kMaxKV + 12 mbarriers and the
// TMEM address.
struct AttnSmem {
  uint8_t* kv_ring;
  uint8_t* q_ring;
  uint8_t* staging;
  uint64_t* kv_full;    // [kMaxKV] producer -> issuers
  uint64_t* kv_empty;   // [kMaxKV] PV issuer (commit) -> producer
  uint64_t* q_full;     // [2] producer -> QK issuer
  uint64_t* q_empty;    // [2] QK issuer (commit) -> producer
  uint64_t* s_ready;    // [2] QK issuer (commit) -> softmax group
  uint64_t* p_ready;    // [2] softmax group (4 warps) -> PV issuer
  uint64_t* pv_done;    // [2] PV issuer (commit) -> softmax group (O complete; long kernel: also QK issuer, P read)
  uint64_t* slot_free;  // [2] softmax group (4 warps, O read out) -> QK issuer
  uint32_t* tmem_ptr;
};
__device__ __forceinline__ AttnSmem attn_smem(uint8_t* smem_raw, int kv_ring_bytes, int q_tile_bytes = kQTileBytes) {
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  AttnSmem m;
  m.kv_ring = smem;
  m.q_ring = smem + kv_ring_bytes;
  m.staging = m.q_ring + 2 * q_tile_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(m.staging + kSoftmaxWarps * kStgWarpBytes);
  m.kv_full = bars;
  m.kv_empty = bars + kMaxKV;
  m.q_full = bars + 2 * kMaxKV;
  m.q_empty = m.q_full + 2;
  m.s_ready = m.q_empty + 2;
  m.p_ready = m.s_ready + 2;
  m.pv_done = m.p_ready + 2;
  m.slot_free = m.pv_done + 2;
  m.tmem_ptr = reinterpret_cast<uint32_t*>(m.slot_free + 2);
  return m;
}

// Tensor-map prefetch, barrier init (kv_empty completes after kv_empty_count commits), TMEM allocation (2 slots), PDL.
// Returns the TMEM base; the previous kernel's output (qkv) is complete from here on.
__device__ __forceinline__ uint32_t attn_prologue(int warp, const AttnSmem& sm, const CUtensorMap* tmQ, const CUtensorMap* tmKV,
                                                  const CUtensorMap* tmO, uint32_t kv_empty_count) {
  if (warp == kProdWarp && ptx::elect_one()) {
    ptx::prefetch_tmap(tmQ);
    ptx::prefetch_tmap(tmKV);
    ptx::prefetch_tmap(tmO);
    for (int s = 0; s < kMaxKV; ++s) {
      ptx::mbar_init(&sm.kv_full[s], 1);
      ptx::mbar_init(&sm.kv_empty[s], kv_empty_count);
    }
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&sm.q_full[s], 1);
      ptx::mbar_init(&sm.q_empty[s], 1);
      ptx::mbar_init(&sm.s_ready[s], 1);
      ptx::mbar_init(&sm.p_ready[s], 4);
      ptx::mbar_init(&sm.pv_done[s], 1);
      ptx::mbar_init(&sm.slot_free[s], 4);
    }
    ptx::fence_mbar_init();
  }
  if (warp == kQKWarp) ptx::tmem_alloc<2 * kSlotCols>(sm.tmem_ptr);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *sm.tmem_ptr;
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();
  return tmem_base;
}

// Context of one query tile, run by each softmax warp once its P is handed over: wait for O = P V (pv_done, phase), read the
// warp's 32 rows of O (TMEM lane row t_row), release the slot (slot_free), then O * hm / sum -> bf16, row per thread, into
// the warp's 128B-swizzled staging tile (16-byte piece i of row r at piece i ^ (r & 7)) and a 3-D TMA store of the tile at
// (col, row, img); rows past the end of the tensor map are clipped.  A warp with no live row only takes part in the barriers.
// HD = 80: O columns 64..79 go straight from registers to `tail` (this thread's row, 32 bytes; null for a row past Sq).
template <int HD = 64>
__device__ __forceinline__ void store_context(float sum, float hm, bool warp_live, uint64_t* pv_done, uint32_t phase,
                                              uint64_t* slot_free, uint32_t t_row, uint8_t* stg, const CUtensorMap* tmO, int col,
                                              int row, int img, __nv_bfloat16* tail = nullptr) {
  static_assert(HD == 64 || HD == 80, "head size 64 or 80");
  const int lane = threadIdx.x & 31;
  const float inv = ptx::rcp_approx(sum) * hm;  // sum >= 1 (the maximum contributes 2^0)
  if (warp_live && ptx::elect_one()) ptx::bulk_wait_read<0>();  // the previous context tile has left the staging buffer
  ptx::mbar_wait(pv_done, phase);
  ptx::tc_fence_after();
  if constexpr (HD == 80) {  // columns 64..79 first, so that they are never live beside the other 64
    if (warp_live) {
      uint32_t o2[16];
      ptx::tmem_ld_x16(t_row + kOCol + 64, o2);
      ptx::tmem_ld_wait();
      if (tail != nullptr) {
        uint32_t w[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) w[j] = ptx::pack_bf16x2(__uint_as_float(o2[2 * j]) * inv, __uint_as_float(o2[2 * j + 1]) * inv);
        reinterpret_cast<uint4*>(tail)[0] = make_uint4(w[0], w[1], w[2], w[3]);
        reinterpret_cast<uint4*>(tail)[1] = make_uint4(w[4], w[5], w[6], w[7]);
      }
    }
  }
  uint32_t o0[32], o1[32];
  if (warp_live) {
    ptx::tmem_ld_x32(t_row + kOCol, o0);
    ptx::tmem_ld_x32(t_row + kOCol + 32, o1);
    ptx::tmem_ld_wait();
  }
  ptx::tc_fence_before();
  __syncwarp();
  if (lane == 0) ptx::mbar_arrive(slot_free);  // the slot can take the next S while we convert and store
  if (!warp_live) return;
  uint8_t* stg_row = stg + lane * 128;
  const int sw = lane & 7;
#pragma unroll
  for (int half = 0; half < 2; ++half) {
#pragma unroll
    for (int jj = 0; jj < 32; jj += 8) {
      const uint32_t* r = half == 0 ? &o0[jj] : &o1[jj];
      const uint32_t x = ptx::pack_bf16x2(__uint_as_float(r[0]) * inv, __uint_as_float(r[1]) * inv);
      const uint32_t y = ptx::pack_bf16x2(__uint_as_float(r[2]) * inv, __uint_as_float(r[3]) * inv);
      const uint32_t z = ptx::pack_bf16x2(__uint_as_float(r[4]) * inv, __uint_as_float(r[5]) * inv);
      const uint32_t w = ptx::pack_bf16x2(__uint_as_float(r[6]) * inv, __uint_as_float(r[7]) * inv);
      const int piece = half * 4 + (jj >> 3);
      ptx::sts_u4(ptx::smem_u32(stg_row) + ((piece ^ sw) << 4), x, y, z, w);  // explicit STS (a C++ store here is generic)
    }
  }
  ptx::fence_proxy_async_smem();
  __syncwarp();
  if (ptx::elect_one()) {
    ptx::tma_store_3d(tmO, stg, col, row, img);
    ptx::bulk_commit();
  }
}

__device__ __forceinline__ void attn_teardown(int warp, uint32_t tmem_base) {
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == kQKWarp) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<2 * kSlotCols>(tmem_base);
  }
}

__global__ void __launch_bounds__(kThreads2, 1)
attention2_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmKV,
                  const __grid_constant__ CUtensorMap tmO, const Attn2Params p) {
  extern __shared__ uint8_t smem_raw[];
  const int kv_bytes = p.SK * 128;
  const AttnSmem sm = attn_smem(smem_raw, p.n_kv * 2 * kv_bytes);  // ring: n_kv x (K | V)
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int a = p.heads * kHD;
  const int total_units = p.B * p.heads * (p.q_tiles / p.n_mt);
  const int my_units = (total_units - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);
  const int n_items = my_units * p.n_mt;
  const uint32_t tmem_base = attn_prologue(warp, sm, &tmQ, &tmKV, &tmO, p.n_mt);  // n_mt commits release K and V of a unit

  if (warp == kProdWarp) {
    // ------------------------------------------------------------ TMA producer
    if (ptx::elect_one()) {
      int kst = 0;
      uint32_t kph = 0;
      int j = 0;
      for (int ql = 0; ql < my_units; ++ql) {
        const Unit u = unit_of(p, ql);
        const int row0 = u.b * p.S;
        ptx::mbar_wait(&sm.kv_empty[kst], kph ^ 1);
        uint8_t* sK = sm.kv_ring + kst * 2 * kv_bytes;
        ptx::mbar_arrive_expect_tx(&sm.kv_full[kst], 2 * kv_bytes);
        ptx::tma_load_2d(sK, &tmKV, &sm.kv_full[kst], a + u.h * kHD, row0);
        ptx::tma_load_2d(sK + kv_bytes, &tmKV, &sm.kv_full[kst], 2 * a + u.h * kHD, row0);
        for (int s = 0; s < p.n_mt; ++s, ++j) {
          const int g = j & 1;
          ptx::mbar_wait(&sm.q_empty[g], ((j >> 1) & 1) ^ 1);
          ptx::mbar_arrive_expect_tx(&sm.q_full[g], kQTileBytes);
          const int mt = tile_of(p, u, ql, s);
#pragma unroll
          for (int q = 0; q < 4; ++q)  // rows past the end of the image (and whole empty blocks) arrive as zeros
            ptx::tma_load_3d(sm.q_ring + g * kQTileBytes + q * kStgWarpBytes, &tmQ, &sm.q_full[g], u.h * kHD, 32 * block_of(mt, q, ql & 3), u.b);
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
        ptx::mbar_wait(&sm.kv_full[kst], kph);
        const uint64_t kd = ptx::smem_desc_sw128(ptx::smem_u32(sm.kv_ring + kst * 2 * kv_bytes));
        for (int s = 0; s < p.n_mt; ++s, ++j) {
          const int g = j & 1;
          const uint32_t ph = (j >> 1) & 1;
          ptx::mbar_wait(&sm.q_full[g], ph);
          ptx::mbar_wait(&sm.slot_free[g], ph ^ 1);
          ptx::tc_fence_after();
          const uint64_t qd = ptx::smem_desc_sw128(ptx::smem_u32(sm.q_ring + g * kQTileBytes));
          const uint32_t slot = tmem_base + g * kSlotCols;
#pragma unroll
          for (int k = 0; k < kHD / 16; ++k) ptx::mma_f16_ss(slot, qd + 2 * k, kd + 2 * k, idesc_qk, k != 0 ? 1u : 0u);
          ptx::mma_commit(&sm.s_ready[g]);
          ptx::mma_commit(&sm.q_empty[g]);  // the Q tile can be replaced as soon as these MMAs have read it
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
        ptx::mbar_wait(&sm.kv_full[kst], kph);  // complete long ago (S of this unit exists); taken for the memory ordering
        const uint64_t vd = ptx::smem_desc_sw128(ptx::smem_u32(sm.kv_ring + kst * 2 * kv_bytes + kv_bytes));
        for (int s = 0; s < p.n_mt; ++s, ++j) {
          const int g = j & 1;
          ptx::mbar_wait(&sm.p_ready[g], (j >> 1) & 1);
          ptx::tc_fence_after();
          const uint32_t slot = tmem_base + g * kSlotCols;
          // P from TMEM (8 columns per K = 16), V MN-major (2048 B per step)
          for (int k = 0; k < nk; ++k)
            ptx::mma_f16_ts(slot + kOCol, slot + 8 * k, vd + static_cast<uint64_t>(128 * k), idesc_pv, k != 0 ? 1u : 0u);
          ptx::mma_commit(&sm.pv_done[g]);
          ptx::mma_commit(&sm.kv_empty[kst]);  // n_mt arrivals release K and V of the unit
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
    uint8_t* stg = sm.staging + warp * kStgWarpBytes;
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
      ptx::mbar_wait(&sm.s_ready[grp], ph);
      ptx::tc_fence_after();
      float sum = 1.f;
      if (warp_live) {
        sum = softmax_row(t_row, n16, last_valid, p.scale_log2e);
        ptx::tmem_st_wait();
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&sm.p_ready[grp]);
      store_context(sum, hm, warp_live, &sm.pv_done[grp], ph, &sm.slot_free[grp], t_row, stg, &tmO, u.h * kHD, qrow0, u.b);
    }
    if (ptx::elect_one()) ptx::bulk_wait<0>();
  }
  attn_teardown(warp, tmem_base);
}

// ------------------------------------------------------------------------------------------------------------
// Long sequences (256 < S <= EVT_ATTN_MAX_TOKENS).  A score row of a head no longer fits in TMEM and one head's K + V no
// longer fits twice in shared memory, so every 128-row query tile runs against 128-key blocks with an online softmax.
// Same warp roles, TMEM slots and context store as attention2_kernel:
//
//   work item          (image b, head h, 128-row query tile mt), flattened with mt fastest: the tiles of one (image, head)
//                      run on neighbouring CTAs at the same time, so the K / V blocks they all re-read come from L2.  A CTA
//                      takes units of two consecutive items, one per softmax group.
//   warp 8 (1 thread)  TMA producer: each item's Q tile (four 32-row boxes, one Q buffer per group), then K and V of every
//                      128-key block of both items, interleaved group 0 / group 1, into a ring of kLongStages stages.  The
//                      3-D map clips at the image end: keys past it arrive as zeros and are masked to probability 0 (a
//                      zero key scores 0, not -inf).
//   warp 9 (1 thread)  S = Q K_blk^T (M = 128, N = 128) into columns [0, 128) of the group's slot, once O = P V of the
//                      previous block has read its P.
//   warp 10 (1 thread) O += P V_blk: P bf16 from TMEM [0, 64), O at [128, 192).
//   warps 0-3 / 4-7    softmax groups, one thread per query row.  The running maximum is lazy: a row's P, O and sum stay
//                      relative to the maximum it last used (mu) until a block's maximum exceeds mu by more than
//                      kRescaleLog2 (log2 units); only then are O and the sum multiplied by 2^(mu - mu_new).  In between
//                      P <= 2^kRescaleLog2, and O and the sum share the same stale maximum, so the quotient is exact.
//                      Every decision is per row: a row comes out the same whatever Sq is and whatever its neighbours hold.
//
// Head size 80 (attention_long_kernel<80>, every S from 1 to EVT_ATTN_MAX_TOKENS): a 160-byte bf16 row is wider than one
// 128-byte swizzle atom, so every Q tile and K / V block is two operands: columns 0..63 as before (SW128, tmQ / tmKV) and
// columns 64..79 as a 32-byte-swizzled one (SW32, tmQ32 / tmKV32).  S = Q K^T is four SW128 K-steps plus one SW32 K-step;
// O = P V is N = 64 from the SW128 V plus N = 16 from the SW32 V (both MN-major) into TMEM columns [128, 208).  A ring stage
// is 40 KB, so the ring has 3 stages instead of 4.  O columns 64..79 leave by direct 32-byte stores beside the TMA store.
constexpr int kKeyBlock = 128;
constexpr int kKeyBlockBytes = kKeyBlock * 128;  // 128 keys (or query rows) x 64 bf16: the SW128 part of a block or Q tile
constexpr int kLongStages = 4;
static_assert(kLongStages == kMaxKV, "attn_prologue initialises kMaxKV K/V stages");
constexpr float kRescaleLog2 = 8.f;

struct AttnLongParams {
  const float* head_mask;
  int S, Sq, heads;
  int n_kb;      // 128-key blocks per item
  int q_tiles;   // query tiles per (image, head)
  int n_items;   // B * heads * q_tiles
  float scale_log2e;
  __nv_bfloat16* ctx;  // head size 80: context columns 64..79 are stored through this ([B*Sq, ldc])
  long long ldc;
};
template <int HD>
struct LongShape {
  static constexpr int kStages = HD == 64 ? kLongStages : 3;
  static constexpr int kBlockBytes = kKeyBlock * HD * 2;  // one K or V block: the SW128 part, then (HD = 80) the SW32 part
  static constexpr int kQBytes = kQRows * HD * 2;
};

struct LongItem {
  int b, h, mt;
};
__device__ __forceinline__ LongItem long_item(const AttnLongParams& p, int it) {
  LongItem r;
  const int bh = it / p.q_tiles;
  r.mt = it - bh * p.q_tiles;
  r.b = bh / p.heads;
  r.h = bh - r.b * p.heads;
  return r;
}

// Item of softmax group g in unit ql of this CTA; the group-1 item of the very last unit may not exist.
__device__ __forceinline__ int item_index(int ql, int g) {
  return 2 * (static_cast<int>(blockIdx.x) + ql * static_cast<int>(gridDim.x)) + g;
}
__device__ __forceinline__ int groups_of(const AttnLongParams& p, int ql) { return item_index(ql, 1) < p.n_items ? 2 : 1; }

// One 128-key block of the online softmax for the query row at t_row (nvalid: valid keys in the block, 1..128).  mu is
// the row's current maximum times scale * log2(e), sum its running sum; both are updated, and O (TMEM columns
// [kOCol, kOCol + HD)) is rescaled with them when the maximum moves (has_o: O already holds earlier blocks).
// bf16 P is written over the consumed S columns; the caller issues tcgen05.wait::st.
template <int HD, bool MASKED>
__device__ __forceinline__ void softmax_block(uint32_t t_row, int nvalid, bool has_o, float scale_log2e, float& mu, float& sum) {
  const uint64_t scale2 = ptx::pk2(scale_log2e, scale_log2e);
  uint32_t ra[16], rb[16];
  float m[4] = {-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F};
  ptx::tmem_ld_x16(t_row, ra);
#pragma unroll 1
  for (int c = 0; c < kKeyBlock / 16; c += 2) {
    ptx::tmem_ld_wait();
    ptx::tmem_ld_x16(t_row + (c + 1) * 16, rb);
    chunk_max<16, MASKED>(ra, nvalid - c * 16, m);
    ptx::tmem_ld_wait();
    if (c + 2 < kKeyBlock / 16) ptx::tmem_ld_x16(t_row + (c + 2) * 16, ra);
    chunk_max<16, MASKED>(rb, nvalid - (c + 1) * 16, m);
  }
  const float bm = fmaxf(fmaxf(m[0], m[1]), fmaxf(m[2], m[3])) * scale_log2e;
  const bool grow = bm > mu + kRescaleLog2;  // always on the first block (mu = -inf)
  float alpha = 1.f;
  if (grow) {
    alpha = ptx::ex2_approx(mu - bm);  // 0 on the first block
    mu = bm;
    sum *= alpha;
  }
  if (has_o && __any_sync(0xffffffffu, grow)) {
    if constexpr (HD % 32 != 0) {  // O columns [64, 80)
      ptx::tmem_ld_x16(t_row + kOCol + HD - 16, ra);
      ptx::tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 16; ++j) ra[j] = __float_as_uint(__uint_as_float(ra[j]) * alpha);
      ptx::tmem_st_x16(t_row + kOCol + HD - 16, ra);
    }
#pragma unroll
    for (int c = 0; c + 1 < HD / 16; c += 2) {
      ptx::tmem_ld_x16(t_row + kOCol + c * 16, ra);
      ptx::tmem_ld_x16(t_row + kOCol + (c + 1) * 16, rb);
      ptx::tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        ra[j] = __float_as_uint(__uint_as_float(ra[j]) * alpha);
        rb[j] = __float_as_uint(__uint_as_float(rb[j]) * alpha);
      }
      ptx::tmem_st_x16(t_row + kOCol + c * 16, ra);
      ptx::tmem_st_x16(t_row + kOCol + (c + 1) * 16, rb);
    }
  }
  const uint64_t negm2 = ptx::pk2(-mu, -mu);
  uint64_t sum2[2] = {0ull, 0ull};
  uint32_t pk[8];
  ptx::tmem_ld_x16(t_row, ra);
#pragma unroll 1
  for (int c = 0; c < kKeyBlock / 16; c += 2) {
    ptx::tmem_ld_wait();
    ptx::tmem_ld_x16(t_row + (c + 1) * 16, rb);
    chunk_exp<16, MASKED>(ra, nvalid - c * 16, scale2, negm2, sum2, pk);
    ptx::tmem_st_x8(t_row + c * 8, pk);
    ptx::tmem_ld_wait();
    if (c + 2 < kKeyBlock / 16) ptx::tmem_ld_x16(t_row + (c + 2) * 16, ra);
    chunk_exp<16, MASKED>(rb, nvalid - (c + 1) * 16, scale2, negm2, sum2, pk);
    ptx::tmem_st_x8(t_row + (c + 1) * 8, pk);
  }
  float s0, s1, s2, s3;
  ptx::upk2(sum2[0], s0, s1);
  ptx::upk2(sum2[1], s2, s3);
  sum += (s0 + s1) + (s2 + s3);
}

template <int HD>
__global__ void __launch_bounds__(kThreads2, 1)
attention_long_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmKV,
                      const __grid_constant__ CUtensorMap tmO, const AttnLongParams p, const __grid_constant__ CUtensorMap tmQ32,
                      const __grid_constant__ CUtensorMap tmKV32) {
  using LS = LongShape<HD>;
  extern __shared__ uint8_t smem_raw[];
  const AttnSmem sm = attn_smem(smem_raw, LS::kStages * 2 * LS::kBlockBytes, LS::kQBytes);  // ring: kStages x (K | V) blocks
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int a = p.heads * HD;
  const int n_units = (p.n_items + 1) / 2;
  const int my_units = (n_units - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);
  const uint32_t tmem_base = attn_prologue(warp, sm, &tmQ, &tmKV, &tmO, 1);

  // The three single-thread roles walk the same sequence of (unit, key block, group) stages.
  if (warp == kProdWarp) {
    // ------------------------------------------------------------ TMA producer
    if (ptx::elect_one()) {
      int t = 0;
      uint32_t kph = 0;
      for (int ql = 0; ql < my_units; ++ql) {
        const int n_g = groups_of(p, ql);
        for (int g = 0; g < n_g; ++g) {
          const LongItem it = long_item(p, item_index(ql, g));
          ptx::mbar_wait(&sm.q_empty[g], (ql & 1) ^ 1);
          ptx::mbar_arrive_expect_tx(&sm.q_full[g], LS::kQBytes);
#pragma unroll
          for (int q = 0; q < 4; ++q)  // rows past Sq arrive as zeros
            ptx::tma_load_3d(sm.q_ring + g * LS::kQBytes + q * kStgWarpBytes, &tmQ, &sm.q_full[g], it.h * HD, it.mt * kQRows + 32 * q, it.b);
          if constexpr (HD == 80)
            ptx::tma_load_3d(sm.q_ring + g * LS::kQBytes + kKeyBlockBytes, &tmQ32, &sm.q_full[g], it.h * HD + 64, it.mt * kQRows, it.b);
        }
        for (int kb = 0; kb < p.n_kb; ++kb) {
          for (int g = 0; g < n_g; ++g) {
            const LongItem it = long_item(p, item_index(ql, g));
            ptx::mbar_wait(&sm.kv_empty[t], kph ^ 1);
            uint8_t* sK = sm.kv_ring + t * 2 * LS::kBlockBytes;
            ptx::mbar_arrive_expect_tx(&sm.kv_full[t], 2 * LS::kBlockBytes);
            ptx::tma_load_3d(sK, &tmKV, &sm.kv_full[t], a + it.h * HD, kb * kKeyBlock, it.b);
            ptx::tma_load_3d(sK + LS::kBlockBytes, &tmKV, &sm.kv_full[t], 2 * a + it.h * HD, kb * kKeyBlock, it.b);
            if constexpr (HD == 80) {
              ptx::tma_load_3d(sK + kKeyBlockBytes, &tmKV32, &sm.kv_full[t], a + it.h * HD + 64, kb * kKeyBlock, it.b);
              ptx::tma_load_3d(sK + LS::kBlockBytes + kKeyBlockBytes, &tmKV32, &sm.kv_full[t], 2 * a + it.h * HD + 64, kb * kKeyBlock, it.b);
            }
            if (++t == LS::kStages) {
              t = 0;
              kph ^= 1;
            }
          }
        }
      }
    }
  } else if (warp == kQKWarp) {
    // ------------------------------------------------------------ S = Q K^T issuer
    if (ptx::elect_one()) {
      const uint32_t idesc_qk = ptx::make_idesc(kQRows, kKeyBlock, 1, 0, 0);
      int t = 0;
      uint32_t kph = 0;
      for (int ql = 0; ql < my_units; ++ql) {
        const int n_g = groups_of(p, ql);
        for (int kb = 0; kb < p.n_kb; ++kb) {
          for (int g = 0; g < n_g; ++g) {
            ptx::mbar_wait(&sm.kv_full[t], kph);
            if (kb == 0) {
              ptx::mbar_wait(&sm.q_full[g], ql & 1);
              ptx::mbar_wait(&sm.slot_free[g], (ql & 1) ^ 1);  // the previous item's O has been read out
            } else {
              ptx::mbar_wait(&sm.pv_done[g], (ql * p.n_kb + kb - 1) & 1);  // the previous block's P has been read
            }
            ptx::tc_fence_after();
            const uint64_t qd = ptx::smem_desc_sw128(ptx::smem_u32(sm.q_ring + g * LS::kQBytes));
            const uint64_t kd = ptx::smem_desc_sw128(ptx::smem_u32(sm.kv_ring + t * 2 * LS::kBlockBytes));
            const uint32_t slot = tmem_base + g * kSlotCols;
#pragma unroll
            for (int k = 0; k < 64 / 16; ++k) ptx::mma_f16_ss(slot, qd + 2 * k, kd + 2 * k, idesc_qk, k != 0 ? 1u : 0u);
            if constexpr (HD == 80)
              ptx::mma_f16_ss(slot, ptx::smem_desc_sw32(ptx::smem_u32(sm.q_ring + g * LS::kQBytes + kKeyBlockBytes)),
                              ptx::smem_desc_sw32(ptx::smem_u32(sm.kv_ring + t * 2 * LS::kBlockBytes + kKeyBlockBytes)), idesc_qk, 1u);
            ptx::mma_commit(&sm.s_ready[g]);
            if (kb == p.n_kb - 1) ptx::mma_commit(&sm.q_empty[g]);
            if (++t == LS::kStages) {
              t = 0;
              kph ^= 1;
            }
          }
        }
      }
    }
  } else if (warp == kPVWarp) {
    // ------------------------------------------------------------ O += P V issuer
    if (ptx::elect_one()) {
      const uint32_t idesc_pv = ptx::make_idesc(kQRows, 64, 1, 0, 1);
      const uint32_t idesc_pv16 = ptx::make_idesc(kQRows, 16, 1, 0, 1);
      int t = 0;
      uint32_t kph = 0;
      for (int ql = 0; ql < my_units; ++ql) {
        const int n_g = groups_of(p, ql);
        for (int kb = 0; kb < p.n_kb; ++kb) {
          for (int g = 0; g < n_g; ++g) {
            ptx::mbar_wait(&sm.kv_full[t], kph);  // complete long ago (S of this block exists); taken for the memory ordering
            ptx::mbar_wait(&sm.p_ready[g], (ql * p.n_kb + kb) & 1);
            ptx::tc_fence_after();
            const uint32_t v_addr = ptx::smem_u32(sm.kv_ring + t * 2 * LS::kBlockBytes + LS::kBlockBytes);
            const uint64_t vd = ptx::smem_desc_sw128(v_addr);
            const uint32_t slot = tmem_base + g * kSlotCols;
#pragma unroll
            for (int k = 0; k < kKeyBlock / 16; ++k) {
              ptx::mma_f16_ts(slot + kOCol, slot + 8 * k, vd + static_cast<uint64_t>(128 * k), idesc_pv, (kb | k) != 0 ? 1u : 0u);
              if constexpr (HD == 80)  // 16 keys x 32 B = 512 B per K-step
                ptx::mma_f16_ts(slot + kOCol + 64, slot + 8 * k, ptx::smem_desc_sw32(v_addr + kKeyBlockBytes) + static_cast<uint64_t>(32 * k),
                                idesc_pv16, (kb | k) != 0 ? 1u : 0u);
            }
            ptx::mma_commit(&sm.pv_done[g]);
            ptx::mma_commit(&sm.kv_empty[t]);
            if (++t == LS::kStages) {
              t = 0;
              kph ^= 1;
            }
          }
        }
      }
    }
  } else {
    // ------------------------------------------------------------ softmax groups
    const int grp = warp >> 2;
    const int quad = warp & 3;
    const uint32_t t_row = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + grp * kSlotCols;
    const int last_valid = p.S - (p.n_kb - 1) * kKeyBlock;  // valid keys in the last block (1..128)
    uint8_t* stg = sm.staging + warp * kStgWarpBytes;
#pragma unroll 1
    for (int ql = 0; ql < my_units; ++ql) {
      const int idx = item_index(ql, grp);
      if (idx >= p.n_items) break;
      const LongItem u = long_item(p, idx);
      const int qrow0 = u.mt * kQRows + quad * 32;
      const bool warp_live = qrow0 < p.Sq;  // rows past Sq (or past S in the last tile): nothing to compute
      float hm = 1.f;
      if (p.head_mask != nullptr) hm = p.head_mask[u.h];
      const int c0 = ql * p.n_kb;  // this group's block count before the item: the barrier phases below
      float mu = -CUDART_INF_F, sum = 0.f;
#pragma unroll 1
      for (int kb = 0; kb < p.n_kb; ++kb) {
        ptx::mbar_wait(&sm.s_ready[grp], (c0 + kb) & 1);
        if (kb != 0) ptx::mbar_wait(&sm.pv_done[grp], (c0 + kb - 1) & 1);  // O may be rescaled below
        ptx::tc_fence_after();
        if (warp_live) {
          if (kb != p.n_kb - 1) softmax_block<HD, false>(t_row, kKeyBlock, kb != 0, p.scale_log2e, mu, sum);
          else softmax_block<HD, true>(t_row, last_valid, kb != 0, p.scale_log2e, mu, sum);
          ptx::tmem_st_wait();
        }
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&sm.p_ready[grp]);
      }
      __nv_bfloat16* tail = nullptr;
      if constexpr (HD == 80) {
        if (qrow0 + lane < p.Sq) tail = p.ctx + (static_cast<long long>(u.b) * p.Sq + qrow0 + lane) * p.ldc + u.h * HD + 64;
      }
      store_context<HD>(sum, hm, warp_live, &sm.pv_done[grp], (c0 + p.n_kb - 1) & 1, &sm.slot_free[grp], t_row, stg, &tmO, u.h * HD,
                        qrow0, u.b, tail);
    }
    if (ptx::elect_one()) ptx::bulk_wait<0>();
  }
  attn_teardown(warp, tmem_base);
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

// S > 256 (head size 64) or any S (head size 80): attention_long_kernel.  Argument checks are the caller's.
template <int HD>
int attention_long_launch(const void* qkv, int64_t ldq, void* ctx, int64_t ldc, const float* head_mask, int B, int S, int Sq,
                          int heads, float scale, cudaStream_t stream) {
  using LS = LongShape<HD>;
  AttnLongParams q;
  q.head_mask = head_mask;
  q.S = S;
  q.Sq = Sq;
  q.heads = heads;
  q.n_kb = (S + kKeyBlock - 1) / kKeyBlock;
  q.q_tiles = (Sq + kQRows - 1) / kQRows;
  const long long n_items = static_cast<long long>(B) * heads * q.q_tiles;
  EVT_CHECK_ARG(n_items < (1ll << 30), "attention: B * heads * query tiles too large");
  q.n_items = static_cast<int>(n_items);
  q.scale_log2e = scale * 1.4426950408889634f;
  q.ctx = static_cast<__nv_bfloat16*>(ctx);
  q.ldc = ldc;
  CUtensorMap tmQ, tmKV, tmO, tmQ32, tmKV32;
  // K / V: 128-key blocks of one image (keys past S arrive as zeros); Q: the first Sq rows of every image; context packed
  int rc = make_tmap_3d_rows(&tmKV, qkv, 2, 3ull * heads * HD, static_cast<uint64_t>(S), static_cast<uint64_t>(B),
                             static_cast<uint64_t>(ldq), kKeyBlock, 64, static_cast<uint64_t>(S));
  if (rc != EVT_OK) return rc;
  rc = make_tmap_3d_rows(&tmQ, qkv, 2, 3ull * heads * HD, static_cast<uint64_t>(Sq), static_cast<uint64_t>(B),
                         static_cast<uint64_t>(ldq), 32, 64, static_cast<uint64_t>(S));
  if (rc != EVT_OK) return rc;
  rc = make_tmap_3d_rows(&tmO, ctx, 2, static_cast<uint64_t>(heads) * HD, static_cast<uint64_t>(Sq), static_cast<uint64_t>(B),
                         static_cast<uint64_t>(ldc), 32, 64);
  if (rc != EVT_OK) return rc;
  if (HD == 80) {  // the SW32 parts: head columns 64..79
    rc = make_tmap_3d_rows_sw32(&tmKV32, qkv, 3ull * heads * HD, static_cast<uint64_t>(S), static_cast<uint64_t>(B),
                                static_cast<uint64_t>(ldq), kKeyBlock, static_cast<uint64_t>(S));
    if (rc != EVT_OK) return rc;
    rc = make_tmap_3d_rows_sw32(&tmQ32, qkv, 3ull * heads * HD, static_cast<uint64_t>(Sq), static_cast<uint64_t>(B),
                                static_cast<uint64_t>(ldq), kQRows, static_cast<uint64_t>(S));
    if (rc != EVT_OK) return rc;
  } else {
    tmQ32 = tmQ;  // not read
    tmKV32 = tmKV;
  }
  const long long units = (n_items + 1) / 2;
  const int grid = units < num_sms() ? static_cast<int>(units) : num_sms();
  const int smem = 1024 + LS::kStages * 2 * LS::kBlockBytes + 2 * LS::kQBytes + kSoftmaxWarps * kStgWarpBytes +
                   (2 * kMaxKV + 12) * 8 + 16;
  EVT_TRY(opt_in_smem<attention_long_kernel<HD>>(smem));
  const bool pdl = pdl_for_work(static_cast<long long>(B) * S, static_cast<long long>(heads) * HD);
  EVT_CUDA(launch_pdl(attention_long_kernel<HD>, dim3(grid), dim3(kThreads2), smem, stream, pdl, tmQ, tmKV, tmO, q, tmQ32, tmKV32));
  EVT_LAUNCH_CHECK("attention_long_kernel");
  return EVT_OK;
}

}  // namespace

int attention_launch(const void* qkv, int64_t ldq, void* ctx, int64_t ldc, const float* head_mask, int B, int S, int Sq,
                     int heads, int head_size, float scale, cudaStream_t stream) {
  EVT_CHECK_ARG(qkv && ctx, "attention: null pointer");
  EVT_CHECK_ARG(B > 0 && S > 0 && heads > 0, "attention: B, S, heads must be positive");
  EVT_CHECK_ARG(Sq > 0 && Sq <= S, "attention: query rows must be in 1..S");
  if (head_size != kHD && head_size != 80) return fail(EVT_ERR_UNSUPPORTED, "attention: only head sizes 64 and 80 are implemented");
  if (S > EVT_ATTN_MAX_TOKENS)
    return fail(EVT_ERR_UNSUPPORTED, "attention: sequence length above " + std::to_string(EVT_ATTN_MAX_TOKENS) + " is not implemented");
  if (head_size == 80) {  // the key-blocked kernel at every S
    EVT_CHECK_ARG(ldq >= 3ll * heads * 80 && ldc >= static_cast<int64_t>(heads) * 80, "attention: leading dimension too small");
    EVT_CHECK_ARG(ldc % 8 == 0 && reinterpret_cast<uintptr_t>(ctx) % 16 == 0, "attention: ctx must be 16-byte aligned rows");
    EVT_CHECK_ARG(static_cast<int64_t>(B) * S < (1ll << 31) - 512, "attention: B*S too large");
    return attention_long_launch<80>(qkv, ldq, ctx, ldc, head_mask, B, S, Sq, heads, scale, stream);
  }
  return attention_any_length_launch(qkv, ldq, ctx, ldc, head_mask, B, S, Sq, heads, scale, stream);
}

// Nothing in attention_long_kernel depends on S beyond the B*S bound checked here: its shared and tensor memory are per
// 128-key block, its item count B * heads * ceil(Sq / 128) is checked against 2^30 by attention_long_launch, and its TMA
// coordinates (head column, row within the image, image) stay below 2^31 for any B*S that passes.  The public cap is
// EVT_ATTN_MAX_TOKENS (attention_launch); the T2T token transformer runs one head over 3136 tokens through here.
int attention_any_length_launch(const void* qkv, int64_t ldq, void* ctx, int64_t ldc, const float* head_mask, int B, int S, int Sq,
                                int heads, float scale, cudaStream_t stream) {
  EVT_CHECK_ARG(qkv && ctx, "attention: null pointer");
  EVT_CHECK_ARG(B > 0 && S > 0 && heads > 0, "attention: B, S, heads must be positive");
  EVT_CHECK_ARG(Sq > 0 && Sq <= S, "attention: query rows must be in 1..S");
  EVT_CHECK_ARG(ldq >= 3ll * heads * kHD && ldc >= static_cast<int64_t>(heads) * kHD, "attention: leading dimension too small");
  EVT_CHECK_ARG(ldc % 8 == 0 && reinterpret_cast<uintptr_t>(ctx) % 16 == 0, "attention: ctx must be 16-byte aligned rows");
  EVT_CHECK_ARG(static_cast<int64_t>(B) * S < (1ll << 31) - 512, "attention: B*S too large");
  if (S > 256) return attention_long_launch<kHD>(qkv, ldq, ctx, ldc, head_mask, B, S, Sq, heads, scale, stream);
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
