// Device code shared by the 1-CTA (gemm.cu) and 2-CTA (gemm2.cu) tcgen05 GEMM kernels: parameters, the GELU epilogue
// math, and the per-warp epilogue of one accumulator tile.
#pragma once
#include <cuda_bf16.h>

#include "common.h"
#include "ptx.cuh"

namespace evt {
namespace gemm_detail {


constexpr int BM = 128;
constexpr int kStageRowBytes = 128;  // one swizzle row: 64 bf16 or 32 tf32 of K
constexpr int kEpiWarps = 8;
constexpr int kProducerWarp = kEpiWarps;
constexpr int kMmaWarp = kEpiWarps + 1;
constexpr int kThreads = 32 * (kEpiWarps + 2);
constexpr int kStgBytes = 32 * 128;  // per epilogue warp: 32 dense 128-byte rows, 128B-swizzled

template <int BN>
struct Cfg {
  static constexpr int kABytes = BM * kStageRowBytes;
  static constexpr int kBBytes = BN * kStageRowBytes;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kStages = BN == 256 ? 4 : BN == 192 ? 4 : BN == 128 ? 6 : 8;
  static constexpr int kTmemCols = BN == 256 ? 512 : BN == 192 ? 512 : BN == 128 ? 256 : 128;
  static constexpr int kStagingBytes = kEpiWarps * kStgBytes;
  static constexpr int kBarBytes = (2 * kStages + 4) * 8 + 16;
  static constexpr int kSmemBytes = 1024 /*align slack*/ + kStages * kStageBytes + kStagingBytes + kBarBytes;
  static_assert(kSmemBytes <= 232448, "exceeds the 227 KB of shared memory a CTA can opt in to");
};

struct GemmParams {
  const float* bias;
  const float* residual;
  void* out;
  long long ldr, ldo;
  int M, N, K;
  int res_row_mod, res_row_off;
  int out_group, out_group_stride, out_group_off;
  int tiles_m, tiles_n, num_kb;
  int k_splits, kb_per_split;  // 1-CTA kernel: K range per work item (split K for reduce-add outputs at small M)
  int k_step;  // elements of K per stage (64 bf16 / 32 tf32)
  int vec_ok;  // out / residual / bias allow 16-byte vector access
  int round_tf32;  // f32 output feeds a tf32 tensor-core op: round to nearest tf32 when written
  int w_static;    // W is not written by the preceding kernel on the stream (model weights): its first tiles may be
                   // requested before griddepcontrol.wait (1-CTA kernel, latency path)
};

__device__ __forceinline__ long long map_out_row(const GemmParams& p, long long row) {
  if (p.out_group <= 0) return row;
  const long long g = row / p.out_group;
  return g * p.out_group_stride + p.out_group_off + (row - g * p.out_group);
}
// the epilogue math is written with the packed f32x2 and approximate-math primitives of ptx.cuh
using ptx::add2;
using ptx::ex2_approx;
using ptx::fma2;
using ptx::mul2;
using ptx::pack_bf16x2;
using ptx::pk2;
using ptx::rcp_approx;
using ptx::upk2;

// erf-GELU of a pair, in place.  erfc(z) = exp2(z Q(z)) on z = |x|/sqrt(2) in [0, 4] with Q a minimax fit of
// log2(erfc(z))/z (tools/fit_erfc.py; erfc(4) = 1.5e-8 is below f32 resolution of 1, so z is clamped there).  The
// polynomial is written in a = |x| (powers of 1/sqrt(2) folded into the coefficients) and the exponent carries an extra
// -1, so e = erfc/2 and   gelu(x) = x/2 (1 + sign(x)(1 - erfc)) = max(x, 0) - |x| e.
//   HI (f32 output):  degree 6, |gelu error| < 7e-7 absolute, < 7e-6 relative
//   !HI (bf16 output): degree 5, < 6e-6 absolute, < 4e-5 relative = 1 % of a bf16 ulp
// Per element: 1 MUFU (ex2), DEG + 2 FMA-pipe lane operations (packed two per instruction), 2 ALU-pipe min/max, against
// 2 MUFU + 13 FMA for the textbook A&S 7.1.26 form -- the FMA pipe is what the FC1 epilogue saturates.
template <bool HI>
__device__ __forceinline__ void gelu_erf_pair(float& x0, float& x1) {
  constexpr float kAmax = 5.65685424949238f;  // 4 sqrt(2)
  const uint64_t a = pk2(fminf(fabsf(x0), kAmax), fminf(fabsf(x1), kAmax));
  uint64_t q;
  if (HI) {
    q = fma2(a, pk2(-1.765649017e-06f, -1.765649017e-06f), pk2(6.025074981e-05f, 6.025074981e-05f));
    q = fma2(q, a, pk2(-9.201008943e-04f, -9.201008943e-04f));
    q = fma2(q, a, pk2(8.467212319e-03f, 8.467212319e-03f));
    q = fma2(q, a, pk2(-5.387612060e-02f, -5.387612060e-02f));
    q = fma2(q, a, pk2(-4.585517347e-01f, -4.585517347e-01f));
    q = fma2(q, a, pk2(-1.151212096e+00f, -1.151212096e+00f));
  } else {
    q = fma2(a, pk2(2.554092680e-05f, 2.554092680e-05f), pk2(-6.528479280e-04f, -6.528479280e-04f));
    q = fma2(q, a, pk2(7.452332415e-03f, 7.452332415e-03f));
    q = fma2(q, a, pk2(-5.191940814e-02f, -5.191940814e-02f));
    q = fma2(q, a, pk2(-4.602991641e-01f, -4.602991641e-01f));
    q = fma2(q, a, pk2(-1.150684714e+00f, -1.150684714e+00f));
  }
  float t0, t1;
  upk2(fma2(q, a, pk2(-1.0f, -1.0f)), t0, t1);
  const float e0 = ex2_approx(t0), e1 = ex2_approx(t1);
  x0 = fmaf(-fabsf(x0), e0, fmaxf(x0, 0.0f));
  x1 = fmaf(-fabsf(x1), e1, fmaxf(x1, 0.0f));
}
// tanh-GELU of a pair: 0.5 x (1 + tanh(u)) == x * sigmoid(2u) ; u = sqrt(2/pi) (x + 0.044715 x^3)
__device__ __forceinline__ void gelu_tanh_pair(float& x0, float& x1) {
  constexpr float k0 = -2.0f * 1.4426950408889634f * 0.7978845608028654f;  // exponent of 2 is -2 log2(e) u
  constexpr float k1 = k0 * 0.044715f;
  const uint64_t x = pk2(x0, x1);
  const uint64_t w = fma2(mul2(x, x), pk2(k1, k1), pk2(k0, k0));
  float t0, t1;
  upk2(mul2(x, w), t0, t1);
  x0 *= rcp_approx(1.0f + ex2_approx(t0));
  x1 *= rcp_approx(1.0f + ex2_approx(t1));
}
template <int ACT, bool EXACT, bool HI>
__device__ __forceinline__ void apply_act_pair(float& x0, float& x1) {
  if (ACT == EVT_ACT_GELU_ERF) {
    if (EXACT) {
      x0 = 0.5f * x0 * (1.0f + erff(x0 * 0.70710678118654752f));
      x1 = 0.5f * x1 * (1.0f + erff(x1 * 0.70710678118654752f));
    } else {
      gelu_erf_pair<HI>(x0, x1);
    }
  } else if (ACT == EVT_ACT_GELU_TANH) {
    if (EXACT) {
      x0 = 0.5f * x0 * (1.0f + tanhf(0.7978845608028654f * (x0 + 0.044715f * x0 * x0 * x0)));
      x1 = 0.5f * x1 * (1.0f + tanhf(0.7978845608028654f * (x1 + 0.044715f * x1 * x1 * x1)));
    } else {
      gelu_tanh_pair(x0, x1);
    }
  }
}
// v[j] = act(v[j] + bias[n0 + j]) for the CH columns of one chunk (columns >= N are don't-care).
template <int CH, int ACT, bool EXACT, bool HI>
__device__ __forceinline__ void bias_act(float (&v)[CH], const float* __restrict__ bias, int n0, int N, bool full) {
  if (bias != nullptr) {
    if (full) {
      const float4* b4 = reinterpret_cast<const float4*>(bias + n0);
#pragma unroll
      for (int i = 0; i < CH / 4; ++i) {
        const float4 b = __ldg(b4 + i);
        upk2(add2(pk2(v[4 * i], v[4 * i + 1]), pk2(b.x, b.y)), v[4 * i], v[4 * i + 1]);
        upk2(add2(pk2(v[4 * i + 2], v[4 * i + 3]), pk2(b.z, b.w)), v[4 * i + 2], v[4 * i + 3]);
      }
    } else {
#pragma unroll
      for (int j = 0; j < CH; ++j)
        if (n0 + j < N) v[j] += __ldg(bias + n0 + j);
    }
  }
  if (ACT != EVT_ACT_NONE) {
#pragma unroll
    for (int j = 0; j < CH; j += 2) apply_act_pair<ACT, EXACT, HI>(v[j], v[j + 1]);
  }
}


// Bias lines of this warp's chunks of the coming tile -> L1, issued before the accumulator wait: with 227 KB of shared
// memory the L1 is tiny and the bias loads of the epilogue otherwise pay an L2 round trip per chunk (ncu: ~10 % of the
// FC1 kernel's warp samples stalled on them).  No registers are held across the wait.
template <int BN, bool OUT_F32, int NGRP = 2>
__device__ __forceinline__ void prefetch_bias(const GemmParams& p, int grp, int lane, int nt0) {
  constexpr int CH = OUT_F32 ? 32 : 64;
  constexpr int NCH = BN / CH;
  if (p.bias == nullptr) return;
  // lane l covers 32-float (128-byte) line l of the warp's chunks: chunk k of this warp = grp + NGRP k
  constexpr int kLinesPerChunk = CH / 32;
  const int k = lane / kLinesPerChunk;
  const int c = grp + NGRP * k;
  const int col = nt0 + c * CH + (lane % kLinesPerChunk) * 32;
  if (c < NCH && col < p.N) asm volatile("prefetch.global.L1 [%0];" ::"l"(p.bias + col));
}

// Epilogue of one 32-row x BN-column accumulator block by one warp.  Warp w reads TMEM lanes 32*(w%4).. (the
// hardware's lane-quadrant rule) and takes the 128-byte output chunks (64 bf16 / 32 f32 columns) c = grp, grp+2, ...
// (grp = w/4; NGRP = epilogue warps / 4 groups share every row block: 2 in the 1-CTA kernels, up to 4 in the CTA-pair kernel).  Thread == accumulator row while the bias / activation math runs
// on packed f32x2 pairs; the converted chunk then goes through a 128B-swizzled 4 KB smem tile (stg) to a TMA store /
// TMA f32 reduce-add, or to coalesced global stores on the generic path.
//   m0: first global row of this warp's block; nt0: first column of the tile; t_row: TMEM address (lane | column).
template <int BN, bool TF32, bool OUT_F32, int ACT, bool TMA_OUT, int NGRP = 2>
__device__ __forceinline__ void epilogue_tile(const GemmParams& p, const CUtensorMap* tmO, uint8_t* stg, int grp, int lane,
                                              int m0, int nt0, uint32_t t_row) {
  constexpr int CH = OUT_F32 ? 32 : 64;
  constexpr int NCH = BN / CH;
  const int sw = lane & 7;
  const bool has_res = p.residual != nullptr;
  const int rows_here = min(32, p.M - m0);  // may be <= 0 for a fully out-of-range warp
  // Residual rows of this warp's 32x32 chunk, one float4 per (4-row group, lane): issued one chunk ahead so
  // the HBM latency of the skip connection hides behind the previous chunk (and behind the MMA wait).
  float4 rnext[8];
  auto load_res = [&](int n0c) {
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      const int rr = it * 4 + (lane >> 3);
      rnext[it] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (rr < rows_here && p.vec_ok && n0c + CH <= p.N) {
        const long long row = m0 + rr;
        const long long rrow = p.res_row_mod > 0 ? p.res_row_off + row % p.res_row_mod : map_out_row(p, row);
        rnext[it] = *reinterpret_cast<const float4*>(p.residual + rrow * p.ldr + n0c + (lane & 7) * 4);
      }
    }
  };
  if constexpr (OUT_F32 && !TMA_OUT) {
    if (has_res && grp < NCH) load_res(nt0 + grp * CH);
  }
  if (rows_here > 0) {
#pragma unroll 1
    for (int c = grp; c < NCH; c += NGRP) {
      const int n0 = nt0 + c * CH;
      if (n0 >= p.N) break;
      float v[CH];
      {
        uint32_t r[32];
        ptx::tmem_ld_x32(t_row + c * CH, r);
        if constexpr (CH == 64) {
          uint32_t r2[32];
          ptx::tmem_ld_x32(t_row + c * CH + 32, r2);
          ptx::tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) v[32 + j] = __uint_as_float(r2[j]);
        } else {
          ptx::tmem_ld_wait();
        }
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
      }
      const bool full = p.vec_ok && (n0 + CH <= p.N);
      float4 rcur[8];
      if constexpr (OUT_F32 && !TMA_OUT) {
        if (has_res) {
#pragma unroll
          for (int it = 0; it < 8; ++it) rcur[it] = rnext[it];
          if (c + NGRP < NCH && n0 + NGRP * CH < p.N) load_res(n0 + NGRP * CH);
        }
      }
      bias_act<CH, ACT, TF32, OUT_F32>(v, p.bias, n0, p.N, full);
      if constexpr (OUT_F32) {
        if (p.round_tf32) {
#pragma unroll
          for (int j = 0; j < CH; ++j) v[j] = ptx::round_tf32(v[j]);
        }
      }
      if constexpr (!OUT_F32) if (has_res && lane < rows_here) {  // rare combination: add before rounding to bf16
        const long long orow = map_out_row(p, m0 + lane);
        const long long rrow = p.res_row_mod > 0 ? p.res_row_off + (m0 + lane) % p.res_row_mod : orow;
#pragma unroll
        for (int j = 0; j < CH; ++j)
          if (n0 + j < p.N) v[j] += p.residual[rrow * p.ldr + n0 + j];
      }
      // stage: dense 128-byte rows, 16-byte pieces XOR-swizzled by (row & 7) -- the layout a SWIZZLE_128B
      // tensor map expects, and conflict-free for both the row-per-thread writes and the row-segment reads.
      if constexpr (TMA_OUT) {
        if (ptx::elect_one()) ptx::bulk_wait_read<0>();  // the previous store of this warp has finished reading stg
      }
      __syncwarp();
      // explicit st.shared: through the C++ pointer these were generic ST.E with descriptor set-up (see ptx.cuh)
      const uint32_t sb = ptx::smem_u32(stg) + lane * 128;
      if constexpr (OUT_F32) {
#pragma unroll
        for (int i = 0; i < 8; ++i) ptx::sts_f4(sb + ((i ^ sw) << 4), v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i)
          ptx::sts_u4(sb + ((i ^ sw) << 4), pack_bf16x2(v[8 * i], v[8 * i + 1]), pack_bf16x2(v[8 * i + 2], v[8 * i + 3]),
                      pack_bf16x2(v[8 * i + 4], v[8 * i + 5]), pack_bf16x2(v[8 * i + 6], v[8 * i + 7]));
      }
      if constexpr (TMA_OUT) {
        // The TMA engine does the coalescing, the M/N clipping and (for the skip connection) the f32 add into
        // the residual stream at L2 -- the SM never reads the residual.
        ptx::fence_proxy_async_smem();
        __syncwarp();
        if (ptx::elect_one()) {  // the same thread every time (elect.sync is deterministic for a full mask): bulk groups are per thread
          if (has_res) ptx::tma_reduce_add_2d(tmO, stg, n0, m0);
          else ptx::tma_store_2d(tmO, stg, n0, m0);
          ptx::bulk_commit();
        }
        continue;
      }
      __syncwarp();
      // store: lanes 8k..8k+7 cover one 128-byte row segment; 4 rows per instruction
      const int piece = lane & 7;
#pragma unroll
      for (int it = 0; it < 8; ++it) {
        const int rr = it * 4 + (lane >> 3);
        if (rr < rows_here) {
          const long long row = m0 + rr;
          const long long orow = map_out_row(p, row);
          const uint8_t* src = stg + rr * 128 + ((piece ^ (rr & 7)) << 4);
          if constexpr (OUT_F32) {
            float4 val = *reinterpret_cast<const float4*>(src);
            const int col = n0 + piece * 4;
            float* dst = reinterpret_cast<float*>(p.out) + orow * p.ldo + col;
            if (full) {
              if (has_res) {
                const float4 rs = rcur[it];
                val.x += rs.x;
                val.y += rs.y;
                val.z += rs.z;
                val.w += rs.w;
              }
              *reinterpret_cast<float4*>(dst) = val;
            } else {
              const float e[4] = {val.x, val.y, val.z, val.w};
              const long long rrow = p.res_row_mod > 0 ? p.res_row_off + row % p.res_row_mod : orow;
#pragma unroll
              for (int q = 0; q < 4; ++q)
                if (col + q < p.N) dst[q] = e[q] + (has_res ? p.residual[rrow * p.ldr + col + q] : 0.f);
            }
          } else {
            const uint4 val = *reinterpret_cast<const uint4*>(src);
            const int col = n0 + piece * 8;
            __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(p.out) + orow * p.ldo + col;
            if (full) {
              *reinterpret_cast<uint4*>(dst) = val;
            } else {
              const uint32_t e[4] = {val.x, val.y, val.z, val.w};
#pragma unroll
              for (int q = 0; q < 8; ++q)
                if (col + q < p.N) {
                  const uint16_t h = static_cast<uint16_t>(e[q >> 1] >> ((q & 1) * 16));
                  reinterpret_cast<uint16_t*>(dst)[q] = h;
                }
            }
          }
        }
      }
    }
  }
}

// CTA-pair kernels (gemm2.cu): bf16 operands, TMA epilogue.  p.tiles_m is recomputed for 256-row tiles.
bool pair_supported(int bn);
int gemm_pair_launch(int bn, const void* W, int64_t ldw, const CUtensorMap& tmA, const CUtensorMap& tmO, const GemmParams& p,
                     bool out_f32, int act, cudaStream_t stream);

}  // namespace gemm_detail
}  // namespace evt
