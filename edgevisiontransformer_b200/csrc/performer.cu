// T2T-ViT front-end kernels (modeling/models/t2t_vit.py:43-88, modeling/layers/transformer_encoder.py:39-101).
//
//   unfold_ln     soft split (tf_Unfold, channel-last, depth order (kh,kw,c), zero pad) fused with the performer's
//                 first LayerNorm: one warp gathers one window, normalises it in registers and writes the bf16 row
//                 that feeds the kqv GEMM -- the unfolded tensor never exists un-normalised in HBM.
//   performer     linear attention with positive random features (m = 32, emb = 64):
//                   kp = exp(w k - |k|^2/2)/sqrt(m);  ksum = sum_t kp;  kptv = sum_t v kp^T      (reduce, per image)
//                   qp = exp(w q - |q|^2/2)/sqrt(m);  y = (qp kptv^T) / (qp.ksum + 1e-8)          (apply, per token)
//                 The reduction over tokens is two-level with a fixed summation order (deterministic, no atomics).
// The dense layers around them (kqv, attn_output, MLP, project) run on the tcgen05 GEMM with fused epilogues.
#include <cuda_bf16.h>

#include "common.h"
#include "gemm_common.cuh"
#include "ops.h"
#include "ptx.cuh"

namespace evt {
namespace {

constexpr int kEmb = 64;
constexpr int kM = 32;

// ---------------------------------------------------------------------------------------------- unfold (+ LN)
// One warp per output row; lane l owns the column pairs (64 i + 2 l, + 1), so stores are packed bf16x2 (128 B per warp
// instruction).  KK / CC > 0 fix the window and channel count at compile time (T2T: 7 x 7 x 3 and 3 x 3 x 64) -- the
// column -> (ky, kx, c) decomposition is then multiply-shift arithmetic instead of integer divisions by run-time values,
// which is what the run-time-generic version (KK = 0) spent most of its instructions on (0.94 ms -> see DESIGN.md).
// Row length L = k*k*C <= 64 * kMaxPairs.
constexpr int kMaxPairs = 9;  // 576 / 64

template <typename TIN, bool LN, int KK, int CC>
__global__ void __launch_bounds__(256) unfold_ln_kernel(const TIN* __restrict__ x, __nv_bfloat16* __restrict__ out,
                                                        long long ldo, const float* __restrict__ gamma,
                                                        const float* __restrict__ beta, float eps, int B, int H, int W,
                                                        int C_rt, int k_rt, int s, int p, int oh, int ow, long long rows) {
  const int lane = threadIdx.x & 31;
  const long long row = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int k = KK > 0 ? KK : k_rt;
  const int C = CC > 0 ? CC : C_rt;
  const int L = k * k * C;
  constexpr int NP = KK > 0 ? (KK * KK * CC + 63) / 64 : kMaxPairs;
  const int ox = static_cast<int>(row % ow);
  const int oy = static_cast<int>((row / ow) % oh);
  const long long b = row / (static_cast<long long>(ow) * oh);
  const int kC = k * C;
  const int ix0 = ox * s - p, iy0 = oy * s - p;
  const TIN* xb = x + b * H * static_cast<long long>(W) * C;
  auto fetch = [&](int col) -> float {
    if (col >= L) return 0.f;
    const int ky = col / kC;
    const int rem = col - ky * kC;  // kx*C + c : contiguous in the input row
    const int kx = rem / C;
    const int iy = iy0 + ky, ix = ix0 + kx;
    if (iy < 0 || iy >= H || ix < 0 || ix >= W) return 0.f;
    return static_cast<float>(xb[(static_cast<long long>(iy) * W + ix0) * C + rem]);
  };
  float v0[NP], v1[NP];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < NP; ++i) {
    const int col = i * 64 + 2 * lane;
    if constexpr (CC > 0 && CC % 2 == 0 && sizeof(TIN) == 4) {
      // both columns of the pair lie in the same (ky, kx) cell: one 8-byte load
      float2 t = make_float2(0.f, 0.f);
      if (col < L) {
        const int ky = col / kC;
        const int rem = col - ky * kC;
        const int kx = rem / C;
        const int iy = iy0 + ky, ix = ix0 + kx;
        if (iy >= 0 && iy < H && ix >= 0 && ix < W)
          t = *reinterpret_cast<const float2*>(reinterpret_cast<const float*>(xb) + (static_cast<long long>(iy) * W + ix0) * C + rem);
      }
      v0[i] = t.x;
      v1[i] = t.y;
    } else {
      v0[i] = fetch(col);
      v1[i] = fetch(col + 1);
    }
    sum += v0[i] + v1[i];
  }
  float mean = 0.f, rstd = 1.f;
  if (LN) {
    mean = ptx::warp_sum(sum) / static_cast<float>(L);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < NP; ++i) {
      const int col = i * 64 + 2 * lane;
      const float d0 = v0[i] - mean, d1 = v1[i] - mean;
      if (col < L) q += d0 * d0;
      if (col + 1 < L) q += d1 * d1;
    }
    rstd = rsqrtf(ptx::warp_sum(q) / static_cast<float>(L) + eps);
  }
  __nv_bfloat16* orow = out + row * ldo;  // ldo is even and the base 4-byte aligned (checked by the launcher)
#pragma unroll
  for (int i = 0; i < NP; ++i) {
    const int col = i * 64 + 2 * lane;
    if (col < ldo) {
      float o0 = 0.f, o1 = 0.f;
      if (col < L) o0 = LN ? (v0[i] - mean) * rstd * gamma[col] + beta[col] : v0[i];
      if (col + 1 < L) o1 = LN ? (v1[i] - mean) * rstd * gamma[col + 1] + beta[col + 1] : v1[i];
      *reinterpret_cast<__nv_bfloat162*>(orow + col) = __floats2bfloat162_rn(o0, o1);
    }
  }
}

// The 7 x 7 x 3 soft split of T2T's first stage (147 elements per output row = 7 runs of 21 contiguous floats), written for
// instruction count: the generic kernel above issued ~660 warp instructions per output row here (ncu: issue slots 85 % busy --
// per-element validity branches, 64-bit address arithmetic, gamma / beta reloaded per row) and ran at 283 us per 256 images
// against a 61 us HBM floor; one row per warp with row-invariant registers still took ~220 (205 us, issue slots 76 %).
// Here EIGHT lanes share an output row (four rows per warp at a time): lane j of the group owns elements j, j + 8, ..., j + 144
// (19 each, 8 x 19 = 152 = the padded row length), so a row costs three shuffle levels per reduction instead of five, the
// per-row bookkeeping is shared by four rows, and 19 independent loads per lane are in flight.  Offsets and affine parameters
// of the lane's elements are row-invariant registers; a group of four windows that are all interior (83 % of a 56 x 56 grid)
// takes a path without any bounds test.
template <typename TIN, bool LN, int ITER>
__global__ void __launch_bounds__(256) unfold773_kernel(const TIN* __restrict__ x, __nv_bfloat16* __restrict__ out, long long ldo,
                                                        const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                                                        int H, int W, int s, int p, int oh, int ow, long long rows) {
  constexpr int KK = 7, CC = 3, L = KK * KK * CC, kRun = KK * CC, NE = 19;  // 147, 21; 8 lanes x 19 elements = 152
  const int lane = threadIdx.x & 31;
  const int j = lane & 7, slot = lane >> 3;
  const long long warp_id = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int off[NE];
  float g[NE], be[NE];
#pragma unroll
  for (int i = 0; i < NE; ++i) {
    const int e = j + 8 * i;
    const bool in = e < L;
    const int ky = in ? e / kRun : 0;
    off[i] = in ? ky * W * CC + (e - ky * kRun) : -1;
    g[i] = (LN && in) ? gamma[e] : 0.f;
    be[i] = (LN && in) ? beta[e] : 0.f;
  }
#pragma unroll 1
  for (int it = 0; it < ITER; ++it) {
    const long long row = (warp_id * ITER + it) * 4 + slot;
    const bool live = row < rows;
    const long long rc = live ? row : rows - 1;  // dead slots recompute the last row and store nothing (shuffles stay uniform)
    const int ox = static_cast<int>(rc % ow);
    const long long t = rc / ow;
    const int oy = static_cast<int>(t % oh);
    const long long b = t / oh;
    const int iy0 = oy * s - p, ix0 = ox * s - p;
    const TIN* base = x + ((b * H + iy0) * static_cast<long long>(W) + ix0) * CC;
    const bool interior = iy0 >= 0 && iy0 + KK <= H && ix0 >= 0 && ix0 + KK <= W;
    float v[NE];
    if (__all_sync(0xffffffffu, interior)) {
#pragma unroll
      for (int i = 0; i < NE - 1; ++i) v[i] = static_cast<float>(base[off[i]]);
      v[NE - 1] = off[NE - 1] >= 0 ? static_cast<float>(base[off[NE - 1]]) : 0.f;
    } else {
#pragma unroll
      for (int i = 0; i < NE; ++i) {
        const int e = j + 8 * i;
        const int ky = e / kRun, kx = (e - ky * kRun) / CC;
        const int iy = iy0 + ky, ix = ix0 + kx;
        const bool ok = off[i] >= 0 && iy >= 0 && iy < H && ix >= 0 && ix < W;
        v[i] = ok ? static_cast<float>(base[off[i]]) : 0.f;
      }
    }
    float mean = 0.f, rstd = 1.f;
    if (LN) {
      float sum = 0.f;
#pragma unroll
      for (int i = 0; i < NE; ++i) sum += v[i];
      sum += __shfl_xor_sync(0xffffffffu, sum, 1);
      sum += __shfl_xor_sync(0xffffffffu, sum, 2);
      sum += __shfl_xor_sync(0xffffffffu, sum, 4);
      mean = sum / static_cast<float>(L);
      float q = 0.f;
#pragma unroll
      for (int i = 0; i < NE - 1; ++i) {
        const float d = v[i] - mean;
        q += d * d;
      }
      if (off[NE - 1] >= 0) {
        const float d = v[NE - 1] - mean;
        q += d * d;
      }
      q += __shfl_xor_sync(0xffffffffu, q, 1);
      q += __shfl_xor_sync(0xffffffffu, q, 2);
      q += __shfl_xor_sync(0xffffffffu, q, 4);
      rstd = rsqrtf(q / static_cast<float>(L) + eps);
    }
    if (live) {
      __nv_bfloat16* orow = out + row * ldo + j;
#pragma unroll
      for (int i = 0; i < NE; ++i) {
        float o = LN ? (v[i] - mean) * rstd * g[i] + be[i] : v[i];
        if (i == NE - 1 && off[i] < 0) o = 0.f;  // elements 147 .. 151: the zero padding of the row
        orow[8 * i] = __float2bfloat16_rn(o);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------- performer
// Both kernels are chains of small matrix products per 16-token tile and run them on the warp-level tensor path
// (mma.sync m16n8k16, bf16 operands, f32 accumulate) -- the first version walked them with 128 warp shuffles per token
// and was shuffle-issue bound (0.61 + 0.94 ms for 802 816 tokens; now HBM-bound).  Orientation is chosen so that every
// accumulator fragment is directly the A fragment of the next product (no transposes through shared memory except V):
//   reduce : WTX^T[32 x 16] = W[32 x 64] K^T[64 x 16]  ->  kp^T = exp(WTX^T - |k|^2/2)/sqrt(32)
//            kptv^T[32 x 64] += kp^T[32 x 16] V[16 x 64]       (V via ldmatrix.trans from a swizzled 2 KB tile)
//   apply  : WTX[16 x 32] = Q[16 x 64] W^T[64 x 32]     ->  qp = exp(WTX - |q|^2/2)/sqrt(32)
//            Y[16 x 64] = qp[16 x 32] kptv^T[32 x 64];  D = qp . ksum (f32)
// The random-feature matrix w enters as a bf16 hi + lo pair (two MMAs), i.e. with 16 mantissa bits: rounding w itself to
// bf16 would shift every exponent by up to ~0.02.  k, q, v are bf16 already; kp / qp / kptv are rounded to bf16 only as
// tensor-core operands (like P in attention) while ksum and D stay f32.
constexpr int kTileTok = 16;
constexpr int kChunk = 256;  // tokens per block: 4 warps x 4 tiles
constexpr float kInvSqrtM = 0.17677669529663687f;  // 1/sqrt(32)

// (hi, lo) bf16 pairs of two consecutive f32 values: x ~= hi + lo with 16 mantissa bits
__device__ __forceinline__ void split2(float a, float b, uint32_t& hi, uint32_t& lo) {
  const __nv_bfloat16 ha = __float2bfloat16_rn(a), hb = __float2bfloat16_rn(b);
  hi = ptx::pack_bf16x2(__bfloat162float(ha), __bfloat162float(hb));
  lo = ptx::pack_bf16x2(a - __bfloat162float(ha), b - __bfloat162float(hb));
}
__device__ __forceinline__ float sumsq_bf16x2(uint32_t v) {
  const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&v));
  return f.x * f.x + f.y * f.y;
}
__device__ __forceinline__ float quad_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  return v;
}

// kqv: bf16 [B*T, ld] with k at cols [0,64), q at [64,128), v at [128,192).
// partial: f32 [B, nsplit, 32 + 64*32]  (ksum[m] | kptv[n][m])
__global__ void __launch_bounds__(128) performer_reduce_kernel(const __nv_bfloat16* __restrict__ kqv, long long ld,
                                                               const float* __restrict__ w, float* __restrict__ partial,
                                                               int T, int nsplit) {
  __shared__ float red[4][kM + kEmb * kM];
  __shared__ __align__(128) uint8_t vtile[4][kTileTok * 128];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int split = blockIdx.x, b = blockIdx.y;
  // A fragments of W[32 features x 64]: m-tile mi, k-step ks
  uint32_t whi[2][4][4], wlo[2][4][4];
#pragma unroll
  for (int mi = 0; mi < 2; ++mi)
#pragma unroll
    for (int ks = 0; ks < 4; ++ks)
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const float2 x = *reinterpret_cast<const float2*>(w + (mi * 16 + g + (r & 1) * 8) * kEmb + ks * 16 + (r >> 1) * 8 + 2 * t);
        split2(x.x, x.y, whi[mi][ks][r], wlo[mi][ks][r]);
      }
  float ksum[2][2] = {{0.f, 0.f}, {0.f, 0.f}};  // features mi*16 + g, mi*16 + g + 8 (summed over this lane's token columns)
  float kacc[2][8][4];                           // kptv^T: (feature mi*16 + g (+8), emb ne*8 + 2t (+1))
#pragma unroll
  for (int mi = 0; mi < 2; ++mi)
#pragma unroll
    for (int ne = 0; ne < 8; ++ne) kacc[mi][ne][0] = kacc[mi][ne][1] = kacc[mi][ne][2] = kacc[mi][ne][3] = 0.f;
  const int t0 = split * kChunk, t1 = min(T, t0 + kChunk);
  const uint32_t vt = ptx::smem_u32(vtile[warp]);
  for (int tb = t0 + warp * kTileTok; tb < t1; tb += 4 * kTileTok) {
    const __nv_bfloat16* base = kqv + (static_cast<long long>(b) * T + tb) * ld;
    // V tile -> shared memory (16 rows x 128 B, 16-byte chunks XOR-swizzled by row & 7); rows past t1 are zero
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int c = lane + 32 * i, row = c >> 3, ch = c & 7;
      uint4 val = make_uint4(0, 0, 0, 0);
      if (tb + row < t1) val = *reinterpret_cast<const uint4*>(base + row * ld + 128 + ch * 8);
      *reinterpret_cast<uint4*>(vtile[warp] + row * 128 + ((ch ^ (row & 7)) << 4)) = val;
    }
    // K fragments (B operand, n = token): n-tile nj = tokens 8 nj + g
    uint32_t kb[2][4][2];
    float xd[2];
#pragma unroll
    for (int nj = 0; nj < 2; ++nj) {
      const bool ok = tb + nj * 8 + g < t1;
      const __nv_bfloat16* rp = base + (nj * 8 + g) * ld + 2 * t;
      float sq = 0.f;
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        kb[nj][ks][0] = ok ? *reinterpret_cast<const uint32_t*>(rp + ks * 16) : 0u;
        kb[nj][ks][1] = ok ? *reinterpret_cast<const uint32_t*>(rp + ks * 16 + 8) : 0u;
        sq += sumsq_bf16x2(kb[nj][ks][0]) + sumsq_bf16x2(kb[nj][ks][1]);
      }
      xd[nj] = 0.5f * quad_sum(sq);  // |k|^2 / 2 of token 8 nj + g, in all four lanes of the quad
    }
    __syncwarp();
    uint32_t pa[2][4];  // kp^T as A fragments (features x 16 tokens)
#pragma unroll
    for (int mi = 0; mi < 2; ++mi) {
#pragma unroll
      for (int nj = 0; nj < 2; ++nj) {
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
          ptx::mma_bf16_16816(acc, whi[mi][ks], kb[nj][ks][0], kb[nj][ks][1]);
          ptx::mma_bf16_16816(acc, wlo[mi][ks], kb[nj][ks][0], kb[nj][ks][1]);
        }
        // columns of this lane: tokens 8 nj + 2t, + 1
        const float x0 = __shfl_sync(0xffffffffu, xd[nj], (2 * t) * 4);
        const float x1 = __shfl_sync(0xffffffffu, xd[nj], (2 * t + 1) * 4);
        const bool ok0 = tb + nj * 8 + 2 * t < t1, ok1 = tb + nj * 8 + 2 * t + 1 < t1;
        const float p0 = ok0 ? __expf(acc[0] - x0) * kInvSqrtM : 0.f;
        const float p1 = ok1 ? __expf(acc[1] - x1) * kInvSqrtM : 0.f;
        const float p2 = ok0 ? __expf(acc[2] - x0) * kInvSqrtM : 0.f;
        const float p3 = ok1 ? __expf(acc[3] - x1) * kInvSqrtM : 0.f;
        ksum[mi][0] += p0 + p1;
        ksum[mi][1] += p2 + p3;
        pa[mi][nj * 2] = ptx::pack_bf16x2(p0, p1);
        pa[mi][nj * 2 + 1] = ptx::pack_bf16x2(p2, p3);
      }
    }
    // kptv^T += kp^T V
#pragma unroll
    for (int np = 0; np < 4; ++np) {
      uint32_t vb[4];  // {b0, b1} of emb n-tile 2 np, {b0, b1} of 2 np + 1
      const int row = (lane & 7) + ((lane >> 3) & 1) * 8, ch = np * 2 + (lane >> 4);
      ptx::ldmatrix_x4_trans(vt + row * 128 + ((ch ^ (row & 7)) << 4), vb);
#pragma unroll
      for (int mi = 0; mi < 2; ++mi) {
        ptx::mma_bf16_16816(kacc[mi][2 * np], pa[mi], vb[0], vb[1]);
        ptx::mma_bf16_16816(kacc[mi][2 * np + 1], pa[mi], vb[2], vb[3]);
      }
    }
  }
  // per-warp results -> shared memory in the [ksum | kptv[n][m]] layout, then a fixed-order sum over the four warps
#pragma unroll
  for (int mi = 0; mi < 2; ++mi) {
    const float s0 = quad_sum(ksum[mi][0]), s1 = quad_sum(ksum[mi][1]);
    if (t == 0) {
      red[warp][mi * 16 + g] = s0;
      red[warp][mi * 16 + g + 8] = s1;
    }
#pragma unroll
    for (int ne = 0; ne < 8; ++ne) {
      const int n = ne * 8 + 2 * t, m = mi * 16 + g;
      red[warp][kM + n * kM + m] = kacc[mi][ne][0];
      red[warp][kM + (n + 1) * kM + m] = kacc[mi][ne][1];
      red[warp][kM + n * kM + m + 8] = kacc[mi][ne][2];
      red[warp][kM + (n + 1) * kM + m + 8] = kacc[mi][ne][3];
    }
  }
  __syncthreads();
  float* dst = partial + (static_cast<long long>(b) * nsplit + split) * (kM + kEmb * kM);
  for (int i = threadIdx.x; i < kM + kEmb * kM; i += 128) dst[i] = ((red[0][i] + red[1][i]) + red[2][i]) + red[3][i];
}

__global__ void __launch_bounds__(256) performer_reduce_final_kernel(const float* __restrict__ partial,
                                                                     float* __restrict__ stats, int nsplit) {
  const int b = blockIdx.x;
  const int n = kM + kEmb * kM;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    float s = 0.f;
    for (int k = 0; k < nsplit; ++k) s += partial[(static_cast<long long>(b) * nsplit + k) * n + i];
    stats[static_cast<long long>(b) * n + i] = s;
  }
}

// ---------------------------------------------------------------------------------------------- performer tail
// Everything the Token_performer does after the attention contraction (modeling/layers/transformer_encoder.py:93-99), for 64-wide
// tokens, in ONE pass over the rows:
//     y  = v + attn_output(ya)            (Dense 64 -> 64; v = the f32 copy of the value rows the apply kernel wrote)
//     y += mlp(LayerNorm(y))              (Dense 64 -> 64, tanh-GELU, Dense 64 -> 64)
// Before: GEMM (f32 reduce-add), LayerNorm kernel, GEMM + GELU, GEMM (reduce-add) -- four launches moving 1920 bytes per token;
// here 640 (ya in, y in, y out).  Per 16-token tile a warp chains three m16n8k16 products whose accumulator fragments are the
// next product's A fragments (two adjacent n-tiles = one k-step), the LayerNorm statistics are quad reductions over the
// accumulator fragment (f32, centred variance), the three 64 x 64 weights sit in shared memory with rows padded to 144 bytes
// (conflict-free B-fragment loads).  Same arithmetic as the four kernels (bf16 operands, f32 accumulation, f32 skip), so the
// results agree with them to summation order.
constexpr int kWRow = 72;  // bf16 elements per padded weight row

struct TailWeights {
  const __nv_bfloat16 *wo, *w1, *w2;   // [64 out, 64 in] dense
  const float *bo, *gamma, *beta, *b1, *b2;
  float eps;
};
struct TailSmem {
  __align__(16) __nv_bfloat16 ws[3][kEmb * kWRow];
  __align__(16) float vec[5][kEmb];  // bo, gamma, beta, b1, b2
};

// cooperative load by the whole block (128 threads); the caller synchronises afterwards
__device__ __forceinline__ void tail_load(TailSmem& sm, const TailWeights& w) {
  for (int i = threadIdx.x; i < 3 * kEmb * 8; i += blockDim.x) {  // 16-byte pieces: 8 per 64-element row
    const int m = i / (kEmb * 8), r = (i / 8) % kEmb, c = i % 8;
    const __nv_bfloat16* src = m == 0 ? w.wo : m == 1 ? w.w1 : w.w2;
    *reinterpret_cast<uint4*>(&sm.ws[m][r * kWRow + c * 8]) = *reinterpret_cast<const uint4*>(src + r * kEmb + c * 8);
  }
  for (int i = threadIdx.x; i < 5 * kEmb; i += blockDim.x) {
    const int m = i / kEmb, c = i % kEmb;
    const float* src = m == 0 ? w.bo : m == 1 ? w.gamma : m == 2 ? w.beta : m == 3 ? w.b1 : w.b2;
    sm.vec[m][c] = src != nullptr ? src[c] : 0.f;
  }
}

// One 16-token tile.  a: A fragments of ya (bf16, 4 k-steps); y1: on entry v in accumulator-fragment layout (rows g / g + 8,
// columns 8 nj + 2t, + 1), on exit the performer's output rows.
__device__ __forceinline__ void tail_tile(const TailSmem& sm, uint32_t (&a)[4][4], float (&y1)[8][4], int g, int t, float eps) {
  auto bfrag = [&](int m, int nj, int ks, uint32_t& b0, uint32_t& b1v) {
    const __nv_bfloat16* rp = &sm.ws[m][(nj * 8 + g) * kWRow + ks * 16 + 2 * t];
    b0 = *reinterpret_cast<const uint32_t*>(rp);
    b1v = *reinterpret_cast<const uint32_t*>(rp + 8);
  };
  float acc[8][4];
  // y1 = v + ya wo^T + bo
  float sA = 0.f, sB = 0.f;
#pragma unroll
  for (int nj = 0; nj < 8; ++nj) {
    acc[nj][0] = acc[nj][1] = acc[nj][2] = acc[nj][3] = 0.f;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      uint32_t b0, b1v;
      bfrag(0, nj, ks, b0, b1v);
      ptx::mma_bf16_16816(acc[nj], a[ks], b0, b1v);
    }
    const float2 bb = *reinterpret_cast<const float2*>(&sm.vec[0][nj * 8 + 2 * t]);
    y1[nj][0] += acc[nj][0] + bb.x;
    y1[nj][1] += acc[nj][1] + bb.y;
    y1[nj][2] += acc[nj][2] + bb.x;
    y1[nj][3] += acc[nj][3] + bb.y;
    sA += y1[nj][0] + y1[nj][1];
    sB += y1[nj][2] + y1[nj][3];
  }
  // LayerNorm over the 64 columns of rows g and g + 8 (each spread over the four lanes of a quad)
  const float mA = quad_sum(sA) * (1.0f / kEmb), mB = quad_sum(sB) * (1.0f / kEmb);
  float qA = 0.f, qB = 0.f;
#pragma unroll
  for (int nj = 0; nj < 8; ++nj) {
    const float d0 = y1[nj][0] - mA, d1 = y1[nj][1] - mA, d2 = y1[nj][2] - mB, d3 = y1[nj][3] - mB;
    qA += d0 * d0 + d1 * d1;
    qB += d2 * d2 + d3 * d3;
  }
  const float rA = rsqrtf(quad_sum(qA) * (1.0f / kEmb) + eps), rB = rsqrtf(quad_sum(qB) * (1.0f / kEmb) + eps);
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int nj = 2 * ks + h, col = nj * 8 + 2 * t;
      const float2 gg = *reinterpret_cast<const float2*>(&sm.vec[1][col]);
      const float2 be = *reinterpret_cast<const float2*>(&sm.vec[2][col]);
      a[ks][2 * h] = ptx::pack_bf16x2((y1[nj][0] - mA) * rA * gg.x + be.x, (y1[nj][1] - mA) * rA * gg.y + be.y);
      a[ks][2 * h + 1] = ptx::pack_bf16x2((y1[nj][2] - mB) * rB * gg.x + be.x, (y1[nj][3] - mB) * rB * gg.y + be.y);
    }
  }
  // h = gelu_tanh(z w1^T + b1)
#pragma unroll
  for (int nj = 0; nj < 8; ++nj) {
    acc[nj][0] = acc[nj][1] = acc[nj][2] = acc[nj][3] = 0.f;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      uint32_t b0, b1v;
      bfrag(1, nj, ks, b0, b1v);
      ptx::mma_bf16_16816(acc[nj], a[ks], b0, b1v);
    }
  }
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int nj = 2 * ks + h;
      const float2 bb = *reinterpret_cast<const float2*>(&sm.vec[3][nj * 8 + 2 * t]);
      float h0 = acc[nj][0] + bb.x, h1 = acc[nj][1] + bb.y, h2 = acc[nj][2] + bb.x, h3 = acc[nj][3] + bb.y;
      gemm_detail::gelu_tanh_pair(h0, h1);
      gemm_detail::gelu_tanh_pair(h2, h3);
      a[ks][2 * h] = ptx::pack_bf16x2(h0, h1);
      a[ks][2 * h + 1] = ptx::pack_bf16x2(h2, h3);
    }
  }
  // y = y1 + h w2^T + b2
#pragma unroll
  for (int nj = 0; nj < 8; ++nj) {
    acc[nj][0] = acc[nj][1] = acc[nj][2] = acc[nj][3] = 0.f;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      uint32_t b0, b1v;
      bfrag(2, nj, ks, b0, b1v);
      ptx::mma_bf16_16816(acc[nj], a[ks], b0, b1v);
    }
    const float2 bb = *reinterpret_cast<const float2*>(&sm.vec[4][nj * 8 + 2 * t]);
    y1[nj][0] += acc[nj][0] + bb.x;
    y1[nj][1] += acc[nj][1] + bb.y;
    y1[nj][2] += acc[nj][2] + bb.x;
    y1[nj][3] += acc[nj][3] + bb.y;
  }
}

// per token: yattn (bf16 [B*T, 64]) = (qp kptv^T)/(qp.ksum + eps);  vout (f32 [B*T, 64]) = v (the skip connection that
// the attn_output GEMM then reduce-adds into, transformer_encoder.py:93).
// TAIL: the tile goes straight on through attn_output + LayerNorm + MLP (tail_tile above) -- ya and v never leave the registers,
// vout receives the performer's finished output rows and yattn is not written: 512 bytes of HBM traffic per token (q, v in; y out)
// instead of 640 here + 640 in the tail kernel.  Bit-identical to the two kernels (same roundings, same order).
template <bool TAIL>
__global__ void __launch_bounds__(128) performer_apply_kernel(const __nv_bfloat16* __restrict__ kqv, long long ld,
                                                              const float* __restrict__ w, const float* __restrict__ stats,
                                                              __nv_bfloat16* __restrict__ yattn, float* __restrict__ vout,
                                                              int T, float eps, const TailWeights tw) {
  __shared__ TailSmem sm_tail[1];  // unused (and eliminated) without TAIL
  if (TAIL) {
    tail_load(sm_tail[0], tw);
    __syncthreads();
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int b = blockIdx.y;
  const float* st = stats + static_cast<long long>(b) * (kM + kEmb * kM);
  // B fragments of W^T[64 emb x 32 features]: n-tile nf = features 8 nf + g, k-step ks
  uint32_t whi[4][4][2], wlo[4][4][2];
#pragma unroll
  for (int nf = 0; nf < 4; ++nf)
#pragma unroll
    for (int ks = 0; ks < 4; ++ks)
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const float2 x = *reinterpret_cast<const float2*>(w + (nf * 8 + g) * kEmb + ks * 16 + r * 8 + 2 * t);
        split2(x.x, x.y, whi[nf][ks][r], wlo[nf][ks][r]);
      }
  // B fragments of kptv^T[32 features x 64 emb]: n-tile ne = emb 8 ne + g, k-step ks = features 16 ks ..
  uint32_t kvb[8][2][2];
#pragma unroll
  for (int ne = 0; ne < 8; ++ne)
#pragma unroll
    for (int ks = 0; ks < 2; ++ks)
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const float2 x = *reinterpret_cast<const float2*>(st + kM + (ne * 8 + g) * kM + ks * 16 + r * 8 + 2 * t);
        kvb[ne][ks][r] = ptx::pack_bf16x2(x.x, x.y);
      }
  float ksm[4][2];  // ksum of this lane's feature columns 8 nf + 2t, + 1
#pragma unroll
  for (int nf = 0; nf < 4; ++nf) {
    ksm[nf][0] = st[nf * 8 + 2 * t];
    ksm[nf][1] = st[nf * 8 + 2 * t + 1];
  }
  const int t0 = blockIdx.x * kChunk, t1 = min(T, t0 + kChunk);
  for (int tb = t0 + warp * kTileTok; tb < t1; tb += 4 * kTileTok) {
    const long long r0 = static_cast<long long>(b) * T + tb;
    const __nv_bfloat16* base = kqv + r0 * ld;
    const bool okA = tb + g < t1, okB = tb + g + 8 < t1;  // rows g and g + 8 of the tile
    // Q fragments (A operand): rows = tokens g, g + 8
    uint32_t qa[4][4];
    float sqA = 0.f, sqB = 0.f;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      const __nv_bfloat16* ra = base + g * ld + 64 + ks * 16 + 2 * t;
      const __nv_bfloat16* rb = ra + 8 * ld;
      qa[ks][0] = okA ? *reinterpret_cast<const uint32_t*>(ra) : 0u;
      qa[ks][1] = okB ? *reinterpret_cast<const uint32_t*>(rb) : 0u;
      qa[ks][2] = okA ? *reinterpret_cast<const uint32_t*>(ra + 8) : 0u;
      qa[ks][3] = okB ? *reinterpret_cast<const uint32_t*>(rb + 8) : 0u;
      sqA += sumsq_bf16x2(qa[ks][0]) + sumsq_bf16x2(qa[ks][2]);
      sqB += sumsq_bf16x2(qa[ks][1]) + sumsq_bf16x2(qa[ks][3]);
    }
    const float xA = 0.5f * quad_sum(sqA), xB = 0.5f * quad_sum(sqB);
    uint32_t pa[2][4];  // qp as A fragments of the two k-steps (features 0..15, 16..31)
    float dA = 0.f, dB = 0.f;
#pragma unroll
    for (int nf = 0; nf < 4; ++nf) {
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        ptx::mma_bf16_16816(acc, qa[ks], whi[nf][ks][0], whi[nf][ks][1]);
        ptx::mma_bf16_16816(acc, qa[ks], wlo[nf][ks][0], wlo[nf][ks][1]);
      }
      const float p0 = __expf(acc[0] - xA) * kInvSqrtM, p1 = __expf(acc[1] - xA) * kInvSqrtM;
      const float p2 = __expf(acc[2] - xB) * kInvSqrtM, p3 = __expf(acc[3] - xB) * kInvSqrtM;
      dA = fmaf(p0, ksm[nf][0], fmaf(p1, ksm[nf][1], dA));
      dB = fmaf(p2, ksm[nf][0], fmaf(p3, ksm[nf][1], dB));
      pa[nf >> 1][(nf & 1) * 2] = ptx::pack_bf16x2(p0, p1);
      pa[nf >> 1][(nf & 1) * 2 + 1] = ptx::pack_bf16x2(p2, p3);
    }
    const float invA = 1.0f / (quad_sum(dA) + eps), invB = 1.0f / (quad_sum(dB) + eps);
    uint32_t ya_frag[4][4];  // TAIL: yattn as the A fragments of the attn_output product (n-tiles 2 ks, 2 ks + 1 = k-step ks)
#pragma unroll
    for (int ne = 0; ne < 8; ++ne) {
      float y[4] = {0.f, 0.f, 0.f, 0.f};
      ptx::mma_bf16_16816(y, pa[0], kvb[ne][0][0], kvb[ne][0][1]);
      ptx::mma_bf16_16816(y, pa[1], kvb[ne][1][0], kvb[ne][1][1]);
      const int col = ne * 8 + 2 * t;
      if (TAIL) {
        ya_frag[ne >> 1][(ne & 1) * 2] = ptx::pack_bf16x2(y[0] * invA, y[1] * invA);
        ya_frag[ne >> 1][(ne & 1) * 2 + 1] = ptx::pack_bf16x2(y[2] * invB, y[3] * invB);
      } else {
        if (okA) *reinterpret_cast<uint32_t*>(yattn + (r0 + g) * kEmb + col) = ptx::pack_bf16x2(y[0] * invA, y[1] * invA);
        if (okB) *reinterpret_cast<uint32_t*>(yattn + (r0 + g + 8) * kEmb + col) = ptx::pack_bf16x2(y[2] * invB, y[3] * invB);
      }
    }
    if (TAIL) {
      float y1[8][4];  // v in accumulator-fragment layout
#pragma unroll
      for (int nj = 0; nj < 8; ++nj) {
        const int col = 128 + nj * 8 + 2 * t;
        float2 vA = make_float2(0.f, 0.f), vB = make_float2(0.f, 0.f);
        if (okA) vA = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(base + g * ld + col));
        if (okB) vB = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(base + (g + 8) * ld + col));
        y1[nj][0] = vA.x, y1[nj][1] = vA.y, y1[nj][2] = vB.x, y1[nj][3] = vB.y;
      }
      tail_tile(sm_tail[0], ya_frag, y1, g, t, tw.eps);
#pragma unroll
      for (int nj = 0; nj < 8; ++nj) {
        const int col = nj * 8 + 2 * t;
        if (okA) *reinterpret_cast<float2*>(vout + (r0 + g) * kEmb + col) = make_float2(y1[nj][0], y1[nj][1]);
        if (okB) *reinterpret_cast<float2*>(vout + (r0 + g + 8) * kEmb + col) = make_float2(y1[nj][2], y1[nj][3]);
      }
    } else {
      // vout = v as f32: 16 rows x 32 bf16 pairs, coalesced
#pragma unroll
      for (int i = 0; i < kTileTok; ++i) {
        if (tb + i < t1) {
          const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(base + i * ld + 128 + 2 * lane));
          *reinterpret_cast<float2*>(vout + (r0 + i) * kEmb + 2 * lane) = f;
        }
      }
    }
  }
}



__global__ void __launch_bounds__(128) performer_mlp_kernel(const __nv_bfloat16* __restrict__ ya, float* __restrict__ y, const TailWeights tw,
                                                            long long rows) {
  __shared__ TailSmem sm;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  tail_load(sm, tw);
  __syncthreads();
  const long long tiles = (rows + kTileTok - 1) / kTileTok;
  for (long long tile = static_cast<long long>(blockIdx.x) * 4 + warp; tile < tiles; tile += static_cast<long long>(gridDim.x) * 4) {
    const long long r0 = tile * kTileTok;
    const bool okA = r0 + g < rows, okB = r0 + g + 8 < rows;
    uint32_t a[4][4];
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      const __nv_bfloat16* pa = ya + (r0 + g) * kEmb + ks * 16 + 2 * t;
      a[ks][0] = okA ? *reinterpret_cast<const uint32_t*>(pa) : 0u;
      a[ks][1] = okB ? *reinterpret_cast<const uint32_t*>(pa + 8 * kEmb) : 0u;
      a[ks][2] = okA ? *reinterpret_cast<const uint32_t*>(pa + 8) : 0u;
      a[ks][3] = okB ? *reinterpret_cast<const uint32_t*>(pa + 8 * kEmb + 8) : 0u;
    }
    float y1[8][4];
#pragma unroll
    for (int nj = 0; nj < 8; ++nj) {
      const int col = nj * 8 + 2 * t;
      float2 vA = make_float2(0.f, 0.f), vB = make_float2(0.f, 0.f);
      if (okA) vA = *reinterpret_cast<const float2*>(y + (r0 + g) * kEmb + col);
      if (okB) vB = *reinterpret_cast<const float2*>(y + (r0 + g + 8) * kEmb + col);
      y1[nj][0] = vA.x, y1[nj][1] = vA.y, y1[nj][2] = vB.x, y1[nj][3] = vB.y;
    }
    tail_tile(sm, a, y1, g, t, tw.eps);
#pragma unroll
    for (int nj = 0; nj < 8; ++nj) {
      const int col = nj * 8 + 2 * t;
      if (okA) *reinterpret_cast<float2*>(y + (r0 + g) * kEmb + col) = make_float2(y1[nj][0], y1[nj][1]);
      if (okB) *reinterpret_cast<float2*>(y + (r0 + g + 8) * kEmb + col) = make_float2(y1[nj][2], y1[nj][3]);
    }
  }
}

}  // namespace

template <typename TIN, bool LN>
void unfold_ln_dispatch(const TIN* xi, __nv_bfloat16* o, int64_t ldo, const float* gamma, const float* beta, float eps, int B, int H,
                        int W, int C, int k, int s, int p, int oh, int ow, long long rows, cudaStream_t st) {
  const unsigned grid = static_cast<unsigned>((rows + 7) / 8);
  if (k == 7 && C == 3 && ldo == 152) {
    constexpr int kIter = 2;  // 8 warps x 4 rows x 2 iterations = 64 rows per block
    const unsigned g773 = static_cast<unsigned>((rows + 64 - 1) / 64);
    unfold773_kernel<TIN, LN, kIter><<<g773, 256, 0, st>>>(xi, o, ldo, gamma, beta, eps, H, W, s, p, oh, ow, rows);
  }
  else if (k == 7 && C == 3) unfold_ln_kernel<TIN, LN, 7, 3><<<grid, 256, 0, st>>>(xi, o, ldo, gamma, beta, eps, B, H, W, C, k, s, p, oh, ow, rows);
  else if (k == 3 && C == 64) unfold_ln_kernel<TIN, LN, 3, 64><<<grid, 256, 0, st>>>(xi, o, ldo, gamma, beta, eps, B, H, W, C, k, s, p, oh, ow, rows);
  else unfold_ln_kernel<TIN, LN, 0, 0><<<grid, 256, 0, st>>>(xi, o, ldo, gamma, beta, eps, B, H, W, C, k, s, p, oh, ow, rows);
}

int unfold_ln_launch(const void* x, int x_dtype, void* out, int64_t ldo, const float* gamma, const float* beta, float eps,
                     int B, int H, int W, int C, int k, int s, int p, cudaStream_t st) {
  EVT_CHECK_ARG(x && out, "unfold_ln: null pointer");
  EVT_CHECK_ARG(B > 0 && H > 0 && W > 0 && C > 0 && k > 0 && s > 0 && p >= 0, "unfold_ln: bad sizes");
  const int L = k * k * C;
  EVT_CHECK_ARG(ldo >= L, "unfold_ln: ldo smaller than k*k*C");
  EVT_CHECK_ARG(ldo % 2 == 0 && reinterpret_cast<uintptr_t>(out) % 4 == 0, "unfold_ln: ldo must be even and out 4-byte aligned");
  if (ldo > 64 * kMaxPairs) return fail(EVT_ERR_UNSUPPORTED, "unfold_ln: rows longer than 576 elements are not implemented");
  EVT_CHECK_ARG((gamma == nullptr) == (beta == nullptr), "unfold_ln: gamma and beta must both be given or both be null");
  const int oh = (H + 2 * p - k) / s + 1, ow = (W + 2 * p - k) / s + 1;
  EVT_CHECK_ARG(oh > 0 && ow > 0, "unfold_ln: empty output");
  const long long rows = static_cast<long long>(B) * oh * ow;
  __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(out);
  const bool ln = gamma != nullptr;
  if (x_dtype == EVT_F32) {
    const float* xi = reinterpret_cast<const float*>(x);
    EVT_CHECK_ARG(reinterpret_cast<uintptr_t>(x) % 8 == 0, "unfold_ln: x must be 8-byte aligned");
    if (ln) unfold_ln_dispatch<float, true>(xi, o, ldo, gamma, beta, eps, B, H, W, C, k, s, p, oh, ow, rows, st);
    else unfold_ln_dispatch<float, false>(xi, o, ldo, gamma, beta, eps, B, H, W, C, k, s, p, oh, ow, rows, st);
  } else if (x_dtype == EVT_BF16) {
    const __nv_bfloat16* xi = reinterpret_cast<const __nv_bfloat16*>(x);
    if (ln) unfold_ln_dispatch<__nv_bfloat16, true>(xi, o, ldo, gamma, beta, eps, B, H, W, C, k, s, p, oh, ow, rows, st);
    else unfold_ln_dispatch<__nv_bfloat16, false>(xi, o, ldo, gamma, beta, eps, B, H, W, C, k, s, p, oh, ow, rows, st);
  } else {
    return fail(EVT_ERR_INVALID, "unfold_ln: x dtype must be f32 or bf16");
  }
  EVT_LAUNCH_CHECK("unfold_ln");
  return EVT_OK;
}

}  // namespace evt

using namespace evt;

extern "C" int evt_unfold_ln_nhwc(const void* x, int x_dtype, void* out, int64_t ldo, const float* gamma,
                                  const float* beta, float eps, int B, int H, int W, int C, int k, int s, int p,
                                  evt_stream stream) {
  int rc = evt_device_check();
  if (rc != EVT_OK) return rc;
  return unfold_ln_launch(x, x_dtype, out, ldo, gamma, beta, eps, B, H, W, C, k, s, p, static_cast<cudaStream_t>(stream));
}

extern "C" int evt_performer_workspace_bytes(int B, int T, size_t* out) {
  EVT_CHECK_ARG(out != nullptr && B > 0 && T > 0, "performer_workspace_bytes: bad arguments");
  *out = evt::performer_workspace_bytes(B, T);
  return EVT_OK;
}

extern "C" int evt_performer_mlp_fwd(const void* ya, float* y, const void* wo, const float* bo, const float* gamma, const float* beta,
                                     const void* w1, const float* b1, const void* w2, const float* b2, int64_t rows, float eps,
                                     evt_stream stream) {
  int rc = evt_device_check();
  if (rc != EVT_OK) return rc;
  return evt::performer_mlp_launch(ya, y, wo, bo, gamma, beta, w1, b1, w2, b2, rows, eps, static_cast<cudaStream_t>(stream));
}

extern "C" int evt_performer_block_fwd(const void* kqv, int64_t ld, const float* w, float* y, void* workspace, int B, int T, float eps,
                                       const void* wo, const float* bo, const float* gamma, const float* beta, const void* w1,
                                       const float* b1, const void* w2, const float* b2, float ln_eps, evt_stream stream) {
  int rc = evt_device_check();
  if (rc != EVT_OK) return rc;
  return evt::performer_block_launch(kqv, ld, w, y, workspace, B, T, eps, wo, bo, gamma, beta, w1, b1, w2, b2, ln_eps,
                                     static_cast<cudaStream_t>(stream));
}

extern "C" int evt_performer_fwd(const void* kqv, int64_t ld, const float* w, void* yattn, float* vout, void* workspace,
                                 int B, int T, int emb, int m, float eps, evt_stream stream) {
  int rc = evt_device_check();
  if (rc != EVT_OK) return rc;
  return evt::performer_launch(kqv, ld, w, yattn, vout, workspace, B, T, emb, m, eps, static_cast<cudaStream_t>(stream));
}

namespace evt {

size_t performer_workspace_bytes(int B, int T) {
  const size_t nsplit = (T + kChunk - 1) / kChunk;
  return static_cast<size_t>(B) * (nsplit + 1) * (kM + kEmb * kM) * sizeof(float);
}

int performer_mlp_launch(const void* ya, float* y, const void* wo, const float* bo, const float* gamma, const float* beta, const void* w1,
                         const float* b1, const void* w2, const float* b2, int64_t rows, float eps, cudaStream_t st) {
  EVT_CHECK_ARG(ya && y && wo && gamma && beta && w1 && w2, "performer_mlp: null pointer");
  EVT_CHECK_ARG(rows > 0, "performer_mlp: rows must be positive");
  for (const void* p : {ya, static_cast<const void*>(y), wo, w1, w2})
    EVT_CHECK_ARG(reinterpret_cast<uintptr_t>(p) % 16 == 0, "performer_mlp: operands must be 16-byte aligned");
  const long long tiles = (rows + kTileTok - 1) / kTileTok;
  const long long want = (tiles + 3) / 4;
  const long long cap = static_cast<long long>(num_sms()) * 16;  // 4-warp blocks: grid-stride beyond 16 resident blocks per SM
  const unsigned grid = static_cast<unsigned>(want < cap ? want : cap);
  TailWeights tw;
  tw.wo = reinterpret_cast<const __nv_bfloat16*>(wo), tw.w1 = reinterpret_cast<const __nv_bfloat16*>(w1), tw.w2 = reinterpret_cast<const __nv_bfloat16*>(w2);
  tw.bo = bo, tw.gamma = gamma, tw.beta = beta, tw.b1 = b1, tw.b2 = b2, tw.eps = eps;
  performer_mlp_kernel<<<grid, 128, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(ya), y, tw, rows);
  EVT_LAUNCH_CHECK("performer_mlp");
  return EVT_OK;
}

int performer_launch(const void* kqv, int64_t ld, const float* w, void* yattn, float* vout, void* workspace, int B, int T, int emb,
                     int m, float eps, cudaStream_t st) {
  EVT_CHECK_ARG(kqv && w && yattn && vout && workspace, "performer: null pointer");
  EVT_CHECK_ARG(B > 0 && T > 0 && B <= 65535, "performer: B in 1..65535 and T > 0");
  if (emb != kEmb || m != kM) return fail(EVT_ERR_UNSUPPORTED, "performer: only emb = 64, m = 32 (T2T token_size 64, kernel_ratio 0.5) is implemented");
  EVT_CHECK_ARG(ld >= 3 * kEmb && ld % 8 == 0 && reinterpret_cast<uintptr_t>(kqv) % 16 == 0,
                "performer: kqv rows must be 16-byte aligned with a leading dimension >= 192");
  EVT_CHECK_ARG(reinterpret_cast<uintptr_t>(w) % 8 == 0 && reinterpret_cast<uintptr_t>(workspace) % 8 == 0 &&
                    reinterpret_cast<uintptr_t>(yattn) % 4 == 0 && reinterpret_cast<uintptr_t>(vout) % 8 == 0,
                "performer: w / workspace / outputs must be 8-byte aligned");
  const int nsplit = (T + kChunk - 1) / kChunk;
  float* partial = reinterpret_cast<float*>(workspace);
  float* stats = partial + static_cast<size_t>(B) * nsplit * (kM + kEmb * kM);
  dim3 grid(nsplit, B);
  performer_reduce_kernel<<<grid, 128, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(kqv), ld, w, partial, T, nsplit);
  EVT_LAUNCH_CHECK("performer_reduce");
  performer_reduce_final_kernel<<<B, 256, 0, st>>>(partial, stats, nsplit);
  EVT_LAUNCH_CHECK("performer_reduce_final");
  performer_apply_kernel<false><<<grid, 128, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(kqv), ld, w, stats,
                                                      reinterpret_cast<__nv_bfloat16*>(yattn), vout, T, eps, TailWeights{});
  EVT_LAUNCH_CHECK("performer_apply");
  return EVT_OK;
}

// The whole Token_performer after the kqv projection: attention contraction + attn_output + LayerNorm + MLP; y f32 [B*T, 64]
int performer_block_launch(const void* kqv, int64_t ld, const float* w, float* y, void* workspace, int B, int T, float eps, const void* wo,
                           const float* bo, const float* gamma, const float* beta, const void* w1, const float* b1, const void* w2,
                           const float* b2, float ln_eps, cudaStream_t st) {
  EVT_CHECK_ARG(kqv && w && y && workspace && wo && gamma && beta && w1 && w2, "performer_block: null pointer");
  EVT_CHECK_ARG(B > 0 && T > 0 && B <= 65535, "performer_block: B in 1..65535 and T > 0");
  EVT_CHECK_ARG(ld >= 3 * kEmb && ld % 8 == 0 && reinterpret_cast<uintptr_t>(kqv) % 16 == 0,
                "performer_block: kqv rows must be 16-byte aligned with a leading dimension >= 192");
  for (const void* p : {static_cast<const void*>(w), static_cast<const void*>(workspace), static_cast<const void*>(y), wo, w1, w2})
    EVT_CHECK_ARG(reinterpret_cast<uintptr_t>(p) % 16 == 0, "performer_block: operands must be 16-byte aligned");
  const int nsplit = (T + kChunk - 1) / kChunk;
  float* partial = reinterpret_cast<float*>(workspace);
  float* stats = partial + static_cast<size_t>(B) * nsplit * (kM + kEmb * kM);
  dim3 grid(nsplit, B);
  performer_reduce_kernel<<<grid, 128, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(kqv), ld, w, partial, T, nsplit);
  EVT_LAUNCH_CHECK("performer_reduce");
  performer_reduce_final_kernel<<<B, 256, 0, st>>>(partial, stats, nsplit);
  EVT_LAUNCH_CHECK("performer_reduce_final");
  TailWeights tw;
  tw.wo = reinterpret_cast<const __nv_bfloat16*>(wo), tw.w1 = reinterpret_cast<const __nv_bfloat16*>(w1), tw.w2 = reinterpret_cast<const __nv_bfloat16*>(w2);
  tw.bo = bo, tw.gamma = gamma, tw.beta = beta, tw.b1 = b1, tw.b2 = b2, tw.eps = ln_eps;
  performer_apply_kernel<true><<<grid, 128, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(kqv), ld, w, stats, nullptr, y, T, eps, tw);
  EVT_LAUNCH_CHECK("performer_apply_tail");
  return EVT_OK;
}

}  // namespace evt
