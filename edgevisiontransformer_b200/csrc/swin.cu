// Kernels of the Swin shifted-window block (SURVEY.md section 8f rank 4; the model tools.py:265-292 export_onnx_swin /
// utils.py:14-47 get_swin builds; arithmetic = SwinLayer / SwinSelfAttention / SwinPatchMerging,
// SITE/models/swin/modeling_swin.py:141-160, 326-349, 410-459, 591-654).
//
// Layout decision: inside a stage the token rows are kept in WINDOW ORDER of the current block (image, window, token
// in window), so the QKV / out-proj / FC1 / FC2 GEMMs and their TMA reduce-add epilogues work on plain row-major
// matrices and a window's 49 tokens are 49 consecutive rows.  Changing the order (cyclic shift on / off, raster ->
// windows after the patch embedding, the 2x2 neighbourhood gather of patch merging) is a row gather fused into the
// LayerNorm that follows it anyway:
//
//   gather_ln_kernel          out row r = LayerNorm( concat_g x[ image(r) * T_in + idx[(r % T_out) * G + g] ] ), G = 1 | 4;
//                             optionally also the raw gathered row as f32 (the permuted residual stream).  HBM-bound.
//   window_attention_kernel   softmax(q k^T * scale + bias_table) v for 49-token windows, head size 32, one warp per
//                             (window, head): q, k, v staged with cp.async into swizzled shared memory, mma.sync
//                             m16n8k16 bf16 with the probabilities kept in registers (accumulator fragments re-used as A
//                             fragments).  A 49 x 49 x 32 problem fills 38 % of a 128-row tcgen05 tile and its time is
//                             exp / load bound, so the warp-level tensor path is used here (a tcgen05 kernel with two
//                             windows per tile was measured slower, DESIGN.md).
//   window_attention144_kernel the same for 12 x 12 windows (144 tokens, swin_*_window12_384); K and V fragments are
//                             re-read from shared memory per query m-tile instead of held in registers.
//   ln_mean_tokens_kernel     final LayerNorm + average pool over the tokens of an image (SwinModel.layernorm + pooler).
#include <cuda_bf16.h>
#include <math_constants.h>

#include "ops.h"
#include "ptx.cuh"

namespace evt {
namespace {

// ---------------------------------------------------------------------------------------------------- gather + LN
// One warp per output row of D = G * C floats (C % 4 == 0, D <= 128 * NV).
template <int NV, int OUT>
__global__ void __launch_bounds__(256) gather_ln_kernel(const float* __restrict__ x, const int* __restrict__ idx,
                                                        const float* __restrict__ gamma, const float* __restrict__ beta,
                                                        void* __restrict__ y, float* __restrict__ copy, long long rows_out,
                                                        int T_in, int T_out, int G, int C, float eps) {
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();
  const int lane = threadIdx.x & 31;
  const long long row = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows_out) return;
  const int D = G * C;
  const long long img = row / T_out;
  const int t = static_cast<int>(row - img * T_out);
  const float* xb = x + img * T_in * static_cast<long long>(C);
  const int* ir = idx + static_cast<long long>(t) * G;
  float4 v[NV];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = i * 128 + lane * 4;
    v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c < D) {
      const int g = c / C;
      const int src = __ldg(ir + g);
      v[i] = *reinterpret_cast<const float4*>(xb + static_cast<long long>(src) * C + (c - g * C));
      s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    }
  }
  if (copy != nullptr) {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = i * 128 + lane * 4;
      if (c < D) *reinterpret_cast<float4*>(copy + row * D + c) = v[i];
    }
  }
  if (y == nullptr) return;
  const float mean = ptx::warp_sum(s) / static_cast<float>(D);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = i * 128 + lane * 4;
    if (c < D) {
      const float a0 = v[i].x - mean, a1 = v[i].y - mean, a2 = v[i].z - mean, a3 = v[i].w - mean;
      q += (a0 * a0 + a1 * a1) + (a2 * a2 + a3 * a3);
    }
  }
  const float rstd = rsqrtf(ptx::warp_sum(q) / static_cast<float>(D) + eps);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = i * 128 + lane * 4;
    if (c < D) {
      const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + c));
      const float4 b = __ldg(reinterpret_cast<const float4*>(beta + c));
      ptx::store_ln4<OUT>(v[i], mean, rstd, g, b, y, D, nullptr, 0, row, c);
    }
  }
}

// G = 1 with narrow rows (C = 96 / 192: Swin stages 1 and 2): 32 / LPR rows per warp, every lane carries NV float4
// (a whole warp per 96-float row leaves a quarter of the lanes idle; these launches cover 802 816 rows at batch 256).
template <int LPR, int NV, int OUT>
__global__ void __launch_bounds__(256) gather_ln_sub_kernel(const float* __restrict__ x, const int* __restrict__ idx,
                                                            const float* __restrict__ gamma, const float* __restrict__ beta,
                                                            void* __restrict__ y, float* __restrict__ copy, long long rows_out,
                                                            int T_in, int T_out, float eps) {
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();
  constexpr int C = 4 * LPR * NV;
  constexpr int RPW = 32 / LPR;
  const int lane = threadIdx.x & 31;
  const int sub = lane / LPR, l = lane % LPR;
  const long long row = (static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5)) * RPW + sub;
  const bool live = row < rows_out;
  const long long r = live ? row : 0;
  const long long img = r / T_out;
  const int src = __ldg(idx + static_cast<int>(r - img * T_out));
  const float* xr = x + (img * T_in + src) * static_cast<long long>(C);
  float4 v[NV];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    v[i] = *reinterpret_cast<const float4*>(xr + (i * LPR + l) * 4);
    s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  }
  if (live && copy != nullptr) {
#pragma unroll
    for (int i = 0; i < NV; ++i) *reinterpret_cast<float4*>(copy + row * C + (i * LPR + l) * 4) = v[i];
  }
  if (y == nullptr) return;
  const float mean = ptx::group_sum<LPR>(s) / static_cast<float>(C);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const float a0 = v[i].x - mean, a1 = v[i].y - mean, a2 = v[i].z - mean, a3 = v[i].w - mean;
    q += (a0 * a0 + a1 * a1) + (a2 * a2 + a3 * a3);
  }
  const float rstd = rsqrtf(ptx::group_sum<LPR>(q) / static_cast<float>(C) + eps);
  if (!live) return;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = (i * LPR + l) * 4;
    const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + c));
    const float4 b = __ldg(reinterpret_cast<const float4*>(beta + c));
    ptx::store_ln4<OUT>(v[i], mean, rstd, g, b, y, C, nullptr, 0, row, c);
  }
}

template <int LPR, int NV>
int launch_gather_ln_sub(const float* x, const int* idx, const float* gamma, const float* beta, void* y, int y_dtype, float* copy,
                         long long rows_out, int T_in, int T_out, float eps, cudaStream_t st) {
  constexpr int RPW = 32 / LPR;
  const unsigned grid = static_cast<unsigned>((rows_out + 8 * RPW - 1) / (8 * RPW));
  const bool pdl = pdl_for_work(rows_out, 4 * LPR * NV);
  if (y_dtype == EVT_BF16)
    EVT_CUDA(launch_pdl(gather_ln_sub_kernel<LPR, NV, EVT_BF16>, dim3(grid), dim3(256), 0, st, pdl, x, idx, gamma, beta, y, copy, rows_out,
                        T_in, T_out, eps));
  else
    EVT_CUDA(launch_pdl(gather_ln_sub_kernel<LPR, NV, EVT_F32>, dim3(grid), dim3(256), 0, st, pdl, x, idx, gamma, beta, y, copy, rows_out,
                        T_in, T_out, eps));
  EVT_LAUNCH_CHECK("gather_ln_sub_kernel");
  return EVT_OK;
}

template <int NV>
int launch_gather_ln(const float* x, const int* idx, const float* gamma, const float* beta, void* y, int y_dtype, float* copy,
                     long long rows_out, int T_in, int T_out, int G, int C, float eps, cudaStream_t st) {
  const unsigned grid = static_cast<unsigned>((rows_out + 7) / 8);
  const bool pdl = pdl_for_work(rows_out, static_cast<long long>(G) * C);
  if (y_dtype == EVT_BF16)
    EVT_CUDA(launch_pdl(gather_ln_kernel<NV, EVT_BF16>, dim3(grid), dim3(256), 0, st, pdl, x, idx, gamma, beta, y, copy, rows_out, T_in,
                        T_out, G, C, eps));
  else
    EVT_CUDA(launch_pdl(gather_ln_kernel<NV, EVT_F32>, dim3(grid), dim3(256), 0, st, pdl, x, idx, gamma, beta, y, copy, rows_out, T_in,
                        T_out, G, C, eps));
  EVT_LAUNCH_CHECK("gather_ln_kernel");
  return EVT_OK;
}

// ---------------------------------------------------------------------------------------------------- window attention
constexpr int kWTok = 49;     // 7 x 7 window
constexpr int kWHd = 32;      // head size of every Swin variant (C / heads = 96 / 3 = ... = 32)
constexpr int kWRows = 64;    // query / key rows per matrix in shared memory (49 + zero padding)
constexpr int kWKeyCols = 56; // key columns of the score tile (7 n-tiles of 8); columns 49..55 carry -inf in the table
constexpr int kWWarps = 4;
constexpr int kWMatBytes = kWRows * kWHd * 2;  // 4 KB

// 12 x 12 windows (swin_*_window12_384): 144 = 9 m16 query tiles x 18 n8 key tiles, no padding
constexpr int kW12Tok = 144;
constexpr int kW12Warps = 4;                    // 4 x 27 KB per CTA: 2 CTAs = 8 warps per SM
constexpr int kW12MatBytes = kW12Tok * kWHd * 2;  // 9 KB

// byte offset of (row, 16-byte chunk) in a [rows][64 bytes] matrix: chunks XOR-swizzled by (row / 2) % 4, so the
// eight 16-byte rows an ldmatrix phase reads fall into eight different bank groups
__device__ __forceinline__ uint32_t wofs(int row, int chunk) { return row * 64 + ((chunk ^ ((row >> 1) & 3)) << 4); }

// cp.async the q, k and v slices of head h of the window whose first row is row0 (TOK rows each) into the warp's three
// swizzled matrices at aQ, aQ + MAT, aQ + 2 MAT, and wait for them
template <int TOK, int MAT>
__device__ __forceinline__ void stage_window(const __nv_bfloat16* __restrict__ qkv, long long ldq, long long row0, int C, int h,
                                             uint32_t aQ, int lane) {
  for (int c = lane; c < 3 * TOK * 4; c += 32) {
    const int mat = c / (TOK * 4), rc = c - mat * (TOK * 4);
    const int row = rc >> 2, ch = rc & 3;
    const __nv_bfloat16* src = qkv + (row0 + row) * ldq + mat * C + h * kWHd + ch * 8;
    const uint32_t dst = aQ + mat * MAT + wofs(row, ch);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
  }
  asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory");
}

// Scores of the rows g and g + 8 of one m-tile (NT n-tiles) -> log2 domain plus the table rows t0 / t1 (columns
// 8 nt + 2 t, + 1); m0 / m1 = the row maxima over the quad
template <int NT>
__device__ __forceinline__ void scores_rowmax(float (&s)[NT][4], const float* __restrict__ t0, const float* __restrict__ t1,
                                              float scale_log2e, float& m0, float& m1) {
  m0 = -CUDART_INF_F, m1 = -CUDART_INF_F;
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) {
    const float2 b0 = __ldg(reinterpret_cast<const float2*>(t0 + nt * 8));
    const float2 b1 = __ldg(reinterpret_cast<const float2*>(t1 + nt * 8));
    s[nt][0] = fmaf(s[nt][0], scale_log2e, b0.x);
    s[nt][1] = fmaf(s[nt][1], scale_log2e, b0.y);
    s[nt][2] = fmaf(s[nt][2], scale_log2e, b1.x);
    s[nt][3] = fmaf(s[nt][3], scale_log2e, b1.y);
    m0 = fmaxf(m0, fmaxf(s[nt][0], s[nt][1]));
    m1 = fmaxf(m1, fmaxf(s[nt][2], s[nt][3]));
  }
  m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1));
  m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 2));
  m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1));
  m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 2));
}

// Probabilities 2^(s - m) as the A fragments of the (NT + 1) / 2 k-steps of P V (an odd NT leaves the last k-step's upper
// half zero: those keys do not exist); l0 / l1 = the row sums over the quad
template <int NT>
__device__ __forceinline__ void exp_rowsum(const float (&s)[NT][4], float m0, float m1, uint32_t (&pa)[(NT + 1) / 2][4], float& l0,
                                           float& l1) {
  l0 = 0.f, l1 = 0.f;
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) {
    const float p0 = ptx::ex2_approx(s[nt][0] - m0), p1 = ptx::ex2_approx(s[nt][1] - m0);
    const float p2 = ptx::ex2_approx(s[nt][2] - m1), p3 = ptx::ex2_approx(s[nt][3] - m1);
    l0 += p0 + p1;
    l1 += p2 + p3;
    pa[nt >> 1][(nt & 1) * 2] = ptx::pack_bf16x2(p0, p1);
    pa[nt >> 1][(nt & 1) * 2 + 1] = ptx::pack_bf16x2(p2, p3);
  }
  if (NT & 1) pa[NT >> 1][2] = pa[NT >> 1][3] = 0u;
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
  l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
}

// qkv  bf16 [n_windows * 49, ldq], columns q | k | v (each heads * 32), head h at h * 32 inside each
// tab  f32 [n_tab, heads, 64, 56] = (relative position bias + shift mask) * log2(e); key columns >= 49 hold -inf
// ctx  bf16 [n_windows * 49, ldc]
__global__ void __launch_bounds__(kWWarps * 32) window_attention_kernel(const __nv_bfloat16* __restrict__ qkv, long long ldq,
                                                                        __nv_bfloat16* __restrict__ ctx, long long ldc,
                                                                        const float* __restrict__ tab, int n_tab, int heads,
                                                                        long long n_items, float scale_log2e) {
  extern __shared__ __align__(128) uint8_t wsm[];
  ptx::grid_dep_launch();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint8_t* sQ = wsm + warp * 3 * kWMatBytes;
  uint8_t* sK = sQ + kWMatBytes;
  uint8_t* sV = sK + kWMatBytes;
  // zero the padding rows 49..63 once (cp.async never touches them): P = 0 there must meet finite V, and padded K
  // rows only feed columns the table masks
  for (int i = lane; i < 3 * (kWRows - kWTok) * 4; i += 32) {
    const int mat = i / ((kWRows - kWTok) * 4), rc = i % ((kWRows - kWTok) * 4);
    *reinterpret_cast<uint4*>(sQ + mat * kWMatBytes + wofs(kWTok + rc / 4, rc % 4)) = make_uint4(0, 0, 0, 0);
  }
  ptx::grid_dep_wait();
  const int C = heads * kWHd;
  const int g = lane >> 2, t = lane & 3;
  const uint32_t aQ = ptx::smem_u32(sQ), aK = ptx::smem_u32(sK), aV = ptx::smem_u32(sV);
  for (long long item = static_cast<long long>(blockIdx.x) * kWWarps + warp; item < n_items;
       item += static_cast<long long>(gridDim.x) * kWWarps) {
    const long long w = item / heads;
    const int h = static_cast<int>(item - w * heads);
    const long long row0 = w * kWTok;
    __syncwarp();  // every lane is done with the previous item's shared memory
    stage_window<kWTok, kWMatBytes>(qkv, ldq, row0, C, h, aQ, lane);
    __syncwarp();
    // K fragments (B operand of S = Q K^T): n-tile nt = keys 8 nt .. 8 nt + 7; registers {ks0.b0, ks0.b1, ks1.b0, ks1.b1}
    uint32_t kb[7][4];
#pragma unroll
    for (int nt = 0; nt < 7; ++nt) ptx::ldmatrix_x4(aK + wofs(nt * 8 + (lane & 7), lane >> 3), kb[nt]);
    // V fragments (B operand of O = P V): k-step kk = keys 16 kk .. +15, dims chunk pair cp: {n 2cp: b0, b1, n 2cp+1: b0, b1}
    uint32_t vb[4][2][4];
#pragma unroll
    for (int kk = 0; kk < 4; ++kk)
#pragma unroll
      for (int cp = 0; cp < 2; ++cp)
        ptx::ldmatrix_x4_trans(aV + wofs(kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8, cp * 2 + (lane >> 4)), vb[kk][cp]);
    const float* tb = tab + ((w % n_tab) * heads + h) * static_cast<long long>(kWRows * kWKeyCols);
#pragma unroll 1
    for (int mt = 0; mt < 4; ++mt) {
      uint32_t qa[2][4];
#pragma unroll
      for (int ks = 0; ks < 2; ++ks) ptx::ldmatrix_x4(aQ + wofs(mt * 16 + (lane & 7) + ((lane >> 3) & 1) * 8, ks * 2 + (lane >> 4)), qa[ks]);
      float s[7][4];
#pragma unroll
      for (int nt = 0; nt < 7; ++nt) {
        s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
        ptx::mma_bf16_16816(s[nt], qa[0], kb[nt][0], kb[nt][1]);
        ptx::mma_bf16_16816(s[nt], qa[1], kb[nt][2], kb[nt][3]);
      }
      // scores -> log2 domain with bias / mask; rows g and g + 8 of this m-tile, columns 8 nt + 2 t, + 1
      const float* t0 = tb + (mt * 16 + g) * kWKeyCols + 2 * t;
      const float* t1 = t0 + 8 * kWKeyCols;
      float m0, m1, l0, l1;
      scores_rowmax<7>(s, t0, t1, scale_log2e, m0, m1);
      uint32_t pa[4][4];  // probabilities as A fragments of the four k-steps (keys 56..63 do not exist -> 0)
      exp_rowsum<7>(s, m0, m1, pa, l0, l1);
      float o[4][4];
#pragma unroll
      for (int n = 0; n < 4; ++n) o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f;
#pragma unroll
      for (int kk = 0; kk < 4; ++kk)
#pragma unroll
        for (int n = 0; n < 4; ++n) ptx::mma_bf16_16816(o[n], pa[kk], vb[kk][n >> 1][(n & 1) * 2], vb[kk][n >> 1][(n & 1) * 2 + 1]);
      const float i0 = 1.0f / l0, i1 = 1.0f / l1;  // l >= 1: the row maximum contributes 2^0
      const int r0 = mt * 16 + g, r1 = r0 + 8;
#pragma unroll
      for (int n = 0; n < 4; ++n) {
        const int col = h * kWHd + n * 8 + 2 * t;
        if (r0 < kWTok) *reinterpret_cast<uint32_t*>(ctx + (row0 + r0) * ldc + col) = ptx::pack_bf16x2(o[n][0] * i0, o[n][1] * i0);
        if (r1 < kWTok) *reinterpret_cast<uint32_t*>(ctx + (row0 + r1) * ldc + col) = ptx::pack_bf16x2(o[n][2] * i1, o[n][3] * i1);
      }
    }
  }
}

// The same for 144-token windows.  All K fragments (18 n-tiles x 4) and V fragments (9 k-steps x 8) would take 144
// registers beside the 72 of the score tile, so both are re-read from shared memory with ldmatrix for every query m-tile
// (18 + 18 ldmatrix.x4 against 72 mma per m-tile); the score tile of one m-tile holds every key, so the softmax needs no
// rescale.
// qkv  bf16 [n_windows * 144, ldq], columns q | k | v (each heads * 32), head h at h * 32 inside each
// tab  f32 [n_tab, heads, 144, 144] = (relative position bias + shift mask) * log2(e)
// ctx  bf16 [n_windows * 144, ldc]
__global__ void __launch_bounds__(kW12Warps * 32) window_attention144_kernel(const __nv_bfloat16* __restrict__ qkv, long long ldq,
                                                                            __nv_bfloat16* __restrict__ ctx, long long ldc,
                                                                            const float* __restrict__ tab, int n_tab, int heads,
                                                                            long long n_items, float scale_log2e) {
  constexpr int NT = kW12Tok / 8, KS = kW12Tok / 16;
  extern __shared__ __align__(128) uint8_t wsm[];
  ptx::grid_dep_launch();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t aQ = ptx::smem_u32(wsm + warp * 3 * kW12MatBytes), aK = aQ + kW12MatBytes, aV = aK + kW12MatBytes;
  ptx::grid_dep_wait();
  const int C = heads * kWHd;
  const int g = lane >> 2, t = lane & 3;
  for (long long item = static_cast<long long>(blockIdx.x) * kW12Warps + warp; item < n_items;
       item += static_cast<long long>(gridDim.x) * kW12Warps) {
    const long long w = item / heads;
    const int h = static_cast<int>(item - w * heads);
    const long long row0 = w * kW12Tok;
    __syncwarp();  // every lane is done with the previous item's shared memory
    stage_window<kW12Tok, kW12MatBytes>(qkv, ldq, row0, C, h, aQ, lane);
    __syncwarp();
    const float* tb = tab + ((w % n_tab) * heads + h) * static_cast<long long>(kW12Tok * kW12Tok);
#pragma unroll 1
    for (int mt = 0; mt < KS; ++mt) {
      uint32_t qa[2][4];
#pragma unroll
      for (int ks = 0; ks < 2; ++ks) ptx::ldmatrix_x4(aQ + wofs(mt * 16 + (lane & 7) + ((lane >> 3) & 1) * 8, ks * 2 + (lane >> 4)), qa[ks]);
      float s[NT][4];
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        uint32_t kb[4];  // keys 8 nt .. 8 nt + 7: {ks0.b0, ks0.b1, ks1.b0, ks1.b1}
        ptx::ldmatrix_x4(aK + wofs(nt * 8 + (lane & 7), lane >> 3), kb);
        s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
        ptx::mma_bf16_16816(s[nt], qa[0], kb[0], kb[1]);
        ptx::mma_bf16_16816(s[nt], qa[1], kb[2], kb[3]);
      }
      const float* t0 = tb + (mt * 16 + g) * kW12Tok + 2 * t;
      float m0, m1, l0, l1;
      scores_rowmax<NT>(s, t0, t0 + 8 * kW12Tok, scale_log2e, m0, m1);
      uint32_t pa[KS][4];
      exp_rowsum<NT>(s, m0, m1, pa, l0, l1);
      float o[4][4];
#pragma unroll
      for (int n = 0; n < 4; ++n) o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f;
#pragma unroll
      for (int kk = 0; kk < KS; ++kk) {
        uint32_t vb[2][4];  // keys 16 kk .. +15, dims chunk pair cp: {n 2cp: b0, b1, n 2cp+1: b0, b1}
#pragma unroll
        for (int cp = 0; cp < 2; ++cp)
          ptx::ldmatrix_x4_trans(aV + wofs(kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8, cp * 2 + (lane >> 4)), vb[cp]);
#pragma unroll
        for (int n = 0; n < 4; ++n) ptx::mma_bf16_16816(o[n], pa[kk], vb[n >> 1][(n & 1) * 2], vb[n >> 1][(n & 1) * 2 + 1]);
      }
      const float i0 = 1.0f / l0, i1 = 1.0f / l1;  // l >= 1: the row maximum contributes 2^0
      const long long r0 = row0 + mt * 16 + g, r1 = r0 + 8;
#pragma unroll
      for (int n = 0; n < 4; ++n) {
        const int col = h * kWHd + n * 8 + 2 * t;
        *reinterpret_cast<uint32_t*>(ctx + r0 * ldc + col) = ptx::pack_bf16x2(o[n][0] * i0, o[n][1] * i0);
        *reinterpret_cast<uint32_t*>(ctx + r1 * ldc + col) = ptx::pack_bf16x2(o[n][2] * i1, o[n][3] * i1);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------- final LN + pool
// One CTA (8 warps) per image: every warp normalises tokens warp, warp + 8, ... and accumulates them; the warps' sums meet
// in shared memory.  D % 4 == 0, D <= 128 * NV.
template <int NV>
__global__ void __launch_bounds__(256) ln_mean_tokens_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                                             const float* __restrict__ beta, __nv_bfloat16* __restrict__ y,
                                                             int T, int D, float eps) {
  __shared__ float acc_s[8][128 * NV];
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float* xb = x + static_cast<long long>(blockIdx.x) * T * D;
  float4 acc[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int tk = warp; tk < T; tk += 8) {
    const float* xr = xb + static_cast<long long>(tk) * D;
    float4 v[NV];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = i * 128 + lane * 4;
      v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c < D) {
        v[i] = *reinterpret_cast<const float4*>(xr + c);
        s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
      }
    }
    const float mean = ptx::warp_sum(s) / static_cast<float>(D);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = i * 128 + lane * 4;
      if (c < D) {
        const float a0 = v[i].x - mean, a1 = v[i].y - mean, a2 = v[i].z - mean, a3 = v[i].w - mean;
        q += (a0 * a0 + a1 * a1) + (a2 * a2 + a3 * a3);
      }
    }
    const float rstd = rsqrtf(ptx::warp_sum(q) / static_cast<float>(D) + eps);
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      acc[i].x += (v[i].x - mean) * rstd;
      acc[i].y += (v[i].y - mean) * rstd;
      acc[i].z += (v[i].z - mean) * rstd;
      acc[i].w += (v[i].w - mean) * rstd;
    }
  }
#pragma unroll
  for (int i = 0; i < NV; ++i) *reinterpret_cast<float4*>(&acc_s[warp][i * 128 + lane * 4]) = acc[i];
  __syncthreads();
  // mean_t(LN(x_t)) = gamma * mean_t(xhat_t) + beta
  const float inv_t = 1.0f / static_cast<float>(T);
  for (int c = threadIdx.x; c < D; c += blockDim.x) {
    float s = 0.f;
#pragma unroll
    for (int w8 = 0; w8 < 8; ++w8) s += acc_s[w8][c];
    y[static_cast<long long>(blockIdx.x) * D + c] = __float2bfloat16_rn(s * inv_t * gamma[c] + beta[c]);
  }
}

// ---------------------------------------------------------------------------------------------------- im2col, P % 4 == 0
// One thread = 4 consecutive pixels of one image row (16 B in, 8 B out); same (c, i, j) K order as im2col_kernel.
__global__ void __launch_bounds__(256) im2col4_kernel(const float* __restrict__ px, __nv_bfloat16* __restrict__ cols, int H,
                                                      int W, int P, long long total) {
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();
  const long long tid = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (tid >= total) return;
  const int w4 = W / 4;
  const int x4 = static_cast<int>(tid % w4);
  long long r = tid / w4;
  const int y = static_cast<int>(r % H);
  r /= H;
  const int c = static_cast<int>(r % 3);
  const long long b = r / 3;
  const float4 v = *reinterpret_cast<const float4*>(px + tid * 4);
  const int x = x4 * 4;
  const int py = y / P, i = y % P, pxi = x / P, j = x % P;
  const long long row = (b * (H / P) + py) * (W / P) + pxi;
  const int k = (c * P + i) * P + j;
  uint2 o;
  o.x = ptx::pack_bf16x2(v.x, v.y);
  o.y = ptx::pack_bf16x2(v.z, v.w);
  *reinterpret_cast<uint2*>(cols + row * (3ll * P * P) + k) = o;
}

}  // namespace

int im2col4_launch(const float* pixels, void* cols, int B, int H, int W, int P, cudaStream_t st) {
  const long long total = static_cast<long long>(B) * 3 * H * (W / 4);
  EVT_CUDA(launch_pdl(im2col4_kernel, dim3(static_cast<unsigned>((total + 255) / 256)), dim3(256), 0, st, false, pixels,
                      reinterpret_cast<__nv_bfloat16*>(cols), H, W, P, total));
  EVT_LAUNCH_CHECK("im2col4_kernel");
  return EVT_OK;
}

int gather_layernorm_launch(const float* x, const int* idx, const float* gamma, const float* beta, void* y, int y_dtype, float* copy_f32,
                            int64_t images, int T_in, int T_out, int G, int C, float eps, cudaStream_t st) {
  EVT_CHECK_ARG(x && idx, "gather_layernorm: null pointer");
  EVT_CHECK_ARG(y != nullptr || copy_f32 != nullptr, "gather_layernorm: nothing to write");
  EVT_CHECK_ARG(y == nullptr || (gamma && beta), "gather_layernorm: LayerNorm output needs gamma and beta");
  EVT_CHECK_ARG(images > 0 && T_in > 0 && T_out > 0 && (G == 1 || G == 4), "gather_layernorm: bad sizes (G must be 1 or 4)");
  EVT_CHECK_ARG(C > 0 && C % 4 == 0 && G * C <= 3072, "gather_layernorm: C must be a multiple of 4 with G*C <= 3072");
  EVT_CHECK_ARG(y_dtype == EVT_BF16 || y_dtype == EVT_F32, "gather_layernorm: y dtype must be bf16 or f32");
  EVT_CHECK_ARG(eps >= 0.f, "gather_layernorm: negative eps");
  const long long rows = images * T_out;
  const int D = G * C;
  if (G == 1 && C == 96) return launch_gather_ln_sub<8, 3>(x, idx, gamma, beta, y, y_dtype, copy_f32, rows, T_in, T_out, eps, st);
  if (G == 1 && C == 192) return launch_gather_ln_sub<16, 3>(x, idx, gamma, beta, y, y_dtype, copy_f32, rows, T_in, T_out, eps, st);
  const int nv = (D + 127) / 128;
  if (nv <= 1) return launch_gather_ln<1>(x, idx, gamma, beta, y, y_dtype, copy_f32, rows, T_in, T_out, G, C, eps, st);
  if (nv <= 2) return launch_gather_ln<2>(x, idx, gamma, beta, y, y_dtype, copy_f32, rows, T_in, T_out, G, C, eps, st);
  if (nv <= 3) return launch_gather_ln<3>(x, idx, gamma, beta, y, y_dtype, copy_f32, rows, T_in, T_out, G, C, eps, st);
  if (nv <= 6) return launch_gather_ln<6>(x, idx, gamma, beta, y, y_dtype, copy_f32, rows, T_in, T_out, G, C, eps, st);
  if (nv <= 12) return launch_gather_ln<12>(x, idx, gamma, beta, y, y_dtype, copy_f32, rows, T_in, T_out, G, C, eps, st);
  return launch_gather_ln<24>(x, idx, gamma, beta, y, y_dtype, copy_f32, rows, T_in, T_out, G, C, eps, st);
}

int window_attention_launch(const void* qkv, int64_t ldq, void* ctx, int64_t ldc, const float* table, int n_tab, int64_t n_windows,
                            int window_tokens, int heads, int head_size, float scale, cudaStream_t st) {
  EVT_CHECK_ARG(qkv && ctx && table, "window_attention: null pointer");
  EVT_CHECK_ARG(n_windows > 0 && heads > 0 && n_tab > 0, "window_attention: sizes must be positive");
  if ((window_tokens != kWTok && window_tokens != kW12Tok) || head_size != kWHd)
    return fail(EVT_ERR_UNSUPPORTED,
                "window_attention: only 7x7 (49-token) and 12x12 (144-token) windows with head size 32 are implemented");
  EVT_CHECK_ARG(ldq >= 3ll * heads * kWHd && ldc >= static_cast<int64_t>(heads) * kWHd, "window_attention: leading dimension too small");
  EVT_CHECK_ARG(ldq % 8 == 0 && reinterpret_cast<uintptr_t>(qkv) % 16 == 0, "window_attention: qkv rows must be 16-byte aligned");
  EVT_CHECK_ARG(ldc % 2 == 0 && reinterpret_cast<uintptr_t>(ctx) % 4 == 0, "window_attention: ctx rows must be 4-byte aligned");
  const long long items = n_windows * heads;
  if (window_tokens == kW12Tok) {
    const int smem = kW12Warps * 3 * kW12MatBytes;
    EVT_TRY(opt_in_smem<window_attention144_kernel>(smem));
    const long long ctas_needed = (items + kW12Warps - 1) / kW12Warps;
    const long long cap = static_cast<long long>(num_sms()) * 2;  // 2 CTAs of 108 KB per SM, grid-stride over the rest
    const unsigned grid = static_cast<unsigned>(ctas_needed < cap ? ctas_needed : cap);
    EVT_CUDA(launch_pdl(window_attention144_kernel, dim3(grid), dim3(kW12Warps * 32), smem, st,
                        pdl_for_work(n_windows * kW12Tok, static_cast<long long>(heads) * kWHd), reinterpret_cast<const __nv_bfloat16*>(qkv),
                        static_cast<long long>(ldq), reinterpret_cast<__nv_bfloat16*>(ctx), static_cast<long long>(ldc), table, n_tab, heads,
                        items, scale * 1.4426950408889634f));
    EVT_LAUNCH_CHECK("window_attention144_kernel");
    return EVT_OK;
  }
  const int smem = kWWarps * 3 * kWMatBytes;
  EVT_TRY(opt_in_smem<window_attention_kernel>(smem));
  const long long ctas_needed = (items + kWWarps - 1) / kWWarps;
  const long long cap = static_cast<long long>(num_sms()) * 4;  // 4 CTAs of 48 KB per SM, grid-stride over the rest
  const unsigned grid = static_cast<unsigned>(ctas_needed < cap ? ctas_needed : cap);
  EVT_CUDA(launch_pdl(window_attention_kernel, dim3(grid), dim3(kWWarps * 32), smem, st,
                      pdl_for_work(n_windows * kWTok, static_cast<long long>(heads) * kWHd), reinterpret_cast<const __nv_bfloat16*>(qkv), static_cast<long long>(ldq),
                      reinterpret_cast<__nv_bfloat16*>(ctx), static_cast<long long>(ldc), table, n_tab, heads, items,
                      scale * 1.4426950408889634f));
  EVT_LAUNCH_CHECK("window_attention_kernel");
  return EVT_OK;
}

int layernorm_mean_tokens_launch(const float* x, const float* gamma, const float* beta, void* y, int64_t images, int T, int D, float eps,
                                 cudaStream_t st) {
  EVT_CHECK_ARG(x && gamma && beta && y, "layernorm_mean_tokens: null pointer");
  EVT_CHECK_ARG(images > 0 && T > 0 && D > 0 && D % 4 == 0 && D <= 1536, "layernorm_mean_tokens: D must be a multiple of 4, <= 1536");
  const dim3 grid(static_cast<unsigned>(images));
  __nv_bfloat16* yo = reinterpret_cast<__nv_bfloat16*>(y);
  const int nv = (D + 127) / 128;
  if (nv <= 3) EVT_CUDA(launch_pdl(ln_mean_tokens_kernel<3>, grid, dim3(256), 0, st, false, x, gamma, beta, yo, T, D, eps));
  else if (nv <= 6) EVT_CUDA(launch_pdl(ln_mean_tokens_kernel<6>, grid, dim3(256), 0, st, false, x, gamma, beta, yo, T, D, eps));
  else EVT_CUDA(launch_pdl(ln_mean_tokens_kernel<12>, grid, dim3(256), 0, st, false, x, gamma, beta, yo, T, D, eps));
  EVT_LAUNCH_CHECK("ln_mean_tokens_kernel");
  return EVT_OK;
}

}  // namespace evt

extern "C" int evt_gather_layernorm(const float* x, const int* idx, const float* gamma, const float* beta, void* y, int y_dtype,
                                    float* copy_f32, int64_t images, int T_in, int T_out, int G, int C, float eps,
                                    evt_stream stream) {
  int rc = evt_device_check();
  if (rc != EVT_OK) return rc;
  return evt::gather_layernorm_launch(x, idx, gamma, beta, y, y_dtype, copy_f32, images, T_in, T_out, G, C, eps,
                                      static_cast<cudaStream_t>(stream));
}

extern "C" int evt_window_attention_fwd(const void* qkv, int64_t ldq, void* ctx, int64_t ldc, const float* table, int n_tab,
                                        int64_t n_windows, int window_tokens, int heads, int head_size, float scale,
                                        evt_stream stream) {
  int rc = evt_device_check();
  if (rc != EVT_OK) return rc;
  return evt::window_attention_launch(qkv, ldq, ctx, ldc, table, n_tab, n_windows, window_tokens, heads, head_size, scale,
                                      static_cast<cudaStream_t>(stream));
}

extern "C" int evt_layernorm_mean_tokens(const float* x, const float* gamma, const float* beta, void* y, int64_t images, int T,
                                         int D, float eps, evt_stream stream) {
  int rc = evt_device_check();
  if (rc != EVT_OK) return rc;
  return evt::layernorm_mean_tokens_launch(x, gamma, beta, y, images, T, D, eps, static_cast<cudaStream_t>(stream));
}
