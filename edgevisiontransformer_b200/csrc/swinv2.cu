// Kernels of the Swin V2 block (SITE/models/swinv2/modeling_swinv2.py: Swinv2SelfAttention.forward :421-470, the continuous
// position bias :490-524, Swinv2Layer.forward :662-716, Swinv2PatchMerging :365-387).  The token rows keep the window order
// of the V1 path (swin.cu): a window's N tokens are N consecutive rows of the qkv / ctx matrices.
//
//   cosine_window_attention_kernel  softmax(normalize(q) normalize(k)^T * exp(min(logit_scale, ln 100)) + bias + mask) v
//                                   for 8 x 8 and 16 x 16 windows, head size 32.  q and k rows are normalised in f32 in
//                                   shared memory and stored back as f16 (|x| <= 1: f16 keeps 3 more mantissa bits than
//                                   bf16 at no range cost); scores from mma.sync m16n8k16 f16, P V in bf16, f32 softmax.
//                                   Each warp owns 64 query rows and runs them against 64-key blocks with an online
//                                   softmax: one block for 64-token windows, four for 256-token windows (whose four warps
//                                   share one (window, head) and its K / V in shared memory).  The relative position bias
//                                   comes from a compact per-head table [(2w-1)^2], staged in shared memory beside q / k / v
//                                   and indexed arithmetically, and the shift-mask region of each (query, key) pair is
//                                   computed from the window index and the token coordinates: no dense
//                                   [windows, heads, N, N] table exists.
//   postnorm_residual_kernel        out = resid + LayerNorm(y) (post-norm residual update; resid nullable: patch
//                                   merging's LayerNorm after the reduction), optionally through a row gather (the next
//                                   block's window order, or patch merging's 2 x 2 concat), writing the f32 stream and /
//                                   or its bf16 copy, the next GEMM's A operand.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <math_constants.h>

#include <cmath>
#include <vector>

#include "ops.h"
#include "ptx.cuh"

namespace evt {

// Index arithmetic shared by the kernel and the host-side dense restatement (evt_swinv2_score_bias).
// Row of the compact (2w-1) x (2w-1) bias table for query (qi, qj) and key (ki, kj) of a w x w window = HF
// relative_position_index (:512-522).
__host__ __device__ __forceinline__ int v2_rel_index(int qi, int qj, int ki, int kj, int ws) {
  return (qi - ki + ws - 1) * (2 * ws - 1) + (qj - kj + ws - 1);
}
// Shift-mask region (0, 1, 2) along one axis of the token at in-window coordinate i of window wc (of nw per axis):
// Swinv2Layer.get_attn_mask's slices (0, -w), (-w, -shift), (-shift, None) of the rolled image.
__host__ __device__ __forceinline__ int v2_region(int wc, int nw, int i, int ws, int shift) {
  return wc < nw - 1 ? 0 : (i < ws - shift ? 1 : 2);
}

namespace {

constexpr int kV2Hd = 32;     // head size of every Swin V2 variant
constexpr int kV2Warps = 4;
constexpr int kV2Rows = 64;   // query rows per warp = keys per softmax block

// byte offset of (row, 16-byte chunk) in a [rows][64 bytes] matrix, chunks XOR-swizzled by (row / 2) % 4 (as swin.cu)
__device__ __forceinline__ uint32_t vofs(int row, int chunk) { return row * 64 + ((chunk ^ ((row >> 1) & 3)) << 4); }

// d += a b, m16n8k16, f16 operands, f32 accumulate
__device__ __forceinline__ void mma_f16_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

__device__ __forceinline__ float quad_max(float v) {
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
  return fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
}

// qkv  bf16 [n_windows * WS^2, ldq], columns q | k | v (heads * 32 each), rows in window order
// tab  f32 [heads, (2 WS - 1)^2] = 16 sigmoid(cpb_mlp(coords)) * log2(e)
// hsc  f32 [heads] = exp(min(logit_scale, ln 100)) * log2(e)
// window w of the launch is window w % nw^2 of its image (nw = windows per image side); shift > 0: masked pairs get
// mask_log2 added (the shift mask times log2(e))
// ctx  bf16 [n_windows * WS^2, ldc]
template <int WS>
__global__ void __launch_bounds__(kV2Warps * 32) cosine_window_attention_kernel(const __nv_bfloat16* __restrict__ qkv, long long ldq,
                                                                               __nv_bfloat16* __restrict__ ctx, long long ldc,
                                                                               const float* __restrict__ tab, const float* __restrict__ hsc,
                                                                               int heads, long long n_items, int nw, int shift,
                                                                               float mask_log2) {
  constexpr int TOK = WS * WS, WPI = TOK / kV2Rows, IPC = kV2Warps / WPI, MAT = TOK * kV2Hd * 2, KB = TOK / kV2Rows;
  constexpr int NTAB = (2 * WS - 1) * (2 * WS - 1);
  extern __shared__ __align__(128) uint8_t wsm[];
  // per slot: q, k, v [TOK][64 B] each; after all slots' matrices, each slot's head bias table (NTAB floats)
  ptx::grid_dep_launch();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int slot = warp / WPI, part = warp % WPI;  // (window, head) slot of the CTA; which 64 query rows of it
  const int tid = part * 32 + lane;                // thread index among the warps of the slot
  uint8_t* sQ = wsm + slot * 3 * MAT;
  float* sTab = reinterpret_cast<float*>(wsm + IPC * 3 * MAT) + slot * NTAB;
  const uint32_t aQ = ptx::smem_u32(sQ), aK = aQ + MAT, aV = aK + MAT;
  ptx::grid_dep_wait();
  const int C = heads * kV2Hd;
  const int g = lane >> 2, t = lane & 3;
  const long long n_groups = (n_items + IPC - 1) / IPC;
  for (long long grp = blockIdx.x; grp < n_groups; grp += gridDim.x) {
    const long long item = grp * IPC + slot;
    const bool live = item < n_items;
    const long long w = live ? item / heads : 0;
    const int h = static_cast<int>(item - w * heads);
    const long long row0 = w * TOK;
    __syncthreads();  // every warp is done with the previous group's shared memory
    if (live) {
      for (int c = tid; c < 3 * TOK * 4; c += 32 * WPI) {
        const int mat = c / (TOK * 4), rc = c - mat * (TOK * 4);
        const int row = rc >> 2, ch = rc & 3;
        const __nv_bfloat16* src = qkv + (row0 + row) * ldq + mat * C + h * kV2Hd + ch * 8;
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(aQ + mat * MAT + vofs(row, ch)), "l"(src) : "memory");
      }
      asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory");
      for (int i = tid; i < NTAB; i += 32 * WPI) sTab[i] = __ldg(tab + static_cast<long long>(h) * NTAB + i);
    }
    __syncthreads();
    // q and k rows -> normalize(x) = x / max(|x|, 1e-12) in f32 (F.normalize), stored back as f16
    if (live) {
      for (int r = tid; r < 2 * TOK; r += 32 * WPI) {
        uint8_t* m = sQ + (r >= TOK ? MAT : 0);
        const int row = r >= TOK ? r - TOK : r;
        float x[32];
        float ss = 0.f;
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
          const uint4 u = *reinterpret_cast<const uint4*>(m + vofs(row, ch));
          const uint32_t wds[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&wds[e]));
            x[ch * 8 + 2 * e] = f.x;
            x[ch * 8 + 2 * e + 1] = f.y;
            ss = fmaf(f.x, f.x, fmaf(f.y, f.y, ss));
          }
        }
        const float inv = 1.0f / fmaxf(sqrtf(ss), 1e-12f);
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
          uint32_t wds[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const __half2 hv = __floats2half2_rn(x[ch * 8 + 2 * e] * inv, x[ch * 8 + 2 * e + 1] * inv);
            wds[e] = *reinterpret_cast<const uint32_t*>(&hv);
          }
          *reinterpret_cast<uint4*>(m + vofs(row, ch)) = make_uint4(wds[0], wds[1], wds[2], wds[3]);
        }
      }
    }
    __syncthreads();
    if (!live) continue;
    const float sc = __ldg(hsc + h);
    const int wi = static_cast<int>(w % (static_cast<long long>(nw) * nw)), wh = wi / nw, ww = wi - wh * nw;
    const bool masked = shift > 0 && (wh == nw - 1 || ww == nw - 1);  // only the last window row / column mixes regions
#pragma unroll 1
    for (int mt = part * 4; mt < part * 4 + 4; ++mt) {
      uint32_t qa[2][4];
#pragma unroll
      for (int ks = 0; ks < 2; ++ks) ptx::ldmatrix_x4(aQ + vofs(mt * 16 + (lane & 7) + ((lane >> 3) & 1) * 8, ks * 2 + (lane >> 4)), qa[ks]);
      const int r0 = mt * 16 + g, r1 = r0 + 8;
      const int qi0 = r0 / WS, qj0 = r0 % WS, qi1 = r1 / WS, qj1 = r1 % WS;
      const int reg0 = v2_region(wh, nw, qi0, WS, shift) * 3 + v2_region(ww, nw, qj0, WS, shift);
      const int reg1 = v2_region(wh, nw, qi1, WS, shift) * 3 + v2_region(ww, nw, qj1, WS, shift);
      float m0 = -CUDART_INF_F, m1 = -CUDART_INF_F, l0 = 0.f, l1 = 0.f;
      float o[4][4];
#pragma unroll
      for (int n = 0; n < 4; ++n) o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f;
#pragma unroll 1
      for (int kb = 0; kb < KB; ++kb) {
        float s[8][4];
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
          uint32_t kf[4];  // keys kb*64 + 8 nt .. + 7: {ks0.b0, ks0.b1, ks1.b0, ks1.b1}
          ptx::ldmatrix_x4(aK + vofs(kb * kV2Rows + nt * 8 + (lane & 7), lane >> 3), kf);
          s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
          mma_f16_16816(s[nt], qa[0], kf[0], kf[1]);
          mma_f16_16816(s[nt], qa[1], kf[2], kf[3]);
        }
        // log2-domain scores: cos * scale + bias (+ mask); rows r0 / r1, keys kb*64 + 8 nt + 2 t + e
        float bm0 = -CUDART_INF_F, bm1 = -CUDART_INF_F;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt)
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int c = kb * kV2Rows + nt * 8 + 2 * t + e, ki = c / WS, kj = c % WS;
            float b0 = sTab[v2_rel_index(qi0, qj0, ki, kj, WS)];
            float b1 = sTab[v2_rel_index(qi1, qj1, ki, kj, WS)];
            if (masked) {
              const int kr = v2_region(wh, nw, ki, WS, shift) * 3 + v2_region(ww, nw, kj, WS, shift);
              if (kr != reg0) b0 += mask_log2;
              if (kr != reg1) b1 += mask_log2;
            }
            s[nt][e] = fmaf(s[nt][e], sc, b0);
            s[nt][2 + e] = fmaf(s[nt][2 + e], sc, b1);
            bm0 = fmaxf(bm0, s[nt][e]);
            bm1 = fmaxf(bm1, s[nt][2 + e]);
          }
        const float mn0 = fmaxf(m0, quad_max(bm0)), mn1 = fmaxf(m1, quad_max(bm1));
        const float a0 = ptx::ex2_approx(m0 - mn0), a1 = ptx::ex2_approx(m1 - mn1);  // 0 on the first block (m = -inf)
        m0 = mn0, m1 = mn1;
        l0 *= a0, l1 *= a1;
#pragma unroll
        for (int n = 0; n < 4; ++n) o[n][0] *= a0, o[n][1] *= a0, o[n][2] *= a1, o[n][3] *= a1;
        uint32_t pa[4][4];  // probabilities as the A fragments of the four 16-key k-steps
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
          const float p0 = ptx::ex2_approx(s[nt][0] - m0), p1 = ptx::ex2_approx(s[nt][1] - m0);
          const float p2 = ptx::ex2_approx(s[nt][2] - m1), p3 = ptx::ex2_approx(s[nt][3] - m1);
          l0 += p0 + p1;
          l1 += p2 + p3;
          pa[nt >> 1][(nt & 1) * 2] = ptx::pack_bf16x2(p0, p1);
          pa[nt >> 1][(nt & 1) * 2 + 1] = ptx::pack_bf16x2(p2, p3);
        }
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          uint32_t vb[2][4];  // keys kb*64 + 16 kk .. +15, dims chunk pair cp: {n 2cp: b0, b1, n 2cp+1: b0, b1}
#pragma unroll
          for (int cp = 0; cp < 2; ++cp)
            ptx::ldmatrix_x4_trans(aV + vofs(kb * kV2Rows + kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8, cp * 2 + (lane >> 4)), vb[cp]);
#pragma unroll
          for (int n = 0; n < 4; ++n) ptx::mma_bf16_16816(o[n], pa[kk], vb[n >> 1][(n & 1) * 2], vb[n >> 1][(n & 1) * 2 + 1]);
        }
      }
      l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
      l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
      l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
      l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
      const float i0 = 1.0f / l0, i1 = 1.0f / l1;  // l >= 1: the row maximum contributes 2^0
#pragma unroll
      for (int n = 0; n < 4; ++n) {
        const int col = h * kV2Hd + n * 8 + 2 * t;
        *reinterpret_cast<uint32_t*>(ctx + (row0 + r0) * ldc + col) = ptx::pack_bf16x2(o[n][0] * i0, o[n][1] * i0);
        *reinterpret_cast<uint32_t*>(ctx + (row0 + r1) * ldc + col) = ptx::pack_bf16x2(o[n][2] * i1, o[n][3] * i1);
      }
    }
  }
}

// One warp per C-float source row: output row r (image r / T_out, token r % T_out), group g of G, reads source row
// src = image * T_in + (idx ? idx[(r % T_out) * G + g] : r % T_out) of y (and of resid), and writes
// v = (resid ? resid[src] : 0) + LayerNorm(y[src]) to columns [g C, g C + C) of row r of out_f32 and / or out_bf16
// (row length G * C).  resid may alias out_f32 when idx is null (every row reads and writes only itself).
template <int NV>
__global__ void __launch_bounds__(256) postnorm_residual_kernel(const float* __restrict__ y, const float* resid, const int* __restrict__ idx,
                                                                const float* __restrict__ gamma, const float* __restrict__ beta, float* out_f32,
                                                                __nv_bfloat16* __restrict__ out_bf16, long long sub_rows, int T_in,
                                                                int T_out, int G, int C, float eps) {
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();
  const int lane = threadIdx.x & 31;
  const long long sr = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (sr >= sub_rows) return;
  const long long row = sr / G;
  const int grp = static_cast<int>(sr - row * G);
  const long long img = row / T_out;
  const int tk = static_cast<int>(row - img * T_out);
  const long long src = img * T_in + (idx != nullptr ? __ldg(idx + static_cast<long long>(tk) * G + grp) : tk);
  const float* yr = y + src * C;
  float4 v[NV];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = i * 128 + lane * 4;
    v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c < C) {
      v[i] = *reinterpret_cast<const float4*>(yr + c);
      s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    }
  }
  const float mean = ptx::warp_sum(s) / static_cast<float>(C);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = i * 128 + lane * 4;
    if (c < C) {
      const float a0 = v[i].x - mean, a1 = v[i].y - mean, a2 = v[i].z - mean, a3 = v[i].w - mean;
      q += (a0 * a0 + a1 * a1) + (a2 * a2 + a3 * a3);
    }
  }
  const float rstd = rsqrtf(ptx::warp_sum(q) / static_cast<float>(C) + eps);
  const long long ob = row * static_cast<long long>(G) * C + static_cast<long long>(grp) * C;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = i * 128 + lane * 4;
    if (c < C) {
      const float4 gm = __ldg(reinterpret_cast<const float4*>(gamma + c));
      const float4 bt = __ldg(reinterpret_cast<const float4*>(beta + c));
      float4 o = make_float4((v[i].x - mean) * rstd * gm.x + bt.x, (v[i].y - mean) * rstd * gm.y + bt.y,
                             (v[i].z - mean) * rstd * gm.z + bt.z, (v[i].w - mean) * rstd * gm.w + bt.w);
      if (resid != nullptr) {
        const float4 r = *reinterpret_cast<const float4*>(resid + src * C + c);
        o.x += r.x, o.y += r.y, o.z += r.z, o.w += r.w;
      }
      if (out_f32 != nullptr) *reinterpret_cast<float4*>(out_f32 + ob + c) = o;
      if (out_bf16 != nullptr) *reinterpret_cast<uint2*>(out_bf16 + ob + c) = make_uint2(ptx::pack_bf16x2(o.x, o.y), ptx::pack_bf16x2(o.z, o.w));
    }
  }
}

template <int NV>
int launch_postnorm(const float* y, const float* resid, const int* idx, const float* gamma, const float* beta, float* out_f32,
                    void* out_bf16, long long sub_rows, int T_in, int T_out, int G, int C, float eps, cudaStream_t st) {
  const unsigned grid = static_cast<unsigned>((sub_rows + 7) / 8);
  EVT_CUDA(launch_pdl(postnorm_residual_kernel<NV>, dim3(grid), dim3(256), 0, st, pdl_for_work(sub_rows / G, static_cast<long long>(G) * C), y,
                      resid, idx, gamma, beta, out_f32, reinterpret_cast<__nv_bfloat16*>(out_bf16), sub_rows, T_in, T_out, G, C, eps));
  EVT_LAUNCH_CHECK("postnorm_residual_kernel");
  return EVT_OK;
}

template <int WS>
int launch_cosine(const void* qkv, int64_t ldq, void* ctx, int64_t ldc, const float* tab, const float* hsc, int64_t n_windows, int heads,
                  int nw, int shift, float mask_log2, cudaStream_t st) {
  constexpr int TOK = WS * WS, IPC = kV2Warps / (TOK / kV2Rows);
  constexpr auto kern = cosine_window_attention_kernel<WS>;
  // 48 KB of q / k / v and 3.5 KB (8 x 8: four tables of 225) or 3.8 KB (16 x 16: one of 961) of bias: four CTAs per SM
  const int smem = IPC * (3 * TOK * kV2Hd * 2 + (2 * WS - 1) * (2 * WS - 1) * 4);
  EVT_TRY(opt_in_smem<kern>(smem));
  const long long items = n_windows * heads;
  const long long groups = (items + IPC - 1) / IPC;
  const long long cap = static_cast<long long>(num_sms()) * 4;  // grid-stride over the rest
  EVT_CUDA(launch_pdl(kern, dim3(static_cast<unsigned>(groups < cap ? groups : cap)), dim3(kV2Warps * 32), smem, st,
                      pdl_for_work(n_windows * TOK, static_cast<long long>(heads) * kV2Hd), reinterpret_cast<const __nv_bfloat16*>(qkv),
                      static_cast<long long>(ldq), reinterpret_cast<__nv_bfloat16*>(ctx), static_cast<long long>(ldc), tab, hsc, heads, items,
                      nw, shift, mask_log2));
  EVT_LAUNCH_CHECK("cosine_window_attention_kernel");
  return EVT_OK;
}

}  // namespace

int cosine_window_attention_launch(const void* qkv, int64_t ldq, void* ctx, int64_t ldc, const float* table, const float* head_scale,
                                   int64_t n_windows, int window, int heads, int head_size, int grid, int shift, float mask, cudaStream_t st) {
  EVT_CHECK_ARG(qkv && ctx && table && head_scale, "cosine_window_attention: null pointer");
  if ((window != 8 && window != 16) || head_size != kV2Hd)
    return fail(EVT_ERR_UNSUPPORTED, "cosine_window_attention: only 8x8 (64-token) and 16x16 (256-token) windows with head size 32 are implemented");
  EVT_CHECK_ARG(n_windows > 0 && heads > 0, "cosine_window_attention: sizes must be positive");
  EVT_CHECK_ARG(grid >= window && grid % window == 0 && n_windows % ((grid / window) * (grid / window)) == 0,
                "cosine_window_attention: grid must be a multiple of the window and n_windows a multiple of (grid / window)^2");
  EVT_CHECK_ARG(shift >= 0 && shift < window && (shift == 0 || grid > window), "cosine_window_attention: shift must be in [0, window), 0 when grid == window");
  EVT_CHECK_ARG(ldq >= 3ll * heads * kV2Hd && ldc >= static_cast<int64_t>(heads) * kV2Hd, "cosine_window_attention: leading dimension too small");
  EVT_CHECK_ARG(ldq % 8 == 0 && reinterpret_cast<uintptr_t>(qkv) % 16 == 0, "cosine_window_attention: qkv rows must be 16-byte aligned");
  EVT_CHECK_ARG(ldc % 2 == 0 && reinterpret_cast<uintptr_t>(ctx) % 4 == 0, "cosine_window_attention: ctx rows must be 4-byte aligned");
  const int nw = grid / window;
  const float ml2 = mask * 1.4426950408889634f;
  if (window == 8) return launch_cosine<8>(qkv, ldq, ctx, ldc, table, head_scale, n_windows, heads, nw, shift, ml2, st);
  return launch_cosine<16>(qkv, ldq, ctx, ldc, table, head_scale, n_windows, heads, nw, shift, ml2, st);
}

int postnorm_residual_launch(const float* y, const float* resid, const int* idx, const float* gamma, const float* beta, float* out_f32,
                             void* out_bf16, int64_t images, int T_in, int T_out, int G, int C, float eps, cudaStream_t st) {
  EVT_CHECK_ARG(y && gamma && beta, "postnorm_residual: null pointer");
  EVT_CHECK_ARG(out_f32 != nullptr || out_bf16 != nullptr, "postnorm_residual: nothing to write");
  EVT_CHECK_ARG(images > 0 && T_in > 0 && T_out > 0 && (G == 1 || G == 4), "postnorm_residual: bad sizes (G must be 1 or 4)");
  EVT_CHECK_ARG(idx != nullptr || (G == 1 && T_in == T_out), "postnorm_residual: without idx, G must be 1 and T_in == T_out");
  EVT_CHECK_ARG(idx == nullptr || out_f32 == nullptr || (out_f32 != resid && out_f32 != y), "postnorm_residual: a gathered out_f32 must not alias its inputs");
  EVT_CHECK_ARG(C > 0 && C % 4 == 0 && C <= 1536, "postnorm_residual: C must be a multiple of 4, <= 1536");
  EVT_CHECK_ARG(eps >= 0.f, "postnorm_residual: negative eps");
  const long long sub = images * T_out * G;
  const int nv = (C + 127) / 128;
  if (nv <= 1) return launch_postnorm<1>(y, resid, idx, gamma, beta, out_f32, out_bf16, sub, T_in, T_out, G, C, eps, st);
  if (nv <= 2) return launch_postnorm<2>(y, resid, idx, gamma, beta, out_f32, out_bf16, sub, T_in, T_out, G, C, eps, st);
  if (nv <= 3) return launch_postnorm<3>(y, resid, idx, gamma, beta, out_f32, out_bf16, sub, T_in, T_out, G, C, eps, st);
  if (nv <= 4) return launch_postnorm<4>(y, resid, idx, gamma, beta, out_f32, out_bf16, sub, T_in, T_out, G, C, eps, st);
  if (nv <= 6) return launch_postnorm<6>(y, resid, idx, gamma, beta, out_f32, out_bf16, sub, T_in, T_out, G, C, eps, st);
  if (nv <= 8) return launch_postnorm<8>(y, resid, idx, gamma, beta, out_f32, out_bf16, sub, T_in, T_out, G, C, eps, st);
  return launch_postnorm<12>(y, resid, idx, gamma, beta, out_f32, out_bf16, sub, T_in, T_out, G, C, eps, st);
}

int swinv2_cpb_table(const float* w1, const float* b1, const float* w2, int heads, int ws, int pws, float* out) {
  EVT_CHECK_ARG(w1 && b1 && w2 && out, "swinv2_cpb_table: null pointer");
  EVT_CHECK_ARG(heads > 0 && ws >= 1 && (pws == 0 || pws >= 2), "swinv2_cpb_table: heads > 0, window >= 1, pretrained window 0 or >= 2");
  constexpr int kHidden = 512;
  const int tw = 2 * ws - 1;
  const double div = pws > 0 ? pws - 1 : (ws > 1 ? ws - 1 : 1);
  std::vector<double> hid(kHidden);
  for (int a = 0; a < tw; ++a)
    for (int b = 0; b < tw; ++b) {
      double c[2] = {(a - (ws - 1)) / div * 8.0, (b - (ws - 1)) / div * 8.0};  // :497-506, then normalised to [-8, 8]
      for (double& x : c) x = (x > 0 ? 1.0 : x < 0 ? -1.0 : 0.0) * std::log2(std::fabs(x) + 1.0) / 3.0;  // / log2(8)
      for (int j = 0; j < kHidden; ++j) {
        const double z = static_cast<double>(w1[2 * j]) * c[0] + static_cast<double>(w1[2 * j + 1]) * c[1] + b1[j];
        hid[j] = z > 0 ? z : 0.0;
      }
      for (int h = 0; h < heads; ++h) {
        double z = 0;
        for (int j = 0; j < kHidden; ++j) z += static_cast<double>(w2[static_cast<size_t>(h) * kHidden + j]) * hid[j];
        out[static_cast<size_t>(h) * tw * tw + a * tw + b] = static_cast<float>(16.0 / (1.0 + std::exp(-z)));
      }
    }
  return EVT_OK;
}

}  // namespace evt

extern "C" int evt_cosine_window_attention_fwd(const void* qkv, int64_t ldq, void* ctx, int64_t ldc, const float* table,
                                               const float* head_scale, int64_t n_windows, int window, int heads, int head_size, int grid,
                                               int shift, float mask, evt_stream stream) {
  int rc = evt_device_check();
  if (rc != EVT_OK) return rc;
  return evt::cosine_window_attention_launch(qkv, ldq, ctx, ldc, table, head_scale, n_windows, window, heads, head_size, grid, shift, mask,
                                             static_cast<cudaStream_t>(stream));
}

extern "C" int evt_postnorm_residual(const float* y, const float* resid, const int* idx, const float* gamma, const float* beta, float* out_f32,
                                     void* out_bf16, int64_t images, int T_in, int T_out, int G, int C, float eps, evt_stream stream) {
  int rc = evt_device_check();
  if (rc != EVT_OK) return rc;
  return evt::postnorm_residual_launch(y, resid, idx, gamma, beta, out_f32, out_bf16, images, T_in, T_out, G, C, eps,
                                       static_cast<cudaStream_t>(stream));
}

extern "C" int evt_swinv2_cpb_table(const float* w1, const float* b1, const float* w2, int heads, int window, int pretrained_window,
                                    float* out) {
  return evt::swinv2_cpb_table(w1, b1, w2, heads, window, pretrained_window, out);
}

extern "C" int evt_swinv2_score_bias(const float* table, int heads, int window, int grid, int shift, float mask, float* out) {
  EVT_CHECK_ARG(table && out, "swinv2_score_bias: null pointer");
  EVT_CHECK_ARG(heads > 0 && window > 0 && grid % window == 0 && shift >= 0 && shift < window, "swinv2_score_bias: bad geometry");
  const int ws = window, N = ws * ws, nw = grid / ws, tw = 2 * ws - 1;
  for (int wi = 0; wi < nw * nw; ++wi) {
    const int wh = wi / nw, ww = wi % nw;
    for (int h = 0; h < heads; ++h)
      for (int a = 0; a < N; ++a)
        for (int b = 0; b < N; ++b) {
          const int qi = a / ws, qj = a % ws, ki = b / ws, kj = b % ws;
          float v = table[static_cast<size_t>(h) * tw * tw + evt::v2_rel_index(qi, qj, ki, kj, ws)];
          if (shift > 0 && evt::v2_region(wh, nw, qi, ws, shift) * 3 + evt::v2_region(ww, nw, qj, ws, shift) !=
                               evt::v2_region(wh, nw, ki, ws, shift) * 3 + evt::v2_region(ww, nw, kj, ws, shift))
            v += mask;
          out[((static_cast<size_t>(wi) * heads + h) * N + a) * N + b] = v;
        }
  }
  return EVT_OK;
}
