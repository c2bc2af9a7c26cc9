// LayerNorm kernels (HBM-bound): one warp per row, 8-byte vector loads, the row lives in registers,
// mean then centred variance (exact for eps = 1e-12 as well as 1e-5), fp32 statistics.
#include <cuda_bf16.h>

#include "common.h"
#include "ptx.cuh"

namespace evt {
namespace {

constexpr int kMaxVec = 16;  // float2 per lane -> D <= 1024 on the fast path

// D even, D <= 1024, strides even.  NV = ceil(D / 64).
template <int NV, int OUT>
__global__ void __launch_bounds__(256) ln_rows_kernel(const float* x, long long x_stride,
                                                      const float* __restrict__ gamma, const float* __restrict__ beta,
                                                      void* __restrict__ y, long long y_stride, float* y_copy,
                                                      long long rows, int D, float eps) {
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();
  const int lane = threadIdx.x & 31;
  const long long row = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const float* xr = x + row * x_stride;
  float2 v[NV];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = i * 64 + lane * 2;
    if (c < D) {
      v[i] = *reinterpret_cast<const float2*>(xr + c);
      s += v[i].x + v[i].y;
    } else {
      v[i] = make_float2(0.f, 0.f);
    }
  }
  const float mean = ptx::warp_sum(s) / static_cast<float>(D);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = i * 64 + lane * 2;
    if (c < D) {
      const float a = v[i].x - mean, b = v[i].y - mean;
      q += a * a + b * b;
    }
  }
  const float rstd = rsqrtf(ptx::warp_sum(q) / static_cast<float>(D) + eps);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = i * 64 + lane * 2;
    if (c < D) {
      const float2 g = *reinterpret_cast<const float2*>(gamma + c);
      const float2 b = *reinterpret_cast<const float2*>(beta + c);
      float o0 = (v[i].x - mean) * rstd * g.x + b.x;
      float o1 = (v[i].y - mean) * rstd * g.y + b.y;
      // the f32 copy (TF dialect: it becomes the skip connection) keeps full precision; only the GEMM operand is rounded
      if (y_copy != nullptr) *reinterpret_cast<float2*>(y_copy + row * x_stride + c) = make_float2(o0, o1);
      if (OUT == EVT_TF32) {
        o0 = ptx::round_tf32(o0);
        o1 = ptx::round_tf32(o1);
      }
      if (OUT == EVT_BF16) {
        __nv_bfloat162 h = __floats2bfloat162_rn(o0, o1);
        *reinterpret_cast<__nv_bfloat162*>(reinterpret_cast<__nv_bfloat16*>(y) + row * y_stride + c) = h;
      } else {
        *reinterpret_cast<float2*>(reinterpret_cast<float*>(y) + row * y_stride + c) = make_float2(o0, o1);
      }
    }
  }
}

// D % 4 == 0, D <= 1024, strides % 4 == 0: 16-byte loads (512 B per warp instruction), 8-byte bf16 / 16-byte f32 stores.
// NV = ceil(D / 128).  The input is read with a streaming (no L1 allocate) hint: nothing here is touched twice.
// PRE (latency path, few rows): gamma / beta are fetched into registers BEFORE griddepcontrol.wait -- they do not depend on
// the previous kernel, so under programmatic dependent launch that round trip overlaps the previous kernel's tail instead of
// following the row statistics (three dependent memory round trips per LayerNorm become two; 25 LayerNorms per forward).
// Not used at large batch: 48 more live registers would halve the occupancy of a kernel that runs at the HBM roofline.
template <int NV, int OUT, bool PRE = false>
__global__ void __launch_bounds__(256) ln_rows4_kernel(const float* x, long long x_stride,
                                                       const float* __restrict__ gamma, const float* __restrict__ beta,
                                                       void* __restrict__ y, long long y_stride, float* y_copy,
                                                       long long rows, int D, float eps) {
  ptx::grid_dep_launch();
  const int lane = threadIdx.x & 31;
  float4 gpre[PRE ? NV : 1], bpre[PRE ? NV : 1];
  if (PRE) {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = i * 128 + lane * 4;
      if (c < D) {
        gpre[i] = __ldg(reinterpret_cast<const float4*>(gamma + c));
        bpre[i] = __ldg(reinterpret_cast<const float4*>(beta + c));
      }
    }
  }
  ptx::grid_dep_wait();
  const long long row = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const float* xr = x + row * x_stride;
  float4 v[NV];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = i * 128 + lane * 4;
    v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c < D) {
      asm volatile("ld.global.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
                   : "=f"(v[i].x), "=f"(v[i].y), "=f"(v[i].z), "=f"(v[i].w)
                   : "l"(xr + c));
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
    const int c = i * 128 + lane * 4;
    if (c < D) {
      const float4 g = PRE ? gpre[i] : __ldg(reinterpret_cast<const float4*>(gamma + c));
      const float4 b = PRE ? bpre[i] : __ldg(reinterpret_cast<const float4*>(beta + c));
      ptx::store_ln4<OUT>(v[i], mean, rstd, g, b, y, y_stride, y_copy, x_stride, row, c);
    }
  }
}

// Narrow rows (D = 4 * LPR * NV with LPR = 8 or 16 lanes per row: 64, 96, 128, 192, ...): 32 / LPR rows per warp so that
// every lane carries exactly NV float4 -- with a whole warp per row a D = 192 row keeps half the lanes at half load and
// a D = 96 row (Swin stage 1) leaves a quarter of them idle (4.5 and 3.4 TB/s instead of ~6).  Statistics are reduced
// with xor-shuffles inside the LPR-lane group.
template <int LPR, int NV, int OUT>
__global__ void __launch_bounds__(256) ln_rows4_sub_kernel(const float* x, long long x_stride, const float* __restrict__ gamma,
                                                           const float* __restrict__ beta, void* __restrict__ y,
                                                           long long y_stride, float* y_copy, long long rows, float eps) {
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();
  constexpr int D = 4 * LPR * NV;
  constexpr int RPW = 32 / LPR;
  const int lane = threadIdx.x & 31;
  const int sub = lane / LPR, l = lane % LPR;
  const long long row = (static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5)) * RPW + sub;
  const bool live = row < rows;  // dead sub-rows still take part in the shuffles
  const float* xr = x + (live ? row : 0) * x_stride;
  float4 v[NV];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = (i * LPR + l) * 4;
    asm volatile("ld.global.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(v[i].x), "=f"(v[i].y), "=f"(v[i].z), "=f"(v[i].w)
                 : "l"(xr + c));
    s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  }
  const float mean = ptx::group_sum<LPR>(s) / static_cast<float>(D);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const float a0 = v[i].x - mean, a1 = v[i].y - mean, a2 = v[i].z - mean, a3 = v[i].w - mean;
    q += (a0 * a0 + a1 * a1) + (a2 * a2 + a3 * a3);
  }
  const float rstd = rsqrtf(ptx::group_sum<LPR>(q) / static_cast<float>(D) + eps);
  if (!live) return;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = (i * LPR + l) * 4;
    const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + c));
    const float4 b = __ldg(reinterpret_cast<const float4*>(beta + c));
    ptx::store_ln4<OUT>(v[i], mean, rstd, g, b, y, y_stride, y_copy, x_stride, row, c);
  }
}

// Any D (odd, > 1024): warp per row, three strided passes over the row (L1/L2 resident).
template <int OUT>
__global__ void __launch_bounds__(256) ln_rows_generic_kernel(const float* x, long long x_stride,
                                                              const float* __restrict__ gamma,
                                                              const float* __restrict__ beta, void* __restrict__ y,
                                                              long long y_stride, float* y_copy, long long rows, int D,
                                                              float eps) {
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();
  const int lane = threadIdx.x & 31;
  const long long row = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const float* xr = x + row * x_stride;
  float s = 0.f;
  for (int c = lane; c < D; c += 32) s += xr[c];
  const float mean = ptx::warp_sum(s) / static_cast<float>(D);
  float q = 0.f;
  for (int c = lane; c < D; c += 32) {
    const float a = xr[c] - mean;
    q += a * a;
  }
  const float rstd = rsqrtf(ptx::warp_sum(q) / static_cast<float>(D) + eps);
  for (int c = lane; c < D; c += 32) {
    float o = (xr[c] - mean) * rstd * gamma[c] + beta[c];
    if (y_copy != nullptr) y_copy[row * x_stride + c] = o;  // unrounded
    if (OUT == EVT_TF32) o = ptx::round_tf32(o);
    if (OUT == EVT_BF16) reinterpret_cast<__nv_bfloat16*>(y)[row * y_stride + c] = __float2bfloat16_rn(o);
    else reinterpret_cast<float*>(y)[row * y_stride + c] = o;
  }
}

// Joint LayerNorm over nh = n*h elements per image (torch_layers dialect): one CTA per image.
__global__ void __launch_bounds__(1024) ln2d_kernel(const float* __restrict__ x, const float* __restrict__ addend,
                                                    const float* __restrict__ gamma, const float* __restrict__ beta,
                                                    float* __restrict__ y, long long nh, float eps) {
  __shared__ float red[32];
  __shared__ float stat;
  const long long base = static_cast<long long>(blockIdx.x) * nh;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = blockDim.x >> 5;
  auto block_sum = [&](float v) -> float {
    v = ptx::warp_sum(v);
    if (lane == 0) red[warp] = v;
    __syncthreads();
    if (warp == 0) {
      float t = lane < nwarp ? red[lane] : 0.f;
      t = ptx::warp_sum(t);
      if (lane == 0) stat = t;
    }
    __syncthreads();
    const float r = stat;
    __syncthreads();
    return r;
  };
  float s = 0.f;
  for (long long i = tid; i < nh; i += blockDim.x) s += x[base + i] + (addend ? addend[base + i] : 0.f);
  const float mean = block_sum(s) / static_cast<float>(nh);
  float q = 0.f;
  for (long long i = tid; i < nh; i += blockDim.x) {
    const float a = x[base + i] + (addend ? addend[base + i] : 0.f) - mean;
    q += a * a;
  }
  const float rstd = rsqrtf(block_sum(q) / static_cast<float>(nh) + eps);
  for (long long i = tid; i < nh; i += blockDim.x) {
    const float a = x[base + i] + (addend ? addend[base + i] : 0.f);
    y[base + i] = (a - mean) * rstd * gamma[i] + beta[i];
  }
}

template <int OUT>
int launch_rows(const float* x, long long xs, const float* g, const float* b, void* y, long long ys, float* yc,
                long long rows, int D, float eps, cudaStream_t st) {
  // warps (= rows, or row groups) per block; 4 measured 2 % faster than 8 at 201 728 x 768 inside the forward
  constexpr int wpb = 4;
  const unsigned grid = static_cast<unsigned>((rows + wpb - 1) / wpb);
  const bool fast = (D % 2 == 0) && D <= 64 * kMaxVec && (xs % 2 == 0) && (ys % 2 == 0) &&
                    (reinterpret_cast<uintptr_t>(x) % 8 == 0) && (reinterpret_cast<uintptr_t>(y) % 8 == 0) &&
                    (reinterpret_cast<uintptr_t>(g) % 8 == 0) && (reinterpret_cast<uintptr_t>(b) % 8 == 0) &&
                    (yc == nullptr || reinterpret_cast<uintptr_t>(yc) % 8 == 0);
  const bool fast4 = (D % 4 == 0) && D <= 1024 && (xs % 4 == 0) && (ys % 4 == 0) &&
                     (reinterpret_cast<uintptr_t>(x) % 16 == 0) && (reinterpret_cast<uintptr_t>(y) % 16 == 0) &&
                     (reinterpret_cast<uintptr_t>(g) % 16 == 0) && (reinterpret_cast<uintptr_t>(b) % 16 == 0) &&
                     (yc == nullptr || reinterpret_cast<uintptr_t>(yc) % 16 == 0);
  // narrow rows: several rows per warp (D = 64, 96, 192 -- T2T performer, Swin stage 1, DeiT-Tiny / Swin stage 2)
  int lpr = 0, nvs = 0;
  if (fast4 && D == 64) lpr = 16, nvs = 1;
  else if (fast4 && D == 96) lpr = 8, nvs = 3;
  else if (fast4 && D == 192) lpr = 16, nvs = 3;
  if (lpr != 0) {
    const int rpw = 32 / lpr;
    const unsigned gsub = static_cast<unsigned>((rows + wpb * rpw - 1) / (wpb * rpw));
    if (D == 64)
      EVT_CUDA(launch_pdl(ln_rows4_sub_kernel<16, 1, OUT>, dim3(gsub), dim3(wpb * 32), 0, st, pdl_for_work(rows, D), x, xs, g, b, y, ys, yc, rows, eps));
    else if (D == 96)
      EVT_CUDA(launch_pdl(ln_rows4_sub_kernel<8, 3, OUT>, dim3(gsub), dim3(wpb * 32), 0, st, pdl_for_work(rows, D), x, xs, g, b, y, ys, yc, rows, eps));
    else
      EVT_CUDA(launch_pdl(ln_rows4_sub_kernel<16, 3, OUT>, dim3(gsub), dim3(wpb * 32), 0, st, pdl_for_work(rows, D), x, xs, g, b, y, ys, yc, rows, eps));
  } else if (fast4) {
    const int nv = (D + 127) / 128;
#define EVT_LN4_CASE(NVV)                                                                          \
  case NVV:                                                                                        \
    if (rows <= 4096)                                                                              \
      EVT_CUDA(launch_pdl(ln_rows4_kernel<NVV, OUT, true>, dim3(grid), dim3(wpb * 32), 0, st, pdl_for_work(rows, D), x, xs, g, b, y, ys, yc, rows, D, eps)); \
    else                                                                                           \
      EVT_CUDA(launch_pdl(ln_rows4_kernel<NVV, OUT>, dim3(grid), dim3(wpb * 32), 0, st, pdl_for_work(rows, D), x, xs, g, b, y, ys, yc, rows, D, eps)); \
    break;
    switch (nv) {
      EVT_LN4_CASE(1) EVT_LN4_CASE(2) EVT_LN4_CASE(3) EVT_LN4_CASE(4) EVT_LN4_CASE(5) EVT_LN4_CASE(6) EVT_LN4_CASE(7)
      EVT_LN4_CASE(8)
    }
#undef EVT_LN4_CASE
  } else if (!fast) {
    EVT_CUDA(launch_pdl(ln_rows_generic_kernel<OUT>, dim3(grid), dim3(wpb * 32), 0, st, pdl_for_work(rows, D), x, xs, g, b, y, ys, yc, rows, D, eps));
  } else {
    const int nv = (D + 63) / 64;
#define EVT_LN_CASE(NVV)                                                                          \
  case NVV:                                                                                       \
    EVT_CUDA(launch_pdl(ln_rows_kernel<NVV, OUT>, dim3(grid), dim3(wpb * 32), 0, st, pdl_for_work(rows, D), x, xs, g, b, y, ys, yc, rows, D, eps)); \
    break;
    switch (nv) {
      EVT_LN_CASE(1) EVT_LN_CASE(2) EVT_LN_CASE(3) EVT_LN_CASE(4) EVT_LN_CASE(5) EVT_LN_CASE(6) EVT_LN_CASE(7)
      EVT_LN_CASE(8) EVT_LN_CASE(9) EVT_LN_CASE(10) EVT_LN_CASE(11) EVT_LN_CASE(12) EVT_LN_CASE(13) EVT_LN_CASE(14)
      EVT_LN_CASE(15) EVT_LN_CASE(16)
    }
#undef EVT_LN_CASE
  }
  EVT_LAUNCH_CHECK("layernorm");
  return EVT_OK;
}

}  // namespace

int layernorm_launch(const float* x, int64_t x_stride, const float* gamma, const float* beta, void* y, int y_dtype,
                     int64_t y_stride, float* y_copy, int64_t rows, int D, float eps, cudaStream_t st) {
  EVT_CHECK_ARG(x && gamma && beta && y, "layernorm: null pointer");
  EVT_CHECK_ARG(rows > 0 && D > 0, "layernorm: rows and D must be positive");
  EVT_CHECK_ARG(x_stride >= D && y_stride >= D, "layernorm: stride smaller than D");
  EVT_CHECK_ARG(y_dtype == EVT_BF16 || y_dtype == EVT_F32 || y_dtype == EVT_TF32, "layernorm: y dtype must be bf16, f32 or tf32");
  EVT_CHECK_ARG(eps >= 0.f, "layernorm: negative eps");
  if (y_dtype == EVT_BF16) return launch_rows<EVT_BF16>(x, x_stride, gamma, beta, y, y_stride, y_copy, rows, D, eps, st);
  if (y_dtype == EVT_TF32) return launch_rows<EVT_TF32>(x, x_stride, gamma, beta, y, y_stride, y_copy, rows, D, eps, st);
  return launch_rows<EVT_F32>(x, x_stride, gamma, beta, y, y_stride, y_copy, rows, D, eps, st);
}

}  // namespace evt

extern "C" int evt_layernorm_fwd(const float* x, int64_t x_stride, const float* gamma, const float* beta, void* y,
                                 int y_dtype, int64_t y_stride, float* y_copy_f32, int64_t rows, int D, float eps,
                                 evt_stream stream) {
  int rc = evt_device_check();
  if (rc != EVT_OK) return rc;
  return evt::layernorm_launch(x, x_stride, gamma, beta, y, y_dtype, y_stride, y_copy_f32, rows, D, eps,
                               static_cast<cudaStream_t>(stream));
}

extern "C" int evt_layernorm2d_fwd(const float* x, const float* addend, const float* gamma, const float* beta, float* y,
                                   int64_t batch, int64_t nh, float eps, evt_stream stream) {
  int rc = evt_device_check();
  if (rc != EVT_OK) return rc;
  EVT_CHECK_ARG(x && gamma && beta && y, "layernorm2d: null pointer");
  EVT_CHECK_ARG(batch > 0 && nh > 0, "layernorm2d: batch and nh must be positive");
  evt::ln2d_kernel<<<static_cast<unsigned>(batch), 1024, 0, static_cast<cudaStream_t>(stream)>>>(x, addend, gamma, beta,
                                                                                                 y, nh, eps);
  EVT_LAUNCH_CHECK("layernorm2d");
  return EVT_OK;
}
