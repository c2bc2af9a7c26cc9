// Memory-bound gather / elementwise kernels around the GEMMs: patch im2col, cls / distillation token
// rows, fp32 -> bf16 cast, T2T soft-split unfold.  All are coalesced 16- or 32-byte-per-thread streams.
#include <cuda_bf16.h>

#include "common.h"
#include "ops.h"
#include "ptx.cuh"

namespace evt {
namespace {

// One thread = 8 consecutive pixels of one image row (32 / 16 / 8 B in for f32 / bf16 / u8 pixels, 16 B of bf16 or 32 B of
// tf32-rounded f32 out).  Thread order follows the input (b, c, y, x8) so reads are perfectly coalesced; writes are full
// 16-byte pieces of patch rows.  Patch p of image b lands in row  b * row_stride + row_off + p  (row_stride = patches,
// row_off = 0: dense patch matrix; row_stride = tokens, row_off = number of prefix tokens: one row per TOKEN, so the
// embedding GEMM's output rows are the rows of the residual stream and its epilogue can be the TMA reduce-add).
// The pixel type conversion is fused here (the C ABI takes f32, bf16 or u8 pixels): u8 pixels are normalised on the fly,
// value = pixel * scale[c] + bias[c]  (= (pixel / 255 - mean[c]) / std[c], the torchvision Normalize the reference's
// data loaders apply, deit_pruning/src/utils.py:118-133), which cuts the host -> device bytes of the e2e path by 4x.
struct PixAffine {
  float scale[3], bias[3];
};
__device__ __forceinline__ void load8(const float* p, float (&v)[8]) {
  const float4 a = *reinterpret_cast<const float4*>(p);
  const float4 b = *reinterpret_cast<const float4*>(p + 4);
  v[0] = a.x, v[1] = a.y, v[2] = a.z, v[3] = a.w, v[4] = b.x, v[5] = b.y, v[6] = b.z, v[7] = b.w;
}
__device__ __forceinline__ void load8(const __nv_bfloat16* p, float (&v)[8]) {
  const uint4 a = *reinterpret_cast<const uint4*>(p);
  const uint32_t w[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    v[2 * i] = __uint_as_float(w[i] << 16);
    v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
  }
}
__device__ __forceinline__ void load8(const uint8_t* p, float (&v)[8]) {
  const uint2 a = *reinterpret_cast<const uint2*>(p);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    v[i] = static_cast<float>((a.x >> (8 * i)) & 0xffu);
    v[4 + i] = static_cast<float>((a.y >> (8 * i)) & 0xffu);
  }
}
template <typename TIN, bool OUT_BF16, bool AFFINE>
__global__ void __launch_bounds__(256) im2col_kernel(const TIN* __restrict__ px, void* __restrict__ cols_, int B, int H, int W,
                                                     int P, long long total, int row_stride, int row_off, const PixAffine af) {
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();
  const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const int w8 = W / 8;
  const int x8 = static_cast<int>(t % w8);
  long long r = t / w8;
  const int y = static_cast<int>(r % H);
  r /= H;
  const int c = static_cast<int>(r % 3);
  const int b = static_cast<int>(r / 3);
  float v[8];
  load8(px + t * 8, v);
  if (AFFINE) {
    const float sc = af.scale[c], bi = af.bias[c];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = fmaf(v[i], sc, bi);
  }
  const int x = x8 * 8;
  const int py = y / P, i = y % P, pxi = x / P, j = x % P;
  const int gw = W / P;
  const long long row = static_cast<long long>(b) * row_stride + row_off + py * gw + pxi;
  const int k = (c * P + i) * P + j;
  if (OUT_BF16) {
    uint4 o;
    o.x = ptx::pack_bf16x2(v[0], v[1]);
    o.y = ptx::pack_bf16x2(v[2], v[3]);
    o.z = ptx::pack_bf16x2(v[4], v[5]);
    o.w = ptx::pack_bf16x2(v[6], v[7]);
    *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(cols_) + row * (3ll * P * P) + k) = o;
  } else {  // tf32 mode keeps the patch matrix in fp32, rounded to nearest tf32 (the tensor core would truncate)
    float* dst = reinterpret_cast<float*>(cols_) + row * (3ll * P * P) + k;
    *reinterpret_cast<float4*>(dst) = make_float4(ptx::round_tf32(v[0]), ptx::round_tf32(v[1]), ptx::round_tf32(v[2]), ptx::round_tf32(v[3]));
    *reinterpret_cast<float4*>(dst + 4) = make_float4(ptx::round_tf32(v[4]), ptx::round_tf32(v[5]), ptx::round_tf32(v[6]), ptx::round_tf32(v[7]));
  }
}

__global__ void __launch_bounds__(256) prefix_tokens_kernel(const float* __restrict__ prefix,
                                                            const float* __restrict__ pos, float* __restrict__ out,
                                                            int B, int tokens, int n_prefix, int D) {
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();
  const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long total = static_cast<long long>(B) * n_prefix * D;
  if (t >= total) return;
  const int d = static_cast<int>(t % D);
  const int tk = static_cast<int>((t / D) % n_prefix);
  const long long b = t / (static_cast<long long>(D) * n_prefix);
  out[(b * tokens + tk) * D + d] = prefix[tk * D + d] + pos[tk * D + d];
}

// Residual stream before the embedding GEMM reduce-adds the patch projections into it:
//   out[b, t, :] = pos[t, :] + (t < n_prefix ? prefix[t, :] : bias[:])     (cls / distillation rows; conv bias elsewhere)
__global__ void __launch_bounds__(256) embed_fill_kernel(const float* __restrict__ prefix, const float* __restrict__ pos,
                                                         const float* __restrict__ bias, float* __restrict__ out,
                                                         long long total4, int tokens, int n_prefix, int D4) {
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  const int d4 = static_cast<int>(i % D4);
  const int tk = static_cast<int>((i / D4) % tokens);
  const float4 a = __ldg(reinterpret_cast<const float4*>(pos) + static_cast<long long>(tk) * D4 + d4);
  const float4 c = tk < n_prefix ? __ldg(reinterpret_cast<const float4*>(prefix) + static_cast<long long>(tk) * D4 + d4)
                                 : __ldg(reinterpret_cast<const float4*>(bias) + d4);
  reinterpret_cast<float4*>(out)[i] = make_float4(a.x + c.x, a.y + c.y, a.z + c.z, a.w + c.w);
}

__global__ void __launch_bounds__(256) cast_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y,
                                                   long long n8, long long n) {
  const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t < n8) {
    const float4 a = *reinterpret_cast<const float4*>(x + t * 8);
    const float4 b = *reinterpret_cast<const float4*>(x + t * 8 + 4);
    uint4 o;
    o.x = ptx::pack_bf16x2(a.x, a.y);
    o.y = ptx::pack_bf16x2(a.z, a.w);
    o.z = ptx::pack_bf16x2(b.x, b.y);
    o.w = ptx::pack_bf16x2(b.z, b.w);
    *reinterpret_cast<uint4*>(y + t * 8) = o;
  } else if (t == n8) {
    for (long long i = n8 * 8; i < n; ++i) y[i] = __float2bfloat16_rn(x[i]);
  }
}

// tf_Unfold (channel-last): out[(b, oy, ox), (ky, kx, c)] = x[b, oy*s - p + ky, ox*s - p + kx, c], zero outside.
// One thread per output element pair-of-channels would be wasteful for C = 3, so: one thread per output
// element, consecutive threads along the output row (kx, c fastest) -> contiguous writes and, within a
// window row, contiguous reads of kx*C values.
template <typename TIN>
__global__ void __launch_bounds__(256) unfold_kernel(const TIN* __restrict__ x, __nv_bfloat16* __restrict__ out,
                                                     long long ldo, int B, int H, int W, int C, int k, int s, int p,
                                                     int oh, int ow, long long total) {
  const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const int col = static_cast<int>(t % ldo);
  const long long row = t / ldo;
  const int kkc = k * k * C;
  float v = 0.f;
  if (col < kkc) {
    const int c = col % C;
    const int kx = (col / C) % k;
    const int ky = col / (C * k);
    const int ox = static_cast<int>(row % ow);
    const int oy = static_cast<int>((row / ow) % oh);
    const long long b = row / (static_cast<long long>(ow) * oh);
    const int iy = oy * s - p + ky, ix = ox * s - p + kx;
    if (iy >= 0 && iy < H && ix >= 0 && ix < W) v = static_cast<float>(x[((b * H + iy) * W + ix) * C + c]);
  }
  out[row * ldo + col] = __float2bfloat16_rn(v);
}

}  // namespace

namespace {

template <typename TIN, bool AFFINE>
int im2col_typed(const void* pixels, void* cols, int out_dtype, int B, int H, int W, int P, cudaStream_t st, int row_stride,
                 int row_off, const PixAffine& af) {
  const long long total = static_cast<long long>(B) * 3 * H * (W / 8);
  const dim3 grid(static_cast<unsigned>((total + 255) / 256));
  const bool pdl = pdl_for_rows(static_cast<long long>(B) * 256);
  const TIN* px = reinterpret_cast<const TIN*>(pixels);
  if (out_dtype == EVT_BF16)
    EVT_CUDA(launch_pdl(im2col_kernel<TIN, true, AFFINE>, grid, dim3(256), 0, st, pdl, px, cols, B, H, W, P, total, row_stride, row_off, af));
  else
    EVT_CUDA(launch_pdl(im2col_kernel<TIN, false, AFFINE>, grid, dim3(256), 0, st, pdl, px, cols, B, H, W, P, total, row_stride, row_off, af));
  EVT_LAUNCH_CHECK("im2col");
  return EVT_OK;
}

}  // namespace

int im2col_launch(const void* pixels, int pixel_dtype, const float* scale3, const float* bias3, void* cols, int out_dtype, int B,
                  int H, int W, int P, cudaStream_t st, int row_stride, int row_off) {
  if (row_stride <= 0) row_stride = (H / (P > 0 ? P : 1)) * (W / (P > 0 ? P : 1)), row_off = 0;
  EVT_CHECK_ARG(pixels && cols, "im2col: null pointer");
  EVT_CHECK_ARG(B > 0 && H > 0 && W > 0 && P > 0, "im2col: sizes must be positive");
  EVT_CHECK_ARG(H % P == 0 && W % P == 0, "im2col: image size must be a multiple of the patch size");
  EVT_CHECK_ARG(reinterpret_cast<uintptr_t>(cols) % 16 == 0, "im2col: output pointer must be 16-byte aligned");
  const int in_bytes = pixel_dtype == EVT_PIX_F32 ? 4 : pixel_dtype == EVT_PIX_BF16 ? 2 : 1;
  EVT_CHECK_ARG(pixel_dtype == EVT_PIX_F32 || pixel_dtype == EVT_PIX_BF16 || pixel_dtype == EVT_PIX_U8, "im2col: unknown pixel dtype");
  EVT_CHECK_ARG(reinterpret_cast<uintptr_t>(pixels) % (8 * in_bytes) == 0, "im2col: pixel pointer must be aligned to 8 pixels");
  if (P % 8 != 0 && P % 4 == 0 && out_dtype == EVT_BF16 && row_off == 0 && pixel_dtype == EVT_PIX_F32)
    return im2col4_launch(reinterpret_cast<const float*>(pixels), cols, B, H, W, P, st);  // Swin: P = 4
  EVT_CHECK_ARG(P % 8 == 0 && W % 8 == 0, "im2col: patch width must be a multiple of 8 (f32 pixels, bf16 output: of 4)");
  PixAffine af = {{1.f, 1.f, 1.f}, {0.f, 0.f, 0.f}};
  if (pixel_dtype == EVT_PIX_U8) {
    EVT_CHECK_ARG(scale3 && bias3, "im2col: u8 pixels need a per-channel scale and bias");
    for (int c = 0; c < 3; ++c) af.scale[c] = scale3[c], af.bias[c] = bias3[c];
    return im2col_typed<uint8_t, true>(pixels, cols, out_dtype, B, H, W, P, st, row_stride, row_off, af);
  }
  if (pixel_dtype == EVT_PIX_BF16) return im2col_typed<__nv_bfloat16, false>(pixels, cols, out_dtype, B, H, W, P, st, row_stride, row_off, af);
  return im2col_typed<float, false>(pixels, cols, out_dtype, B, H, W, P, st, row_stride, row_off, af);
}

int embed_fill_launch(const float* prefix, const float* pos, const float* bias, float* out, int B, int tokens, int n_prefix, int D,
                      cudaStream_t st) {
  EVT_CHECK_ARG(prefix && pos && bias && out, "embed_fill: null pointer");
  EVT_CHECK_ARG(B > 0 && tokens > 0 && n_prefix > 0 && n_prefix <= tokens && D > 0 && D % 4 == 0, "embed_fill: bad sizes");
  const long long total4 = static_cast<long long>(B) * tokens * (D / 4);
  EVT_CUDA(launch_pdl(embed_fill_kernel, dim3(static_cast<unsigned>((total4 + 255) / 256)), dim3(256), 0, st,
                      pdl_for_rows(static_cast<long long>(B) * tokens), prefix, pos, bias, out, total4, tokens, n_prefix, D / 4));
  EVT_LAUNCH_CHECK("embed_fill");
  return EVT_OK;
}

int prefix_tokens_launch(const float* prefix, const float* pos, float* out, int B, int tokens, int n_prefix, int D,
                         cudaStream_t st) {
  EVT_CHECK_ARG(prefix && pos && out, "prefix_tokens: null pointer");
  EVT_CHECK_ARG(B > 0 && tokens > 0 && n_prefix > 0 && n_prefix <= tokens && D > 0, "prefix_tokens: bad sizes");
  const long long total = static_cast<long long>(B) * n_prefix * D;
  EVT_CUDA(launch_pdl(prefix_tokens_kernel, dim3(static_cast<unsigned>((total + 255) / 256)), dim3(256), 0, st, pdl_for_rows(static_cast<long long>(B) * tokens), prefix, pos,
                      out, B, tokens, n_prefix, D));
  EVT_LAUNCH_CHECK("prefix_tokens");
  return EVT_OK;
}

int cast_launch(const float* x, void* y, int64_t n, cudaStream_t st) {
  EVT_CHECK_ARG(x && y && n > 0, "cast: bad arguments");
  EVT_CHECK_ARG(reinterpret_cast<uintptr_t>(x) % 16 == 0 && reinterpret_cast<uintptr_t>(y) % 16 == 0,
                "cast: pointers must be 16-byte aligned");
  const long long n8 = n / 8;
  const long long threads = n8 + 1;
  cast_kernel<<<static_cast<unsigned>((threads + 255) / 256), 256, 0, st>>>(x, reinterpret_cast<__nv_bfloat16*>(y), n8, n);
  EVT_LAUNCH_CHECK("cast");
  return EVT_OK;
}

int unfold_launch(const void* x, int x_dtype, void* out, int64_t ldo, int B, int H, int W, int C, int k, int s, int p,
                  cudaStream_t st) {
  EVT_CHECK_ARG(x && out, "unfold: null pointer");
  EVT_CHECK_ARG(B > 0 && H > 0 && W > 0 && C > 0 && k > 0 && s > 0 && p >= 0, "unfold: bad sizes");
  EVT_CHECK_ARG(ldo >= static_cast<int64_t>(k) * k * C, "unfold: ldo smaller than k*k*C");
  const int oh = (H + 2 * p - k) / s + 1, ow = (W + 2 * p - k) / s + 1;
  EVT_CHECK_ARG(oh > 0 && ow > 0, "unfold: empty output");
  const long long total = static_cast<long long>(B) * oh * ow * ldo;
  const unsigned grid = static_cast<unsigned>((total + 255) / 256);
  if (x_dtype == EVT_F32)
    unfold_kernel<float><<<grid, 256, 0, st>>>(reinterpret_cast<const float*>(x), reinterpret_cast<__nv_bfloat16*>(out), ldo,
                                               B, H, W, C, k, s, p, oh, ow, total);
  else if (x_dtype == EVT_BF16)
    unfold_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(x),
                                                       reinterpret_cast<__nv_bfloat16*>(out), ldo, B, H, W, C, k, s, p, oh,
                                                       ow, total);
  else
    return fail(EVT_ERR_INVALID, "unfold: x dtype must be f32 or bf16");
  EVT_LAUNCH_CHECK("unfold");
  return EVT_OK;
}

}  // namespace evt

extern "C" int evt_im2col_patch(const float* pixels, void* cols, int B, int H, int W, int P, evt_stream stream) {
  int rc = evt_device_check();
  if (rc != EVT_OK) return rc;
  return evt::im2col_launch(pixels, EVT_PIX_F32, nullptr, nullptr, cols, EVT_BF16, B, H, W, P, static_cast<cudaStream_t>(stream));
}
// ViTEmbeddings.forward as ONE op-level call (SURVEY.md section 8 rows a1 + a2): the same three launches the model runtime
// issues -- patch gather with one row per TOKEN (prefix rows zero), residual rows preset to pos + (prefix token | conv bias),
// tcgen05 GEMM whose TMA reduce-add epilogue adds the projections.
extern "C" int evt_patch_embed_workspace_bytes(int B, int H, int W, int P, int n_prefix, size_t* out) {
  EVT_CHECK_ARG(out != nullptr, "patch_embed: null out");
  EVT_CHECK_ARG(B > 0 && H > 0 && W > 0 && P > 0 && n_prefix > 0 && H % P == 0 && W % P == 0, "patch_embed: bad sizes");
  const size_t tokens = static_cast<size_t>(n_prefix) + static_cast<size_t>(H / P) * (W / P);
  *out = static_cast<size_t>(B) * tokens * 3 * P * P * 2;
  return EVT_OK;
}
extern "C" int evt_patch_embed_fwd(const void* pixels, int pixel_dtype, const float* pixel_scale, const float* pixel_bias,
                                   const void* W, int64_t ldw, const float* bias, const float* prefix, const float* pos,
                                   float* out, void* workspace, int B, int H, int Wd, int P, int D, int n_prefix,
                                   evt_stream stream) {
  int rc = evt_device_check();
  if (rc != EVT_OK) return rc;
  EVT_CHECK_ARG(pixels && W && bias && prefix && pos && out && workspace, "patch_embed: null pointer");
  EVT_CHECK_ARG(B > 0 && H > 0 && Wd > 0 && P > 0 && D > 0 && n_prefix > 0, "patch_embed: sizes must be positive");
  EVT_CHECK_ARG(H % P == 0 && Wd % P == 0, "patch_embed: image size must be a multiple of the patch size");
  const int K = 3 * P * P;
  EVT_CHECK_ARG(D % 4 == 0 && ldw >= K && ldw % 8 == 0, "patch_embed: D must be a multiple of 4, ldw a multiple of 8 and >= 3*P*P");
  EVT_CHECK_ARG(reinterpret_cast<uintptr_t>(workspace) % 1024 == 0, "patch_embed: workspace must be 1 KiB aligned");
  const int tokens = n_prefix + (H / P) * (Wd / P);
  const long long M = static_cast<long long>(B) * tokens;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t row_bytes = static_cast<size_t>(K) * 2;
  EVT_CUDA(cudaMemset2DAsync(workspace, tokens * row_bytes, 0, n_prefix * row_bytes, B, st));
  rc = evt::im2col_launch(pixels, pixel_dtype, pixel_scale, pixel_bias, workspace, EVT_BF16, B, H, Wd, P, st, tokens, n_prefix);
  if (rc != EVT_OK) return rc;
  rc = evt::embed_fill_launch(prefix, pos, bias, out, B, tokens, n_prefix, D, st);
  if (rc != EVT_OK) return rc;
  return evt::gemm_launch(
      {.A = workspace, .lda = K, .W = W, .ldw = ldw, .residual = out, .ldr = D, .out = out, .out_dtype = EVT_F32, .ldo = D, .M = M, .N = D, .K = K}, st);
}
extern "C" int evt_prefix_tokens(const float* prefix, const float* pos, float* out, int B, int tokens, int n_prefix,
                                 int D, evt_stream stream) {
  int rc = evt_device_check();
  if (rc != EVT_OK) return rc;
  return evt::prefix_tokens_launch(prefix, pos, out, B, tokens, n_prefix, D, static_cast<cudaStream_t>(stream));
}
extern "C" int evt_cast_f32_bf16(const float* x, void* y, int64_t n, evt_stream stream) {
  int rc = evt_device_check();
  if (rc != EVT_OK) return rc;
  return evt::cast_launch(x, y, n, static_cast<cudaStream_t>(stream));
}
extern "C" int evt_unfold_nhwc(const void* x, int x_dtype, void* out, int64_t ldo, int B, int H, int W, int C, int k,
                               int s, int p, evt_stream stream) {
  int rc = evt_device_check();
  if (rc != EVT_OK) return rc;
  return evt::unfold_launch(x, x_dtype, out, ldo, B, H, W, C, k, s, p, static_cast<cudaStream_t>(stream));
}
