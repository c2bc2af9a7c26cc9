// Internal launchers shared between the op-level C ABI and the model runtimes.
#pragma once
#include "common.h"

namespace evt {

// out[M, N] = act(A[M, K] W[N, K]^T + bias) (+ residual), row-major with leading dimensions in elements.  Call sites name the
// fields with designated initializers, in declaration order.
struct GemmOp {
  // Rows of out and of the residual for outputs that are not one dense block (evt_gemm_bias_act in include/evt.h); the default
  // is the identity.
  struct RowMap {
    int res_row_mod = 0, res_row_off = 0;
    int out_group = 0, out_group_stride = 0, out_group_off = 0;
  };
  const void* A = nullptr;
  int64_t lda = 0;
  const void* W = nullptr;
  int64_t ldw = 0;
  int in_dtype = EVT_BF16;  // EVT_BF16 (kind::f16) or EVT_F32 (kind::tf32: operands read as fp32, truncated to tf32 by the MMA)
  const float* bias = nullptr;
  const float* residual = nullptr;
  int64_t ldr = 0;
  void* out = nullptr;
  int out_dtype = EVT_BF16;
  int64_t ldo = 0;
  int64_t M = 0;
  int N = 0, K = 0;
  int act = EVT_ACT_NONE;
  RowMap map = {};
  int max_k_splits = 0;  // upper bound on the K splits of a small-M reduce-add (0 = no bound; 1 = fixed summation order)
};
int gemm_launch(const GemmOp& op, cudaStream_t stream);
int gemm_k_splits(const GemmOp& op);  // the K splits gemm_launch would use for `op` (1 = none)

// x <- x + A W^T + bias (f32 residual stream, in place) and xn <- LayerNorm(x) gamma + beta (bf16) for row lengths 192 / 384,
// with whole rows resident in tensor memory (gemm_rowln.cu); copy_ln: the residual stream receives the normalised rows (TF
// dialect).  Supported = large M only (every CTA pair gets a 256-row block).
bool gemm_rowln_supported(int64_t M, int N, int K, bool copy_ln);
bool gemm_rowln_pays(int N, int K, bool copy_ln);  // model runtime: the fused kernel beats GEMM + LayerNorm for this projection
int gemm_rowln_launch(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias, float* resid, int64_t ldr,
                      const float* gamma, const float* beta, float eps, bool copy_ln, void* xn, int64_t ldxn, int64_t M, int N,
                      int K, cudaStream_t stream);

// Sq: query rows per image (1..S; S = all), K and V span all S rows; ctx receives Sq rows per image, packed
int attention_launch(const void* qkv, int64_t ldq, void* ctx, int64_t ldc, const float* head_mask, int B, int S, int Sq,
                     int heads, int head_size, float scale, cudaStream_t stream);

// attention_launch without the EVT_ATTN_MAX_TOKENS cap (any S with B*S < 2^31 - 512; S > 256 runs attention_long_kernel):
// the T2T token transformer's single-head attention over 3136 and 784 tokens
int attention_any_length_launch(const void* qkv, int64_t ldq, void* ctx, int64_t ldc, const float* head_mask, int B, int S, int Sq,
                                int heads, float scale, cudaStream_t stream);

int attention_tf32_launch(const float* qkv, int64_t ldq, float* ctx, int64_t ldc, const float* head_mask, int B, int S,
                          int heads, int head_size, float scale, cudaStream_t stream);

int layernorm_launch(const float* x, int64_t x_stride, const float* gamma, const float* beta, void* y, int y_dtype,
                     int64_t y_stride, float* y_copy, int64_t rows, int D, float eps, cudaStream_t st);

// row_stride > 0: patch p of image b is written to row b * row_stride + row_off + p (one row per token); 0 = dense patch matrix
// pixel_dtype: evt_pixel_dtype; scale3 / bias3 (host, 3 floats each): per-channel affine applied to u8 pixels
// Columns of a patch-matrix row: 3 * P * P, except P = 14, whose 588 are padded with zero columns to kPatchLd14 (16-byte rows).
constexpr int kPatchLd14 = 592;
inline int patch_k(int P) { return P == 14 ? kPatchLd14 : 3 * P * P; }
int im2col_launch(const void* pixels, int pixel_dtype, const float* scale3, const float* bias3, void* cols, int out_dtype, int B,
                  int H, int W, int P, cudaStream_t st, int row_stride = 0, int row_off = 0);
int embed_fill_launch(const float* prefix, const float* pos, const float* bias, float* out, int B, int tokens, int n_prefix, int D,
                      cudaStream_t st);
// swin.cu, P % 4 == 0; out_dtype EVT_BF16 or EVT_TF32
int im2col4_launch(const float* pixels, void* cols, int out_dtype, int B, int H, int W, int P, cudaStream_t st);
// swin.cu: evt_gather_layernorm, evt_window_attention_fwd(_tf32) and evt_layernorm_mean_tokens_ex without the device check
int gather_layernorm_launch(const float* x, const int* idx, const float* gamma, const float* beta, void* y, int y_dtype, float* copy_f32,
                            int64_t images, int T_in, int T_out, int G, int C, float eps, cudaStream_t st);
int window_attention_launch(const void* qkv, int64_t ldq, void* ctx, int64_t ldc, const float* table, int n_tab, int64_t n_windows,
                            int window_tokens, int heads, int head_size, float scale, cudaStream_t st);
int window_attention_tf32_launch(const float* qkv, int64_t ldq, float* ctx, int64_t ldc, const float* table, int n_tab, int64_t n_windows,
                                 int window_tokens, int heads, int head_size, float scale, cudaStream_t st);
int layernorm_mean_tokens_launch(const float* x, const float* gamma, const float* beta, void* y, int y_dtype, int64_t images, int T, int D,
                                 float eps, cudaStream_t st);
int prefix_tokens_launch(const float* prefix, const float* pos, float* out, int B, int tokens, int n_prefix, int D,
                         cudaStream_t st);
int cast_launch(const float* x, void* y, int64_t n, cudaStream_t st);
// T2T front-end pieces (performer.cu)
int unfold_ln_launch(const void* x, int x_dtype, void* out, int64_t ldo, const float* gamma, const float* beta, float eps, int B,
                     int H, int W, int C, int k, int s, int p, cudaStream_t st);
size_t performer_workspace_bytes(int B, int T);
int performer_launch(const void* kqv, int64_t ld, const float* w, void* yattn, float* vout, void* workspace, int B, int T, int emb,
                     int m, float eps, cudaStream_t st);
// y <- v + attn_output(ya); y += mlp(LayerNorm(y)) for 64-wide performer tokens: ya bf16 [rows, 64], y f32 [rows, 64] holding v on
// entry; wo / w1 / w2 bf16 [64 out, 64 in] dense; tanh-GELU
int performer_mlp_launch(const void* ya, float* y, const void* wo, const float* bo, const float* gamma, const float* beta, const void* w1,
                         const float* b1, const void* w2, const float* b2, int64_t rows, float eps, cudaStream_t st);
// the whole Token_performer after the kqv projection in three launches: y f32 [B*T, 64] = the performer's output rows
int performer_block_launch(const void* kqv, int64_t ld, const float* w, float* y, void* workspace, int B, int T, float eps, const void* wo,
                           const float* bo, const float* gamma, const float* beta, const void* w1, const float* b1, const void* w2,
                           const float* b2, float ln_eps, cudaStream_t st, int act = EVT_ACT_GELU_TANH);  // act: the MLP's GELU (evt_act)
// the first soft split of the PyTorch T2T-ViT (nn.Unfold(7, stride 4, padding 2) over NCHW pixels [B,3,H,W] of an evt_pixel_dtype;
// u8 takes scale3 / bias3) + the performer's norm1 -> bf16 [B*oh*ow, 152], columns in (kh, kw, c) order, 147.. zero
int unfold773_nchw_launch(const void* pixels, int pixel_dtype, const float* scale3, const float* bias3, void* out, const float* gamma,
                          const float* beta, float eps, int B, int H, int W, cudaStream_t st);
// T2T Token_transformer after its qkv projection (attention + the performer tail with v from the qkv matrix, erf-GELU): qkv bf16 [B*T, ld],
// q | k | v in columns [0,64) [64,128) [128,192); y f32 [B*T, 64]; workspace token_transformer_workspace_bytes(B, T) bytes
size_t token_transformer_workspace_bytes(int B, int T);
int token_transformer_block_launch(const void* qkv, int64_t ld, float* y, void* workspace, int B, int T, float scale, const void* wo,
                                   const float* bo, const float* gamma, const float* beta, const void* w1, const float* b1, const void* w2,
                                   const float* b2, float ln_eps, cudaStream_t st);
int unfold_launch(const void* x, int x_dtype, void* out, int64_t ldo, int B, int H, int W, int C, int k, int s, int p,
                  cudaStream_t st);

}  // namespace evt
