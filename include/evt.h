/*
 * libevt -- B200-native (sm_100a) ViT / DeiT / T2T inference forward behind a C ABI.
 *
 * The reference (xudoong/EdgeVisionTransformer) has no FFI for this path: callers invoke a
 * Python nn.Module (`model(images).logits`, deit_pruning/src/utils.py:194-195,
 * are_16_heads/classifier_eval.py:69-70; op-level models utils.py:322-365).  This header is the
 * boundary a binding for that path would use; INTEGRATION.md shows the ctypes stub.  Each entry
 * point cites the reference interface it replaces.
 *
 * Conventions
 *   - every function returns int: 0 = EVT_OK, negative = EVT_ERR_*; never throws.
 *   - evt_last_error() returns a thread-local message for the last failing call.
 *   - all data pointers are DEVICE pointers unless the name says host; `stream` is a cudaStream_t.
 *   - calls are asynchronous on `stream`: no allocation, no host sync, CUDA-graph capturable,
 *     unless stated otherwise.
 *   - there is no CPU fallback: a device that is not compute capability 10.x -> EVT_ERR_UNSUPPORTED.
 *   - bf16 matrices given to the GEMM / attention ops need 16-byte aligned base pointers and
 *     leading dimensions that are multiples of 8 elements (TMA requirement).
 */
#ifndef EVT_H_
#define EVT_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EVT_VERSION 100

enum evt_status {
  EVT_OK = 0,
  EVT_ERR_INVALID = -1,      /* bad argument (maps to ValueError in the Python wrapper)   */
  EVT_ERR_CUDA = -2,         /* a CUDA runtime / driver call failed                        */
  EVT_ERR_UNSUPPORTED = -3,  /* not an sm_100 device, or shape outside the kernel's range  */
  EVT_ERR_STATE = -4         /* call order violated (e.g. forward before weights loaded)   */
};

/* EVT_TF32 is f32 storage whose values are rounded (to nearest) to tf32 precision when written: use it for
 * outputs that feed a tf32 GEMM / attention, whose tensor cores would otherwise truncate. */
enum evt_dtype { EVT_F32 = 0, EVT_BF16 = 1, EVT_TF32 = 2 };

/* activation fused in the GEMM epilogue.  ERF: HF `hidden_act="gelu"`
 * (SITE/models/vit/modeling_vit.py:291-299); TANH: modeling/torch_layers/activation.py:4-7. */
enum evt_act { EVT_ACT_NONE = 0, EVT_ACT_GELU_ERF = 1, EVT_ACT_GELU_TANH = 2 };

typedef void* evt_stream;

const char* evt_last_error(void);
int evt_version(void);
/* EVT_OK when the current CUDA device can run the kernels (compute capability 10.x). */
int evt_device_check(void);
/* Number of kernel launches issued by this library on the calling thread since the last reset. */
int64_t evt_launch_count(void);
void evt_launch_count_reset(void);
/* GEMM kernel choice: -1 = automatic (CTA-pair kernel, tcgen05 cta_group::2, for problems with at least one
 * 256-row tile per SM), 0 = always the single-CTA kernel, 1 = the CTA-pair kernel whenever it is applicable.
 * Results are identical either way (same K order, same epilogue); the switch exists for tests and tuning.
 * Initial value: environment variable EVT_GEMM_PAIR if set, else -1. */
void evt_gemm_set_pair_mode(int mode);
/* Split K across idle SMs for residual (reduce-add) GEMMs whose tile count leaves most of the GPU idle -- the batch-1
 * latency path (DeiT-Base batch 1: 1.03 -> 0.62 ms).  The partial products meet in the f32 residual stream through TMA
 * reduce-adds whose order is not fixed, so with splitting on (the default) small-batch bf16 results can differ from run
 * to run and from one batch size to another by a last-bit f32 difference in the residual stream (which bf16 roundings
 * downstream turn into logit differences of a few 1e-3, inside the 2e-2 parity budget); 0 turns it off (bit-reproducible,
 * batch-invariant results).  Large batches never split, and neither does the tf32 accuracy mode (splitting would take
 * DeiT-Tiny batch 1 from 0.48 to 0.43 ms, but the logit error would stop being reproducible: 7.5e-4 -> 9.2e-4 of the 1e-3 budget).
 * Initial value: environment variable EVT_GEMM_SPLIT_K if set, else 1. */
void evt_gemm_set_split_k(int enable);
/* Promise, for the evt_gemm_bias_act* calls the calling thread makes while the count is positive, that W is a weight matrix:
 * not written by the launch that precedes the GEMM on its stream.  The GEMM then requests its first W tiles before the
 * programmatic dependency wait, overlapping their HBM round trip with the previous kernel's tail (batch-1 latency path:
 * weights are cold, each is read once per forward).  delta = +1 to enter such a region, -1 to leave it (nestable).  The
 * model-level entry points do this themselves; it is for forwards composed from the op-level calls (Swin, T2T front-end). */
void evt_gemm_weights_static(int delta);

/* ------------------------------------------------------------------ op level ------------- */

/* LayerNorm over the last dim of `rows` rows of length D (nn.LayerNorm,
 * SITE/models/vit/modeling_vit.py:325-326,333,340,455; modeling/layers/norm.py:6).
 * x: f32, row stride x_stride elements.  y: bf16 or f32 (y_dtype), row stride y_stride.
 * y_copy_f32 (nullable): also write the normalised row as f32 with stride x_stride -- may alias x
 * (TF dialect: the skip connection carries LN(x), modeling/layers/norm.py:10-12 + residual.py:8). */
int evt_layernorm_fwd(const float* x, int64_t x_stride, const float* gamma, const float* beta,
                      void* y, int y_dtype, int64_t y_stride, float* y_copy_f32,
                      int64_t rows, int D, float eps, evt_stream stream);

/* Joint LayerNorm over the last TWO dims [n,h] of x[B,n,h] (+ optional addend of the same shape
 * before normalising), affine gamma/beta [n,h]: modeling/torch_layers/norm.py:4-15 as built at
 * utils.py:338,364.  All f32. */
int evt_layernorm2d_fwd(const float* x, const float* addend, const float* gamma, const float* beta,
                        float* y, int64_t batch, int64_t nh, float eps, evt_stream stream);

/* out[M,N] = epilogue( A[M,K] . W[N,K]^T )   -- nn.Linear (modeling/torch_layers/attention.py:19-22,
 * ffn.py:10-11; SITE/models/vit/modeling_vit.py:216-218,262,290,305,640-642).
 *   A, W : bf16 row-major, leading dims lda / ldw (multiples of 8)
 *   bias : f32 [N] or NULL
 *   act  : evt_act, applied after bias
 *   residual : f32 or NULL; added after the activation.  Row r of the output reads residual row
 *              (res_row_mod > 0 ? res_row_off + r % res_row_mod : out_row(r)), leading dim ldr.
 *   out  : bf16 or f32 (out_dtype), leading dim ldo.  out_row(r) = r when out_group == 0, else
 *          (r / out_group) * out_group_stride + out_group_off + r % out_group   (patch-embed rows
 *          1..196 of each image's 197-token block, SITE/models/vit/modeling_vit.py:117-126).
 *   residual may alias out (in-place residual stream update). */
int evt_gemm_bias_act(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias,
                      const float* residual, int64_t ldr, int res_row_mod, int res_row_off,
                      void* out, int out_dtype, int64_t ldo,
                      int out_group, int out_group_stride, int out_group_off,
                      int64_t M, int N, int K, int act, evt_stream stream);

/* tf32 flavour of evt_gemm_bias_act: A and W are f32 (read as tf32 by the tensor core, f32 accumulate),
 * out is f32; leading dims multiples of 4.  Used by the tf32 accuracy mode (max-abs 1e-3 on logits). */
int evt_gemm_bias_act_tf32(const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias,
                           const float* residual, int64_t ldr, int res_row_mod, int res_row_off,
                           float* out, int64_t ldo, int out_group, int out_group_stride, int out_group_off,
                           int64_t M, int N, int K, int act, evt_stream stream);

/* out[M,N] (bf16) = act( LayerNorm(x)[M,K] W[N,K]^T + bias ) -- the LayerNorm that precedes a projection, run inside
 * the GEMM as the producer of its A operand: layernorm_before -> query|key|value and layernorm_after ->
 * intermediate.dense of a ViT layer (SITE/models/vit/modeling_vit.py:333-340) for narrow residual streams, where the
 * stand-alone LayerNorm pass is HBM traffic the encoder cannot afford (DeiT-Tiny / -Small, T2T-ViT).
 *   x : f32 [M, ldx] (ldx % 4 == 0, 16-byte aligned); K = row length, one of 64, 128, 192, 256, 384
 *   x_copy_f32 (nullable, may alias x): the normalised rows written back as f32 (TF dialect skip connection)
 *   W : bf16 [N, ldw]; bias f32 [N] or NULL; out bf16 [M, ldo] (ldo % 8 == 0)
 * Statistics are f32 with a centred variance, exactly as evt_layernorm_fwd computes them. */
int evt_layernorm_gemm(const float* x, int64_t ldx, const float* gamma, const float* beta, float eps, float* x_copy_f32,
                       const void* W, int64_t ldw, const float* bias, void* out, int64_t ldo, int64_t M, int N, int K,
                       int act, evt_stream stream);

/* Residual projection with the following LayerNorm fused into the epilogue (bf16 A and W):
 *     resid[M,N] <- resid + A[M,K] W[N,K]^T + bias        (f32, in place)
 *     xn[M,N]    <- LayerNorm(resid) * gamma + beta        (bf16)
 * = ViTSelfOutput.dense + the skip connection + layernorm_after, and ViTOutput.dense + skip + the next layer's
 * layernorm_before (SITE/models/vit/modeling_vit.py:265-268, 308-312, 333-340), without re-reading the residual
 * stream from HBM.  Statistics are fp32 with a centred variance (exact for constant rows with eps = 1e-12).
 * N must be a multiple of 64 in [64, 1024]; returns EVT_ERR_UNSUPPORTED otherwise (callers fall back to
 * evt_gemm_bias_act + evt_layernorm_fwd, which compute the same thing). */
int evt_gemm_residual_layernorm(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias,
                                float* resid, int64_t ldr, const float* gamma, const float* beta, float eps,
                                void* xn, int64_t ldxn, int64_t M, int N, int K, evt_stream stream);
/* Same, with the reference's TF dialect as an option: copy_ln != 0 makes the residual stream receive the (unrounded f32)
 * normalised rows instead of the sum (modeling/models/vit.py: the skip connection starts from LN(x)).  For N = 192 or 384 and
 * enough rows to give every CTA pair a 256-row block this is ONE kernel that keeps whole rows in tensor memory
 * (csrc/gemm_rowln.cu: the old residual arrives through a TMA ring, the LayerNorm passes read TMEM only); other shapes issue
 * evt_gemm_bias_act + evt_layernorm_fwd.  Any N >= 1 with ldr, ldxn >= N. */
int evt_gemm_residual_layernorm_ex(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias,
                                   float* resid, int64_t ldr, const float* gamma, const float* beta, float eps, int copy_ln,
                                   void* xn, int64_t ldxn, int64_t M, int N, int K, evt_stream stream);

/* Longest sequence the bf16 attention accepts: ViT / DeiT-B/16 at 512 px with a cls and a distillation token
 * (32 * 32 + 2 tokens). */
#define EVT_ATTN_MAX_TOKENS 1026

/* Fused softmax(Q K^T * scale) V, head size 64, any S from 1 to EVT_ATTN_MAX_TOKENS.  S <= 256 keeps every key of a head
 * on chip; longer sequences run query tiles against 128-key blocks with an online softmax (no score tensor in HBM either way):
 * eager_attention_forward SITE/models/vit/modeling_vit.py:171-196 ==
 * modeling/torch_layers/attention.py:36-45 == modeling/layers/attention.py:30-33.
 *   qkv : bf16 [B*S, ldq]; q of head h at columns [h*64, h*64+64), k at [heads*64 + h*64, ...),
 *         v at [2*heads*64 + h*64, ...)
 *   ctx : bf16 [B*S, ldc]; head h written to columns [h*64, h*64+64)
 *   head_mask : f32 [heads] or NULL; ctx of head h is multiplied by head_mask[h]
 *               (are_16_heads `mask_heads`, are_16_heads/run_classifier.py:247-250). */
int evt_attention_fwd(const void* qkv, int64_t ldq, void* ctx, int64_t ldc, const float* head_mask,
                      int B, int S, int heads, int head_size, float scale, evt_stream stream);

/* evt_attention_fwd for the first Sq (1..S) query rows of every image against all S keys: ctx is bf16 [B*Sq, ldc].
 * Those rows are bit-identical to the same rows of evt_attention_fwd. */
int evt_attention_query_rows_fwd(const void* qkv, int64_t ldq, void* ctx, int64_t ldc, const float* head_mask,
                                 int B, int S, int Sq, int heads, int head_size, float scale, evt_stream stream);

/* tf32 flavour of evt_attention_fwd: qkv and ctx are f32 (leading dims multiples of 4); S <= 256 only. */
int evt_attention_fwd_tf32(const float* qkv, int64_t ldq, float* ctx, int64_t ldc, const float* head_mask,
                           int B, int S, int heads, int head_size, float scale, evt_stream stream);

/* Non-overlapping patch gather: pixels f32 NCHW [B,3,H,W] -> bf16 [B*(H/P)*(W/P), 3*P*P] with
 * K order (c, i, j) -- the im2col of Conv2d(3,D,P,P) (SITE/models/vit/modeling_vit.py:151-167).  P a multiple of 4
 * (ViT / DeiT: 16; Swin: 4). */
int evt_im2col_patch(const float* pixels, void* cols, int B, int H, int W, int P, evt_stream stream);

/* ViTEmbeddings.forward as one op-level call (SITE/models/vit/modeling_vit.py:95-126 = cls / distillation token,
 * position embeddings; :151-167 = ViTPatchEmbeddings, Conv2d(3, D, P, P) as an im2col GEMM):
 *   out[b, t, :] = pos[t, :] + (t < n_prefix ? prefix[t, :] : bias + W . patch(b, t - n_prefix))
 * pixels    NCHW [B,3,H,W] of pixel_dtype (evt_pixel_dtype: f32, bf16 or raw u8; u8 takes pixel_scale / pixel_bias,
 *           3 HOST floats each, applied as x * scale[c] + bias[c] inside the patch gather; NULL otherwise)
 * W         bf16 [D, ldw], K order (c, i, j) = conv.weight.reshape(D, -1); ldw >= 3*P*P, multiple of 8
 * bias      f32 [D]; prefix f32 [n_prefix, D] (cls, or cls + distillation token); pos f32 [tokens, D]
 * out       f32 [B * tokens, D], tokens = n_prefix + (H/P)*(W/P)
 * workspace evt_patch_embed_workspace_bytes bytes, 1 KiB aligned (the bf16 patch matrix, one row per token)
 * P a multiple of 8.  Three launches (patch gather, row preset, tcgen05 GEMM with a TMA reduce-add epilogue). */
int evt_patch_embed_workspace_bytes(int B, int H, int W, int P, int n_prefix, size_t* out);
int evt_patch_embed_fwd(const void* pixels, int pixel_dtype, const float* pixel_scale, const float* pixel_bias,
                        const void* W, int64_t ldw, const float* bias, const float* prefix, const float* pos,
                        float* out, void* workspace, int B, int H, int Wd, int P, int D, int n_prefix,
                        evt_stream stream);

/* Rows [0, n_prefix) of each image's token block: out[b, t, :] = prefix[t, :] + pos[t, :]
 * (cls / distillation token + position embedding, SITE/models/vit/modeling_vit.py:117-126). */
int evt_prefix_tokens(const float* prefix, const float* pos, float* out, int B, int tokens, int n_prefix,
                      int D, evt_stream stream);

/* f32 -> bf16 cast of n elements (n multiple of 1; pointers 16-byte aligned). */
int evt_cast_f32_bf16(const float* x, void* y, int64_t n, evt_stream stream);

/* T2T soft split (tf_Unfold, modeling/models/t2t_vit.py:20-40): x NHWC [B,H,W,C] (f32 or bf16) ->
 * bf16 [B*oh*ow, ldo] with depth order (kh, kw, c), zero padding p; ldo >= k*k*C, pad cols zeroed. */
int evt_unfold_nhwc(const void* x, int x_dtype, void* out, int64_t ldo, int B, int H, int W, int C,
                    int k, int s, int p, evt_stream stream);

/* T2T soft split fused with the following LayerNorm (TokenPerformer.norm1, transformer_encoder.py:49,97): like
 * evt_unfold_nhwc, each output row normalised over its k*k*C elements (gamma/beta f32 [k*k*C]; both NULL = no LN). */
int evt_unfold_ln_nhwc(const void* x, int x_dtype, void* out, int64_t ldo, const float* gamma, const float* beta,
                       float eps, int B, int H, int W, int C, int k, int s, int p, evt_stream stream);

/* TokenPerformer.single_attn core (modeling/layers/transformer_encoder.py:67-94) for emb = 64, m = 32:
 *   kqv   : bf16 [B*T, ld], k | q | v in columns [0,64) [64,128) [128,192)   (output of the kqv Dense)
 *   w     : f32 [32, 64], already multiplied by sqrt(m) (transformer_encoder.py:65)
 *   yattn : bf16 [B*T, 64] = (qp kptv^T) / (qp.ksum + eps)
 *   vout  : f32 [B*T, 64]  = v (the skip input that attn_output's GEMM is then added into)
 *   workspace : evt_performer_workspace_bytes(B, T) bytes. */
int evt_performer_workspace_bytes(int B, int T, size_t* out);
int evt_performer_fwd(const void* kqv, int64_t ld, const float* w, void* yattn, float* vout, void* workspace,
                      int B, int T, int emb, int m, float eps, evt_stream stream);

/* What Token_performer does after the attention contraction (modeling/layers/transformer_encoder.py:93-99), 64-wide tokens, one
 * kernel:   y <- y + attn_output(ya) ;  y <- y + fc2(gelu_tanh(fc1(LayerNorm(y))))
 *   ya : bf16 [rows, 64] (evt_performer_fwd's yattn);  y : f32 [rows, 64], holds v on entry (evt_performer_fwd's vout), in place
 *   wo, w1, w2 : bf16 [64 out, 64 in] dense;  bo, b1, b2 : f32 [64] or NULL;  gamma, beta : f32 [64] (norm2);  all 16-byte aligned
 * Same arithmetic as evt_gemm_bias_act (f32 residual) + evt_layernorm_fwd + evt_gemm_bias_act (tanh-GELU) + evt_gemm_bias_act,
 * which it replaces in the T2T front-end: 640 instead of 1920 bytes of HBM traffic per token. */
int evt_performer_mlp_fwd(const void* ya, float* y, const void* wo, const float* bo, const float* gamma, const float* beta,
                          const void* w1, const float* b1, const void* w2, const float* b2, int64_t rows, float eps,
                          evt_stream stream);

/* evt_performer_fwd + evt_performer_mlp_fwd in three launches instead of four: the apply kernel carries each 16-token tile straight
 * on through attn_output + LayerNorm + MLP, so yattn and v never go to HBM (512 bytes per token: q, v in; y out).  Bit-identical to
 * the two calls.  y : f32 [B*T, 64] out = the Token_performer's output rows; ln_eps = norm2's epsilon. */
int evt_performer_block_fwd(const void* kqv, int64_t ld, const float* w, float* y, void* workspace, int B, int T, float eps,
                            const void* wo, const float* bo, const float* gamma, const float* beta, const void* w1,
                            const float* b1, const void* w2, const float* b2, float ln_eps, evt_stream stream);

/* ---- Swin shifted-window block (tools.py:265-292 export_onnx_swin, utils.py:14-47 get_swin; arithmetic:
 * SITE/models/swin/modeling_swin.py).  Token rows are kept in the window order of the current block, see
 * edgevisiontransformer_b200/modeling_swin.py. */

/* Row gather fused with LayerNorm: output row r (image r / T_out, token t = r % T_out) is the concatenation of the G
 * input rows  image * T_in + idx[t * G + g]  (g = 0..G-1, each C floats) of x, normalised over its G*C elements.
 *   G = 1: window partition / cyclic shift / reverse (SwinLayer.forward :606-637) folded into layernorm_before;
 *          copy_f32 (nullable) receives the gathered, un-normalised rows = the residual stream in the new order
 *   G = 4: SwinPatchMerging (:326-349): 2x2 neighbourhood concat + LayerNorm(4C)
 *   y (nullable when copy_f32 is given): bf16 or f32 [images * T_out, G*C]; idx: int32 [T_out * G] (device). */
int evt_gather_layernorm(const float* x, const int* idx, const float* gamma, const float* beta, void* y, int y_dtype,
                         float* copy_f32, int64_t images, int T_in, int T_out, int G, int C, float eps, evt_stream stream);

/* Window attention (SwinSelfAttention.forward :410-459) for 7x7 (window_tokens = 49) or 12x12 (window_tokens = 144)
 * windows, head size 32; anything else is EVT_ERR_UNSUPPORTED:
 *   ctx = softmax(q k^T * scale + relative_position_bias + shift_mask) v   per (window, head)
 *   qkv   : bf16 [n_windows * N, ldq] (N = window_tokens), columns q | k | v (heads*32 each), rows in window order
 *   table : (bias[h] + mask[w % n_tab]) * log2(e), the shift mask being HF's 0 / -100; n_tab = windows per image for
 *           shifted blocks, 1 otherwise
 *           N = 49 : f32 [n_tab, heads, 64, 56], key columns 49..55 = -inf, rows 49..63 finite
 *           N = 144: f32 [n_tab, heads, 144, 144]
 *   ctx   : bf16 [n_windows * N, ldc]. */
int evt_window_attention_fwd(const void* qkv, int64_t ldq, void* ctx, int64_t ldc, const float* table, int n_tab,
                             int64_t n_windows, int window_tokens, int heads, int head_size, float scale, evt_stream stream);

/* y[image, :] (bf16) = mean over the T tokens of LayerNorm(x[image, t, :]) -- SwinModel.layernorm + AdaptiveAvgPool1d
 * (:899-904).  x f32 [images, T, D]. */
int evt_layernorm_mean_tokens(const float* x, const float* gamma, const float* beta, void* y, int64_t images, int T, int D,
                              float eps, evt_stream stream);

/* ------------------------------------------------------------------ model level ---------- */

typedef struct evt_model evt_model;

#define EVT_MAX_LAYERS 64

/* arithmetic mode of the whole forward.  BF16: bf16 GEMM / attention operands, f32 accumulate, f32 residual
 * stream (logits within 2e-2 of the f32 reference).  TF32: f32 activations and weights read as tf32 by the
 * tensor cores (logits within 1e-3). */
enum evt_precision { EVT_PREC_BF16 = 0, EVT_PREC_TF32 = 1 };

enum evt_dialect {
  EVT_DIALECT_HF = 0,   /* HF ViT/DeiT: pre-LN, qkv bias, final LN + Linear head            */
  EVT_DIALECT_TF = 1    /* modeling/models/vit.py: skip carries LN(x), no qkv bias, no final
                           LN, 2-layer MLP head; also the T2T-ViT encoder (final LN + Dense) */
};

typedef struct evt_model_spec {
  int dialect;                 /* evt_dialect */
  int hidden;                  /* D */
  int layers;                  /* L <= EVT_MAX_LAYERS */
  int tokens;                  /* patches + 1 (cls) or + 2 (DeiT distillation token): 197 / 198 at 224 px, 577 / 578 at
                                  384 px; up to EVT_ATTN_MAX_TOKENS in bf16, up to 256 in the tf32 mode */
  int image, patch;            /* 224, 16 */
  int head_size;               /* 64 */
  int num_labels;              /* 1000 */
  int act;                     /* evt_act for the FFN */
  float eps;                   /* LayerNorm epsilon */
  int heads[EVT_MAX_LAYERS];   /* surviving heads per layer (HF prune_heads semantics)       */
  int inter[EVT_MAX_LAYERS];   /* FFN width per layer (optimize_model semantics), any int>0  */
  int final_ln;                /* 1: LayerNorm before the head (HF, T2T); 0: TF-dialect DeiT */
  int head_hidden;             /* 0: single Linear head; >0: Dense(head_hidden, gelu)->Dense */
  int t2t;                     /* 1: T2T front-end (NHWC input) instead of the patch embed   */
  int precision;               /* evt_precision: 0 bf16 operands, 1 tf32 operands (f32 activations) */
  int embed_k;                 /* 0: 3*patch*patch.  >0: K of the token-embedding GEMM when the caller builds the
                                  patch matrix itself (T2T: 3*3*64 = 576) and calls evt_model_forward_embedded */
  int head_rows;               /* 0 / 1: the classifier reads the cls row.  2: HF DeiTForImageClassificationWithTeacher
                                  (SITE/models/deit/modeling_deit.py, logits = (cls_classifier(x[:,0]) +
                                  distillation_classifier(x[:,1])) / 2): rows 0 and 1 are normalised into one 2D-wide row
                                  and "classifier.weight" is [num_labels, 2D] = [W_cls | W_dist] / 2, "classifier.bias"
                                  = (b_cls + b_dist) / 2 (the Python loader builds both); needs tokens = patches + 2 */
} evt_model_spec;

typedef struct evt_tensor_view {
  const char* name;            /* weight name, see INTEGRATION.md (HF state_dict keys)        */
  const void* data;            /* f32, contiguous, DEVICE pointer                              */
  int ndim;
  int64_t shape[4];
} evt_tensor_view;

/* Validate the spec and allocate an empty model on the current device (allocates; not async). */
int evt_model_create(const evt_model_spec* spec, evt_model** out);
/* Repack weights into the library's own padded bf16 / f32 buffers (allocates; synchronises `stream`).
 * The caller keeps ownership of the views.  Missing or mis-shaped tensors -> EVT_ERR_INVALID. */
int evt_model_load_weights(evt_model* m, const evt_tensor_view* tensors, int n, evt_stream stream);
/* Bytes of caller-provided scratch needed for a forward at `batch`. */
int evt_model_workspace_bytes(const evt_model* m, int batch, size_t* out);
/* logits[batch, num_labels] (f32) = forward(pixels f32 NCHW [batch,3,image,image]); async on stream. */
int evt_model_forward(evt_model* m, const float* pixels, int batch, float* logits,
                      void* workspace, size_t workspace_bytes, evt_stream stream);
/* Pixel storage accepted by evt_model_forward_ex: the conversion is fused into the patch gather (im2col), so a caller that
 * keeps bf16 or raw u8 images in pinned host memory moves 2x / 4x fewer bytes over PCIe than with f32. */
enum evt_pixel_dtype { EVT_PIX_F32 = 0, EVT_PIX_BF16 = 1, EVT_PIX_U8 = 2 };

/* Optional inputs / outputs of one forward.  A zero-initialised struct == evt_model_forward. */
typedef struct evt_forward_opts {
  int pixel_dtype;           /* evt_pixel_dtype of `pixels` (NCHW [batch,3,image,image])                                    */
  float pixel_scale[3];      /* EVT_PIX_U8 only: value = pixel * scale[c] + bias[c], i.e. scale = 1/(255 std[c]),           */
  float pixel_bias[3];       /*   bias = -mean[c]/std[c] -- torchvision Normalize, deit_pruning/src/utils.py:118-133        */
  const float* head_mask;    /* NULL, or DEVICE f32 [layers, head_mask_ld]: head h of layer l is multiplied by              */
  int head_mask_ld;          /*   head_mask[l*ld + h] (h < heads[l]) -- HF forward(head_mask=...) and are_16_heads           */
                             /*   `model.vit.mask_heads(to_prune)`, are_16_heads/run_classifier.py:247-250                   */
  void* const* ctx_out;      /* NULL, or HOST array of `layers` DEVICE pointers (entries may be NULL): layer l's attention   */
                             /*   context before the output projection, [batch*tokens, heads[l]*64] in the operand type      */
                             /*   (bf16; f32 in tf32 mode) = `context_layer_val` of are_16_heads/classifier_eval.py:183-191  */
                             /*   (reshape to [batch, tokens, heads, 64] and permute to [batch, heads, tokens, 64])          */
} evt_forward_opts;

/* evt_model_forward with options (opts may be NULL).  Same launch count, same workspace. */
int evt_model_forward_ex(evt_model* m, const void* pixels, const evt_forward_opts* opts, int batch, float* logits,
                         void* workspace, size_t workspace_bytes, evt_stream stream);
/* Same forward, starting from the A operand of the token-embedding GEMM instead of pixels: patch_matrix is
 * [batch*patches, ld] in the operand type of the model's precision (bf16, or f32 for tf32).  Used by the T2T front-end
 * (tokens-to-token module, modeling/models/t2t_vit.py:63-88), whose last soft split produces exactly that matrix. */
int evt_model_forward_embedded(evt_model* m, const void* patch_matrix, int64_t ld, int batch, float* logits,
                               void* workspace, size_t workspace_bytes, evt_stream stream);
/* Number of kernel launches one forward issues at small batch (3 + 7 per layer + head; T2T front-end extra).  At large batch
 * a model with hidden size 192 or 384 issues up to two fewer per layer: the LayerNorm that follows a residual projection runs
 * in that projection's epilogue (evt_gemm_residual_layernorm_ex).  evt_launch_count() reports what was actually launched;
 * bench.py's gpu_launches is taken from it. */
int evt_model_launches_per_forward(const evt_model* m);
/* Measurement aid (bench.py's roofline): between begin and end every forward on `m` records a CUDA event on its
 * stream before its first launch and after every launch.  end synchronises on the last event, adds the elapsed time
 * between consecutive events to the stage of the launch they bracket (sum over all forwards since begin) and returns
 * the number of launches per stage.  Forwards issued while profiling is on must not be stream-captured. */
enum evt_stage {
  EVT_STAGE_EMBED = 0,  /* im2col, patch GEMM, cls/pos rows   */
  EVT_STAGE_LN = 1,     /* layernorm_before / layernorm_after */
  EVT_STAGE_QKV = 2,
  EVT_STAGE_ATTN = 3,
  EVT_STAGE_OPROJ = 4,
  EVT_STAGE_FC1 = 5,
  EVT_STAGE_FC2 = 6,
  EVT_STAGE_HEAD = 7,   /* final LN on cls rows + classifier  */
  EVT_STAGE_COUNT = 8
};
int evt_model_profile_begin(evt_model* m);
int evt_model_profile_end(evt_model* m, float* stage_ms /* [EVT_STAGE_COUNT] */, int* stage_launches /* [EVT_STAGE_COUNT] */);
int evt_model_destroy(evt_model* m);

/* ------------------------------------------------------------------ Swin model level ----- */

/* The shifted-window classifier the reference builds with utils.get_swin (utils.py:14-47) and exports / benchmarks in
 * tools.py:265-292 (swin_{tiny,small,base}_patch4_window7_224), arithmetic as in SITE/models/swin/modeling_swin.py;
 * also the 384-pixel swin_{base,large}_patch4_window12_384 (12 x 12 windows).
 * One call = the whole forward as a fixed launch sequence on `stream` (CUDA-graph capturable).  bf16 operands, f32
 * accumulate / residual stream / LayerNorm / softmax. */
typedef struct evt_swin evt_swin;

#define EVT_SWIN_MAX_STAGES 8

typedef struct evt_swin_spec {
  int image, patch, window;          /* 224, 4, 7 (swin_*_window7_224) or 384, 4, 12 (swin_*_window12_384); window 7 or 12 */
  int embed_dim;                     /* 96 (tiny / small), 128 (base), 192 (large); head size is 32 in every stage */
  int stages;                        /* 4 */
  int depths[EVT_SWIN_MAX_STAGES];   /* blocks per stage, e.g. 2, 2, 6, 2 */
  int heads[EVT_SWIN_MAX_STAGES];    /* heads per stage, e.g. 3, 6, 12, 24 */
  int num_labels;
  float eps;                         /* LayerNorm epsilon (1e-5) */
} evt_swin_spec;

int evt_swin_create(const evt_swin_spec* spec, evt_swin** out);
/* Weights under their HF names (swin.embeddings..., swin.encoder.layers.{s}.blocks.{b}..., swin.layernorm, classifier),
 * f32 DEVICE tensors.  The window orders, cyclic-shift gathers, patch-merging gathers and the (relative position bias +
 * shift mask) tables are computed here on the host from the geometry and the bias tables.  Allocates; synchronises. */
int evt_swin_load_weights(evt_swin* m, const evt_tensor_view* tensors, int n, evt_stream stream);
int evt_swin_workspace_bytes(const evt_swin* m, int batch, size_t* out);
/* logits[batch, num_labels] (f32) = forward(pixels f32 NCHW [batch,3,image,image]) */
int evt_swin_forward(evt_swin* m, const float* pixels, int batch, float* logits, void* workspace, size_t workspace_bytes,
                     evt_stream stream);
int evt_swin_launches_per_forward(const evt_swin* m);
int evt_swin_destroy(evt_swin* m);

#ifdef __cplusplus
}
#endif
#endif /* EVT_H_ */
