// Whole-model runtime: owns repacked weights, lays out the caller's workspace, and issues the forward
// as a fixed sequence of kernel launches on one stream (no allocation, no sync -> CUDA-graph capturable).
//
// Forward (HF dialect; SITE/models/vit/modeling_vit.py:620-653, ViTLayer :328-346):
//   im2col -> patch GEMM (+bias +pos, rows 1.. of each token block) -> cls(+dist) rows
//   L x [ LN -> QKV GEMM -> attention -> out-proj GEMM (+residual) -> LN -> FC1 GEMM (+GELU) -> FC2 GEMM (+residual) ]
//   LN on the cls rows only -> classifier GEMM
// The residual stream is fp32 in HBM; GEMM operands are bf16; LN statistics, softmax and accumulation fp32.
// TF dialect (modeling/models/vit.py, modeling/layers/norm.py:10-12): LN writes its result back into the
// residual stream, because there the skip connection carries LN(x).
#include <cuda_bf16.h>

#include <string>
#include <vector>

#include "loader.h"
#include "ops.h"
#include "ptx.cuh"

namespace evt {
namespace {

__device__ __forceinline__ void store_as(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
__device__ __forceinline__ void store_as(float* p, float v) { *p = ptx::round_tf32(v); }  // f32 storage == tf32 operand

template <typename T>
__global__ void __launch_bounds__(256) convert_pad_kernel(const float* __restrict__ src, T* __restrict__ dst, long long rows,
                                                          int cols, int ld) {
  const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= rows * ld) return;
  const int c = static_cast<int>(t % ld);
  const long long r = t / ld;
  store_as(dst + t, c < cols ? src[r * cols + c] : 0.f);
}

// dst[n, k] (bf16, leading dimension ld, zero padded) = src[k, n]: a Keras Dense kernel [in, out] as the [out, in] weight
__global__ void __launch_bounds__(256) convert_pad_transposed_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst,
                                                                     int rows_out, int cols_out, int ld) {
  const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= static_cast<long long>(rows_out) * ld) return;
  const int c = static_cast<int>(t % ld);
  const int r = static_cast<int>(t / ld);
  dst[t] = __float2bfloat16_rn(c < cols_out ? src[static_cast<long long>(c) * rows_out + r] : 0.f);
}

// bf16 rows gathered with a stride from an f32 matrix (cls rows for a head without final LN)
template <typename T>
__global__ void __launch_bounds__(256) gather_rows_cast_kernel(const float* __restrict__ x, long long x_stride,
                                                               T* __restrict__ y, long long rows, int D) {
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();
  const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= rows * D) return;
  const int c = static_cast<int>(t % D);
  const long long r = t / D;
  store_as(y + t, x[r * x_stride + c]);
}

inline int padn(int v, int n) { return (v + n - 1) / n * n; }

struct LayerW {
  uint8_t *wqkv = nullptr, *wo = nullptr, *w1 = nullptr, *w2 = nullptr;  // bf16 or f32 (tf32 mode) matrices
  float *bqkv = nullptr, *bo = nullptr, *b1 = nullptr, *b2 = nullptr;
  float *ln1_g = nullptr, *ln1_b = nullptr, *ln2_g = nullptr, *ln2_b = nullptr;
  float* rel_tab = nullptr;  // BEiT relative position bias: [heads, (2W-1)^2 + 3] times log2(e), or null
  int a = 0, inter = 0, inter_ld = 0;
};

// one TokenPerformer of the T2T front-end (modeling/layers/transformer_encoder.py:39-101), emb = 64, m = 32; with spec.t2t = 3 one
// Token_transformer (PyTorch T2T-ViT, tokens_type='transformer'): wkqv = the bias-free qkv projection (rows q | k | v), no w
struct PerformerW {
  int in_dim = 0, in_ld = 0;            // 147 / 576, leading dimension of the unfolded rows (multiple of 8)
  float *g1 = nullptr, *b1 = nullptr;   // norm1 over the unfolded row
  __nv_bfloat16 *wkqv = nullptr, *wo = nullptr, *w1 = nullptr, *w2 = nullptr;
  float *bkqv = nullptr, *w = nullptr, *bo = nullptr, *g2 = nullptr, *b2 = nullptr, *bb1 = nullptr, *bb2 = nullptr;
};

}  // namespace
}  // namespace evt

struct evt_model {
  evt_model_spec spec;
  int device = 0;
  bool loaded = false;
  int patches = 0, n_prefix = 0, patch_k = 0;
  int es = 2;    // bytes per GEMM operand element: 2 (bf16) or 4 (tf32 mode)
  int pad = 8;   // elements per 16 bytes
  std::vector<evt::LayerW> layers;
  uint8_t* w_patch = nullptr;
  float* b_patch = nullptr;
  float* prefix = nullptr;  // [n_prefix, D]
  float* pos = nullptr;     // [tokens, D]
  float *lnf_g = nullptr, *lnf_b = nullptr;
  uint8_t* w_pre = nullptr;
  float* b_pre = nullptr;
  uint8_t* w_cls = nullptr;
  float* b_cls = nullptr;
  evt::PerformerW perf[2];   // spec.t2t: the two TokenPerformers of the tokens-to-token module
  int rel_grid = 0;          // W of the BEiT relative position bias (layers[l].rel_tab), 0 without it
  std::vector<void*> allocs;
  // evt_model_profile_begin/end: one event before the first launch and one after every launch of a forward
  bool profiling = false;
  std::vector<cudaEvent_t> prof_events;      // pool, reused across forwards
  size_t prof_used = 0;
  std::vector<std::pair<int, std::pair<size_t, size_t>>> prof_spans;  // (stage, (event before, event after))
};

namespace evt {
namespace {

struct Workspace {
  float* resid;
  uint8_t *xn, *qkv, *ctx, *big, *clsn, *hh;  // activations in the GEMM operand type (bf16, or f32 in tf32 mode)
  // T2T front-end (spec.t2t): per performer stage the unfolded + normalised rows, k|q|v, the f32 token
  // stream y and the performer scratch; `pm` = the patch matrix of the embedding GEMM
  uint8_t *t_x[2], *t_kqv[2], *t_ws[2], *t_pm;
  float* t_y[2];
  size_t bytes;
};

// token grid of the T2T soft splits for a square image: unfold(7,4,2) -> unfold(3,2,1) -> unfold(3,2,1)
inline int t2t_side(int image, int stage) {
  int s = (image + 2 * 2 - 7) / 4 + 1;
  for (int i = 0; i < stage; ++i) s = (s + 2 * 1 - 3) / 2 + 1;
  return s;
}

Workspace plan_workspace(const evt_model* m, int batch, uint8_t* base) {
  const evt_model_spec& s = m->spec;
  const size_t M = static_cast<size_t>(batch) * s.tokens;
  const size_t Mp = static_cast<size_t>(batch) * m->patches;
  int amax = 0, imax_ld = 0;
  for (int l = 0; l < s.layers; ++l) {
    amax = std::max(amax, s.heads[l] * s.head_size);
    imax_ld = std::max(imax_ld, padn(s.inter[l], m->pad));
  }
  WorkspaceCarver c{base};
  Workspace w;
  const size_t es = m->es;
  w.resid = c.take<float>(M * s.hidden * 4);
  w.xn = c.take(M * s.hidden * es);
  w.qkv = c.take(M * 3 * amax * es);
  w.ctx = c.take(M * amax * es);
  // the patch matrix has one row per TOKEN when the library builds it (pixels path), see forward_impl
  w.big = c.take(std::max(M * imax_ld, (s.embed_k > 0 ? Mp : M) * static_cast<size_t>(m->patch_k)) * es);
  w.clsn = c.take(static_cast<size_t>(batch) * s.hidden * (s.head_rows > 1 ? s.head_rows : 1) * es);
  w.hh = c.take(static_cast<size_t>(batch) * std::max(padn(s.head_hidden, m->pad), 8) * es);
  if (s.t2t) {
    for (int i = 0; i < 2; ++i) {
      const size_t T = static_cast<size_t>(t2t_side(s.image, i)) * t2t_side(s.image, i) * batch;
      const size_t in_ld = i == 0 ? 152 : 576;
      w.t_x[i] = c.take(T * in_ld * 2);
      w.t_kqv[i] = c.take(T * 192 * 2);
      w.t_y[i] = c.take<float>(T * 64 * 4);
      const int Ti = t2t_side(s.image, i) * t2t_side(s.image, i);
      w.t_ws[i] = c.take(s.t2t == 3 ? token_transformer_workspace_bytes(batch, Ti) : performer_workspace_bytes(batch, Ti));
    }
    w.t_pm = c.take(Mp * 576 * 2);
  }
  w.bytes = c.bytes;
  return w;
}

int validate_spec(const evt_model_spec* s) {
  EVT_CHECK_ARG(s != nullptr, "model spec is null");
  EVT_CHECK_ARG(s->dialect == EVT_DIALECT_HF || s->dialect == EVT_DIALECT_TF, "unknown dialect");
  EVT_CHECK_ARG(s->hidden > 0 && s->hidden % 8 == 0, "hidden size must be a positive multiple of 8");
  EVT_CHECK_ARG(s->layers > 0 && s->layers <= EVT_MAX_LAYERS, "layer count out of range");
  EVT_CHECK_ARG(s->patch > 0 && s->image > 0 && s->image % s->patch == 0, "image size must be a multiple of the patch size");
  EVT_CHECK_ARG(s->patch % 8 == 0 || s->patch == 14, "patch size must be a multiple of 8, or 14");
  const int patches = (s->image / s->patch) * (s->image / s->patch);
  EVT_CHECK_ARG(s->tokens == patches + 1 || s->tokens == patches + 2, "tokens must be patches + 1 (cls) or + 2 (cls, distillation)");
  if (s->tokens > EVT_ATTN_MAX_TOKENS)
    return fail(EVT_ERR_UNSUPPORTED, "more than " + std::to_string(EVT_ATTN_MAX_TOKENS) + " tokens per image is not implemented");
  if (s->tokens > 256 && s->precision == EVT_PREC_TF32)  // its attention keeps every key of a head on chip
    return fail(EVT_ERR_UNSUPPORTED, "the tf32 mode supports at most 256 tokens per image; use the bf16 mode");
  if (s->head_size != 64 && s->head_size != 80) return fail(EVT_ERR_UNSUPPORTED, "only head sizes 64 and 80 are implemented");
  if (s->head_size == 80 && s->precision != EVT_PREC_BF16)
    return fail(EVT_ERR_UNSUPPORTED, "head size 80 is implemented in the bf16 mode only");
  EVT_CHECK_ARG(s->num_labels > 0, "num_labels must be positive");
  EVT_CHECK_ARG(s->act == EVT_ACT_GELU_ERF || s->act == EVT_ACT_GELU_TANH, "FFN activation must be erf- or tanh-GELU");
  EVT_CHECK_ARG(s->eps > 0.f, "LayerNorm eps must be positive");
  EVT_CHECK_ARG(s->head_hidden >= 0, "head_hidden must be >= 0");
  EVT_CHECK_ARG(s->head_rows >= 0 && s->head_rows <= 2, "head_rows must be 0 / 1 (cls row) or 2 (cls + distillation rows)");
  if (s->head_rows == 2)
    EVT_CHECK_ARG(s->tokens == patches + 2 && s->final_ln != 0 && s->head_hidden == 0,
                  "head_rows = 2 (two-head distilled DeiT) needs 198 tokens, the final LayerNorm and a single Linear head");
  EVT_CHECK_ARG(s->precision == EVT_PREC_BF16 || s->precision == EVT_PREC_TF32, "precision must be bf16 (0) or tf32 (1)");
  EVT_CHECK_ARG(s->final_ln >= 0 && s->final_ln <= 2, "final_ln must be 0 (none), 1 (LayerNorm, classifier on the cls row) or 2 (LayerNorm "
                                                      "of the mean of the patch rows)");
  if (s->final_ln == 2) {
    if (s->precision != EVT_PREC_BF16) return fail(EVT_ERR_UNSUPPORTED, "final_ln = 2 (mean-pooled head) is implemented in the bf16 mode only");
    EVT_CHECK_ARG(s->tokens == patches + 1 && s->head_rows <= 1, "final_ln = 2 (mean-pooled head) needs tokens = patches + 1 and head_rows 0 or 1");
    if (s->hidden % 4 != 0 || s->hidden > 1024)
      return fail(EVT_ERR_UNSUPPORTED, "final_ln = 2 (mean-pooled head) is implemented for hidden sizes that are multiples of 4 up to 1024");
  }
  EVT_CHECK_ARG(s->embed_k >= 0 && s->embed_k % 8 == 0, "embed_k must be a non-negative multiple of 8");
  EVT_CHECK_ARG(s->t2t >= 0 && s->t2t <= 3, "t2t must be 0 (patch embedding), 1 (T2T front-end, NHWC f32 pixels), 2 (T2T front-end, "
                                            "NCHW pixels) or 3 (T2T front-end with token transformers, NCHW pixels)");
  if (s->t2t) {
    EVT_CHECK_ARG(s->embed_k == 576 && s->precision == EVT_PREC_BF16, "the T2T front-end needs embed_k = 576 (3 x 3 x 64) and the bf16 mode");
    EVT_CHECK_ARG(t2t_side(s->image, 2) * t2t_side(s->image, 2) == patches, "image size does not give image/16 squared T2T tokens");
  }
  for (int l = 0; l < s->layers; ++l) {
    EVT_CHECK_ARG(s->heads[l] > 0, "every layer must keep at least one head");
    EVT_CHECK_ARG(s->inter[l] > 0, "every layer must keep at least one FFN unit");
  }
  return EVT_OK;
}

}  // namespace

int Loader::index(const evt_tensor_view* tensors, int n) {
  for (int i = 0; i < n; ++i) {
    EVT_CHECK_ARG(tensors[i].name != nullptr, "tensor view without a name");
    EVT_CHECK_ARG(tensors[i].ndim >= 1 && tensors[i].ndim <= 4, "tensor view rank must be 1..4");
    by_name[tensors[i].name] = &tensors[i];
  }
  return EVT_OK;
}

const evt_tensor_view* Loader::find(const std::string& name) const {
  auto it = by_name.find(name);
  return it == by_name.end() ? nullptr : it->second;
}

int Loader::need(const std::string& name, int64_t n, const evt_tensor_view** out) const {
  const evt_tensor_view* v = find(name);
  if (!v) return fail(EVT_ERR_INVALID, "missing weight '" + name + "'");
  if (!v->data) return fail(EVT_ERR_INVALID, "weight '" + name + "' has a null data pointer");
  int64_t numel = 1;
  for (int i = 0; i < v->ndim; ++i) numel *= v->shape[i];
  if (numel != n)
    return fail(EVT_ERR_INVALID, "weight '" + name + "' has " + std::to_string(numel) + " elements, expected " + std::to_string(n));
  *out = v;
  return EVT_OK;
}

int Loader::alloc(size_t bytes, void** out) {
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, std::max<size_t>(bytes, 16));
  if (e != cudaSuccess) return fail(EVT_ERR_CUDA, std::string("cudaMalloc: ") + cudaGetErrorString(e));
  allocs->push_back(p);
  *out = p;
  return EVT_OK;
}

int Loader::vec_into(const std::string& name, int64_t n, bool optional, float* dst) {
  const evt_tensor_view* v = find(name);
  if (!v && optional) {
    EVT_CUDA(cudaMemsetAsync(dst, 0, n * 4, st));
  } else {
    EVT_TRY(need(name, n, &v));
    EVT_CUDA(cudaMemcpyAsync(dst, v->data, n * 4, cudaMemcpyDeviceToDevice, st));
  }
  return EVT_OK;
}

int Loader::vec(const std::string& name, int64_t n, bool optional, float** out) {
  void* p;
  EVT_TRY(alloc(n * 4, &p));
  *out = static_cast<float*>(p);
  return vec_into(name, n, optional, *out);
}

int Loader::mat_into(const std::string& name, int64_t rows, int cols, int ld, void* dst) {
  const evt_tensor_view* v;
  EVT_TRY(need(name, rows * cols, &v));
  const long long total = rows * ld;
  const unsigned grid = static_cast<unsigned>((total + 255) / 256);
  const float* src = static_cast<const float*>(v->data);
  if (es == 2) convert_pad_kernel<<<grid, 256, 0, st>>>(src, static_cast<__nv_bfloat16*>(dst), rows, cols, ld);
  else convert_pad_kernel<<<grid, 256, 0, st>>>(src, static_cast<float*>(dst), rows, cols, ld);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(EVT_ERR_CUDA, std::string("convert_pad: ") + cudaGetErrorString(e));
  return EVT_OK;
}

int Loader::mat_t(const std::string& name, int rows_out, int cols_out, int ld, __nv_bfloat16** out) {
  const evt_tensor_view* v;
  EVT_TRY(need(name, static_cast<int64_t>(rows_out) * cols_out, &v));
  void* p;
  EVT_TRY(alloc(static_cast<size_t>(rows_out) * ld * 2, &p));
  *out = static_cast<__nv_bfloat16*>(p);
  const long long total = static_cast<long long>(rows_out) * ld;
  convert_pad_transposed_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, st>>>(static_cast<const float*>(v->data), *out,
                                                                                             rows_out, cols_out, ld);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(EVT_ERR_CUDA, std::string("convert_pad_transposed: ") + cudaGetErrorString(e));
  return EVT_OK;
}

int Loader::host_copy(const std::string& name, int64_t n, std::vector<float>* out) {
  const evt_tensor_view* v;
  EVT_TRY(need(name, n, &v));
  out->resize(n);
  EVT_CUDA(cudaMemcpyAsync(out->data(), v->data, n * 4, cudaMemcpyDeviceToHost, st));
  EVT_CUDA(cudaStreamSynchronize(st));
  return EVT_OK;
}

}  // namespace evt

using namespace evt;

extern "C" int evt_model_create(const evt_model_spec* spec, evt_model** out) {
  int rc = evt_device_check();
  if (rc != EVT_OK) return rc;
  EVT_CHECK_ARG(out != nullptr, "evt_model_create: out is null");
  rc = validate_spec(spec);
  if (rc != EVT_OK) return rc;
  evt_model* m = new evt_model();
  m->spec = *spec;
  cudaGetDevice(&m->device);
  m->patches = (spec->image / spec->patch) * (spec->image / spec->patch);
  m->n_prefix = spec->tokens - m->patches;
  m->patch_k = spec->embed_k > 0 ? spec->embed_k : patch_k(spec->patch);  // P = 14: 588 columns + 4 zero ones
  m->es = spec->precision == EVT_PREC_TF32 ? 4 : 2;
  m->pad = 16 / m->es;
  m->layers.resize(spec->layers);
  *out = m;
  return EVT_OK;
}

extern "C" int evt_model_destroy(evt_model* m) {
  if (!m) return EVT_OK;
  for (void* p : m->allocs) cudaFree(p);
  for (cudaEvent_t ev : m->prof_events) cudaEventDestroy(ev);
  delete m;
  return EVT_OK;
}

extern "C" int evt_model_load_weights(evt_model* m, const evt_tensor_view* tensors, int n, evt_stream stream) {
  EVT_CHECK_ARG(m != nullptr && tensors != nullptr && n > 0, "evt_model_load_weights: bad arguments");
  if (m->loaded) return fail(EVT_ERR_STATE, "weights already loaded; create a new model to reload");
  const evt_model_spec& s = m->spec;
  Loader L{&m->allocs, static_cast<cudaStream_t>(stream), m->es};
  EVT_TRY(L.index(tensors, n));
  const int D = s.hidden;
  const std::string e = "vit.embeddings.";
  EVT_TRY(L.mat(e + "patch_embeddings.projection.weight", D, s.embed_k > 0 ? m->patch_k : 3 * s.patch * s.patch, m->patch_k, &m->w_patch));
  EVT_TRY(L.vec(e + "patch_embeddings.projection.bias", D, false, &m->b_patch));
  EVT_TRY(L.vec(e + "position_embeddings", static_cast<int64_t>(s.tokens) * D, false, &m->pos));
  {
    void* p;
    EVT_TRY(L.alloc(static_cast<size_t>(m->n_prefix) * D * 4, &p));
    m->prefix = reinterpret_cast<float*>(p);
    EVT_TRY(L.vec_into(e + "cls_token", D, false, m->prefix));
    if (m->n_prefix == 2) EVT_TRY(L.vec_into(e + "distillation_token", D, false, m->prefix + D));
  }
  for (int l = 0; l < s.layers; ++l) {
    LayerW& w = m->layers[l];
    const std::string p = "vit.encoder.layer." + std::to_string(l) + ".";
    w.a = s.heads[l] * s.head_size;
    w.inter = s.inter[l];
    w.inter_ld = padn(w.inter, m->pad);
    void* q;
    EVT_TRY(L.alloc(static_cast<size_t>(3) * w.a * D * m->es, &q));
    w.wqkv = reinterpret_cast<uint8_t*>(q);
    EVT_TRY(L.alloc(static_cast<size_t>(3) * w.a * 4, &q));
    w.bqkv = reinterpret_cast<float*>(q);
    const char* names[3] = {"query", "key", "value"};
    for (int t = 0; t < 3; ++t) {
      const std::string base = p + "attention.attention." + names[t];
      EVT_TRY(L.mat_into(base + ".weight", w.a, D, D, w.wqkv + static_cast<size_t>(t) * w.a * D * m->es));
      EVT_TRY(L.vec_into(base + ".bias", w.a, true, w.bqkv + t * w.a));
    }
    EVT_TRY(L.mat(p + "attention.output.dense.weight", D, w.a, w.a, &w.wo));
    EVT_TRY(L.vec(p + "attention.output.dense.bias", D, true, &w.bo));
    EVT_TRY(L.mat(p + "intermediate.dense.weight", w.inter, D, D, &w.w1));
    EVT_TRY(L.vec(p + "intermediate.dense.bias", w.inter, true, &w.b1));
    EVT_TRY(L.mat(p + "output.dense.weight", D, w.inter, w.inter_ld, &w.w2));
    EVT_TRY(L.vec(p + "output.dense.bias", D, true, &w.b2));
    EVT_TRY(L.vec(p + "layernorm_before.weight", D, false, &w.ln1_g));
    EVT_TRY(L.vec(p + "layernorm_before.bias", D, false, &w.ln1_b));
    EVT_TRY(L.vec(p + "layernorm_after.weight", D, false, &w.ln2_g));
    EVT_TRY(L.vec(p + "layernorm_after.bias", D, false, &w.ln2_b));
  }
  if (s.t2t == 3) {  // Token_transformer (INTEGRATION.md §3), Dense kernels [in, out]; norm1 / qkv rows in (kh, kw, c) order
    for (int i = 0; i < 2; ++i) {
      PerformerW& pw = m->perf[i];
      const std::string p = "t2t.transformer" + std::to_string(i + 1) + ".";
      pw.in_dim = i == 0 ? 7 * 7 * 3 : 3 * 3 * 64;
      pw.in_ld = padn(pw.in_dim, 8);
      EVT_TRY(L.vec(p + "norm1.gamma", pw.in_dim, false, &pw.g1));
      EVT_TRY(L.vec(p + "norm1.beta", pw.in_dim, false, &pw.b1));
      EVT_TRY(L.mat_t(p + "qkv.kernel", 192, pw.in_dim, pw.in_ld, &pw.wkqv));
      EVT_TRY(L.mat_t(p + "attn_output.kernel", 64, 64, 64, &pw.wo));
      EVT_TRY(L.vec(p + "attn_output.bias", 64, true, &pw.bo));
      EVT_TRY(L.vec(p + "norm2.gamma", 64, false, &pw.g2));
      EVT_TRY(L.vec(p + "norm2.beta", 64, false, &pw.b2));
      EVT_TRY(L.mat_t(p + "mlp.fc1.kernel", 64, 64, 64, &pw.w1));
      EVT_TRY(L.vec(p + "mlp.fc1.bias", 64, true, &pw.bb1));
      EVT_TRY(L.mat_t(p + "mlp.fc2.kernel", 64, 64, 64, &pw.w2));
      EVT_TRY(L.vec(p + "mlp.fc2.bias", 64, true, &pw.bb2));
    }
  } else if (s.t2t) {  // Keras variable names of T2T_module (modeling/models/t2t_vit.py:47-59), Dense kernels [in, out]
    for (int i = 0; i < 2; ++i) {
      PerformerW& pw = m->perf[i];
      const std::string p = "t2t.performer" + std::to_string(i + 1) + ".";
      pw.in_dim = i == 0 ? 7 * 7 * 3 : 3 * 3 * 64;
      pw.in_ld = padn(pw.in_dim, 8);
      EVT_TRY(L.vec(p + "norm1.gamma", pw.in_dim, false, &pw.g1));
      EVT_TRY(L.vec(p + "norm1.beta", pw.in_dim, false, &pw.b1));
      EVT_TRY(L.mat_t(p + "kqv.kernel", 192, pw.in_dim, pw.in_ld, &pw.wkqv));
      EVT_TRY(L.vec(p + "kqv.bias", 192, true, &pw.bkqv));
      EVT_TRY(L.vec(p + "w", 32 * 64, false, &pw.w));
      EVT_TRY(L.mat_t(p + "attn_output.kernel", 64, 64, 64, &pw.wo));
      EVT_TRY(L.vec(p + "attn_output.bias", 64, true, &pw.bo));
      EVT_TRY(L.vec(p + "norm2.gamma", 64, false, &pw.g2));
      EVT_TRY(L.vec(p + "norm2.beta", 64, false, &pw.b2));
      EVT_TRY(L.mat_t(p + "mlp.fc1.kernel", 64, 64, 64, &pw.w1));
      EVT_TRY(L.vec(p + "mlp.fc1.bias", 64, true, &pw.bb1));
      EVT_TRY(L.mat_t(p + "mlp.fc2.kernel", 64, 64, 64, &pw.w2));
      EVT_TRY(L.vec(p + "mlp.fc2.bias", 64, true, &pw.bb2));
    }
  }
  // BEiT relative position bias: per layer [(2W-1)^2 + 3, heads] in the HF layout, repacked to [heads, n] times log2(e) (the
  // attention kernels' softmax runs in log2 units)
  auto tab_name = [](int l) {
    return "vit.encoder.layer." + std::to_string(l) + ".attention.attention.relative_position_bias.relative_position_bias_table";
  };
  if (L.find(tab_name(0)) != nullptr) {
    const int W = s.image / s.patch, n = (2 * W - 1) * (2 * W - 1) + 3;
    if (s.precision != EVT_PREC_BF16) return fail(EVT_ERR_UNSUPPORTED, "the relative position bias (BEiT) is implemented in the bf16 mode only");
    if (s.tokens != W * W + 1)
      return fail(EVT_ERR_UNSUPPORTED, "the relative position bias (BEiT) needs tokens = patches + 1 (no distillation token)");
    if (s.head_size != 64) return fail(EVT_ERR_UNSUPPORTED, "the relative position bias (BEiT) is implemented for head size 64 only");
    for (int l = 0; l < s.layers; ++l) {
      const int h = s.heads[l];
      std::vector<float> t;
      EVT_TRY(L.host_copy(tab_name(l), static_cast<int64_t>(n) * h, &t));
      std::vector<float> r(t.size());
      for (int i = 0; i < n; ++i)
        for (int j = 0; j < h; ++j) r[static_cast<size_t>(j) * n + i] = static_cast<float>(static_cast<double>(t[static_cast<size_t>(i) * h + j]) * 1.4426950408889634);
      EVT_TRY(L.upload(r, &m->layers[l].rel_tab));
    }
    m->rel_grid = W;
  } else {
    for (int l = 1; l < s.layers; ++l)
      if (L.find(tab_name(l)) != nullptr)
        return fail(EVT_ERR_INVALID, "relative position bias tables must be given for every layer or for none (layer 0 has none, layer " +
                                         std::to_string(l) + " has one)");
  }
  if (s.final_ln) {
    EVT_TRY(L.vec("vit.layernorm.weight", D, false, &m->lnf_g));
    EVT_TRY(L.vec("vit.layernorm.bias", D, false, &m->lnf_b));
  }
  int cls_in = D * (s.head_rows > 1 ? s.head_rows : 1);
  if (s.head_hidden > 0) {
    EVT_TRY(L.mat("pre_classifier.weight", s.head_hidden, D, D, &m->w_pre));
    EVT_TRY(L.vec("pre_classifier.bias", s.head_hidden, true, &m->b_pre));
    cls_in = s.head_hidden;
  }
  EVT_TRY(L.mat("classifier.weight", s.num_labels, cls_in, padn(cls_in, m->pad), &m->w_cls));
  EVT_TRY(L.vec("classifier.bias", s.num_labels, true, &m->b_cls));
  EVT_CUDA(cudaStreamSynchronize(L.st));
  m->loaded = true;
  return EVT_OK;
}

extern "C" int evt_model_workspace_bytes(const evt_model* m, int batch, size_t* out) {
  EVT_CHECK_ARG(m != nullptr && out != nullptr, "evt_model_workspace_bytes: null argument");
  EVT_CHECK_ARG(batch > 0, "batch must be positive");
  *out = plan_workspace(m, batch, nullptr).bytes + 1024;  // slack to align the caller's pointer
  return EVT_OK;
}

extern "C" int evt_model_launches_per_forward(const evt_model* m) {
  if (!m) return 0;
  const evt_model_spec& s = m->spec;
  // T2T front-end: per performer unfold+LN, kqv, 3 performer kernels (the last one carries attn_output + MLP); per token
  // transformer (t2t = 3) unfold+LN, qkv, attention, tail; then the last soft split
  return (s.t2t == 3 ? 2 * 4 + 1 : s.t2t ? 2 * 5 + 1 : 0) + (s.embed_k > 0 ? 2 : 3) + 7 * s.layers + (s.final_ln && s.head_rows > 1 ? s.head_rows : 1) + (s.head_hidden > 0 ? 2 : 1);
}

static int forward_impl(evt_model* m, const void* pixels, const evt_forward_opts* opts, const void* patch_matrix, int64_t patch_ld,
                        int batch, float* logits, void* workspace, size_t workspace_bytes, evt_stream stream) {
  EVT_CHECK_ARG(m != nullptr, "evt_model_forward: model is null");
  if (!m->loaded) return fail(EVT_ERR_STATE, "evt_model_forward called before evt_model_load_weights");
  EVT_CHECK_ARG((pixels || patch_matrix) && logits && workspace, "evt_model_forward: null pointer");
  EVT_CHECK_ARG(batch > 0 && batch <= 65535, "batch must be in 1..65535");
  const evt_model_spec& s = m->spec;
  static const evt_forward_opts kNoOpts = {};
  const evt_forward_opts& o = opts != nullptr ? *opts : kNoOpts;
  EVT_CHECK_ARG(o.head_mask == nullptr || o.head_mask_ld > 0, "head_mask_ld must be positive when a head mask is given");
  Workspace w;
  EVT_TRY(place_workspace(workspace, workspace_bytes, [&](uint8_t* base) { return plan_workspace(m, batch, base); }, &w,
                          "workspace too small for this batch (see evt_model_workspace_bytes)"));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  StaticWeightsScope weights_are_static;  // every GEMM below multiplies by a weight matrix this model owns
  const int D = s.hidden;
  const int64_t M = static_cast<int64_t>(batch) * s.tokens;
  const int64_t Mp = static_cast<int64_t>(batch) * m->patches;
  const bool tf = s.dialect == EVT_DIALECT_TF;
  const float scale = 1.0f / sqrtf(static_cast<float>(s.head_size));
  // profiling tap: events on the launching stream between launches (no effect on the launches themselves)
  auto mark = [&](int stage) -> int {
    if (!m->profiling) return EVT_OK;
    if (m->prof_used == m->prof_events.size()) {
      cudaEvent_t ev;
      EVT_CUDA(cudaEventCreate(&ev));
      m->prof_events.push_back(ev);
    }
    EVT_CUDA(cudaEventRecord(m->prof_events[m->prof_used], st));
    if (stage >= 0) m->prof_spans.push_back({stage, {m->prof_used - 1, m->prof_used}});
    ++m->prof_used;
    return EVT_OK;
  };
#define EVT_STAGE(stage, expr) \
  do {                         \
    EVT_TRY(expr);             \
    EVT_TRY(mark(stage));      \
  } while (0)
  EVT_TRY(mark(-1));
  const bool tf32 = s.precision == EVT_PREC_TF32;
  const int dt = tf32 ? EVT_F32 : EVT_BF16;   // GEMM operand type
  const int adt = tf32 ? EVT_TF32 : EVT_BF16;  // type activations are WRITTEN in (tf32: f32 storage, rounded to nearest)
  // tokens-to-token front-end (T2T_module.call, modeling/models/t2t_vit.py:63-88).  spec.t2t = 1: NHWC f32 pixels (the TF T2T);
  // 2: NCHW pixels of any evt_pixel_dtype (the PyTorch T2T: nn.Unfold over the image, whose stage-1 columns the first kernel writes
  // in the same (kh, kw, c) order -- the loader permuted the weights).  Stages 2 and 3 read the token-major [B, T, 64] performer
  // output either way.  The performer MLP's GELU is spec.act (tanh for the TF T2T, erf for the PyTorch one).  spec.t2t = 3: the
  // PyTorch T2T with Token_transformers (tokens_type='transformer') -- the same soft splits; per stage the bias-free qkv GEMM, exact
  // single-head softmax attention over all T = 3136 / 784 tokens of an image, with Attention.scale = in_dim ** -0.5 (147 / 576)
  // passed to the kernel, and the tail y = v + proj(ctx); y += mlp(norm2(y)) with erf-GELU (nn.GELU).
  if (s.t2t && patch_matrix == nullptr) {
    const float tf_eps = 1e-5f;   // tf.keras.layers.LayerNormalization(epsilon=1e-5), transformer_encoder.py:49-50; nn.LayerNorm's default
    const void* src = pixels;
    int src_dt = EVT_F32, side = s.image, ch = 3;
    const bool nchw = s.t2t >= 2;
    EVT_CHECK_ARG(nchw || o.pixel_dtype == EVT_PIX_F32, "the T2T front-end with spec.t2t = 1 takes f32 NHWC pixels");
    for (int i = 0; i < 2; ++i) {
      const PerformerW& pw = m->perf[i];
      const int k = i == 0 ? 7 : 3, st_ = i == 0 ? 4 : 2, pad_ = i == 0 ? 2 : 1;
      const int so = t2t_side(s.image, i), T = so * so;
      const int64_t rows = static_cast<int64_t>(batch) * T;
      if (i == 0 && nchw)
        EVT_STAGE(EVT_STAGE_EMBED, unfold773_nchw_launch(pixels, o.pixel_dtype, o.pixel_scale, o.pixel_bias, w.t_x[0], pw.g1, pw.b1, tf_eps,
                                                         batch, s.image, s.image, st));
      else
        EVT_STAGE(EVT_STAGE_EMBED, unfold_ln_launch(src, src_dt, w.t_x[i], pw.in_ld, pw.g1, pw.b1, tf_eps, batch, side, side, ch, k, st_, pad_, st));
      EVT_STAGE(EVT_STAGE_EMBED, gemm_launch({.A = w.t_x[i], .lda = pw.in_ld, .W = pw.wkqv, .ldw = pw.in_ld, .bias = pw.bkqv, .out = w.t_kqv[i],
                                              .out_dtype = EVT_BF16, .ldo = 192, .M = rows, .N = 192, .K = pw.in_dim}, st));
      if (s.t2t == 3) {
        EVT_TRY(token_transformer_block_launch(w.t_kqv[i], 192, w.t_y[i], w.t_ws[i], batch, T, 1.0f / sqrtf(static_cast<float>(pw.in_dim)),
                                               pw.wo, pw.bo, pw.g2, pw.b2, pw.w1, pw.bb1, pw.w2, pw.bb2, tf_eps, st));
        EVT_TRY(mark(EVT_STAGE_EMBED));
        src = w.t_y[i], src_dt = EVT_F32, side = so, ch = 64;
        continue;
      }
      // single_attn + attn_output + LayerNorm + MLP (transformer_encoder.py:67-99): the attention contraction's apply kernel carries
      // each tile through the tail, y = the performer's output rows
      EVT_TRY(performer_block_launch(w.t_kqv[i], 192, pw.w, w.t_y[i], w.t_ws[i], batch, T, 1e-8f, pw.wo, pw.bo, pw.g2, pw.b2, pw.w1,
                                     pw.bb1, pw.w2, pw.bb2, tf_eps, st, s.act));
      EVT_TRY(mark(EVT_STAGE_EMBED));
      src = w.t_y[i], src_dt = EVT_F32, side = so, ch = 64;
    }
    EVT_STAGE(EVT_STAGE_EMBED, unfold_ln_launch(src, src_dt, w.t_pm, 576, nullptr, nullptr, tf_eps, batch, side, side, 64, 3, 2, 1, st));
    patch_matrix = w.t_pm;
    patch_ld = 576;
  }
  // embeddings
  if (patch_matrix == nullptr) {
    // Pixels path: the patch matrix gets one row per token (prefix rows zero), so the embedding GEMM is a plain
    // M = batch * tokens problem whose output rows ARE the residual rows -> CTA-pair kernel + TMA reduce-add epilogue.
    // The residual stream is first filled with pos + (cls | conv bias); the GEMM then adds the patch projections.
    // (Before: remapped output rows forced the generic epilogue -- 1.0 ms of a 41 ms forward at batch 1024, now 0.4.)
    EVT_CHECK_ARG(s.embed_k == 0, "this model takes a caller-built patch matrix (evt_model_forward_embedded)");
    const size_t row_bytes = static_cast<size_t>(m->patch_k) * m->es;
    EVT_CUDA(cudaMemset2DAsync(w.big, s.tokens * row_bytes, 0, m->n_prefix * row_bytes, batch, st));
    EVT_STAGE(EVT_STAGE_EMBED, im2col_launch(pixels, o.pixel_dtype, o.pixel_scale, o.pixel_bias, w.big, dt, batch, s.image, s.image, s.patch, st,
                                             s.tokens, m->n_prefix));
    EVT_STAGE(EVT_STAGE_EMBED, embed_fill_launch(m->prefix, m->pos, m->b_patch, w.resid, batch, s.tokens, m->n_prefix, D, st));
    EVT_STAGE(EVT_STAGE_EMBED, gemm_launch({.A = w.big, .lda = m->patch_k, .W = m->w_patch, .ldw = m->patch_k, .in_dtype = dt, .residual = w.resid,
                                            .ldr = D, .out = w.resid, .out_dtype = EVT_F32, .ldo = D, .M = M, .N = D, .K = m->patch_k}, st));
  } else {
    EVT_CHECK_ARG(patch_ld >= m->patch_k, "patch matrix leading dimension smaller than the embedding K");
    // patch row p of image b: output row b * tokens + n_prefix + p, position-embedding row n_prefix + p
    EVT_STAGE(EVT_STAGE_EMBED,
              gemm_launch({.A = patch_matrix, .lda = patch_ld, .W = m->w_patch, .ldw = m->patch_k, .in_dtype = dt, .bias = m->b_patch,
                           .residual = m->pos, .ldr = D, .out = w.resid, .out_dtype = EVT_F32, .ldo = D, .M = Mp, .N = D, .K = m->patch_k,
                           .map = {.res_row_mod = m->patches, .res_row_off = m->n_prefix, .out_group = m->patches,
                                   .out_group_stride = s.tokens, .out_group_off = m->n_prefix}}, st));
    EVT_STAGE(EVT_STAGE_EMBED, prefix_tokens_launch(m->prefix, m->pos, w.resid, batch, s.tokens, m->n_prefix, D, st));
  }
  // encoder.  Narrow residual streams at large batch (D = 192 / 384: DeiT-Tiny / -Small, T2T): whole rows of a 256-row block
  // fit in tensor memory, so the LayerNorm that FOLLOWS each residual projection runs in that projection's epilogue
  // (gemm_rowln.cu): 5 launches per layer instead of 7 and the LayerNorm kernel's read of the f32 residual stream never happens.
  const bool row_ln = !tf32 && gemm_rowln_supported(M, D, D, tf);  // per projection: gemm_rowln_pays
  // Classification-row tail: the head reads only row 0 of every image, and after the K / V of the last layer everything
  // in that layer is row-wise, so its attention runs for the cls query alone (all keys), and the out-projection, LN2,
  // FC1 and FC2 run on `batch` rows: row i is image i's cls row (residual stream stride tokens * D, context and FC1
  // output packed).  Same launches, same kernels, so the cls row gets the same bits as in a full layer.  Full layer
  // instead when a caller asks for the last layer's context of every row (ctx_out), in the tf32 mode (its attention
  // kernel has no query-row count), for the two-head distilled DeiT (rows 0 and 1 of every image are not one strided
  // row set) and for the mean-pooled head (final_ln = 2: it reads every patch row).
  const int64_t tok_stride = static_cast<int64_t>(s.tokens) * D;
  const bool cls_tail = !tf32 && s.head_rows <= 1 && s.final_ln != 2 && !(o.ctx_out != nullptr && o.ctx_out[s.layers - 1] != nullptr);
  bool xn_ready = false;  // w.xn already holds LN1 of the current layer (written by the previous layer's FC2 epilogue)
  for (int l = 0; l < s.layers; ++l) {
    const LayerW& lw = m->layers[l];
    const int a = lw.a;
    const bool tail = cls_tail && l == s.layers - 1;
    const int64_t rows = tail ? batch : M;        // rows after attention
    const int64_t rs = tail ? tok_stride : D;     // their stride in the residual stream
    // A residual GEMM of the tail splits K only where the full-size one would: no unordered reduce-adds are added to a
    // forward whose full-size launches have a fixed summation order.
    auto on_rows = [&](GemmOp op) {
      if (!tail) return op;
      op.max_k_splits = gemm_k_splits(op) > 1 ? 0 : 1;
      op.M = rows;
      op.ldr = op.ldo = rs;
      return op;
    };
    if (!xn_ready)
      EVT_STAGE(EVT_STAGE_LN, layernorm_launch(w.resid, D, lw.ln1_g, lw.ln1_b, w.xn, adt, D, tf ? w.resid : nullptr, M, D, s.eps, st));
    EVT_STAGE(EVT_STAGE_QKV, gemm_launch({.A = w.xn, .lda = D, .W = lw.wqkv, .ldw = D, .in_dtype = dt, .bias = lw.bqkv, .out = w.qkv,
                                          .out_dtype = adt, .ldo = 3 * a, .M = M, .N = 3 * a, .K = D}, st));
    xn_ready = false;
    // head mask row of this layer (are_16_heads mask_heads) and, on request, the context written straight into the caller's
    // buffer (context_layer_val): the output projection then reads its A operand from there
    const float* hmask = o.head_mask != nullptr ? o.head_mask + static_cast<size_t>(l) * o.head_mask_ld : nullptr;
    EVT_CHECK_ARG(hmask == nullptr || o.head_mask_ld >= s.heads[l], "head_mask_ld smaller than a layer's head count");
    uint8_t* ctx = (o.ctx_out != nullptr && o.ctx_out[l] != nullptr) ? reinterpret_cast<uint8_t*>(o.ctx_out[l]) : w.ctx;
    EVT_CHECK_ARG(reinterpret_cast<uintptr_t>(ctx) % 16 == 0, "ctx_out pointers must be 16-byte aligned");
    if (tf32)
      EVT_STAGE(EVT_STAGE_ATTN, attention_tf32_launch(reinterpret_cast<const float*>(w.qkv), 3 * a, reinterpret_cast<float*>(ctx), a, hmask,
                                    batch, s.tokens, s.heads[l], s.head_size, scale, st));
    else if (lw.rel_tab != nullptr)
      EVT_STAGE(EVT_STAGE_ATTN, attention_rel_bias_launch(w.qkv, 3 * a, ctx, a, hmask, lw.rel_tab, m->rel_grid, batch, s.tokens,
                                                          tail ? 1 : s.tokens, s.heads[l], s.head_size, scale, st));
    else
      EVT_STAGE(EVT_STAGE_ATTN, attention_launch(w.qkv, 3 * a, ctx, a, hmask, batch, s.tokens, tail ? 1 : s.tokens, s.heads[l], s.head_size,
                                                 scale, st));
    if (!tail && row_ln && gemm_rowln_pays(D, a, tf)) {
      EVT_STAGE(EVT_STAGE_OPROJ, gemm_rowln_launch(ctx, a, lw.wo, a, lw.bo, w.resid, D, lw.ln2_g, lw.ln2_b, s.eps, tf, w.xn, D, M, D, a, st));
    } else {
      EVT_STAGE(EVT_STAGE_OPROJ, gemm_launch(on_rows({.A = ctx, .lda = a, .W = lw.wo, .ldw = a, .in_dtype = dt, .bias = lw.bo, .residual = w.resid,
                                                      .ldr = D, .out = w.resid, .out_dtype = EVT_F32, .ldo = D, .M = M, .N = D, .K = a}), st));
      EVT_STAGE(EVT_STAGE_LN, layernorm_launch(w.resid, rs, lw.ln2_g, lw.ln2_b, w.xn, adt, D, tf ? w.resid : nullptr, rows, D, s.eps, st));
    }
    EVT_STAGE(EVT_STAGE_FC1, gemm_launch({.A = w.xn, .lda = D, .W = lw.w1, .ldw = D, .in_dtype = dt, .bias = lw.b1, .out = w.big,
                                          .out_dtype = adt, .ldo = lw.inter_ld, .M = rows, .N = lw.inter, .K = D, .act = s.act}, st));
    if (row_ln && l + 1 < s.layers && gemm_rowln_pays(D, lw.inter, tf)) {
      const LayerW& nx = m->layers[l + 1];
      EVT_STAGE(EVT_STAGE_FC2, gemm_rowln_launch(w.big, lw.inter_ld, lw.w2, lw.inter_ld, lw.b2, w.resid, D, nx.ln1_g, nx.ln1_b, s.eps, tf, w.xn,
                                                 D, M, D, lw.inter, st));
      xn_ready = true;
    } else {
      EVT_STAGE(EVT_STAGE_FC2, gemm_launch(on_rows({.A = w.big, .lda = lw.inter_ld, .W = lw.w2, .ldw = lw.inter_ld, .in_dtype = dt, .bias = lw.b2,
                                                    .residual = w.resid, .ldr = D, .out = w.resid, .out_dtype = EVT_F32, .ldo = D, .M = M, .N = D,
                                                    .K = lw.inter}), st));
    }
  }
  // head: only the cls row of every image is consumed (SITE/models/vit/modeling_vit.py:641)
  const int head_rows = s.head_rows > 1 ? s.head_rows : 1;
  if (s.final_ln == 2) {  // BeitPooler with use_mean_pooling: LayerNorm of the mean of the patch rows
    EVT_STAGE(EVT_STAGE_HEAD, layernorm_patch_mean_launch(w.resid, m->lnf_g, m->lnf_b, w.clsn, batch, s.tokens, D, s.eps, st));
  } else if (s.final_ln) {
    // head_rows = 2 (DeiTForImageClassificationWithTeacher, SITE/models/deit/modeling_deit.py: logits = (cls_classifier(x[:, 0]) +
    // distillation_classifier(x[:, 1])) / 2): rows 0 and 1 of every image are normalised side by side into one 2D-wide row, and
    // ONE classifier GEMM with K = 2D over [W_cls | W_dist] / 2 produces the averaged logits.
    for (int r = 0; r < head_rows; ++r)
      EVT_STAGE(EVT_STAGE_HEAD, layernorm_launch(w.resid + static_cast<size_t>(r) * D, tok_stride, m->lnf_g, m->lnf_b,
                                                 w.clsn + static_cast<size_t>(r) * D * m->es, adt, static_cast<int64_t>(head_rows) * D, nullptr,
                                                 batch, D, s.eps, st));
  } else {
    const long long total = static_cast<long long>(batch) * D;
    const unsigned grid = static_cast<unsigned>((total + 255) / 256);
    const long long nrows = batch;
    if (tf32)
      EVT_CUDA(launch_pdl(gather_rows_cast_kernel<float>, dim3(grid), dim3(256), 0, st, pdl_for_rows(M), static_cast<const float*>(w.resid), tok_stride,
                          reinterpret_cast<float*>(w.clsn), nrows, D));
    else
      EVT_CUDA(launch_pdl(gather_rows_cast_kernel<__nv_bfloat16>, dim3(grid), dim3(256), 0, st, pdl_for_rows(M), static_cast<const float*>(w.resid),
                          tok_stride, reinterpret_cast<__nv_bfloat16*>(w.clsn), nrows, D));
    EVT_LAUNCH_CHECK("gather_rows_cast");
    EVT_TRY(mark(EVT_STAGE_HEAD));
  }
  if (s.head_hidden > 0) {
    const int hl = padn(s.head_hidden, m->pad);
    EVT_STAGE(EVT_STAGE_HEAD, gemm_launch({.A = w.clsn, .lda = D, .W = m->w_pre, .ldw = D, .in_dtype = dt, .bias = m->b_pre, .out = w.hh,
                                           .out_dtype = adt, .ldo = hl, .M = batch, .N = s.head_hidden, .K = D, .act = EVT_ACT_GELU_TANH}, st));
    EVT_STAGE(EVT_STAGE_HEAD, gemm_launch({.A = w.hh, .lda = hl, .W = m->w_cls, .ldw = hl, .in_dtype = dt, .bias = m->b_cls, .out = logits,
                                           .out_dtype = EVT_F32, .ldo = s.num_labels, .M = batch, .N = s.num_labels, .K = s.head_hidden}, st));
  } else {
    const int kc = head_rows * D;
    EVT_STAGE(EVT_STAGE_HEAD, gemm_launch({.A = w.clsn, .lda = kc, .W = m->w_cls, .ldw = kc, .in_dtype = dt, .bias = m->b_cls, .out = logits,
                                           .out_dtype = EVT_F32, .ldo = s.num_labels, .M = batch, .N = s.num_labels, .K = kc}, st));
  }
#undef EVT_STAGE
  return EVT_OK;
}

extern "C" int evt_model_profile_begin(evt_model* m) {
  EVT_CHECK_ARG(m != nullptr, "evt_model_profile_begin: model is null");
  m->profiling = true;
  m->prof_used = 0;
  m->prof_spans.clear();
  return EVT_OK;
}

extern "C" int evt_model_profile_end(evt_model* m, float* stage_ms, int* stage_launches) {
  EVT_CHECK_ARG(m != nullptr && stage_ms != nullptr && stage_launches != nullptr, "evt_model_profile_end: null argument");
  if (!m->profiling) return fail(EVT_ERR_STATE, "evt_model_profile_end without evt_model_profile_begin");
  m->profiling = false;
  for (int i = 0; i < EVT_STAGE_COUNT; ++i) stage_ms[i] = 0.f, stage_launches[i] = 0;
  if (m->prof_used > 0) EVT_CUDA(cudaEventSynchronize(m->prof_events[m->prof_used - 1]));
  for (const auto& sp : m->prof_spans) {
    float ms = 0.f;
    EVT_CUDA(cudaEventElapsedTime(&ms, m->prof_events[sp.second.first], m->prof_events[sp.second.second]));
    stage_ms[sp.first] += ms;
    stage_launches[sp.first] += 1;
  }
  m->prof_spans.clear();
  m->prof_used = 0;
  return EVT_OK;
}

extern "C" int evt_model_forward(evt_model* m, const float* pixels, int batch, float* logits, void* workspace,
                                 size_t workspace_bytes, evt_stream stream) {
  EVT_CHECK_ARG(pixels != nullptr, "evt_model_forward: pixels is null");
  return forward_impl(m, pixels, nullptr, nullptr, 0, batch, logits, workspace, workspace_bytes, stream);
}

extern "C" int evt_model_forward_ex(evt_model* m, const void* pixels, const evt_forward_opts* opts, int batch, float* logits,
                                    void* workspace, size_t workspace_bytes, evt_stream stream) {
  EVT_CHECK_ARG(pixels != nullptr, "evt_model_forward_ex: pixels is null");
  return forward_impl(m, pixels, opts, nullptr, 0, batch, logits, workspace, workspace_bytes, stream);
}

extern "C" int evt_model_forward_embedded(evt_model* m, const void* patch_matrix, int64_t ld, int batch, float* logits,
                                          void* workspace, size_t workspace_bytes, evt_stream stream) {
  EVT_CHECK_ARG(patch_matrix != nullptr, "evt_model_forward_embedded: patch_matrix is null");
  return forward_impl(m, nullptr, nullptr, patch_matrix, ld, batch, logits, workspace, workspace_bytes, stream);
}

extern "C" int evt_gemm_residual_layernorm_ex(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias, float* resid,
                                              int64_t ldr, const float* gamma, const float* beta, float eps, int copy_ln, void* xn,
                                              int64_t ldxn, int64_t M, int N, int K, evt_stream stream) {
  int rc = evt_device_check();
  if (rc != EVT_OK) return rc;
  EVT_CHECK_ARG(A != nullptr && W != nullptr && resid != nullptr && xn != nullptr && gamma != nullptr && beta != nullptr,
                "gemm_residual_layernorm: null pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (gemm_rowln_supported(M, N, K, copy_ln != 0))
    return gemm_rowln_launch(A, lda, W, ldw, bias, resid, ldr, gamma, beta, eps, copy_ln != 0, xn, ldxn, M, N, K, st);
  EVT_TRY(gemm_launch({.A = A, .lda = lda, .W = W, .ldw = ldw, .bias = bias, .residual = resid, .ldr = ldr, .out = resid,
                       .out_dtype = EVT_F32, .ldo = ldr, .M = M, .N = N, .K = K}, st));
  return layernorm_launch(resid, ldr, gamma, beta, xn, EVT_BF16, ldxn, copy_ln ? resid : nullptr, M, N, eps, st);
}

// A single-kernel version measured slower than the two kernels it replaces (DESIGN.md, negative results): the entry point
// issues those two kernels.
extern "C" int evt_gemm_residual_layernorm(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias, float* resid,
                                           int64_t ldr, const float* gamma, const float* beta, float eps, void* xn, int64_t ldxn,
                                           int64_t M, int N, int K, evt_stream stream) {
  int rc = evt_device_check();
  if (rc != EVT_OK) return rc;
  EVT_CHECK_ARG(resid != nullptr && xn != nullptr && gamma != nullptr && beta != nullptr, "gemm_residual_layernorm: null pointer");
  if (N % 64 != 0 || N < 64 || N > 1024) return fail(EVT_ERR_UNSUPPORTED, "gemm+ln: N must be a multiple of 64 in [64, 1024]");
  return evt_gemm_residual_layernorm_ex(A, lda, W, ldw, bias, resid, ldr, gamma, beta, eps, 0, xn, ldxn, M, N, K, stream);
}
