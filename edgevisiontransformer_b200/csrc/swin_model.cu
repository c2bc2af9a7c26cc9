// Whole-model runtime of the Swin shifted-window classifier: owns repacked weights and the host-computed tables
// (window orders, cyclic shifts, relative position bias + shift mask), lays out the caller's workspace and issues the
// forward as a fixed sequence of launches on one stream -- no allocation, no host sync, CUDA-graph capturable.
//
// Reference: the network the reference builds with utils.get_swin (utils.py:14-47) and exports in tools.py:265-292;
// arithmetic as in SITE/models/swin/modeling_swin.py (SwinModel / SwinStage / SwinLayer / SwinPatchMerging).
//
// Data layout (see modeling_swin.py): inside a stage the f32 residual stream [B*T, C] is kept in the WINDOW ORDER of the
// current block.  A block whose cyclic shift differs from the previous one starts with a row gather fused into its
// layernorm_before (gather_layernorm_launch); patch merging is the same kernel with a 4-row gather.
#include <cuda_bf16.h>

#include <cmath>
#include <string>
#include <vector>

#include "loader.h"
#include "ops.h"

namespace evt {
namespace {

constexpr float kLog2e = 1.4426950408889634f;

// raster index (y*W + x) of every position of the window order: r = ((wh*nWw + ww)*ws + i)*ws + j holds the token at
// y = (wh*ws + i + shift) % H, x = (ww*ws + j + shift) % W   (roll by -shift, then window_partition; SwinLayer.forward :606-613)
std::vector<int> window_order(int H, int ws, int shift) {
  std::vector<int> o(static_cast<size_t>(H) * H);
  const int nw = H / ws;
  size_t r = 0;
  for (int wh = 0; wh < nw; ++wh)
    for (int ww = 0; ww < nw; ++ww)
      for (int i = 0; i < ws; ++i)
        for (int j = 0; j < ws; ++j) o[r++] = ((wh * ws + i + shift) % H) * H + (ww * ws + j + shift) % H;
  return o;
}
std::vector<int> inverse(const std::vector<int>& p) {
  std::vector<int> inv(p.size());
  for (size_t i = 0; i < p.size(); ++i) inv[p[i]] = static_cast<int>(i);
  return inv;
}
// [nW, ws*ws, ws*ws] additive 0 / -100 mask of SW-MSA (SwinLayer.get_attn_mask, :556-582)
std::vector<float> shift_mask(int H, int ws, int shift) {
  std::vector<int> img(static_cast<size_t>(H) * H);
  auto region = [&](int v) { return v < H - ws ? 0 : v < H - shift ? 1 : 2; };
  for (int y = 0; y < H; ++y)
    for (int x = 0; x < H; ++x) img[y * H + x] = region(y) * 3 + region(x);
  const int nw = H / ws, N = ws * ws;
  std::vector<float> m(static_cast<size_t>(nw) * nw * N * N);
  for (int wh = 0; wh < nw; ++wh)
    for (int ww = 0; ww < nw; ++ww) {
      float* mw = m.data() + static_cast<size_t>(wh * nw + ww) * N * N;
      for (int a = 0; a < N; ++a)
        for (int b = 0; b < N; ++b) {
          const int ca = img[(wh * ws + a / ws) * H + ww * ws + a % ws], cb = img[(wh * ws + b / ws) * H + ww * ws + b % ws];
          mw[a * N + b] = ca != cb ? -100.f : 0.f;
        }
    }
  return m;
}
// (relative position bias [+ shift mask]) * log2(e) in the window-attention kernel's layout: [n_tab, heads, 64, 56] for
// 7 x 7 windows (key columns 49..55 -inf, rows 49..63 finite), [n_tab, heads, 144, 144] for 12 x 12;
// bias_table [(2ws-1)^2, heads] (SwinSelfAttention :420-438)
std::vector<float> attention_table(const std::vector<float>& bias_table, int heads, int ws, const std::vector<float>* mask, int n_tab) {
  const int N = ws * ws;
  const int rows = N == 49 ? 64 : N, cols = N == 49 ? 56 : N;
  std::vector<float> out(static_cast<size_t>(n_tab) * heads * rows * cols, 0.f);
  for (int t = 0; t < n_tab; ++t)
    for (int h = 0; h < heads; ++h) {
      float* o = out.data() + (static_cast<size_t>(t) * heads + h) * rows * cols;
      for (int r = 0; r < rows; ++r)
        for (int c = N; c < cols; ++c) o[r * cols + c] = -INFINITY;
      for (int a = 0; a < N; ++a)
        for (int b = 0; b < N; ++b) {
          const int dy = a / ws - b / ws + ws - 1, dx = a % ws - b % ws + ws - 1;
          float v = bias_table[static_cast<size_t>(dy * (2 * ws - 1) + dx) * heads + h];
          if (mask) v += (*mask)[(static_cast<size_t>(t) * N + a) * N + b];
          o[a * cols + b] = v * kLog2e;
        }
    }
  return out;
}

struct SwinBlock {
  int* idx = nullptr;  // nullable: row gather into this block's window order
  float *ln1_g = nullptr, *ln1_b = nullptr, *ln2_g = nullptr, *ln2_b = nullptr;
  __nv_bfloat16 *wqkv = nullptr, *wo = nullptr, *w1 = nullptr, *w2 = nullptr;
  float *bqkv = nullptr, *bo = nullptr, *b1 = nullptr, *b2 = nullptr;
  float* table = nullptr;
  int n_tab = 1;
};
struct SwinStage {
  int C = 0, heads = 0, H = 0;
  std::vector<SwinBlock> blocks;
  bool merge = false;
  int* m_idx = nullptr;
  float *m_g = nullptr, *m_b = nullptr;
  __nv_bfloat16* m_w = nullptr;
};

}  // namespace
}  // namespace evt

struct evt_swin {
  evt_swin_spec spec;
  bool loaded = false;
  int grid = 0, patch_k = 0, patch_ld = 0;
  __nv_bfloat16* w_patch = nullptr;
  float *b_patch = nullptr, *g_embed = nullptr, *b_embed = nullptr, *g_final = nullptr, *b_final = nullptr, *b_cls = nullptr;
  __nv_bfloat16* w_cls = nullptr;
  int* idx_embed = nullptr;
  std::vector<evt::SwinStage> stages;
  std::vector<void*> allocs;
};

using namespace evt;

namespace {

struct SwinWs {
  uint8_t *cols, *xn, *qkv, *ctx, *h, *pooled;
  float *ra, *rb;
  size_t bytes;
};

SwinWs plan(const evt_swin* m, int batch, uint8_t* base) {
  const evt_swin_spec& s = m->spec;
  const size_t T0 = static_cast<size_t>(m->grid) * m->grid * batch;
  const size_t C0 = s.embed_dim;
  WorkspaceCarver c{base};
  SwinWs w;
  // T * C is largest in stage 1 and halves with every patch merging
  w.cols = c.take(T0 * m->patch_ld * 2);
  w.ra = c.take<float>(T0 * C0 * 4);
  w.rb = c.take<float>(T0 * C0 * 4);
  w.xn = c.take(T0 * C0 * 2);
  w.qkv = c.take(T0 * 3 * C0 * 2);
  w.ctx = c.take(T0 * C0 * 2);
  w.h = c.take(T0 * 4 * C0 * 2);
  w.pooled = c.take(static_cast<size_t>(batch) * C0 * (1u << (s.stages - 1)) * 2);
  w.bytes = c.bytes;
  return w;
}

}  // namespace

extern "C" int evt_swin_create(const evt_swin_spec* s, evt_swin** out) {
  int rc = evt_device_check();
  if (rc != EVT_OK) return rc;
  EVT_CHECK_ARG(s != nullptr && out != nullptr, "evt_swin_create: null argument");
  EVT_CHECK_ARG(s->stages >= 1 && s->stages <= EVT_SWIN_MAX_STAGES, "stage count out of range");
  if (s->window != 7 && s->window != 12) return fail(EVT_ERR_UNSUPPORTED, "only 7 x 7 and 12 x 12 windows are implemented");
  EVT_CHECK_ARG(s->patch == 4, "only patch size 4 is implemented (swin_*_patch4_window{7,12})");
  EVT_CHECK_ARG(s->image > 0 && s->image % s->patch == 0, "image size must be a multiple of the patch size");
  const int grid = s->image / s->patch;
  EVT_CHECK_ARG(grid % (s->window << (s->stages - 1)) == 0, "image / patch must be a multiple of window * 2^(stages-1)");
  EVT_CHECK_ARG(s->num_labels > 0 && s->eps > 0.f && s->embed_dim > 0 && s->embed_dim % 32 == 0, "bad num_labels / eps / embed_dim");
  for (int i = 0; i < s->stages; ++i) {
    EVT_CHECK_ARG(s->depths[i] > 0 && s->heads[i] > 0, "depths / heads must be positive");
    if ((s->embed_dim << i) != 32 * s->heads[i]) return fail(EVT_ERR_UNSUPPORTED, "only head size 32 is implemented");
  }
  evt_swin* m = new evt_swin();
  m->spec = *s;
  m->grid = grid;
  m->patch_k = 3 * s->patch * s->patch;
  m->patch_ld = (m->patch_k + 7) / 8 * 8;
  *out = m;
  return EVT_OK;
}

extern "C" int evt_swin_destroy(evt_swin* m) {
  if (!m) return EVT_OK;
  for (void* p : m->allocs) cudaFree(p);
  delete m;
  return EVT_OK;
}

extern "C" int evt_swin_load_weights(evt_swin* m, const evt_tensor_view* tensors, int n, evt_stream stream) {
  EVT_CHECK_ARG(m != nullptr && tensors != nullptr && n > 0, "evt_swin_load_weights: bad arguments");
  if (m->loaded) return fail(EVT_ERR_STATE, "weights already loaded; create a new model to reload");
  const evt_swin_spec& s = m->spec;
  Loader L{&m->allocs, static_cast<cudaStream_t>(stream), 2};
  EVT_TRY(L.index(tensors, n));
  const int ws = s.window;
  const std::string e = "swin.embeddings.";
  const int C0 = s.embed_dim;
  // patch-embedding weight [C0, 3, 4, 4] -> bf16 [C0, patch_ld]
  EVT_TRY(L.mat(e + "patch_embeddings.projection.weight", C0, m->patch_k, m->patch_ld, &m->w_patch));
  EVT_TRY(L.vec(e + "patch_embeddings.projection.bias", C0, false, &m->b_patch));
  EVT_TRY(L.vec(e + "norm.weight", C0, false, &m->g_embed));
  EVT_TRY(L.vec(e + "norm.bias", C0, false, &m->b_embed));
  int H = m->grid;
  std::vector<int> order(static_cast<size_t>(H) * H);
  for (size_t i = 0; i < order.size(); ++i) order[i] = static_cast<int>(i);  // raster after the patch embedding
  {
    const std::vector<int> first = window_order(H, ws, 0), inv = inverse(order);
    std::vector<int> idx(first.size());
    for (size_t i = 0; i < first.size(); ++i) idx[i] = inv[first[i]];
    EVT_TRY(L.upload(idx, &m->idx_embed));
    order = first;
  }
  m->stages.resize(s.stages);
  for (int si = 0; si < s.stages; ++si) {
    SwinStage& stg = m->stages[si];
    stg.C = C0 << si;
    stg.heads = s.heads[si];
    stg.H = H;
    const int C = stg.C;
    stg.blocks.resize(s.depths[si]);
    for (int bi = 0; bi < s.depths[si]; ++bi) {
      SwinBlock& blk = stg.blocks[bi];
      const std::string p = "swin.encoder.layers." + std::to_string(si) + ".blocks." + std::to_string(bi) + ".";
      const int shift = (bi % 2 == 1 && H > ws) ? ws / 2 : 0;
      const std::vector<int> want = window_order(H, ws, shift);
      if (want != order) {
        const std::vector<int> inv = inverse(order);
        std::vector<int> idx(want.size());
        for (size_t i = 0; i < want.size(); ++i) idx[i] = inv[want[i]];
        EVT_TRY(L.upload(idx, &blk.idx));
        order = want;
      }
      EVT_TRY(L.vec(p + "layernorm_before.weight", C, false, &blk.ln1_g));
      EVT_TRY(L.vec(p + "layernorm_before.bias", C, false, &blk.ln1_b));
      void* q;
      EVT_TRY(L.alloc(static_cast<size_t>(3) * C * C * 2, &q));
      blk.wqkv = reinterpret_cast<__nv_bfloat16*>(q);
      EVT_TRY(L.alloc(static_cast<size_t>(3) * C * 4, &q));
      blk.bqkv = reinterpret_cast<float*>(q);
      const char* names[3] = {"query", "key", "value"};
      for (int t = 0; t < 3; ++t) {
        EVT_TRY(L.mat_into(p + "attention.self." + names[t] + ".weight", C, C, C, blk.wqkv + static_cast<size_t>(t) * C * C));
        EVT_TRY(L.vec_into(p + "attention.self." + names[t] + ".bias", C, false, blk.bqkv + t * C));
      }
      std::vector<float> bias_table;
      EVT_TRY(L.host_copy(p + "attention.self.relative_position_bias_table", static_cast<int64_t>(2 * ws - 1) * (2 * ws - 1) * stg.heads, &bias_table));
      if (shift > 0) {
        const std::vector<float> mask = shift_mask(H, ws, shift);
        blk.n_tab = (H / ws) * (H / ws);
        EVT_TRY(L.upload(attention_table(bias_table, stg.heads, ws, &mask, blk.n_tab), &blk.table));
      } else {
        blk.n_tab = 1;
        EVT_TRY(L.upload(attention_table(bias_table, stg.heads, ws, nullptr, 1), &blk.table));
      }
      EVT_TRY(L.mat(p + "attention.output.dense.weight", C, C, C, &blk.wo));
      EVT_TRY(L.vec(p + "attention.output.dense.bias", C, false, &blk.bo));
      EVT_TRY(L.vec(p + "layernorm_after.weight", C, false, &blk.ln2_g));
      EVT_TRY(L.vec(p + "layernorm_after.bias", C, false, &blk.ln2_b));
      EVT_TRY(L.mat(p + "intermediate.dense.weight", 4 * C, C, C, &blk.w1));
      EVT_TRY(L.vec(p + "intermediate.dense.bias", 4 * C, false, &blk.b1));
      EVT_TRY(L.mat(p + "output.dense.weight", C, 4 * C, 4 * C, &blk.w2));
      EVT_TRY(L.vec(p + "output.dense.bias", C, false, &blk.b2));
    }
    if (si + 1 < s.stages) {
      // SwinPatchMerging (:326-349): rows (2y, 2x), (2y+1, 2x), (2y, 2x+1), (2y+1, 2x+1) concatenated; the next stage starts in
      // (unshifted) window order
      const std::string p = "swin.encoder.layers." + std::to_string(si) + ".downsample.";
      const int H2 = H / 2;
      const std::vector<int> nxt = window_order(H2, ws, 0), inv = inverse(order);
      std::vector<int> idx(nxt.size() * 4);
      for (size_t i = 0; i < nxt.size(); ++i) {
        const int y2 = nxt[i] / H2, x2 = nxt[i] % H2;
        idx[4 * i + 0] = inv[(2 * y2) * H + 2 * x2];
        idx[4 * i + 1] = inv[(2 * y2 + 1) * H + 2 * x2];
        idx[4 * i + 2] = inv[(2 * y2) * H + 2 * x2 + 1];
        idx[4 * i + 3] = inv[(2 * y2 + 1) * H + 2 * x2 + 1];
      }
      stg.merge = true;
      EVT_TRY(L.upload(idx, &stg.m_idx));
      EVT_TRY(L.vec(p + "norm.weight", 4 * C, false, &stg.m_g));
      EVT_TRY(L.vec(p + "norm.bias", 4 * C, false, &stg.m_b));
      EVT_TRY(L.mat(p + "reduction.weight", 2 * C, 4 * C, 4 * C, &stg.m_w));
      order = nxt;
      H = H2;
    }
  }
  const int Cf = C0 << (s.stages - 1);
  EVT_TRY(L.vec("swin.layernorm.weight", Cf, false, &m->g_final));
  EVT_TRY(L.vec("swin.layernorm.bias", Cf, false, &m->b_final));
  EVT_TRY(L.mat("classifier.weight", s.num_labels, Cf, Cf, &m->w_cls));
  EVT_TRY(L.vec("classifier.bias", s.num_labels, false, &m->b_cls));
  EVT_CUDA(cudaStreamSynchronize(L.st));
  m->loaded = true;
  return EVT_OK;
}

extern "C" int evt_swin_workspace_bytes(const evt_swin* m, int batch, size_t* out) {
  EVT_CHECK_ARG(m != nullptr && out != nullptr && batch > 0, "evt_swin_workspace_bytes: bad arguments");
  *out = plan(m, batch, nullptr).bytes + 1024;
  return EVT_OK;
}

extern "C" int evt_swin_launches_per_forward(const evt_swin* m) {
  if (!m) return 0;
  int n = 3;  // im2col, patch GEMM, embedding LayerNorm (+ gather into window order)
  for (int si = 0; si < m->spec.stages; ++si) n += 7 * m->spec.depths[si] + (si + 1 < m->spec.stages ? 2 : 0);
  return n + 2;  // final LayerNorm + mean pool, classifier
}

extern "C" int evt_swin_forward(evt_swin* m, const float* pixels, int batch, float* logits, void* workspace, size_t workspace_bytes,
                                evt_stream stream) {
  EVT_CHECK_ARG(m != nullptr && pixels != nullptr && logits != nullptr && workspace != nullptr, "evt_swin_forward: null pointer");
  if (!m->loaded) return fail(EVT_ERR_STATE, "evt_swin_forward called before evt_swin_load_weights");
  EVT_CHECK_ARG(batch > 0 && batch <= 65535, "batch must be in 1..65535");
  const evt_swin_spec& s = m->spec;
  SwinWs w;
  EVT_TRY(place_workspace(workspace, workspace_bytes, [&](uint8_t* base) { return plan(m, batch, base); }, &w,
                          "workspace too small for this batch (see evt_swin_workspace_bytes)"));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  StaticWeightsScope weights_are_static;
  const float eps = s.eps;
  const float scale = 1.0f / sqrtf(32.f);
  const int ws2 = s.window * s.window;
  int T = m->grid * m->grid;
  // SwinEmbeddings (:262-301): 4 x 4 patch conv as im2col + GEMM, LayerNorm, rows gathered into the first window order
  EVT_TRY(im2col4_launch(pixels, w.cols, batch, s.image, s.image, s.patch, st));
  EVT_TRY(gemm_launch({.A = w.cols, .lda = m->patch_ld, .W = m->w_patch, .ldw = m->patch_ld, .bias = m->b_patch, .out = w.rb,
                       .out_dtype = EVT_F32, .ldo = s.embed_dim, .M = static_cast<int64_t>(batch) * T, .N = s.embed_dim, .K = m->patch_k}, st));
  EVT_TRY(gather_layernorm_launch(w.rb, m->idx_embed, m->g_embed, m->b_embed, w.ra, EVT_F32, nullptr, batch, T, T, 1, s.embed_dim, eps, st));
  float* resid = w.ra;
  float* other = w.rb;
  for (int si = 0; si < s.stages; ++si) {
    const SwinStage& stg = m->stages[si];
    const int C = stg.C;
    const int64_t M = static_cast<int64_t>(batch) * T;
    for (const SwinBlock& blk : stg.blocks) {
      if (blk.idx != nullptr) {  // cyclic shift / reverse shift folded into layernorm_before; the residual stream is re-ordered too
        EVT_TRY(gather_layernorm_launch(resid, blk.idx, blk.ln1_g, blk.ln1_b, w.xn, EVT_BF16, other, batch, T, T, 1, C, eps, st));
        std::swap(resid, other);
      } else {
        EVT_TRY(layernorm_launch(resid, C, blk.ln1_g, blk.ln1_b, w.xn, EVT_BF16, C, nullptr, M, C, eps, st));
      }
      EVT_TRY(gemm_launch({.A = w.xn, .lda = C, .W = blk.wqkv, .ldw = C, .bias = blk.bqkv, .out = w.qkv, .out_dtype = EVT_BF16, .ldo = 3 * C,
                           .M = M, .N = 3 * C, .K = C}, st));
      EVT_TRY(window_attention_launch(w.qkv, 3 * C, w.ctx, C, blk.table, blk.n_tab, M / ws2, ws2, stg.heads, 32, scale, st));
      EVT_TRY(gemm_launch({.A = w.ctx, .lda = C, .W = blk.wo, .ldw = C, .bias = blk.bo, .residual = resid, .ldr = C, .out = resid,
                           .out_dtype = EVT_F32, .ldo = C, .M = M, .N = C, .K = C}, st));
      EVT_TRY(layernorm_launch(resid, C, blk.ln2_g, blk.ln2_b, w.xn, EVT_BF16, C, nullptr, M, C, eps, st));
      EVT_TRY(gemm_launch({.A = w.xn, .lda = C, .W = blk.w1, .ldw = C, .bias = blk.b1, .out = w.h, .out_dtype = EVT_BF16, .ldo = 4 * C,
                           .M = M, .N = 4 * C, .K = C, .act = EVT_ACT_GELU_ERF}, st));
      EVT_TRY(gemm_launch({.A = w.h, .lda = 4 * C, .W = blk.w2, .ldw = 4 * C, .bias = blk.b2, .residual = resid, .ldr = C, .out = resid,
                           .out_dtype = EVT_F32, .ldo = C, .M = M, .N = C, .K = 4 * C}, st));
    }
    if (stg.merge) {
      // 2 x 2 neighbourhood concat + LayerNorm(4C) as one gather, then the bias-free reduction to 2C
      EVT_TRY(gather_layernorm_launch(resid, stg.m_idx, stg.m_g, stg.m_b, w.h, EVT_BF16, nullptr, batch, T, T / 4, 4, C, eps, st));
      T /= 4;
      EVT_TRY(gemm_launch({.A = w.h, .lda = 4 * C, .W = stg.m_w, .ldw = 4 * C, .out = other, .out_dtype = EVT_F32, .ldo = 2 * C,
                           .M = static_cast<int64_t>(batch) * T, .N = 2 * C, .K = 4 * C}, st));
      std::swap(resid, other);
    }
  }
  const int Cf = s.embed_dim << (s.stages - 1);
  EVT_TRY(layernorm_mean_tokens_launch(resid, m->g_final, m->b_final, w.pooled, batch, T, Cf, eps, st));
  EVT_TRY(gemm_launch({.A = w.pooled, .lda = Cf, .W = m->w_cls, .ldw = Cf, .bias = m->b_cls, .out = logits, .out_dtype = EVT_F32,
                       .ldo = s.num_labels, .M = batch, .N = s.num_labels, .K = Cf}, st));
  return EVT_OK;
}
