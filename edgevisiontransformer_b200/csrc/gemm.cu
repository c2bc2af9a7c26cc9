// out[M,N] = epilogue(A[M,K] . W[N,K]^T): persistent, warp-specialised tcgen05 GEMM for sm_100a.
//
//   warp 8      TMA producer   : A tile 128x64 and W tile BNx64 (bf16; 128x32 / BNx32 for tf32) into a
//                                 STAGES-deep ring of 128B-swizzled shared-memory buffers
//   warp 9      MMA issuer     : one thread issues tcgen05.mma (M=128, N=BN, K=16|8) into one of two
//                                 TMEM accumulator stages (2 x BN columns), commits to mbarriers
//   warps 0-7   epilogue       : tcgen05.ld the accumulator (lane == row; two warps per TMEM lane quadrant, taking
//                                 alternate 128-byte column chunks), bias / GELU on packed f32x2 pairs, then through
//                                 a 128B-swizzled shared tile to a TMA store / TMA f32 reduce-add (or coalesced
//                                 global stores on the generic path); overlaps the next tile's MMAs
//
// Tiles are walked N-fastest so the CTAs resident at one time share a few A row-blocks (read from HBM
// once) while the whole weight matrix stays in L2.  M, N and K tails are handled by TMA zero fill on the
// load side and by clipping / predication on the store side, so no operand is ever padded in HBM (only leading
// dimensions must be multiples of 16 bytes).
#include "gemm_common.cuh"
#include "ops.h"

namespace evt {
namespace {

using namespace gemm_detail;

template <int BN, bool TF32, bool OUT_F32, int ACT, bool TMA_OUT>
__global__ void __launch_bounds__(kThreads, 1)
gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW,
            const __grid_constant__ CUtensorMap tmO, const GemmParams p) {
  using C = Cfg<BN>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* stage_base = smem;
  uint8_t* staging = smem + C::kStages * C::kStageBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::kStages * C::kStageBytes + C::kStagingBytes);
  uint64_t* full = bars;
  uint64_t* empty = bars + C::kStages;
  uint64_t* tfull = bars + 2 * C::kStages;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tempty + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // work item = (output tile, K split).  k_splits > 1 only for the TMA reduce-add epilogue, where partial products
  // of the same tile simply add up in the residual stream (bias comes from split 0).
  const int num_tiles = p.tiles_m * p.tiles_n * p.k_splits;

  if (warp == kProducerWarp && lane == 0) {
    ptx::prefetch_tmap(&tmA);
    ptx::prefetch_tmap(&tmW);
    if (TMA_OUT) ptx::prefetch_tmap(&tmO);
    for (int s = 0; s < C::kStages; ++s) {
      ptx::mbar_init(&full[s], 1);
      ptx::mbar_init(&empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&tfull[s], 1);
      ptx::mbar_init(&tempty[s], kEpiWarps);
    }
    ptx::fence_mbar_init();
  }
  if (warp == kMmaWarp) ptx::tmem_alloc<C::kTmemCols>(tmem_ptr);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  ptx::grid_dep_launch();  // the next kernel may begin its own prologue
  // Latency path: when the caller vouches that W is not produced by the preceding kernel (model weights), the W tiles of
  // the first pipeline stages are requested BEFORE the dependency wait, so their HBM round trip (weights are cold at batch
  // 1: each is read once per forward) overlaps the previous kernel's tail under programmatic dependent launch.
  int w_pre = 0;
  if (p.w_static && warp == kProducerWarp && static_cast<int>(blockIdx.x) < num_tiles) {
    const int item = blockIdx.x;
    const int tile = item / p.k_splits;
    const int kb0 = (item - tile * p.k_splits) * p.kb_per_split;
    const int kb1 = min(p.num_kb, kb0 + p.kb_per_split);
    const int n0 = (tile % p.tiles_n) * BN;
    w_pre = min(C::kStages, kb1 - kb0);  // warp-uniform; the elected thread of the producer loop below consumes it
    if (ptx::elect_one()) {
      for (int i = 0; i < w_pre; ++i) {
        ptx::mbar_arrive_expect_tx(&full[i], C::kStageBytes);
        ptx::tma_load_2d_hint(stage_base + i * C::kStageBytes + C::kABytes, &tmW, &full[i], (kb0 + i) * p.k_step, n0, ptx::kEvictLast);
      }
    }
  }
  ptx::grid_dep_wait();    // operands / outputs of the previous kernel are complete from here on

  if (warp == kProducerWarp) {
    // ------------------------------------------------------------ TMA producer
    // One thread, chosen with elect.sync rather than `lane == 0`: ptxas then knows the region is single-threaded and keeps
    // descriptors / coordinates in uniform registers.  Under a `lane == 0` guard every UTMALDG / UTCHMMA was wrapped in an
    // ELECT + R2UR.BROADCAST + BRA.U.ANY "waterfall" loop (~16 instructions per MMA, ncu round 2).
    if (ptx::elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int item = blockIdx.x; item < num_tiles; item += gridDim.x) {
        const int tile = item / p.k_splits;
        const int kb0 = (item - tile * p.k_splits) * p.kb_per_split;
        const int kb1 = min(p.num_kb, kb0 + p.kb_per_split);
        const int m0 = (tile / p.tiles_n) * BM;
        const int n0 = (tile % p.tiles_n) * BN;
        for (int kb = kb0; kb < kb1; ++kb) {
          uint8_t* sa = stage_base + stage * C::kStageBytes;
          uint8_t* sb = sa + C::kABytes;
          if (w_pre > 0) {  // first stages of the first item: barrier armed and W already in flight
            --w_pre;
            ptx::tma_load_2d(sa, &tmA, &full[stage], kb * p.k_step, m0);
            if (++stage == C::kStages) {
              stage = 0;
              phase ^= 1;
            }
            continue;
          }
          ptx::mbar_wait(&empty[stage], phase ^ 1);
          ptx::mbar_arrive_expect_tx(&full[stage], C::kStageBytes);
          ptx::tma_load_2d(sa, &tmA, &full[stage], kb * p.k_step, m0);
          ptx::tma_load_2d_hint(sb, &tmW, &full[stage], kb * p.k_step, n0, ptx::kEvictLast);
          if (++stage == C::kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == kMmaWarp) {
    // ------------------------------------------------------------ MMA issuer (one elected thread, see above)
    if (ptx::elect_one()) {
      constexpr uint32_t idesc = ptx::make_idesc(BM, BN, TF32 ? 2 : 1, 0, 0);
      int stage = 0;
      uint32_t phase = 0;
      int as = 0;
      uint32_t aphase = 0;
      for (int item = blockIdx.x; item < num_tiles; item += gridDim.x) {
        const int kb0 = (item % p.k_splits) * p.kb_per_split;
        const int kb1 = min(p.num_kb, kb0 + p.kb_per_split);
        ptx::mbar_wait(&tempty[as], aphase ^ 1);
        ptx::tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN;
        for (int kb = kb0; kb < kb1; ++kb) {
          ptx::mbar_wait(&full[stage], phase);
          ptx::tc_fence_after();
          const uint32_t sa = ptx::smem_u32(stage_base + stage * C::kStageBytes);
          const uint64_t adesc = ptx::smem_desc_sw128(sa);
          const uint64_t bdesc = ptx::smem_desc_sw128(sa + C::kABytes);
#pragma unroll
          for (int k = 0; k < 4; ++k) {  // 4 x 32 bytes of K per stage row
            const uint32_t acc = (kb != kb0 || k != 0) ? 1u : 0u;
            if (TF32) ptx::mma_tf32_ss(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, acc);
            else ptx::mma_f16_ss(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, acc);
          }
          ptx::mma_commit(&empty[stage]);  // frees the smem slot once these MMAs have read it
          if (++stage == C::kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
        ptx::mma_commit(&tfull[as]);  // accumulator complete
        if (++as == 2) {
          as = 0;
          aphase ^= 1;
        }
      }
    }
  } else {
    // ------------------------------------------------------------ epilogue warps 0..7
    const int quad = warp & 3;
    const int grp = warp >> 2;
    uint8_t* stg = staging + warp * kStgBytes;
    int as = 0;
    uint32_t aphase = 0;
    GemmParams pe = p;  // epilogue view of the parameters: K splits other than the first add no bias
    for (int item = blockIdx.x; item < num_tiles; item += gridDim.x) {
      const int tile = item / p.k_splits;
      pe.bias = item - tile * p.k_splits == 0 ? p.bias : nullptr;
      const int m0 = (tile / p.tiles_n) * BM + quad * 32;
      const int nt0 = (tile % p.tiles_n) * BN;
      prefetch_bias<BN, OUT_F32>(pe, grp, lane, nt0);
      ptx::mbar_wait(&tfull[as], aphase);
      ptx::tc_fence_after();
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + as * BN;
      epilogue_tile<BN, TF32, OUT_F32, ACT, TMA_OUT>(pe, &tmO, stg, grp, lane, m0, nt0, t_row);
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&tempty[as]);
      if (++as == 2) {
        as = 0;
        aphase ^= 1;
      }
    }
    if (TMA_OUT && ptx::elect_one()) ptx::bulk_wait<0>();
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<C::kTmemCols>(tmem_base);
  }
}

// Tile width: the one that pads N least; when that leaves SMs without a tile (small M: the latency path), the
// narrower width that puts the most CTAs to work.
int choose_bn(int64_t M, int N) {
  const int cands[4] = {256, 192, 128, 64};
  const long tiles_m = static_cast<long>((M + BM - 1) / BM);
  int best = 256;
  long best_cost = -1;
  for (int bn : cands) {
    long cost = static_cast<long>((N + bn - 1) / bn) * bn;
    if (best_cost < 0 || cost < best_cost) {
      best_cost = cost;
      best = bn;
    }
  }
  const long sms = num_sms();
  if (tiles_m * ((N + best - 1) / best) >= sms) return best;
  long best_busy = -1;
  for (int bn : cands) {
    if (bn > best) continue;
    const long tiles = tiles_m * ((N + bn - 1) / bn);
    const long busy = tiles < sms ? tiles : sms;
    if (busy > best_busy) {  // ties keep the wider tile
      best_busy = busy;
      best = bn;
    }
  }
  return best;
}

template <int BN, bool TF32, bool OUT_F32, int ACT, bool TMA_OUT>
int launch(const CUtensorMap& tmA, const CUtensorMap& tmW, const CUtensorMap& tmO, const GemmParams& p, cudaStream_t stream) {
  using C = Cfg<BN>;
  constexpr auto kern = gemm_kernel<BN, TF32, OUT_F32, ACT, TMA_OUT>;
  EVT_TRY(opt_in_smem<kern>(C::kSmemBytes));
  const int num_tiles = p.tiles_m * p.tiles_n * p.k_splits;
  const int grid = num_tiles < num_sms() ? num_tiles : num_sms();
  EVT_CUDA(launch_pdl(kern, dim3(grid), dim3(kThreads), C::kSmemBytes, stream, pdl_for_gemm(p.M, p.N, p.K), tmA, tmW, tmO, p));
  EVT_LAUNCH_CHECK("gemm_kernel");
  return EVT_OK;
}

template <int BN, bool TF32, bool TMA_OUT>
int dispatch_epi(const CUtensorMap& a, const CUtensorMap& w, const CUtensorMap& o, const GemmParams& p, bool out_f32, int act,
                 cudaStream_t s) {
  if (out_f32) {
    switch (act) {
      case EVT_ACT_NONE: return launch<BN, TF32, true, EVT_ACT_NONE, TMA_OUT>(a, w, o, p, s);
      case EVT_ACT_GELU_ERF: return launch<BN, TF32, true, EVT_ACT_GELU_ERF, TMA_OUT>(a, w, o, p, s);
      default: return launch<BN, TF32, true, EVT_ACT_GELU_TANH, TMA_OUT>(a, w, o, p, s);
    }
  }
  switch (act) {
    case EVT_ACT_NONE: return launch<BN, TF32, false, EVT_ACT_NONE, TMA_OUT>(a, w, o, p, s);
    case EVT_ACT_GELU_ERF: return launch<BN, TF32, false, EVT_ACT_GELU_ERF, TMA_OUT>(a, w, o, p, s);
    default: return launch<BN, TF32, false, EVT_ACT_GELU_TANH, TMA_OUT>(a, w, o, p, s);
  }
}

// TMA epilogue: contiguous output rows, 16-byte aligned, and the skip connection (if any) updated in place
bool tma_out_ok(const GemmOp& op) {
  const int oeb = op.out_dtype != EVT_BF16 ? 4 : 2;
  return op.map.out_group == 0 && op.map.res_row_mod == 0 && reinterpret_cast<uintptr_t>(op.out) % 16 == 0 && (op.ldo * oeb) % 16 == 0 &&
         (op.residual == nullptr || (oeb == 4 && op.residual == reinterpret_cast<const float*>(op.out) && op.ldr == op.ldo));
}

// Split K when a reduce-add epilogue leaves most SMs idle (out-proj / FC2 at batch 1: 6 tiles for 148 SMs).  The
// partial products meet in the f32 residual stream through the same TMA reduce-add; their order is not fixed, so
// results can differ in the last bit from run to run -- only in this small-M regime; evt_gemm_set_split_k(0) turns it
// off, a forced kernel choice (evt_gemm_set_pair_mode) never splits, and op.max_k_splits bounds the count.
// The tf32 (accuracy) mode never splits: DeiT-Tiny batch 1 would drop from 0.477 to 0.427 ms, but the unordered f32
// reduce-adds flip tf32 roundings downstream and the logit error of BASELINE config 1 moves from a reproducible 7.5e-4
// to 9.2e-4 in one run -- a random variable that close to the 1e-3 contract is not worth 0.05 ms.
int k_splits(const GemmOp& op, bool tma_out, long tiles, int num_kb) {
  if (op.in_dtype == EVT_F32 || !tma_out || op.residual == nullptr || gemm_pair_mode() >= 0 || !gemm_split_k_enabled()) return 1;
  if (tiles * 2 > num_sms() || num_kb < 4) return 1;
  int splits = static_cast<int>(num_sms() / tiles);
  if (splits > num_kb / 2) splits = num_kb / 2;  // at least two K blocks per split
  if (op.max_k_splits > 0 && splits > op.max_k_splits) splits = op.max_k_splits;
  return splits > 1 ? splits : 1;
}

}  // namespace

int gemm_k_splits(const GemmOp& op) {
  const int k_step = kStageRowBytes / (op.in_dtype == EVT_F32 ? 4 : 2);
  const int bn = choose_bn(op.M, op.N);
  const long tiles = static_cast<long>((op.M + BM - 1) / BM) * ((op.N + bn - 1) / bn);
  const int num_kb = (op.K + k_step - 1) / k_step;
  const int splits = k_splits(op, tma_out_ok(op), tiles, num_kb);
  if (splits == 1) return 1;
  const int kb_per_split = (num_kb + splits - 1) / splits;
  return (num_kb + kb_per_split - 1) / kb_per_split;
}

int gemm_launch(const GemmOp& op, cudaStream_t stream) {
  EVT_CHECK_ARG(op.A && op.W && op.out, "gemm: null pointer");
  EVT_CHECK_ARG(op.M > 0 && op.N > 0 && op.K > 0, "gemm: M, N, K must be positive");
  EVT_CHECK_ARG(op.M < (1ll << 31) - 256, "gemm: M too large");
  EVT_CHECK_ARG(op.in_dtype == EVT_BF16 || op.in_dtype == EVT_F32, "gemm: input dtype must be bf16 or f32(tf32)");
  EVT_CHECK_ARG(op.out_dtype == EVT_BF16 || op.out_dtype == EVT_F32 || op.out_dtype == EVT_TF32, "gemm: out dtype must be bf16, f32 or tf32");
  EVT_CHECK_ARG(!(op.out_dtype == EVT_TF32 && op.residual != nullptr), "gemm: a tf32-rounded output cannot take a residual");
  EVT_CHECK_ARG(op.act >= EVT_ACT_NONE && op.act <= EVT_ACT_GELU_TANH, "gemm: unknown activation");
  EVT_CHECK_ARG(op.lda >= op.K && op.ldw >= op.K && op.ldo >= op.N, "gemm: leading dimension smaller than the row length");
  EVT_CHECK_ARG(op.map.out_group >= 0 && op.map.res_row_mod >= 0, "gemm: negative row-group parameter");
  EVT_CHECK_ARG(op.residual == nullptr || op.ldr >= op.N, "gemm: residual leading dimension smaller than N");
  const bool tf32 = op.in_dtype == EVT_F32;
  const int eb = tf32 ? 4 : 2;
  const int k_step = kStageRowBytes / eb;
  const int bn = choose_bn(op.M, op.N);
  CUtensorMap tmA, tmW;
  int rc = make_tmap_2d(&tmA, op.A, eb, static_cast<uint64_t>(op.M), static_cast<uint64_t>(op.K), static_cast<uint64_t>(op.lda), BM, k_step);
  if (rc != EVT_OK) return rc;
  rc = make_tmap_2d(&tmW, op.W, eb, static_cast<uint64_t>(op.N), static_cast<uint64_t>(op.K), static_cast<uint64_t>(op.ldw), bn, k_step);
  if (rc != EVT_OK) return rc;
  GemmParams p;
  p.bias = op.bias;
  p.residual = op.residual;
  p.out = op.out;
  p.ldr = op.ldr;
  p.ldo = op.ldo;
  p.M = static_cast<int>(op.M);
  p.N = op.N;
  p.K = op.K;
  p.res_row_mod = op.map.res_row_mod;
  p.res_row_off = op.map.res_row_off;
  p.out_group = op.map.out_group;
  p.out_group_stride = op.map.out_group_stride;
  p.out_group_off = op.map.out_group_off;
  p.tiles_m = static_cast<int>((op.M + BM - 1) / BM);
  p.tiles_n = (op.N + bn - 1) / bn;
  p.num_kb = (op.K + k_step - 1) / k_step;
  p.k_step = k_step;
  p.w_static = gemm_weights_static() ? 1 : 0;
  {
    const int oe = op.out_dtype != EVT_BF16 ? 4 : 2;
    bool ok = reinterpret_cast<uintptr_t>(op.out) % 16 == 0 && (op.ldo * oe) % 16 == 0;
    if (op.bias) ok = ok && reinterpret_cast<uintptr_t>(op.bias) % 16 == 0;
    if (op.residual) ok = ok && reinterpret_cast<uintptr_t>(op.residual) % 16 == 0 && (op.ldr * 4) % 16 == 0;
    p.vec_ok = ok ? 1 : 0;
  }
  const bool of32 = op.out_dtype != EVT_BF16;
  p.round_tf32 = op.out_dtype == EVT_TF32 ? 1 : 0;
  const int oeb = of32 ? 4 : 2;
  const bool tma_out = tma_out_ok(op);
  CUtensorMap tmO = tmA;
  if (tma_out) {
    rc = make_tmap_2d(&tmO, op.out, oeb, static_cast<uint64_t>(op.M), static_cast<uint64_t>(op.N), static_cast<uint64_t>(op.ldo), 32,
                      128 / oeb);
    if (rc != EVT_OK) return rc;
  }
  p.k_splits = 1;
  p.kb_per_split = p.num_kb;
  const int splits = k_splits(op, tma_out, static_cast<long>(p.tiles_m) * p.tiles_n, p.num_kb);
  if (splits > 1) {
    p.kb_per_split = (p.num_kb + splits - 1) / splits;
    p.k_splits = (p.num_kb + p.kb_per_split - 1) / p.kb_per_split;
  }
  // Large problems run on CTA pairs (cta_group::2, 256-row tiles): half the W traffic per SM.  evt_gemm_set_pair_mode
  // forces the choice (tests exercise both kernels on the same shapes).
  if (!tf32 && tma_out && pair_supported(bn)) {
    const int pair_mode = gemm_pair_mode();
    const long pair_tiles = static_cast<long>((op.M + 2 * BM - 1) / (2 * BM)) * p.tiles_n;
    const bool use_pair = pair_mode < 0 ? pair_tiles >= num_sms() : pair_mode != 0;
    if (use_pair) return gemm_pair_launch(bn, op.W, op.ldw, tmA, tmO, p, of32, op.act, stream);
  }
#define EVT_BN_CASE(BNV)                                                                                      \
  case BNV:                                                                                                   \
    if (tma_out)                                                                                              \
      return tf32 ? dispatch_epi<BNV, true, true>(tmA, tmW, tmO, p, of32, op.act, stream)                     \
                  : dispatch_epi<BNV, false, true>(tmA, tmW, tmO, p, of32, op.act, stream);                   \
    return tf32 ? dispatch_epi<BNV, true, false>(tmA, tmW, tmO, p, of32, op.act, stream)                      \
                : dispatch_epi<BNV, false, false>(tmA, tmW, tmO, p, of32, op.act, stream);
  switch (bn) {
    EVT_BN_CASE(256)
    EVT_BN_CASE(192)
    EVT_BN_CASE(128)
    EVT_BN_CASE(64)
  }
#undef EVT_BN_CASE
  return fail(EVT_ERR_INVALID, "gemm: no tile configuration");
}

}  // namespace evt

extern "C" int evt_gemm_bias_act(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias,
                                 const float* residual, int64_t ldr, int res_row_mod, int res_row_off, void* out,
                                 int out_dtype, int64_t ldo, int out_group, int out_group_stride, int out_group_off,
                                 int64_t M, int N, int K, int act, evt_stream stream) {
  int rc = evt_device_check();
  if (rc != EVT_OK) return rc;
  return evt::gemm_launch({.A = A, .lda = lda, .W = W, .ldw = ldw, .in_dtype = EVT_BF16, .bias = bias, .residual = residual, .ldr = ldr,
                           .out = out, .out_dtype = out_dtype, .ldo = ldo, .M = M, .N = N, .K = K, .act = act,
                           .map = {.res_row_mod = res_row_mod, .res_row_off = res_row_off, .out_group = out_group, .out_group_stride = out_group_stride,
                                    .out_group_off = out_group_off}}, static_cast<cudaStream_t>(stream));
}

// tf32 flavour: A and W are f32 (the MMA reads them as tf32); out is f32.
extern "C" int evt_gemm_bias_act_tf32(const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias,
                                      const float* residual, int64_t ldr, int res_row_mod, int res_row_off, float* out,
                                      int64_t ldo, int out_group, int out_group_stride, int out_group_off, int64_t M,
                                      int N, int K, int act, evt_stream stream) {
  int rc = evt_device_check();
  if (rc != EVT_OK) return rc;
  return evt::gemm_launch({.A = A, .lda = lda, .W = W, .ldw = ldw, .in_dtype = EVT_F32, .bias = bias, .residual = residual, .ldr = ldr,
                           .out = out, .out_dtype = EVT_F32, .ldo = ldo, .M = M, .N = N, .K = K, .act = act,
                           .map = {.res_row_mod = res_row_mod, .res_row_off = res_row_off, .out_group = out_group, .out_group_stride = out_group_stride,
                                    .out_group_off = out_group_off}}, static_cast<cudaStream_t>(stream));
}
