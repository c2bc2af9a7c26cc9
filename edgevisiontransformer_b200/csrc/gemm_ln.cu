// out[M,N] = epilogue( LayerNorm(x)[M,K] . W[N,K]^T ) for narrow residual streams (K = D in {64..384}): the LayerNorm
// that precedes the QKV / FC1 projection runs INSIDE the GEMM, as the producer of its A operand.
//
//   ViTLayer: layernorm_before -> query/key/value, layernorm_after -> intermediate.dense
//   (SITE/models/vit/modeling_vit.py:333-340; modeling/layers/norm.py + attention.py / ffn.py for the TF dialect)
//
// Why: for D = 192 / 384 the encoder is HBM-bound (SURVEY.md section 8d) and the stand-alone LayerNorm pass costs a
// read of the f32 residual stream plus a write AND a re-read of its bf16 copy -- 21 % of the pruned DeiT-Tiny forward.
// A whole row (K <= 384 values) is K/64 <= 6 shared-memory k-blocks, so one CTA can normalise its 128 rows once, keep them
// as the (128B-swizzled, K-major) A tiles of ALL N tiles of that row block, and never write the normalised copy to HBM.
// Not applicable to D = 768: 12 k-blocks of A (192 KB) leave no room for the W ring.
//
//   warps 0-7    epilogue (shared code: tcgen05.ld -> bias / GELU -> swizzled staging -> TMA store), tile i while i+1 runs
//   warp  8      TMA producer of the W tiles (BN x 64, ring of kWStages)
//   warp  9      MMA issuer: per row block, for every N tile, K/64 x 4 tcgen05.mma (M = 128, N = BN, K = 16)
//   warp  14     x producer: bulk async copies (cp.async.bulk, mbarrier completion) of 32-row (16 for K > 256) chunks of the
//                f32 residual rows into a 2-deep shared-memory ring -- the loads of the NEXT row block stream in while the
//                tensor core works on the current one.  (A first version had the LayerNorm warps load their rows straight
//                from global memory, two rows in flight per warp: 8 rows in flight per SM could not cover the HBM latency
//                and the fused QKV ran 3.5x SLOWER than LayerNorm kernel + GEMM: 251 vs 72 us on pruned DeiT-Tiny.)
//   warps 10-13  LayerNorm: eight threads per row, 16 rows at a time out of the staged chunk, f32 mean and centred variance
//                (three shuffle levels), bf16 result written straight into the A tiles; optionally the normalised f32
//                row is written back to x (TF dialect: the skip carries LN(x))
//
// The model runtime does not use it: measured on B200 (same box, per launch, batch 1024 / 256):
//   pruned DeiT-Tiny  QKV 83.8 us fused vs 38.3 (LayerNorm) + 33.9 (GEMM);  FC1 94.1 vs 38.3 + 48.1  -> 240 k vs 255 k img/s
//   DeiT-Small        QKV 138 vs 23.6 + 47.0;  FC1 176 vs 23.6 + 72.9 (96 KB of A tiles leave a 2-deep W ring)
// One persistent CTA per SM keeps ~50 KB of the residual stream in flight where the stand-alone LayerNorm kernel keeps
// the whole SM's worth of warps loading.  The op stays available (evt_layernorm_gemm).  See DESIGN.md.
#include "gemm_common.cuh"
#include "ops.h"

namespace evt {
namespace {

using namespace gemm_detail;

constexpr int kLnWarps = 4;
constexpr int kLnProducer = kEpiWarps;       // warp 8: W tiles
constexpr int kLnMma = kEpiWarps + 1;        // warp 9
constexpr int kLnFirst = kEpiWarps + 2;      // warps 10..13
constexpr int kLnXWarp = kLnFirst + kLnWarps;   // warp 14: x chunks
constexpr int kLnThreads = 32 * (kEpiWarps + 3 + kLnWarps);
constexpr int kXStages = 2;

struct LnGemmParams {
  GemmParams g;          // bias / out / ldo / M / N / K / tiles_m / tiles_n / vec_ok ...
  const float* x;        // [M, ldx] f32 residual stream
  float* x_copy;         // nullable: normalised f32 rows written back (may alias x)
  const float* gamma;
  const float* beta;
  long long ldx;
  float eps;
};

template <int BN, int KB>
struct CfgLn {
  static constexpr int kABlock = BM * kStageRowBytes;                 // one k-block of A: 128 rows x 128 B
  static constexpr int kABytes = KB * kABlock;
  static constexpr int kABufs = 1;
  static constexpr int kXRows = KB <= 4 ? 32 : 16;                    // rows per staged chunk of x
  static constexpr int kXBytes = kXRows * KB * 64 * 4;
  static constexpr int kWBytes = BN * kStageRowBytes;
  static constexpr int kStagingBytes = kEpiWarps * kStgBytes;
  static constexpr int kBarBytes = (2 * 8 + 8 + 8) * 8 + 16;
  static constexpr int kFree = 232448 - 1024 - kABufs * kABytes - kXStages * kXBytes - kStagingBytes - kBarBytes;
  static constexpr int kWStages = kFree / kWBytes > 6 ? 6 : kFree / kWBytes;
  static constexpr int kSmemBytes = 1024 + kABufs * kABytes + kXStages * kXBytes + kWStages * kWBytes + kStagingBytes + kBarBytes;
  static constexpr int kTmemCols = BN <= 64 ? 128 : BN <= 128 ? 256 : 512;
  static_assert(kWStages >= 2, "no room for a W ring");
  static_assert(kSmemBytes <= 232448, "exceeds the 227 KB of shared memory a CTA can opt in to");
};

template <int BN, int KB, int ACT>
__global__ void __launch_bounds__(kLnThreads, 1)
gemm_ln_kernel(const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmO, const LnGemmParams p) {
  using C = CfgLn<BN, KB>;
  constexpr int D = KB * 64;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* a_base = smem;
  uint8_t* x_base = smem + C::kABufs * C::kABytes;
  uint8_t* w_base = x_base + kXStages * C::kXBytes;
  uint8_t* staging = w_base + C::kWStages * C::kWBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(staging + C::kStagingBytes);
  uint64_t* w_full = bars;            // [8] W producer -> MMA
  uint64_t* w_empty = bars + 8;       // [8] MMA (commit) -> W producer
  uint64_t* a_full = bars + 16;       // [2] LayerNorm warps (kLnWarps arrivals) -> MMA
  uint64_t* a_empty = a_full + 2;     // [2] MMA (commit) -> LayerNorm warps
  uint64_t* tfull = a_empty + 2;      // [2] MMA (commit) -> epilogue
  uint64_t* tempty = tfull + 2;       // [2] epilogue (kEpiWarps arrivals) -> MMA
  uint64_t* x_full = tempty + 2;      // [4] x producer (bulk-copy bytes) -> LayerNorm warps
  uint64_t* x_empty = x_full + 4;     // [4] LayerNorm warps (kLnWarps arrivals) -> x producer
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(x_empty + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int tiles_m = p.g.tiles_m, tiles_n = p.g.tiles_n;

  if (warp == kLnProducer && ptx::elect_one()) {
    ptx::prefetch_tmap(&tmW);
    ptx::prefetch_tmap(&tmO);
    for (int s = 0; s < 8; ++s) {
      ptx::mbar_init(&w_full[s], 1);
      ptx::mbar_init(&w_empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&a_full[s], kLnWarps);
      ptx::mbar_init(&a_empty[s], 1);
      ptx::mbar_init(&tfull[s], 1);
      ptx::mbar_init(&tempty[s], kEpiWarps);
    }
    for (int s = 0; s < 4; ++s) {
      ptx::mbar_init(&x_full[s], 1);
      ptx::mbar_init(&x_empty[s], kLnWarps);
    }
    ptx::fence_mbar_init();
  }
  if (warp == kLnMma) ptx::tmem_alloc<C::kTmemCols>(tmem_ptr);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();  // x (the previous kernel's output) is complete from here on

  if (warp == kLnProducer) {
    // ------------------------------------------------------------ TMA producer: W tiles
    if (ptx::elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int mt = blockIdx.x; mt < tiles_m; mt += gridDim.x) {
        for (int nt = 0; nt < tiles_n; ++nt) {
          for (int kb = 0; kb < KB; ++kb) {
            ptx::mbar_wait(&w_empty[stage], phase ^ 1);
            ptx::mbar_arrive_expect_tx(&w_full[stage], C::kWBytes);
            ptx::tma_load_2d_hint(w_base + stage * C::kWBytes, &tmW, &w_full[stage], kb * 64, nt * BN, ptx::kEvictLast);
            if (++stage == C::kWStages) {
              stage = 0;
              phase ^= 1;
            }
          }
        }
      }
    }
  } else if (warp == kLnMma) {
    // ------------------------------------------------------------ MMA issuer
    if (ptx::elect_one()) {
      constexpr uint32_t idesc = ptx::make_idesc(BM, BN, 1, 0, 0);
      int stage = 0, as = 0, ab = 0;
      uint32_t phase = 0, aphase = 0, abphase = 0;
      for (int mt = blockIdx.x; mt < tiles_m; mt += gridDim.x) {
        ptx::mbar_wait(&a_full[ab], abphase);
        const uint32_t sa = ptx::smem_u32(a_base + ab * C::kABytes);
        for (int nt = 0; nt < tiles_n; ++nt) {
          ptx::mbar_wait(&tempty[as], aphase ^ 1);
          ptx::tc_fence_after();
          const uint32_t d_tmem = tmem_base + as * BN;
#pragma unroll
          for (int kb = 0; kb < KB; ++kb) {
            ptx::mbar_wait(&w_full[stage], phase);
            ptx::tc_fence_after();
            const uint64_t adesc = ptx::smem_desc_sw128(sa + kb * C::kABlock);
            const uint64_t bdesc = ptx::smem_desc_sw128(ptx::smem_u32(w_base + stage * C::kWBytes));
#pragma unroll
            for (int k = 0; k < 4; ++k) ptx::mma_f16_ss(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
            ptx::mma_commit(&w_empty[stage]);
            if (++stage == C::kWStages) {
              stage = 0;
              phase ^= 1;
            }
          }
          ptx::mma_commit(&tfull[as]);
          if (++as == 2) {
            as = 0;
            aphase ^= 1;
          }
        }
        ptx::mma_commit(&a_empty[ab]);  // every MMA that reads this copy of the row block has completed
        if (C::kABufs == 2) {
          if (++ab == 2) {
            ab = 0;
            abphase ^= 1;
          }
        } else {
          abphase ^= 1;
        }
      }
    }
  } else if (warp == kLnXWarp) {
    // ------------------------------------------------------------ x producer: f32 rows -> shared-memory ring
    if (ptx::elect_one()) {
      int xs = 0;
      uint32_t xph = 0;
      const bool dense = p.ldx == D;  // rows contiguous in memory: one bulk copy per chunk
      for (int mt = blockIdx.x; mt < tiles_m; mt += gridDim.x) {
        for (int c = 0; c < BM / C::kXRows; ++c) {
          const long long row0 = static_cast<long long>(mt) * BM + c * C::kXRows;
          long long nrows = static_cast<long long>(p.g.M) - row0;
          nrows = nrows < 0 ? 0 : nrows > C::kXRows ? C::kXRows : nrows;
          ptx::mbar_wait(&x_empty[xs], xph ^ 1);
          uint8_t* dst = x_base + xs * C::kXBytes;
          if (nrows == 0) {
            ptx::mbar_arrive(&x_full[xs]);  // nothing to load: rows past the end of the matrix are produced as zeros
          } else {
            ptx::mbar_arrive_expect_tx(&x_full[xs], static_cast<uint32_t>(nrows) * D * 4);
            if (dense) {
              ptx::bulk_load(dst, p.x + row0 * p.ldx, static_cast<uint32_t>(nrows) * D * 4, &x_full[xs]);
            } else {
              for (int r = 0; r < nrows; ++r) ptx::bulk_load(dst + r * D * 4, p.x + (row0 + r) * p.ldx, D * 4, &x_full[xs]);
            }
          }
          if (++xs == kXStages) {
            xs = 0;
            xph ^= 1;
          }
        }
      }
    }
  } else if (warp >= kLnFirst) {
    // ------------------------------------------------------------ LayerNorm producers of the A operand
    // Eight threads per row, 16 rows per step over the 128 threads: a thread keeps its NF = D / 32 float4 of the row in
    // registers (single pass over the staged chunk), the row statistics take three shuffle levels, and the eight lanes
    // of a quarter-warp read 128 contiguous bytes of ONE row (conflict-free on dense staged rows).  (One row per warp
    // with 32-lane reductions left the four warps latency-bound: 196 us for the pruned-Tiny QKV against 72 us unfused.)
    constexpr int NF = D / 32;                   // float4 per thread per row
    const int t = threadIdx.x - kLnFirst * 32;   // 0..127
    const int l8 = t & 7;
    const int rstep = t >> 3;                    // row within a 16-row step
    float4 g4[NF], b4[NF];
#pragma unroll
    for (int i = 0; i < NF; ++i) {
      const int col = 4 * (l8 + 8 * i);
      g4[i] = __ldg(reinterpret_cast<const float4*>(p.gamma + col));
      b4[i] = __ldg(reinterpret_cast<const float4*>(p.beta + col));
    }
    uint32_t abphase = 0;
    int xs = 0;
    uint32_t xph = 0;
    for (int mt = blockIdx.x; mt < tiles_m; mt += gridDim.x) {
      ptx::mbar_wait(&a_empty[0], abphase ^ 1);  // the MMAs of the previous row block have read the A tiles
      const long long m0 = static_cast<long long>(mt) * BM;
#pragma unroll 1
      for (int c = 0; c < BM / C::kXRows; ++c) {
        ptx::mbar_wait(&x_full[xs], xph);
        const float* xsm = reinterpret_cast<const float*>(x_base + xs * C::kXBytes);
#pragma unroll
        for (int st = 0; st < C::kXRows / 16; ++st) {
          const int rr = st * 16 + rstep;          // row within the chunk
          const int r = c * C::kXRows + rr;        // row within the tile
          const long long row = m0 + r;
          const bool live = row < p.g.M;
          float4 v[NF];
          float s = 0.f;
#pragma unroll
          for (int i = 0; i < NF; ++i) {
            v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (live) v[i] = *reinterpret_cast<const float4*>(xsm + rr * D + 4 * (l8 + 8 * i));
            s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
          }
          s += __shfl_xor_sync(0xffffffffu, s, 1);
          s += __shfl_xor_sync(0xffffffffu, s, 2);
          s += __shfl_xor_sync(0xffffffffu, s, 4);
          const float mean = s / static_cast<float>(D);
          float q = 0.f;
#pragma unroll
          for (int i = 0; i < NF; ++i) {
            const float a0 = v[i].x - mean, a1 = v[i].y - mean, a2 = v[i].z - mean, a3 = v[i].w - mean;
            q += (a0 * a0 + a1 * a1) + (a2 * a2 + a3 * a3);
          }
          q += __shfl_xor_sync(0xffffffffu, q, 1);
          q += __shfl_xor_sync(0xffffffffu, q, 2);
          q += __shfl_xor_sync(0xffffffffu, q, 4);
          const float rstd = rsqrtf(q / static_cast<float>(D) + p.eps);
#pragma unroll
          for (int i = 0; i < NF; ++i) {
            const int col = 4 * (l8 + 8 * i);
            float o0 = (v[i].x - mean) * rstd * g4[i].x + b4[i].x;
            float o1 = (v[i].y - mean) * rstd * g4[i].y + b4[i].y;
            float o2 = (v[i].z - mean) * rstd * g4[i].z + b4[i].z;
            float o3 = (v[i].w - mean) * rstd * g4[i].w + b4[i].w;
            if (!live) o0 = o1 = o2 = o3 = 0.f;   // rows past the end of the matrix feed zeros to the tensor core
            else if (p.x_copy != nullptr) *reinterpret_cast<float4*>(p.x_copy + row * p.ldx + col) = make_float4(o0, o1, o2, o3);
            // k-block col / 64, row r (128 B), 16-byte chunk (col % 64) / 8 XOR-swizzled by (r & 7), 8-byte half (col % 8) / 4
            const int kb = col >> 6, cc = col & 63;
            uint2 w;
            w.x = pack_bf16x2(o0, o1);
            w.y = pack_bf16x2(o2, o3);
            *reinterpret_cast<uint2*>(a_base + kb * C::kABlock + r * 128 + (((cc >> 3) ^ (r & 7)) << 4) + ((cc & 4) << 1)) = w;
          }
        }
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&x_empty[xs]);  // this warp has read its rows of the chunk
        if (++xs == kXStages) {
          xs = 0;
          xph ^= 1;
        }
      }
      ptx::fence_proxy_async_smem();  // the tensor core (async proxy) reads what these generic-proxy stores wrote
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&a_full[0]);
      abphase ^= 1;
    }
  } else {
    // ------------------------------------------------------------ epilogue warps 0..7
    const int quad = warp & 3;
    const int grp = warp >> 2;
    uint8_t* stg = staging + warp * kStgBytes;
    int as = 0;
    uint32_t aphase = 0;
    for (int mt = blockIdx.x; mt < tiles_m; mt += gridDim.x) {
      const int m0 = mt * BM + quad * 32;
      for (int nt = 0; nt < tiles_n; ++nt) {
        const int nt0 = nt * BN;
        prefetch_bias<BN, false>(p.g, grp, lane, nt0);
        ptx::mbar_wait(&tfull[as], aphase);
        ptx::tc_fence_after();
        const uint32_t t_row = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + as * BN;
        epilogue_tile<BN, false, false, ACT, true>(p.g, &tmO, stg, grp, lane, m0, nt0, t_row);
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&tempty[as]);
        if (++as == 2) {
          as = 0;
          aphase ^= 1;
        }
      }
    }
    if (ptx::elect_one()) ptx::bulk_wait<0>();
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == kLnMma) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<C::kTmemCols>(tmem_base);
  }
}

template <int BN, int KB, int ACT>
int launch_ln(const CUtensorMap& tmW, const CUtensorMap& tmO, const LnGemmParams& p, cudaStream_t stream) {
  using C = CfgLn<BN, KB>;
  constexpr auto kern = gemm_ln_kernel<BN, KB, ACT>;
  EVT_TRY(opt_in_smem<kern>(C::kSmemBytes));
  const int grid = p.g.tiles_m < num_sms() ? p.g.tiles_m : num_sms();
  EVT_CUDA(launch_pdl(kern, dim3(grid), dim3(kLnThreads), C::kSmemBytes, stream, pdl_for_gemm(p.g.M, p.g.N, p.g.K), tmW, tmO, p));
  EVT_LAUNCH_CHECK("gemm_ln_kernel");
  return EVT_OK;
}

template <int BN, int KB>
int dispatch_ln_act(const CUtensorMap& w, const CUtensorMap& o, const LnGemmParams& p, int act, cudaStream_t s) {
  switch (act) {
    case EVT_ACT_NONE: return launch_ln<BN, KB, EVT_ACT_NONE>(w, o, p, s);
    case EVT_ACT_GELU_ERF: return launch_ln<BN, KB, EVT_ACT_GELU_ERF>(w, o, p, s);
    default: return launch_ln<BN, KB, EVT_ACT_GELU_TANH>(w, o, p, s);
  }
}

template <int BN>
int dispatch_ln_kb(int kb, const CUtensorMap& w, const CUtensorMap& o, const LnGemmParams& p, int act, cudaStream_t s) {
  switch (kb) {
    case 1: return dispatch_ln_act<BN, 1>(w, o, p, act, s);
    case 2: return dispatch_ln_act<BN, 2>(w, o, p, act, s);
    case 3: return dispatch_ln_act<BN, 3>(w, o, p, act, s);
    case 4: return dispatch_ln_act<BN, 4>(w, o, p, act, s);
    case 6:
      if constexpr (BN <= 192) return dispatch_ln_act<BN, 6>(w, o, p, act, s);
      break;
  }
  return fail(EVT_ERR_UNSUPPORTED, "layernorm+gemm: K must be 64, 128, 192, 256 or 384");
}

}  // namespace

int gemm_ln_launch(const float* x, int64_t ldx, const float* gamma, const float* beta, float eps, float* x_copy, const void* W,
                   int64_t ldw, const float* bias, void* out, int64_t ldo, int64_t M, int N, int K, int act, cudaStream_t stream) {
  EVT_CHECK_ARG(x && gamma && beta && W && out, "layernorm+gemm: null pointer");
  EVT_CHECK_ARG(M > 0 && N > 0 && M < (1ll << 31) - 256, "layernorm+gemm: bad M / N");
  EVT_CHECK_ARG(K % 64 == 0 && (K == 64 || K == 128 || K == 192 || K == 256 || K == 384), "layernorm+gemm: K must be 64, 128, 192, 256 or 384");
  EVT_CHECK_ARG(ldx >= K && ldw >= K && ldo >= N, "layernorm+gemm: leading dimension smaller than the row length");
  EVT_CHECK_ARG(ldx % 4 == 0 && reinterpret_cast<uintptr_t>(x) % 16 == 0, "layernorm+gemm: x rows must be 16-byte aligned");
  EVT_CHECK_ARG(reinterpret_cast<uintptr_t>(gamma) % 16 == 0 && reinterpret_cast<uintptr_t>(beta) % 16 == 0, "layernorm+gemm: gamma / beta must be 16-byte aligned");
  EVT_CHECK_ARG(ldo % 8 == 0 && reinterpret_cast<uintptr_t>(out) % 16 == 0, "layernorm+gemm: out rows must be 16-byte aligned");
  EVT_CHECK_ARG(act >= EVT_ACT_NONE && act <= EVT_ACT_GELU_TANH, "layernorm+gemm: unknown activation");
  // tile width: the one that pads N least (W tiles are re-streamed per row block, so narrower tiles cost nothing extra)
  const int cands[4] = {256, 192, 128, 64};
  int bn = 0;
  long best = -1;
  for (int c : cands) {
    if (K > 256 && c > 192) continue;  // 96 KB of A tiles + the x ring leave room for a ring of 24 KB W tiles at most
    const long cost = static_cast<long>((N + c - 1) / c) * c;
    if (best < 0 || cost < best) best = cost, bn = c;
  }
  CUtensorMap tmW, tmO;
  int rc = make_tmap_2d(&tmW, W, 2, static_cast<uint64_t>(N), static_cast<uint64_t>(K), static_cast<uint64_t>(ldw), bn, 64);
  if (rc != EVT_OK) return rc;
  rc = make_tmap_2d(&tmO, out, 2, static_cast<uint64_t>(M), static_cast<uint64_t>(N), static_cast<uint64_t>(ldo), 32, 64);
  if (rc != EVT_OK) return rc;
  LnGemmParams p = {};
  p.g.bias = bias;
  p.g.residual = nullptr;
  p.g.out = out;
  p.g.ldo = ldo;
  p.g.M = static_cast<int>(M);
  p.g.N = N;
  p.g.K = K;
  p.g.tiles_m = static_cast<int>((M + BM - 1) / BM);
  p.g.tiles_n = (N + bn - 1) / bn;
  p.g.num_kb = K / 64;
  p.g.k_splits = 1;
  p.g.kb_per_split = p.g.num_kb;
  p.g.k_step = 64;
  p.g.vec_ok = (bias == nullptr || reinterpret_cast<uintptr_t>(bias) % 16 == 0) ? 1 : 0;
  p.x = x;
  p.x_copy = x_copy;
  p.gamma = gamma;
  p.beta = beta;
  p.ldx = ldx;
  p.eps = eps;
  const int kb = K / 64;
  switch (bn) {
    case 256: return dispatch_ln_kb<256>(kb, tmW, tmO, p, act, stream);
    case 192: return dispatch_ln_kb<192>(kb, tmW, tmO, p, act, stream);
    case 128: return dispatch_ln_kb<128>(kb, tmW, tmO, p, act, stream);
    default: return dispatch_ln_kb<64>(kb, tmW, tmO, p, act, stream);
  }
}

}  // namespace evt

extern "C" int evt_layernorm_gemm(const float* x, int64_t ldx, const float* gamma, const float* beta, float eps, float* x_copy_f32,
                                  const void* W, int64_t ldw, const float* bias, void* out, int64_t ldo, int64_t M, int N, int K,
                                  int act, evt_stream stream) {
  int rc = evt_device_check();
  if (rc != EVT_OK) return rc;
  return evt::gemm_ln_launch(x, ldx, gamma, beta, eps, x_copy_f32, W, ldw, bias, out, ldo, M, N, K, act,
                             static_cast<cudaStream_t>(stream));
}
