// Host-side plumbing shared by all translation units of libevt: status / error string, launch
// counting, and TMA tensor-map encoding through the driver entry point (no link-time libcuda).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

#include "../../include/evt.h"

namespace evt {

void set_error(const std::string& msg);
int fail(int code, const std::string& msg);
void count_launch(int n = 1);

#define EVT_CHECK_ARG(cond, msg)                                   \
  do {                                                             \
    if (!(cond)) return ::evt::fail(EVT_ERR_INVALID, (msg));       \
  } while (0)

#define EVT_CUDA(expr)                                                                                   \
  do {                                                                                                   \
    cudaError_t _e = (expr);                                                                             \
    if (_e != cudaSuccess)                                                                               \
      return ::evt::fail(EVT_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));              \
  } while (0)

// After a kernel launch: catch configuration errors without synchronising.
#define EVT_LAUNCH_CHECK(name)                                                                           \
  do {                                                                                                   \
    cudaError_t _e = cudaGetLastError();                                                                 \
    if (_e != cudaSuccess)                                                                               \
      return ::evt::fail(EVT_ERR_CUDA, std::string("launch ") + (name) + ": " + cudaGetErrorString(_e)); \
    ::evt::count_launch();                                                                               \
  } while (0)

// Return the status of a call that failed.
#define EVT_TRY(expr)                     \
  do {                                    \
    const int _rc = (expr);               \
    if (_rc != EVT_OK) return _rc;        \
  } while (0)

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Lays out a workspace: consecutive regions, each starting on a 1 KiB boundary.  A null base only sizes the plan.
struct WorkspaceCarver {
  uint8_t* base;
  size_t bytes = 0;
  template <typename T = uint8_t>
  T* take(size_t n) {
    T* p = reinterpret_cast<T*>(base + bytes);
    bytes = align_up(bytes + n, 1024);
    return p;
  }
};

// Places a workspace plan (a callable from the 1 KiB-aligned base to a struct with `bytes`) on the caller's buffer, rounded up
// to 1 KiB: the *_workspace_bytes queries add 1 KiB of slack for that.
template <typename Plan>
int place_workspace(void* workspace, size_t workspace_bytes, const Plan& plan, decltype(plan(nullptr))* out, const char* too_small) {
  uint8_t* base = reinterpret_cast<uint8_t*>(align_up(reinterpret_cast<uintptr_t>(workspace), 1024));
  *out = plan(base);
  EVT_CHECK_ARG(out->bytes + (base - static_cast<uint8_t*>(workspace)) <= workspace_bytes, too_small);
  return EVT_OK;
}

// Lets `Kernel` use `bytes` of dynamic shared memory, once per device.  The cache is keyed by the kernel pointer, not its type:
// the instantiations of a kernel template that differ only in non-type template arguments share one function type.
template <auto Kernel>
int opt_in_smem(int bytes) {
  static int done_dev = -1;
  int dev = 0;
  EVT_CUDA(cudaGetDevice(&dev));
  if (done_dev != dev) {
    EVT_CUDA(cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    done_dev = dev;
  }
  return EVT_OK;
}

int num_sms();
bool pdl_enabled();  // EVT_PDL=0 launches every kernel with full stream serialization (A/B timing, debugging)
// Programmatic dependent launch pays on the latency path (batch 1: -12 %, the next kernel's prologue hides behind the
// previous kernel's tail); at large batch, where every kernel runs for 100+ us, it measured 2 % SLOWER (CTAs parked in
// griddepcontrol.wait), so only launches over at most this many rows (tokens) ask for it.
constexpr long long kPdlMaxRows = 32768;
long long pdl_max_rows();  // kPdlMaxRows, or EVT_PDL_MAX_ROWS from the environment (tuning: then rows alone decide)
bool pdl_rows_overridden();
inline bool pdl_for_rows(long long rows) { return rows <= pdl_max_rows() && pdl_enabled(); }
// What decides is the kernel's duration, not its row count: launches shorter than ~50-100 us gain from the overlap
// (DeiT-Small batch 256 +2.9 %, pruned DeiT-Tiny batch 1024 +1.5 %, T2T-ViT-14 +1.1 %), longer ones lose (DeiT-Base at
// 50 k rows -1 %, at 200 k rows -1.6 %).  Proxies: elements touched for the memory-bound kernels, FLOPs for the GEMMs.
constexpr long long kPdlMaxElems = 24ll << 20;        // rows x row length
constexpr double kPdlMaxGemmFlops = 100e9;            // 2 M N K
inline bool pdl_for_work(long long rows, long long row_len) {
  if (pdl_rows_overridden()) return pdl_for_rows(rows);
  return (rows <= kPdlMaxRows || rows * row_len <= kPdlMaxElems) && pdl_enabled();
}
inline bool pdl_for_gemm(long long M, long long N, long long K) {
  if (pdl_rows_overridden()) return pdl_for_rows(M);
  return (M <= kPdlMaxRows || 2.0 * static_cast<double>(M) * static_cast<double>(N) * static_cast<double>(K) <= kPdlMaxGemmFlops) &&
         pdl_enabled();
}

// Launch with programmatic dependent launch allowed: the kernel must call ptx::grid_dep_wait() before its first
// global-memory access.  (cudaLaunchKernelEx also honours a compile-time __cluster_dims__.)
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool allow,
                              Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = allow ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
// Model runtime scope: the W operands of the GEMMs launched inside are weights owned by the library (never written by a
// preceding kernel), which lets the small-M kernel prefetch them ahead of the programmatic dependency wait.
bool gemm_weights_static();
void gemm_weights_static_add(int delta);  // evt_gemm_weights_static
struct StaticWeightsScope {
  StaticWeightsScope();
  ~StaticWeightsScope();
};
bool gemm_split_k_enabled();  // evt_gemm_set_split_k / EVT_GEMM_SPLIT_K
int gemm_pair_mode();  // -1 auto, 0 never, 1 whenever applicable (evt_gemm_set_pair_mode / EVT_GEMM_PAIR)

// 2-D row-major tensor map: `rows` x `cols` elements of `elem_bytes`, leading dimension ld (elements),
// box = box_rows x box_cols, 128-byte swizzle (box_cols * elem_bytes must be 128).
int make_tmap_2d(CUtensorMap* out, const void* base, int elem_bytes, uint64_t rows, uint64_t cols, uint64_t ld,
                 uint32_t box_rows, uint32_t box_cols);
// Same with a 64-byte swizzle span (box_cols * elem_bytes == 64): narrow staging tiles (swizzle_bytes 64 or 128).
int make_tmap_2d_sw(CUtensorMap* out, const void* base, int elem_bytes, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows,
                    uint32_t box_cols, int swizzle_bytes);
// 3-D view [batch][rows][cols] of a row-major matrix of batch * rows rows (leading dimension ld): a box is box_rows x
// box_cols of ONE batch entry, so rows past the end of an image are zero-filled on loads and clipped on stores instead of
// running into the next image.  128-byte swizzle.
// batch_rows: matrix rows from one batch entry to the next (0 = rows; more: only the first `rows` of each entry are in view).
int make_tmap_3d_rows(CUtensorMap* out, const void* base, int elem_bytes, uint64_t cols, uint64_t rows, uint64_t batch,
                      uint64_t ld, uint32_t box_rows, uint32_t box_cols, uint64_t batch_rows = 0);
// make_tmap_3d_rows for bf16 boxes 16 columns (32 bytes) wide, 32-byte swizzle: the columns of a head past its first 64.
int make_tmap_3d_rows_sw32(CUtensorMap* out, const void* base, uint64_t cols, uint64_t rows, uint64_t batch, uint64_t ld,
                           uint32_t box_rows, uint64_t batch_rows);

}  // namespace evt
