#include "common.h"

#include <atomic>
#include <cstdlib>
#include <mutex>

namespace evt {

static thread_local std::string g_last_error;
static thread_local int64_t g_launches = 0;

void set_error(const std::string& msg) { g_last_error = msg; }
int fail(int code, const std::string& msg) {
  g_last_error = msg;
  return code;
}
void count_launch(int n) { g_launches += n; }

static thread_local int g_static_weights = 0;
bool gemm_weights_static() { return g_static_weights > 0; }
StaticWeightsScope::StaticWeightsScope() { ++g_static_weights; }
StaticWeightsScope::~StaticWeightsScope() { --g_static_weights; }
void gemm_weights_static_add(int delta) {
  g_static_weights += delta;
  if (g_static_weights < 0) g_static_weights = 0;
}

int num_sms() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(p);
  });
  return fn;
}

static std::atomic<int> g_pair_mode{[] {
  const char* e = getenv("EVT_GEMM_PAIR");
  return e == nullptr ? -1 : atoi(e);
}()};
long long pdl_max_rows() {
  static const long long v = [] {
    const char* e = getenv("EVT_PDL_MAX_ROWS");
    return e ? atoll(e) : kPdlMaxRows;
  }();
  return v;
}

bool pdl_rows_overridden() {
  static const bool v = getenv("EVT_PDL_MAX_ROWS") != nullptr;
  return v;
}

bool pdl_enabled() {
  static const bool on = [] {
    const char* e = getenv("EVT_PDL");
    return e == nullptr || atoi(e) != 0;
  }();
  return on;
}
static std::atomic<int> g_split_k{[] {
  const char* e = getenv("EVT_GEMM_SPLIT_K");
  return e == nullptr ? 1 : (atoi(e) != 0);
}()};
bool gemm_split_k_enabled() { return g_split_k.load(std::memory_order_relaxed) != 0; }
int gemm_pair_mode() { return g_pair_mode.load(std::memory_order_relaxed); }

// What the three map shapes share: the entry point, the alignment checks, the shape's own box check (`box_error`: null when the
// box is valid), then the encode.  A box is box_rows x box_cols of one batch entry (rank 3) or of the whole matrix (rank 2).
static int encode_tmap(CUtensorMap* out, const void* base, int elem_bytes, int rank, uint64_t cols, uint64_t rows, uint64_t batch,
                       uint64_t ld, uint32_t box_rows, uint32_t box_cols, int swizzle_bytes, const char* box_error, const char* what,
                       uint64_t batch_rows = 0) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) return fail(EVT_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0) return fail(EVT_ERR_INVALID, "TMA base pointer not 16-byte aligned");
  if ((ld * elem_bytes) % 16 != 0) return fail(EVT_ERR_INVALID, "TMA leading dimension not a multiple of 16 bytes");
  if (box_error) return fail(EVT_ERR_INVALID, box_error);
  const cuuint64_t dims[3] = {cols, rows, batch};
  const cuuint64_t strides[2] = {ld * static_cast<uint64_t>(elem_bytes), (batch_rows ? batch_rows : rows) * ld * static_cast<uint64_t>(elem_bytes)};
  const cuuint32_t box[3] = {box_cols, box_rows, 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(out, elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, rank, const_cast<void*>(base),
                   dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(EVT_ERR_CUDA, std::string("cuTensorMapEncodeTiled") + what + " failed with CUresult " + std::to_string((int)r));
  return EVT_OK;
}

static const char* box_128_error(int elem_bytes, uint32_t box_rows, uint32_t box_cols) {
  return box_cols * elem_bytes != 128 || box_rows > 256 || box_rows == 0 ? "TMA box must be 128 bytes wide and at most 256 rows" : nullptr;
}

int make_tmap_2d(CUtensorMap* out, const void* base, int elem_bytes, uint64_t rows, uint64_t cols, uint64_t ld,
                 uint32_t box_rows, uint32_t box_cols) {
  const char* err = box_128_error(elem_bytes, box_rows, box_cols);
  if (!err && elem_bytes != 2 && elem_bytes != 4) err = "TMA element size must be 2 or 4";
  return encode_tmap(out, base, elem_bytes, 2, cols, rows, 1, ld, box_rows, box_cols, 128, err, "");
}

int make_tmap_2d_sw(CUtensorMap* out, const void* base, int elem_bytes, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows,
                    uint32_t box_cols, int swizzle_bytes) {
  if (swizzle_bytes == 128) return make_tmap_2d(out, base, elem_bytes, rows, cols, ld, box_rows, box_cols);
  const bool ok = swizzle_bytes == 64 && box_cols * elem_bytes == 64 && box_rows <= 256 && box_rows != 0 && (elem_bytes == 2 || elem_bytes == 4);
  return encode_tmap(out, base, elem_bytes, 2, cols, rows, 1, ld, box_rows, box_cols, 64,
                     ok ? nullptr : "TMA box must be as wide as its swizzle span (64 or 128 bytes) and at most 256 rows", " (64B swizzle)");
}

int make_tmap_3d_rows(CUtensorMap* out, const void* base, int elem_bytes, uint64_t cols, uint64_t rows, uint64_t batch,
                      uint64_t ld, uint32_t box_rows, uint32_t box_cols, uint64_t batch_rows) {
  const char* err = box_128_error(elem_bytes, box_rows, box_cols);
  if (!err && elem_bytes != 2) err = "3-D TMA map: bf16 only";
  if (!err && batch_rows != 0 && batch_rows < rows) err = "3-D TMA map: batch entries closer than their row count";
  return encode_tmap(out, base, elem_bytes, 3, cols, rows, batch, ld, box_rows, box_cols, 128, err, " (3-D)", batch_rows);
}

int make_tmap_3d_rows_sw32(CUtensorMap* out, const void* base, uint64_t cols, uint64_t rows, uint64_t batch, uint64_t ld,
                           uint32_t box_rows, uint64_t batch_rows) {
  const char* err = box_rows > 256 || box_rows == 0 ? "TMA box must be at most 256 rows" : nullptr;
  if (!err && batch_rows != 0 && batch_rows < rows) err = "3-D TMA map: batch entries closer than their row count";
  return encode_tmap(out, base, 2, 3, cols, rows, batch, ld, box_rows, 16, 32, err, " (3-D, 32B swizzle)", batch_rows);
}

}  // namespace evt

extern "C" {

const char* evt_last_error(void) { return evt::g_last_error.c_str(); }
int evt_version(void) { return EVT_VERSION; }
int64_t evt_launch_count(void) { return evt::g_launches; }
void evt_launch_count_reset(void) { evt::g_launches = 0; }
void evt_gemm_set_split_k(int enable) { evt::g_split_k.store(enable != 0, std::memory_order_relaxed); }
void evt_gemm_set_pair_mode(int mode) { evt::g_pair_mode.store(mode < 0 ? -1 : (mode != 0), std::memory_order_relaxed); }

int evt_device_check(void) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return evt::fail(EVT_ERR_CUDA, std::string("cudaGetDevice: ") + cudaGetErrorString(e));
  int major = 0;
  e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (e != cudaSuccess) return evt::fail(EVT_ERR_CUDA, std::string("cudaDeviceGetAttribute: ") + cudaGetErrorString(e));
  if (major != 10)
    return evt::fail(EVT_ERR_UNSUPPORTED, "libevt needs a compute-capability 10.x (sm_100a, B200) device; found major " +
                                              std::to_string(major) + "; there is no CPU or other-GPU fallback");
  return EVT_OK;
}

}  // extern "C"

extern "C" void evt_gemm_weights_static(int delta) { evt::gemm_weights_static_add(delta); }
