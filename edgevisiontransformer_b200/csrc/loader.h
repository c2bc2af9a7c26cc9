// Weight loading shared by the model runtimes: the caller's f32 device tensors, looked up by name, are copied or converted into
// device allocations the model owns, all on one stream.  Defined in model.cu, next to the conversion kernels.
#pragma once
#include <cuda_bf16.h>

#include <map>
#include <string>
#include <vector>

#include "common.h"

namespace evt {

struct Loader {
  std::vector<void*>* allocs;  // the model's allocations, freed when it is destroyed
  cudaStream_t st;
  int es;  // bytes per GEMM operand element: 2 (bf16) or 4 (f32 holding tf32 values)
  std::map<std::string, const evt_tensor_view*> by_name = {};

  int index(const evt_tensor_view* tensors, int n);  // every view needs a name and rank 1..4
  const evt_tensor_view* find(const std::string& name) const;
  int need(const std::string& name, int64_t n, const evt_tensor_view** out) const;  // present, with data and n elements
  int alloc(size_t bytes, void** out);
  // f32 copy of a vector / table; zero-filled when `optional` and absent
  int vec_into(const std::string& name, int64_t n, bool optional, float* dst);
  int vec(const std::string& name, int64_t n, bool optional, float** out);
  // operand-typed [rows, ld] from f32 [rows, cols], zero padded
  int mat_into(const std::string& name, int64_t rows, int cols, int ld, void* dst);
  template <typename T>
  int mat(const std::string& name, int64_t rows, int cols, int ld, T** out) {
    void* p;
    EVT_TRY(alloc(static_cast<size_t>(rows) * ld * es, &p));
    *out = static_cast<T*>(p);
    return mat_into(name, rows, cols, ld, p);
  }
  // bf16 [rows_out, ld] from an f32 Keras kernel [cols_out, rows_out]
  int mat_t(const std::string& name, int rows_out, int cols_out, int ld, __nv_bfloat16** out);
  template <typename T>
  int upload(const std::vector<T>& h, T** out) {
    void* p;
    EVT_TRY(alloc(h.size() * sizeof(T), &p));
    EVT_CUDA(cudaMemcpyAsync(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, st));
    EVT_CUDA(cudaStreamSynchronize(st));  // the host vector goes out of scope
    *out = static_cast<T*>(p);
    return EVT_OK;
  }
  int host_copy(const std::string& name, int64_t n, std::vector<float>* out);
};

}  // namespace evt
