// Host-side kernel selection shared by the kernel files: the public dtype tag -> device element
// type switch, the list of every dtype, and the helpers that launch or preload a selected
// kernel. A launcher launches exactly the pointer its selector returns, and each
// preload*Kernels() walks the same selectors, so the preloaded set is the launchable set.
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <cstdint>
#include <type_traits>

#include "glb/types.h"

namespace glb {
namespace cuda {

// Every dtype the kernels are instantiated for.
inline constexpr DataType kAllDataTypes[] = {DataType::INT8,    DataType::UINT8,   DataType::INT16,
                                             DataType::INT32,   DataType::UINT32,  DataType::INT64,
                                             DataType::UINT64,  DataType::FLOAT32, DataType::FLOAT64,
                                             DataType::FLOAT16, DataType::BFLOAT16};

// Calls f(T{}) with the device element type T of `dt` and returns what f returns.
template <typename F>
auto dispatchType(DataType dt, F&& f) {
  switch (dt) {
    case DataType::INT8: return f(int8_t{});
    case DataType::UINT8: return f(uint8_t{});
    case DataType::INT16: return f(int16_t{});
    case DataType::INT32: return f(int32_t{});
    case DataType::UINT32: return f(uint32_t{});
    case DataType::INT64: return f((long long){});
    case DataType::UINT64: return f((unsigned long long){});
    case DataType::FLOAT32: return f(float{});
    case DataType::FLOAT64: return f(double{});
    case DataType::FLOAT16: return f(__half{});
    case DataType::BFLOAT16: return f(__nv_bfloat16{});
  }
  return decltype(f(float{}))();
}

// Calls f(TI{}, TO{}) for the supported conversions of the cast epilogue (f32 -> f16 / bf16,
// f16 / bf16 -> f32) and returns what f returns; a default value for any other pair.
template <typename F>
auto dispatchCast(DataType in, DataType out, F&& f) {
  if (in == DataType::FLOAT32 && out == DataType::FLOAT16) return f(float{}, __half{});
  if (in == DataType::FLOAT32 && out == DataType::BFLOAT16) return f(float{}, __nv_bfloat16{});
  if (in == DataType::FLOAT16 && out == DataType::FLOAT32) return f(__half{}, float{});
  if (in == DataType::BFLOAT16 && out == DataType::FLOAT32) return f(__nv_bfloat16{}, float{});
  return decltype(f(float{}, __half{}))();
}

// f32 / f16 / bf16: the types with rank-count specialisations and multicast (NVLS) kernels.
template <typename T>
constexpr bool isHotType() {
  return std::is_same<T, float>::value || std::is_same<T, __half>::value || std::is_same<T, __nv_bfloat16>::value;
}

template <typename K>
const void* fn(K kernel) {
  return reinterpret_cast<const void*>(kernel);
}

inline void launchKernel(const void* kernel, int blocks, int threads, void** args, cudaStream_t stream) {
  cudaLaunchKernel(kernel, dim3(static_cast<unsigned>(blocks)), dim3(static_cast<unsigned>(threads)), args, 0, stream);
}

// Force-load one kernel (nullptr: a selector's "no such kernel"). With CUDA's lazy module
// loading the first launch of a kernel may have to synchronise the context; if a peer rank on
// the same device is already spinning inside its collective kernel that launch never happens
// (documented lazy-loading deadlock for kernels that assume concurrency).
inline void touch(const void* kernel) {
  if (kernel == nullptr) return;
  cudaFuncAttributes attr;
  cudaFuncGetAttributes(&attr, kernel);
}

}  // namespace cuda
}  // namespace glb
