// Local (single-device-visible) element-wise kernels:
//   localReduce       dst[i] = dst[i] (op) src[i]   — the building block behind
//                     CudaReductionFunction; 128-bit loads/stores, fp32 accumulate
//                     for fp16/bf16, size_t counts, grid sized to the SM count.
//   localReduceMany   dst = reduce(srcs[0..n)) in one pass (multi-pointer local reduce:
//                     srcs may live on peer devices of the same process).
//   localAllreduceMany every buffer := scale * reduce(all buffers), one pass (fused reduce+broadcast).
//   localBroadcast    copy src to n destinations in one pass.
//   verify            whole-buffer closed-form check on the device (bench / smoke).
//   fill / spin       test helpers (pattern fill; delay kernel that surfaces
//                     missing stream synchronisation).
// Parity: gloo/cuda.cu:274-407 (K1-K5), cuda_private.cu:38-61 (K6),
// test/cuda_base_test.cu:15-27 (K7) — rewritten, not ported: the reference kernels
// are scalar, int-indexed, one element per thread.
#include <cstdio>
#include <string>

#include "glb/common/utils.h"
#include "glb/cuda/device_common.cuh"
#include "glb/cuda/dispatch.cuh"
#include "glb/cuda/kernels.h"

namespace glb {
namespace cuda {

namespace {

constexpr int kLocalThreads = 256;
constexpr int kMaxSrcs = 16;

struct SrcPtrs {
  const void* p[kMaxSrcs];
};
struct DstPtrs {
  void* p[kMaxSrcs];
};

template <typename T>
__global__ void __launch_bounds__(kLocalThreads)
localReduceManyKernel(T* __restrict__ dst, SrcPtrs srcs, int nsrc, size_t count, DevOp op, bool vectorOk) {
  using PT = PackTraits<T>;
  const size_t tid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const size_t nthreads = static_cast<size_t>(gridDim.x) * blockDim.x;
  const size_t nvec = vectorOk ? count / PT::kElems : 0;
  for (size_t v = tid; v < nvec; v += nthreads) {
    typename PT::AccPack acc = PT::widen(ld128_stream(static_cast<const char*>(srcs.p[0]) + v * 16));
    for (int s = 1; s < nsrc; s++) PT::combine(acc, ld128_stream(static_cast<const char*>(srcs.p[s]) + v * 16), op);
    st128(reinterpret_cast<char*>(dst) + v * 16, PT::narrow(acc));
  }
  for (size_t i = nvec * PT::kElems + tid; i < count; i += nthreads) {
    using A = typename AccType<T>::type;
    A acc = toAcc<T>(static_cast<const T*>(srcs.p[0])[i]);
    for (int s = 1; s < nsrc; s++) acc = applyOp<A>(acc, toAcc<T>(static_cast<const T*>(srcs.p[s])[i]), op);
    dst[i] = fromAcc<T, A>(acc);
  }
}

// Fused local allreduce: every one of the n buffers ends up holding scale * reduce(all n),
// in ONE pass (n reads + n writes per element). This is the whole step when a job has a
// single rank with several local pointers (CudaAllreduce* with ptrs.size() > 1, size == 1,
// and CudaAllreduceLocal): previously a reduce pass followed by a broadcast pass.
// U = 128-bit packs per thread and trip (loads of all trips are issued before the first
// store); kTiled: a CTA works on a contiguous tile of U x blockDim packs per trip (fewer DRAM
// pages open at once) instead of striding the whole grid between the U packs.
template <typename T, int U, bool kTiled>
__global__ void __launch_bounds__(kLocalThreads)
localAllreduceManyKernel(DstPtrs bufs, int n, size_t count, DevOp op, float scale, bool vectorOk) {
  using PT = PackTraits<T>;
  const size_t tid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const size_t nthreads = static_cast<size_t>(gridDim.x) * blockDim.x;
  const size_t nvec = vectorOk ? count / PT::kElems : 0;
  const size_t first = kTiled ? static_cast<size_t>(blockIdx.x) * blockDim.x * U + threadIdx.x : tid;
  const size_t inner = kTiled ? blockDim.x : nthreads;  // distance between the U packs of one trip
  for (size_t v0 = first; v0 < nvec; v0 += nthreads * U) {
    typename PT::AccPack acc[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const size_t v = v0 + u * inner;
      if (v < nvec) {
        acc[u] = PT::widen(ld128_stream(static_cast<const char*>(bufs.p[0]) + v * 16));
        for (int s = 1; s < n; s++) PT::combine(acc[u], ld128_stream(static_cast<const char*>(bufs.p[s]) + v * 16), op);
      }
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
      const size_t v = v0 + u * inner;
      if (v < nvec) {
        if (scale != 1.0f) PT::scale(acc[u], scale);
        const Pack16 r = PT::narrow(acc[u]);
        for (int s = 0; s < n; s++) st128_stream(static_cast<char*>(bufs.p[s]) + v * 16, r);
      }
    }
  }
  for (size_t i = nvec * PT::kElems + tid; i < count; i += nthreads) {
    using A = typename AccType<T>::type;
    A acc = toAcc<T>(static_cast<const T*>(bufs.p[0])[i]);
    for (int s = 1; s < n; s++) acc = applyOp<A>(acc, toAcc<T>(static_cast<const T*>(bufs.p[s])[i]), op);
    if (scale != 1.0f) acc = scaleAcc(acc, scale);
    const T res = fromAcc<T, A>(acc);
    for (int s = 0; s < n; s++) static_cast<T*>(bufs.p[s])[i] = res;
  }
}

// Whole-buffer check against the closed form start + stride * i (evaluated in fp64, like
// fillKernel): counts elements outside rtol/atol and remembers the first offender.
template <typename T>
__global__ void verifyKernel(const T* buf, size_t count, double start, double stride, double rtol, double atol,
                             unsigned long long* result /* [0]=mismatches, [1]=first bad index + 1 */) {
  const size_t tid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const size_t nthreads = static_cast<size_t>(gridDim.x) * blockDim.x;
  unsigned long long bad = 0;
  for (size_t i = tid; i < count; i += nthreads) {
    const double want = start + stride * static_cast<double>(i);
    double got;
    if constexpr (std::is_same<T, __half>::value) {
      got = static_cast<double>(__half2float(buf[i]));
    } else if constexpr (std::is_same<T, __nv_bfloat16>::value) {
      got = static_cast<double>(__bfloat162float(buf[i]));
    } else {
      got = static_cast<double>(buf[i]);
    }
    const double err = fabs(got - want);
    if (!(err <= atol + rtol * fabs(want))) {
      bad++;
      atomicMin(&result[1], static_cast<unsigned long long>(i) + 1ull);
    }
  }
  if (bad) atomicAdd(&result[0], bad);
}

__global__ void __launch_bounds__(kLocalThreads)
localBroadcastKernel(DstPtrs dsts, int ndst, const char* __restrict__ src, size_t bytes, bool vectorOk) {
  const size_t tid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const size_t nthreads = static_cast<size_t>(gridDim.x) * blockDim.x;
  const size_t nvec = vectorOk ? bytes / 16 : 0;
  for (size_t v = tid; v < nvec; v += nthreads) {
    const Pack16 p = ld128_stream(src + v * 16);
    for (int d = 0; d < ndst; d++) st128_stream(static_cast<char*>(dsts.p[d]) + v * 16, p);
  }
  for (size_t i = nvec * 16 + tid; i < bytes; i += nthreads) {
    const char c = src[i];
    for (int d = 0; d < ndst; d++) static_cast<char*>(dsts.p[d])[i] = c;
  }
}

template <typename T>
__global__ void fillKernel(T* dst, size_t count, double start, double stride) {
  const size_t tid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const size_t nthreads = static_cast<size_t>(gridDim.x) * blockDim.x;
  for (size_t i = tid; i < count; i += nthreads) {
    const double v = start + stride * static_cast<double>(i);
    if constexpr (std::is_same<T, __half>::value) {
      dst[i] = __float2half_rn(static_cast<float>(v));
    } else if constexpr (std::is_same<T, __nv_bfloat16>::value) {
      dst[i] = __float2bfloat16_rn(static_cast<float>(v));
    } else {
      dst[i] = static_cast<T>(v);
    }
  }
}

__global__ void spinKernel(long long cycles) {
  const long long start = clock64();
  while (clock64() - start < cycles) {
  }
}

// Measured on B200, 2 x 400 MB fp32 (scripts/bench_local.py, profiles/r2/local_shapes.json):
// 4 CTAs/SM x 1 pack 0.269 ms (5.96 TB/s), x 2 packs 0.279, 8 CTAs/SM 0.295, 2 CTAs/SM 0.353.
struct LocalShape {
  int ctasPerSm = 4;
  int unroll = 1;
  bool tiled = false;
};

LocalShape localShapeFromEnv() {
  LocalShape s;
  const std::string v = envStr("LOCAL_SHAPE", "");
  int a = 0, b = 0, c = 0;
  if (!v.empty() && std::sscanf(v.c_str(), "%d,%d,%d", &a, &b, &c) == 3) {
    if (a >= 1 && a <= 8) s.ctasPerSm = a;
    if (b == 1 || b == 2 || b == 4) s.unroll = b;
    s.tiled = c != 0;
  }
  return s;
}

LocalShape& localShape() {
  static LocalShape s = localShapeFromEnv();
  return s;
}

int gridFor(size_t items, int threads, int ctasPerSm = 4) {
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  size_t want = (items + threads - 1) / threads;
  size_t cap = static_cast<size_t>(sms) * static_cast<size_t>(ctasPerSm);
  return static_cast<int>(want < 1 ? 1 : (want > cap ? cap : want));
}

// The instantiation of the fused local allreduce for a launch shape (packs per thread and trip,
// tiled or grid stride); an unroll other than 1 or 4 selects 2.
template <typename T>
const void* localAllreduceFn(int unroll, bool tiled) {
  if (tiled) {
    if (unroll == 4) return fn(localAllreduceManyKernel<T, 4, true>);
    if (unroll == 1) return fn(localAllreduceManyKernel<T, 1, true>);
    return fn(localAllreduceManyKernel<T, 2, true>);
  }
  if (unroll == 4) return fn(localAllreduceManyKernel<T, 4, false>);
  if (unroll == 1) return fn(localAllreduceManyKernel<T, 1, false>);
  return fn(localAllreduceManyKernel<T, 2, false>);
}

bool aligned16(const void* p) { return reinterpret_cast<uintptr_t>(p) % 16 == 0; }

}  // namespace

void launchLocalReduceMany(void* dst, const void* const* srcs, int nsrc, size_t count, DataType dt, ReduceOp op,
                           cudaStream_t stream) {
  if (count == 0 || nsrc == 0) return;
  SrcPtrs sp;
  bool vectorOk = aligned16(dst);
  for (int i = 0; i < nsrc && i < kMaxSrcs; i++) {
    sp.p[i] = srcs[i];
    vectorOk = vectorOk && aligned16(srcs[i]);
  }
  dispatchType(dt, [&](auto tag) {
    using T = decltype(tag);
    const int grid = gridFor(count / PackTraits<T>::kElems + 1, kLocalThreads);
    localReduceManyKernel<T><<<grid, kLocalThreads, 0, stream>>>(static_cast<T*>(dst), sp, nsrc, count,
                                                                static_cast<DevOp>(op), vectorOk);
  });
}

void launchLocalAllreduceMany(void* const* bufs, int n, size_t count, DataType dt, ReduceOp op, float scale,
                              cudaStream_t stream) {
  if (count == 0 || n == 0) return;
  DstPtrs bp;
  bool vectorOk = true;
  for (int i = 0; i < n && i < kMaxSrcs; i++) {
    bp.p[i] = bufs[i];
    vectorOk = vectorOk && aligned16(bufs[i]);
  }
  // Launch shape: measured on B200 (scripts/bench_local.py); GLB_LOCAL_SHAPE = "<ctas per SM>,<unroll>,<tiled>".
  const LocalShape shape = localShape();
  DevOp dop = static_cast<DevOp>(op);
  void* args[] = {&bp, &n, &count, &dop, &scale, &vectorOk};
  dispatchType(dt, [&](auto t) {
    using T = decltype(t);
    const int grid = gridFor(count / PackTraits<T>::kElems / shape.unroll + 1, kLocalThreads, shape.ctasPerSm);
    launchKernel(localAllreduceFn<T>(shape.unroll, shape.tiled), grid, kLocalThreads, args, stream);
  });
}

void launchVerify(const void* buf, size_t count, DataType dt, double start, double stride, double rtol, double atol,
                  unsigned long long* deviceResult, cudaStream_t stream) {
  if (count == 0) return;
  dispatchType(dt, [&](auto tag) {
    using T = decltype(tag);
    verifyKernel<T><<<gridFor(count, 256), 256, 0, stream>>>(static_cast<const T*>(buf), count, start, stride, rtol,
                                                             atol, deviceResult);
  });
}

void launchLocalReduce(void* dst, const void* src, size_t count, DataType dt, ReduceOp op, cudaStream_t stream) {
  const void* srcs[2] = {dst, src};
  launchLocalReduceMany(dst, srcs, 2, count, dt, op, stream);
}

void launchLocalBroadcast(void* const* dsts, int ndst, const void* src, size_t bytes, cudaStream_t stream) {
  if (bytes == 0 || ndst == 0) return;
  DstPtrs dp;
  bool vectorOk = aligned16(src);
  for (int i = 0; i < ndst && i < kMaxSrcs; i++) {
    dp.p[i] = dsts[i];
    vectorOk = vectorOk && aligned16(dsts[i]);
  }
  const int grid = gridFor(bytes / 16 + 1, kLocalThreads);
  localBroadcastKernel<<<grid, kLocalThreads, 0, stream>>>(dp, ndst, static_cast<const char*>(src), bytes, vectorOk);
}

void launchFill(void* dst, size_t count, DataType dt, double start, double stride, cudaStream_t stream) {
  if (count == 0) return;
  dispatchType(dt, [&](auto tag) {
    using T = decltype(tag);
    fillKernel<T><<<gridFor(count, 256), 256, 0, stream>>>(static_cast<T*>(dst), count, start, stride);
  });
}

void launchSpin(long long cycles, cudaStream_t stream) { spinKernel<<<1, 1, 0, stream>>>(cycles); }

void setLocalAllreduceShape(int ctasPerSm, int unroll, bool tiled) {
  LocalShape& s = localShape();
  if (ctasPerSm >= 1 && ctasPerSm <= 8) s.ctasPerSm = ctasPerSm;
  if (unroll == 1 || unroll == 2 || unroll == 4) s.unroll = unroll;
  s.tiled = tiled;
}

void preloadLocalKernels() {
  for (DataType dt : kAllDataTypes) {
    dispatchType(dt, [](auto t) {
      using T = decltype(t);
      touch(fn(localReduceManyKernel<T>));
      touch(fn(verifyKernel<T>));
      touch(fn(fillKernel<T>));
      for (int unroll : {1, 2, 4}) {
        for (bool tiled : {false, true}) touch(localAllreduceFn<T>(unroll, tiled));
      }
    });
  }
  touch(fn(localBroadcastKernel));
  touch(fn(spinKernel));
  cudaGetLastError();
}

}  // namespace cuda
}  // namespace glb
