// Device-side building blocks shared by every collective kernel (sm_100a):
//
//  * CommArgs / SignalPad — per-rank signal page mapped into every peer. A kernel
//    synchronises with its peers by storing a monotonically increasing epoch into
//    the peers' pads (st.release.sys) and spinning on its own pad
//    (ld.acquire.sys): this replaces the host-side stream.wait() + notification
//    Buffers of the reference (cuda_allreduce_ring_chunked.cc:177-208).
//  * 16-byte vector packs with fp32 accumulation for 16-bit types and a runtime
//    reduction op (uniform branch; these kernels are link/HBM bound).
//  * multimem.* wrappers for the NVLS (NVSwitch multicast) path.
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <cstdint>
#include <type_traits>

#include "glb/cuda/comm_types.h"
#include "glb/types.h"

namespace glb {
namespace cuda {

enum class DevOp : int { SUM = 1, PRODUCT = 2, MAX = 3, MIN = 4 };

// ---- memory-ordering primitives -------------------------------------------------

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void st_relaxed_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t ld_relaxed_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

__device__ __forceinline__ unsigned long long globalTimerNs() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// ---- failure detection ------------------------------------------------------------
// The reference bounds every wait with the context timeout and turns a silent peer into an
// IoException (transport/tcp/unbound_buffer.cc:52-94). The device-side equivalent: a flag
// wait that exceeds CommArgs::timeoutNs raises the abort word in every rank's pad and in a
// host-mapped status word, after which every barrier returns false at once and the kernels
// run to their end without touching anything else. PeerContext::checkHealth() turns the
// status word into the exception and poisons the context.
// The slow paths take scalars only: handing `const CommArgs&` (a kernel parameter) to a
// non-inlined function would force a copy of the whole struct into local memory in every
// kernel.
// Returns 0 when the flag arrived, kAbortTimeout when the wait timed out (the local abort
// word is raised here), kAbortPeer when somebody else had raised it.
static __device__ __noinline__ uint32_t waitFlagSlow(const uint32_t* flag, uint32_t want, uint32_t* abortWord,
                                                     unsigned long long timeoutNs) {
  const unsigned long long t0 = globalTimerNs();
  uint32_t polls = 0;
  while (static_cast<int32_t>(ld_acquire_sys(flag) - want) < 0) {
    if ((++polls & 127u) == 0u) {
      if (ld_relaxed_sys(abortWord) != 0u) return kAbortPeer;
      if (timeoutNs != 0ull && globalTimerNs() - t0 > timeoutNs) {
        atomicCAS(abortWord, 0u, static_cast<uint32_t>(kAbortTimeout));
        return kAbortTimeout;
      }
    }
  }
  return 0u;
}

// After a failed wait: tell every peer (their waits end early instead of running into their
// own time-out) and the host.
__device__ __forceinline__ void reportAbort(const CommArgs& a, uint32_t code, int missingPeer) {
  if (code == kAbortTimeout) {
    a.self->abortRank = static_cast<uint32_t>(missingPeer);
    for (int r = 0; r < a.nranks; r++) {
      if (r != a.rank) st_relaxed_sys(&a.sig[r]->abort, static_cast<uint32_t>(kAbortPeer));
    }
  }
  if (a.hostStatus != nullptr && ld_relaxed_sys(a.hostStatus) == 0u) {
    st_relaxed_sys(a.hostStatus, code | (static_cast<uint32_t>(missingPeer) << 8));
  }
  __threadfence_system();
}

// Spin until *flag has reached `want` (wrap-safe). Returns false when the wait was abandoned.
__device__ __forceinline__ bool waitFlag(const CommArgs& a, const uint32_t* flag, uint32_t want, int peer) {
  if (static_cast<int32_t>(ld_acquire_sys(flag) - want) >= 0) return true;
  const uint32_t rc = waitFlagSlow(flag, want, &a.self->abort, a.timeoutNs);
  if (rc == 0u) return true;
  reportAbort(a, rc, peer);
  return false;
}

// All CTAs with the same blockIdx on every rank rendezvous. Everything the
// callers wrote before (including stores into peer memory) is visible to every
// peer's block after it returns (bar.sync + cumulative release/acquire at .sys).
// kRelease=false is for the FIRST barrier of a kernel that has not written anything a
// peer will read: "my kernel has started" needs no fence (the inputs were produced by
// earlier kernels and are already visible system-wide), which saves a MEMBAR.SYS.
// Returns false (on every thread of the CTA) when a peer did not show up in time.
template <bool kRelease = true>
__device__ __forceinline__ bool blockBarrier(const CommArgs& a, uint32_t epoch) {
  __syncthreads();
  int ok = 1;
  if (threadIdx.x < a.nranks) {
    const int peer = threadIdx.x;
    if (kRelease) {
      st_release_sys(&a.sig[peer]->flag[blockIdx.x][a.rank], epoch);
    } else {
      st_relaxed_sys(&a.sig[peer]->flag[blockIdx.x][a.rank], epoch);
    }
    ok = waitFlag(a, &a.self->flag[blockIdx.x][peer], epoch, peer) ? 1 : 0;
  }
  return __syncthreads_and(ok) != 0;
}

// Read the epoch at kernel entry (all CTAs see the same value: it only changes
// when the LAST CTA of a launch retires, after every CTA has read it).
__device__ __forceinline__ uint32_t loadEpoch(const CommArgs& a) { return ld_relaxed_sys(&a.self->epoch); }

// Called by every CTA at the very end; the last one publishes the new counters.
__device__ __forceinline__ void retire(const CommArgs& a, uint32_t barriersUsed, uint32_t stagedLaunch,
                                       uint32_t llLaunch = 0) {
  __syncthreads();
  if (threadIdx.x == 0) {
    SignalPad* me = a.self;
    // No fences: the ticket is an L2 atomic (the last CTA sees every earlier arrival) and
    // the counters are next read by the NEXT launch, after this kernel has retired.
    uint32_t ticket = atomicAdd(&me->done, 1u);
    if (ticket == gridDim.x - 1) {
      me->done = 0;
      me->epoch += barriersUsed;
      me->stageSeq += stagedLaunch;
      me->llSeq += llLaunch;
    }
  }
}

// ---- flag-in-data ("LL") lines ------------------------------------------------------
// A 16-byte line carries 8 bytes of payload and two copies of the launch's sequence
// number: {d0, seq, d1, seq}. Each 8-byte half is written atomically, so a reader that
// sees both flags equal to `seq` has both payload words; no barrier and no MEMBAR.SYS on
// the critical path (one posted store + one poll).
__device__ __forceinline__ void llStore(void* p, uint32_t d0, uint32_t d1, uint32_t seq) {
  asm volatile("st.volatile.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(d0), "r"(seq), "r"(d1), "r"(seq) : "memory");
}
__device__ __forceinline__ bool llTryLoad(const void* p, uint32_t seq, uint32_t& d0, uint32_t& d1) {
  uint32_t f0, f1;
  asm volatile("ld.volatile.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(d0), "=r"(f0), "=r"(d1), "=r"(f1) : "l"(p) : "memory");
  return f0 == seq && f1 == seq;
}
static __device__ __noinline__ uint32_t llLoadSlow(const void* p, uint32_t seq, uint32_t& d0, uint32_t& d1,
                                                   uint32_t* abortWord, unsigned long long timeoutNs) {
  const unsigned long long t0 = globalTimerNs();
  uint32_t polls = 0;
  while (!llTryLoad(p, seq, d0, d1)) {
    if ((++polls & 127u) == 0u) {
      if (ld_relaxed_sys(abortWord) != 0u) return kAbortPeer;
      if (timeoutNs != 0ull && globalTimerNs() - t0 > timeoutNs) {
        atomicCAS(abortWord, 0u, static_cast<uint32_t>(kAbortTimeout));
        return kAbortTimeout;
      }
    }
  }
  return 0u;
}
__device__ __forceinline__ bool llLoad(const CommArgs& a, const void* p, uint32_t seq, uint32_t& d0, uint32_t& d1, int peer) {
  if (llTryLoad(p, seq, d0, d1)) return true;
  const uint32_t rc = llLoadSlow(p, seq, d0, d1, &a.self->abort, a.timeoutNs);
  if (rc == 0u) return true;
  reportAbort(a, rc, peer);
  return false;
}

// ---- 16-byte packs ----------------------------------------------------------------

struct alignas(16) Pack16 {
  uint32_t w[4];
};

__device__ __forceinline__ Pack16 ld128(const void* p) {
  Pack16 v;
  asm volatile("ld.global.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.w[0]), "=r"(v.w[1]), "=r"(v.w[2]), "=r"(v.w[3])
               : "l"(p)
               : "memory");
  return v;
}
// Streaming variants: do not allocate in L1 (peer / single-use data).
__device__ __forceinline__ Pack16 ld128_stream(const void* p) {
  Pack16 v;
  asm volatile("ld.global.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.w[0]), "=r"(v.w[1]), "=r"(v.w[2]), "=r"(v.w[3])
               : "l"(p)
               : "memory");
  return v;
}
__device__ __forceinline__ void st128(void* p, const Pack16& v) {
  asm volatile("st.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.w[0]), "r"(v.w[1]), "r"(v.w[2]), "r"(v.w[3])
               : "memory");
}
__device__ __forceinline__ void st128_stream(void* p, const Pack16& v) {
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.w[0]), "r"(v.w[1]),
               "r"(v.w[2]), "r"(v.w[3])
               : "memory");
}

template <typename T>
__device__ __forceinline__ T applyOp(T a, T b, DevOp op) {
  switch (op) {
    case DevOp::SUM: return a + b;
    case DevOp::PRODUCT: return a * b;
    case DevOp::MAX: return b > a ? b : a;
    default: return b < a ? b : a;
  }
}

// ---- one element at a time ---------------------------------------------------------------
// The scalar paths (sub-pack tails, unaligned buffers, uneven shares) follow the same rule as
// the packs: widen to AccType<T>, reduce and scale there, round once with fromAcc. AccType is
// T itself for every type but the 16-bit floats, so integer / f32 / f64 arithmetic is plain T.
template <typename T>
struct AccType {
  using type = T;
};
template <>
struct AccType<__half> {
  using type = float;
};
template <>
struct AccType<__nv_bfloat16> {
  using type = float;
};

template <typename T>
__device__ __forceinline__ typename AccType<T>::type toAcc(T x) {
  return x;
}
template <>
__device__ __forceinline__ float toAcc<__half>(__half x) {
  return __half2float(x);
}
template <>
__device__ __forceinline__ float toAcc<__nv_bfloat16>(__nv_bfloat16 x) {
  return __bfloat162float(x);
}
template <typename TO, typename A>
__device__ __forceinline__ TO fromAcc(A x) {
  return static_cast<TO>(x);
}
template <>
__device__ __forceinline__ __half fromAcc<__half, float>(float x) {
  return __float2half_rn(x);
}
template <>
__device__ __forceinline__ __nv_bfloat16 fromAcc<__nv_bfloat16, float>(float x) {
  return __float2bfloat16_rn(x);
}
// Epilogue on an accumulator (floating types only; the host rejects a scale on integers).
template <typename A>
__device__ __forceinline__ A scaleAcc(A x, float s) {
  if constexpr (std::is_floating_point<A>::value) return static_cast<A>(x * s);
  return x;
}

// combineOne / scaleOne round to T after every step. Only the literal schedules use them:
// they store each step's partial in T by design. Fused kernels round once (above).
template <typename T>
__device__ __forceinline__ T combineOne(T a, T b, DevOp op) {
  using A = typename AccType<T>::type;
  return fromAcc<T, A>(applyOp<A>(toAcc<T>(a), toAcc<T>(b), op));
}
template <typename T>
__device__ __forceinline__ T scaleOne(T a, float s) {
  return fromAcc<T>(scaleAcc(toAcc<T>(a), s));
}

// Accumulator traits: how one 16-byte pack of T is widened, combined, narrowed.
template <typename T>
struct PackTraits {
  static constexpr int kElems = 16 / sizeof(T);
  using Acc = T;
  struct AccPack {
    T v[kElems];
  };
  __device__ static AccPack widen(const Pack16& p) {
    AccPack a;
    const T* t = reinterpret_cast<const T*>(&p);
#pragma unroll
    for (int i = 0; i < kElems; i++) a.v[i] = t[i];
    return a;
  }
  __device__ static void combine(AccPack& a, const Pack16& p, DevOp op) {
    const T* t = reinterpret_cast<const T*>(&p);
#pragma unroll
    for (int i = 0; i < kElems; i++) a.v[i] = applyOp<T>(a.v[i], t[i], op);
  }
  __device__ static Pack16 narrow(const AccPack& a) {
    Pack16 p;
    T* t = reinterpret_cast<T*>(&p);
#pragma unroll
    for (int i = 0; i < kElems; i++) t[i] = a.v[i];
    return p;
  }
  // Epilogue: multiply the reduced value (floating types only; the host rejects a scale
  // on integer buffers).
  __device__ static void scale(AccPack& a, float s) {
    if constexpr (std::is_floating_point<T>::value) {
#pragma unroll
      for (int i = 0; i < kElems; i++) a.v[i] = static_cast<T>(a.v[i] * s);
    }
  }
};

template <>
struct PackTraits<__half> {
  static constexpr int kElems = 8;
  struct AccPack {
    float v[8];
  };
  __device__ static AccPack widen(const Pack16& p) {
    AccPack a;
    const __half2* h = reinterpret_cast<const __half2*>(&p);
#pragma unroll
    for (int i = 0; i < 4; i++) {
      float2 f = __half22float2(h[i]);
      a.v[2 * i] = f.x;
      a.v[2 * i + 1] = f.y;
    }
    return a;
  }
  __device__ static void combine(AccPack& a, const Pack16& p, DevOp op) {
    const __half2* h = reinterpret_cast<const __half2*>(&p);
#pragma unroll
    for (int i = 0; i < 4; i++) {
      float2 f = __half22float2(h[i]);
      a.v[2 * i] = applyOp<float>(a.v[2 * i], f.x, op);
      a.v[2 * i + 1] = applyOp<float>(a.v[2 * i + 1], f.y, op);
    }
  }
  __device__ static Pack16 narrow(const AccPack& a) {
    Pack16 p;
    __half2* h = reinterpret_cast<__half2*>(&p);
#pragma unroll
    for (int i = 0; i < 4; i++) h[i] = __floats2half2_rn(a.v[2 * i], a.v[2 * i + 1]);
    return p;
  }
  __device__ static void scale(AccPack& a, float s) {
#pragma unroll
    for (int i = 0; i < 8; i++) a.v[i] *= s;
  }
};

template <>
struct PackTraits<__nv_bfloat16> {
  static constexpr int kElems = 8;
  struct AccPack {
    float v[8];
  };
  __device__ static AccPack widen(const Pack16& p) {
    AccPack a;
    // bf16 -> fp32 is a 16-bit shift.
#pragma unroll
    for (int i = 0; i < 4; i++) {
      a.v[2 * i] = __uint_as_float(p.w[i] << 16);
      a.v[2 * i + 1] = __uint_as_float(p.w[i] & 0xffff0000u);
    }
    return a;
  }
  __device__ static void combine(AccPack& a, const Pack16& p, DevOp op) {
#pragma unroll
    for (int i = 0; i < 4; i++) {
      a.v[2 * i] = applyOp<float>(a.v[2 * i], __uint_as_float(p.w[i] << 16), op);
      a.v[2 * i + 1] = applyOp<float>(a.v[2 * i + 1], __uint_as_float(p.w[i] & 0xffff0000u), op);
    }
  }
  __device__ static Pack16 narrow(const AccPack& a) {
    Pack16 p;
    __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&p);
#pragma unroll
    for (int i = 0; i < 4; i++) h[i] = __floats2bfloat162_rn(a.v[2 * i], a.v[2 * i + 1]);
    return p;
  }
  __device__ static void scale(AccPack& a, float s) {
#pragma unroll
    for (int i = 0; i < 8; i++) a.v[i] *= s;
  }
};

// ---- mixed-precision items (cast epilogue) --------------------------------------------
// Eight consecutive elements of T as fp32 lanes: 2 x 16 B for float, 1 x 16 B for the
// 16-bit types. Used by the kernels whose output dtype differs from the input dtype
// (fp32 accumulate -> bf16/fp16 store, or 16-bit inputs -> fp32 result). `widen` turns
// kPacks raw packs into the lanes, for kernels that issue all their loads before using them.
// `store<false>` stores with plain st.global (no L1::no_allocate) for a local output that is
// read again soon, as the same-dtype reduce_scatter does.
template <typename T>  // __half, __nv_bfloat16
struct Item8 {
  static constexpr int kBytes = 16;
  static constexpr int kPacks = 1;
  __device__ static void widen(const Pack16 (&p)[kPacks], float (&v)[8]) {
    const auto a = PackTraits<T>::widen(p[0]);
#pragma unroll
    for (int i = 0; i < 8; i++) v[i] = a.v[i];
  }
  __device__ static void load(const void* p, float (&v)[8]) {
    const auto a = PackTraits<T>::widen(ld128_stream(p));
#pragma unroll
    for (int i = 0; i < 8; i++) v[i] = a.v[i];
  }
  template <bool kStream = true>
  __device__ static void store(void* p, const float (&v)[8]) {
    typename PackTraits<T>::AccPack a;
#pragma unroll
    for (int i = 0; i < 8; i++) a.v[i] = v[i];
    if constexpr (kStream) {
      st128_stream(p, PackTraits<T>::narrow(a));
    } else {
      st128(p, PackTraits<T>::narrow(a));
    }
  }
};
template <>
struct Item8<float> {
  static constexpr int kBytes = 32;
  static constexpr int kPacks = 2;
  __device__ static void widen(const Pack16 (&p)[kPacks], float (&v)[8]) {
#pragma unroll
    for (int i = 0; i < 4; i++) {
      v[i] = __uint_as_float(p[0].w[i]);
      v[4 + i] = __uint_as_float(p[1].w[i]);
    }
  }
  __device__ static void load(const void* p, float (&v)[8]) {
    const Pack16 a = ld128_stream(p), b = ld128_stream(static_cast<const char*>(p) + 16);
#pragma unroll
    for (int i = 0; i < 4; i++) {
      v[i] = __uint_as_float(a.w[i]);
      v[4 + i] = __uint_as_float(b.w[i]);
    }
  }
  template <bool kStream = true>
  __device__ static void store(void* p, const float (&v)[8]) {
    Pack16 a, b;
#pragma unroll
    for (int i = 0; i < 4; i++) {
      a.w[i] = __float_as_uint(v[i]);
      b.w[i] = __float_as_uint(v[4 + i]);
    }
    if constexpr (kStream) {
      st128_stream(p, a);
      st128_stream(static_cast<char*>(p) + 16, b);
    } else {
      st128(p, a);
      st128(static_cast<char*>(p) + 16, b);
    }
  }
};

// ---- NVLS (multimem) --------------------------------------------------------------
// ld_reduce returns the reduction of the same address across every GPU bound to
// the multicast object (performed inside the NVSwitch); st broadcasts to all.

template <typename T>
struct Multimem;  // only add for float / half / bf16; min/max for half/bf16

template <>
struct Multimem<float> {
  __device__ static Pack16 ldReduceAdd(const void* mc) {
    Pack16 v;
    asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(v.w[0]), "=r"(v.w[1]), "=r"(v.w[2]), "=r"(v.w[3])
                 : "l"(mc)
                 : "memory");
    return v;
  }
};
template <>
struct Multimem<__half> {
  __device__ static Pack16 ldReduceAdd(const void* mc) {
    Pack16 v;
    asm volatile("multimem.ld_reduce.relaxed.sys.global.add.acc::f32.v4.f16x2 {%0,%1,%2,%3}, [%4];"
                 : "=r"(v.w[0]), "=r"(v.w[1]), "=r"(v.w[2]), "=r"(v.w[3])
                 : "l"(mc)
                 : "memory");
    return v;
  }
};
template <>
struct Multimem<__nv_bfloat16> {
  __device__ static Pack16 ldReduceAdd(const void* mc) {
    Pack16 v;
    asm volatile("multimem.ld_reduce.relaxed.sys.global.add.acc::f32.v4.bf16x2 {%0,%1,%2,%3}, [%4];"
                 : "=r"(v.w[0]), "=r"(v.w[1]), "=r"(v.w[2]), "=r"(v.w[3])
                 : "l"(mc)
                 : "memory");
    return v;
  }
};

__device__ __forceinline__ void multimemSt128(void* mc, const Pack16& v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(mc), "r"(v.w[0]), "r"(v.w[1]),
               "r"(v.w[2]), "r"(v.w[3])
               : "memory");
}

// ---- building blocks of the fused kernels ---------------------------------------------------

// [begin, end) of rank r's share of n items.
__device__ __forceinline__ void shareOf(size_t n, int parts, int r, size_t& begin, size_t& end) {
  const size_t base = n / parts, rem = n % parts;
  begin = r * base + (static_cast<size_t>(r) < rem ? r : rem);
  end = begin + base + (static_cast<size_t>(r) < rem ? 1 : 0);
}

// Element groups. The barrier pairs CTA b of one rank with CTA b of every peer, so which CTA
// touches which element must not depend on anything rank-local (such as the alignment of a
// user pointer). The staged kernels therefore own 16-byte *groups* of elements by index; a
// group is moved with one 128-bit access when the pointer allows it and element by element
// otherwise (zero padded past `count`).
template <typename T>
__device__ __forceinline__ Pack16 loadGroup(const T* base, size_t g, size_t count, bool aligned) {
  constexpr int K = 16 / sizeof(T);
  const size_t i0 = g * K;
  if (aligned && i0 + K <= count) return ld128_stream(reinterpret_cast<const char*>(base) + g * 16);
  Pack16 p;
  p.w[0] = p.w[1] = p.w[2] = p.w[3] = 0u;
  T* t = reinterpret_cast<T*>(&p);
#pragma unroll
  for (int k = 0; k < K; k++) {
    if (i0 + k < count) t[k] = base[i0 + k];
  }
  return p;
}

// kStream: the 128-bit store does not allocate in L1 (st128_stream) instead of st128.
template <bool kStream, typename T>
__device__ __forceinline__ void storeGroup(T* base, size_t g, size_t count, bool aligned, const Pack16& p) {
  constexpr int K = 16 / sizeof(T);
  const size_t i0 = g * K;
  if (aligned && i0 + K <= count) {
    if constexpr (kStream) {
      st128_stream(reinterpret_cast<char*>(base) + g * 16, p);
    } else {
      st128(reinterpret_cast<char*>(base) + g * 16, p);
    }
    return;
  }
  const T* t = reinterpret_cast<const T*>(&p);
#pragma unroll
  for (int k = 0; k < K; k++) {
    if (i0 + k < count) base[i0 + k] = t[k];
  }
}

template <typename T>
__device__ __forceinline__ Pack16 scalePack(const Pack16& p, float s) {
  using PT = PackTraits<T>;
  typename PT::AccPack acc = PT::widen(p);
  PT::scale(acc, s);
  return PT::narrow(acc);
}

// In place over peer pointers: pack v of the P buffers peer[0..P) is loaded from all of them,
// reduced in peer order, scaled, rounded once and stored to all of them, for v in [vb, ve),
// U packs per thread and trip (kSlots x U independent 128-bit loads in flight).
template <typename T, int kSlots, int U>
__device__ __forceinline__ void peerAllreducePacks(char* const (&peer)[kSlots], int P, size_t vb, size_t ve, DevOp op,
                                                   float scale, size_t tid, size_t nthreads) {
  using PT = PackTraits<T>;
  for (size_t v0 = vb + tid; v0 < ve; v0 += nthreads * U) {
    Pack16 p[U][kSlots];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const size_t v = v0 + static_cast<size_t>(u) * nthreads;
      if (v < ve) {
#pragma unroll
        for (int i = 0; i < kSlots; i++) {
          if (i < P) p[u][i] = ld128_stream(peer[i] + v * 16);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
      const size_t v = v0 + static_cast<size_t>(u) * nthreads;
      if (v < ve) {
        typename PT::AccPack acc = PT::widen(p[u][0]);
#pragma unroll
        for (int i = 1; i < kSlots; i++) {
          if (i < P) PT::combine(acc, p[u][i], op);
        }
        if (scale != 1.0f) PT::scale(acc, scale);
        const Pack16 res = PT::narrow(acc);
#pragma unroll
        for (int i = 0; i < kSlots; i++) {
          if (i < P) st128_stream(peer[i] + v * 16, res);
        }
      }
    }
  }
}

// Element tail of the in-place allreduce (count not a multiple of the pack width, or
// unaligned buffers): rank `rank`'s share of [tailStart, count), reduced across the P buffers
// in AccType<T>, scaled, rounded once and stored to all P.
template <typename T>
__device__ __forceinline__ void allreduceTailInPlace(const PeerPtrs& bufs, int P, int rank, size_t tailStart,
                                                     size_t count, DevOp op, float scale, size_t tid,
                                                     size_t nthreads) {
  using A = typename AccType<T>::type;
  size_t tb, te;
  shareOf(count - tailStart, P, rank, tb, te);
  for (size_t i = tailStart + tb + tid; i < tailStart + te; i += nthreads) {
    A acc = toAcc<T>(static_cast<const T*>(bufs.p[0])[i]);
    for (int r = 1; r < P; r++) acc = applyOp<A>(acc, toAcc<T>(static_cast<const T*>(bufs.p[r])[i]), op);
    if (scale != 1.0f) acc = scaleAcc(acc, scale);
    const T res = fromAcc<T, A>(acc);
    for (int r = 0; r < P; r++) static_cast<T*>(bufs.p[r])[i] = res;
  }
}

}  // namespace cuda
}  // namespace glb
