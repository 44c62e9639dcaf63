// Fused allreduce kernels over NVLink peer memory (sm_100a).
//
//   barrierKernel        flag barrier only.
//   llAllreduce          smallest messages. Flag-in-data ("LL") protocol: every rank stores
//                        its contribution as 16-byte {d0,seq,d1,seq} lines straight into
//                        every peer's pool and polls its own pool for the peers' lines: one
//                        posted NVLink store and one poll on the critical path, no barrier
//                        round, no MEMBAR.SYS.
//   oneShotAllreduce     latency regime above that. Each rank stages its input in its own
//                        symmetric pool (double-buffered by launch parity), one flag
//                        barrier, then every rank reads all P staged copies over NVLink,
//                        reduces in registers (fp32 accumulate for 16-bit types) and writes
//                        its output; a push flavour stores into the peers instead.
//   twoShotAllreduce     bandwidth regime, in place on peer-mapped user buffers.
//                        Rank r owns chunk r: it loads that chunk from all P
//                        buffers (reduce-scatter by direct peer reads), reduces,
//                        and immediately stores the result into all P buffers
//                        (allgather by direct peer writes) — reduce, scatter and
//                        gather fused in one pass; 2·S·(P-1)/P bytes per GPU in
//                        two hops instead of the ring's 2(P-1).
//   nvlsAllreduce        same ownership, but the reduction happens inside the
//                        NVSwitch: multimem.ld_reduce pulls the switch-reduced
//                        chunk, multimem.st broadcasts it; ~S(1+1/P) per direction.
//   castAllreduce        two-shot / NVLS with an output dtype different from the input dtype
//                        (fp32 accumulate -> bf16/fp16 store, or 16-bit in -> fp32 out).
//
// Every variant applies the epilogue `scale` (AVG = 1/P, loss scaling, ...) to the fp32
// accumulator before the single final rounding, and — when a rank passes several local
// pointers — folds them in the same launch (LocalPtrs): no separate elementwise kernel
// runs before or after the collective.
//
// There is no reference counterpart: the reference stages through pinned host
// memory + TCP (cuda_allreduce_ring_chunked.cc:129-273) and reduces on the CPU.
#include "glb/cuda/device_common.cuh"
#include "glb/cuda/dispatch.cuh"
#include "glb/cuda/kernels.h"

namespace glb {
namespace cuda {

__global__ void barrierKernel(CommArgs a) {
  const uint32_t e = loadEpoch(a);
  blockBarrier(a, e + 1);
  retire(a, 1, 0);
}

// Group g of the local contribution: the first pointer, plus the extra local pointers
// folded in (multi-pointer classes) — the fold costs no extra pass.
template <typename T>
__device__ __forceinline__ Pack16 loadLocalGroup(const T* in, const LocalPtrs& extra, size_t g, size_t count,
                                                 bool aligned, DevOp op) {
  using PT = PackTraits<T>;
  Pack16 p = loadGroup(in, g, count, aligned);
  if (extra.n > 0) {
    typename PT::AccPack acc = PT::widen(p);
    for (int k = 0; k < extra.n; k++) PT::combine(acc, loadGroup(static_cast<const T*>(extra.p[k]), g, count, aligned), op);
    p = PT::narrow(acc);
  }
  return p;
}

template <typename T>
__device__ __forceinline__ void storeLocalGroup(T* out, const LocalPtrs& extra, size_t g, size_t count, bool aligned,
                                                const Pack16& p) {
  storeGroup<false>(out, g, count, aligned, p);
  for (int k = 0; k < extra.n; k++) storeGroup<false>(static_cast<T*>(extra.p[k]), g, count, aligned, p);
}

// ---- LL (flag in data) -------------------------------------------------------------------

// `ll.p[r]` is the LL region of rank r's pool: [parity][source rank][line]. A launch uses
// parity = seq & 1; two halves suffice because a rank can run at most one launch ahead of
// its slowest peer (it needs that peer's lines of launch s+1 to finish launch s+1).
// Latency-critical: every loop over ranks / extra pointers is unrolled over a constant range
// with a guard, so kernel parameters are only ever indexed with constants (a dynamic index
// would make the compiler copy the parameter structs to local memory at kernel entry).
template <typename T, typename TO>
__global__ void __launch_bounds__(kThreads)
llAllreduceKernel(CommArgs a, const T* in, TO* out, size_t count, DevOp op, float scale, PeerPtrs ll, char* myLL,
                  size_t srcStride, size_t parityStride, LocalPtrs extra) {
  constexpr int K = 8 / sizeof(T);
  using A = typename AccType<T>::type;
  const uint32_t seq = ld_relaxed_sys(&a.self->llSeq) + 1u;
  const size_t base = (seq & 1u) * parityStride;
  const size_t tid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const size_t nthreads = static_cast<size_t>(gridDim.x) * blockDim.x;
  const size_t nunits = (count + K - 1) / K;
  const int P = a.nranks;
  const int me = a.rank;
  const char* myRegion = myLL + base;
  const size_t mySlot = base + static_cast<size_t>(me) * srcStride;
  const bool inAligned = reinterpret_cast<uintptr_t>(in) % 8 == 0;
  bool alive = true;

  for (size_t u = tid; u < nunits && alive; u += nthreads) {
    const size_t i0 = u * K;
    // my 8 bytes (zero padded past the end; extra local pointers folded in)
    uint32_t w[2] = {0u, 0u};
    T* t = reinterpret_cast<T*>(w);
    if (inAligned && i0 + K <= count) {
      const uint2 v = *reinterpret_cast<const uint2*>(reinterpret_cast<const char*>(in) + u * 8);
      w[0] = v.x;
      w[1] = v.y;
    } else {
#pragma unroll
      for (int k = 0; k < K; k++) {
        if (i0 + k < count) t[k] = in[i0 + k];
      }
    }
    if constexpr (std::is_same<A, T>::value) {
      if (extra.n > 0) {
#pragma unroll
        for (int e = 0; e < kMaxLocal; e++) {
          if (e < extra.n) {
            const T* x = static_cast<const T*>(extra.p[e]);
#pragma unroll
            for (int k = 0; k < K; k++) {
              if (i0 + k < count) t[k] = applyOp<T>(t[k], x[i0 + k], op);
            }
          }
        }
      }
    } else if (extra.n > 0) {
      // the local fold is stored in T (peers read it): accumulate in A, round once
      A f[K];
#pragma unroll
      for (int k = 0; k < K; k++) f[k] = toAcc<T>(t[k]);
#pragma unroll
      for (int e = 0; e < kMaxLocal; e++) {
        if (e < extra.n) {
          const T* x = static_cast<const T*>(extra.p[e]);
#pragma unroll
          for (int k = 0; k < K; k++) {
            if (i0 + k < count) f[k] = applyOp<A>(f[k], toAcc<T>(x[i0 + k]), op);
          }
        }
      }
#pragma unroll
      for (int k = 0; k < K; k++) {
        if (i0 + k < count) t[k] = fromAcc<T, A>(f[k]);
      }
    }
    // push to every peer: posted NVLink stores, no round trip
#pragma unroll
    for (int r = 0; r < kMaxRanks; r++) {
      if (r < P && r != me) llStore(static_cast<char*>(ll.p[r]) + mySlot + u * 16, w[0], w[1], seq);
    }
    // gather in rank order: every rank sums in the same order -> bit-identical results
    A acc[K];
#pragma unroll
    for (int k = 0; k < K; k++) acc[k] = A(0);
#pragma unroll
    for (int r = 0; r < kMaxRanks; r++) {
      if (r < P && alive) {
        uint32_t d[2];
        if (r == me) {
          d[0] = w[0];
          d[1] = w[1];
        } else if (!llLoad(a, myRegion + static_cast<size_t>(r) * srcStride + u * 16, seq, d[0], d[1], r)) {
          alive = false;
        }
        if (alive) {
          const T* x = reinterpret_cast<const T*>(d);
          if (r == 0) {
#pragma unroll
            for (int k = 0; k < K; k++) acc[k] = toAcc<T>(x[k]);
          } else {
#pragma unroll
            for (int k = 0; k < K; k++) acc[k] = applyOp<A>(acc[k], toAcc<T>(x[k]), op);
          }
        }
      }
    }
    if (!alive) break;
    if (scale != 1.0f) {
      if constexpr (std::is_floating_point<A>::value) {
#pragma unroll
        for (int k = 0; k < K; k++) acc[k] = static_cast<A>(acc[k] * scale);
      }
    }
#pragma unroll
    for (int k = 0; k < K; k++) {
      if (i0 + k < count) {
        const TO o = fromAcc<TO, A>(acc[k]);
        out[i0 + k] = o;
        if constexpr (std::is_same<T, TO>::value) {
          if (extra.n > 0) {
#pragma unroll
            for (int e = 0; e < kMaxLocal; e++) {
              if (e < extra.n) static_cast<TO*>(extra.p[e])[i0 + k] = o;
            }
          }
        }
      }
    }
  }
  // Publish the new sequence number. A single-CTA launch needs no completion ticket.
  if (gridDim.x == 1) {
    __syncthreads();
    if (threadIdx.x == 0) a.self->llSeq = seq;
  } else {
    retire(a, 0, 0, 1);
  }
}

// Small reduce_scatter with the same protocol: rank r ships slice j of its input straight to
// rank j as LL lines and reduces the P contributions to its own slice (rank order). Every
// rank hears from every peer, so the two-parity argument of the LL allreduce holds.
template <typename T>
__global__ void __launch_bounds__(kThreads)
llReduceScatterKernel(CommArgs a, const T* in, T* out, size_t per, DevOp op, float scale, PeerPtrs ll, char* myLL,
                      size_t srcStride, size_t parityStride) {
  constexpr int K = 8 / sizeof(T);
  using A = typename AccType<T>::type;
  const uint32_t seq = ld_relaxed_sys(&a.self->llSeq) + 1u;
  const size_t base = (seq & 1u) * parityStride;
  const size_t tid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const size_t nthreads = static_cast<size_t>(gridDim.x) * blockDim.x;
  const size_t nunits = (per + K - 1) / K;
  const int P = a.nranks;
  const int me = a.rank;
  const size_t mySlot = base + static_cast<size_t>(me) * srcStride;
  // send: item = (destination j, unit u)
  for (size_t it = tid; it < static_cast<size_t>(P) * nunits; it += nthreads) {
    const int j = static_cast<int>(it / nunits);
    if (j == me) continue;
    const size_t u = it % nunits;
    uint32_t w[2] = {0u, 0u};
    T* t = reinterpret_cast<T*>(w);
#pragma unroll
    for (int k = 0; k < K; k++) {
      if (u * K + k < per) t[k] = in[static_cast<size_t>(j) * per + u * K + k];
    }
    llStore(static_cast<char*>(ll.p[j]) + mySlot + u * 16, w[0], w[1], seq);
  }
  // reduce my slice
  const char* myRegion = myLL + base;
  bool alive = true;
  for (size_t u = tid; u < nunits && alive; u += nthreads) {
    A acc[K];
#pragma unroll
    for (int k = 0; k < K; k++) acc[k] = A(0);
    for (int r = 0; r < P && alive; r++) {
      uint32_t d[2] = {0u, 0u};
      if (r == me) {
        T* t = reinterpret_cast<T*>(d);
#pragma unroll
        for (int k = 0; k < K; k++) {
          if (u * K + k < per) t[k] = in[static_cast<size_t>(me) * per + u * K + k];
        }
      } else if (!llLoad(a, myRegion + static_cast<size_t>(r) * srcStride + u * 16, seq, d[0], d[1], r)) {
        alive = false;
        break;
      }
      const T* x = reinterpret_cast<const T*>(d);
#pragma unroll
      for (int k = 0; k < K; k++) acc[k] = r == 0 ? toAcc<T>(x[k]) : applyOp<A>(acc[k], toAcc<T>(x[k]), op);
    }
    if (!alive) break;
#pragma unroll
    for (int k = 0; k < K; k++) {
      if (u * K + k < per) {
        A v = acc[k];
        if constexpr (std::is_floating_point<A>::value) {
          if (scale != 1.0f) v = static_cast<A>(v * scale);
        }
        out[u * K + k] = fromAcc<T, A>(v);
      }
    }
  }
  retire(a, 0, 0, 1);
}

// ---- one-shot ---------------------------------------------------------------------

// Push flavour: every rank STORES its contribution into slot `rank` of every peer's pool
// (posted writes, no round trip), one barrier, then reads the P slots from its own memory.
// Saves the remote-load round trip of the pull flavour at the cost of P x the staging
// space, so it is used while P * bytes fits one half.
template <typename T>
__global__ void __launch_bounds__(kThreads)
oneShotPushAllreduceKernel(CommArgs a, const T* in, T* out, size_t count, DevOp op, float scale, PeerPtrs stage,
                           size_t halfBytes, size_t slotBytes, LocalPtrs extra) {
  using PT = PackTraits<T>;
  const uint32_t e = loadEpoch(a);
  const uint32_t parity = ld_relaxed_sys(&a.self->stageSeq) & 1u;
  const size_t tid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const size_t nthreads = static_cast<size_t>(gridDim.x) * blockDim.x;
  const size_t base = parity * halfBytes;
  const size_t ngroups = (count + PT::kElems - 1) / PT::kElems;
  const size_t mySlot = base + static_cast<size_t>(a.rank) * slotBytes;
  const bool inAligned = reinterpret_cast<uintptr_t>(in) % 16 == 0, outAligned = reinterpret_cast<uintptr_t>(out) % 16 == 0;
  bool extraAligned = true;
  for (int k = 0; k < extra.n; k++) extraAligned = extraAligned && reinterpret_cast<uintptr_t>(extra.p[k]) % 16 == 0;

  for (size_t g = tid; g < ngroups; g += nthreads) {
    const Pack16 p = loadLocalGroup(in, extra, g, count, inAligned && extraAligned, op);
#pragma unroll
    for (int r = 0; r < kMaxRanks; r++) {
      if (r < a.nranks) st128_stream(static_cast<char*>(stage.p[r]) + mySlot + g * 16, p);
    }
  }

  if (!blockBarrier(a, e + 1)) {
    retire(a, 1, 1);
    return;
  }

  const char* mine = static_cast<const char*>(stage.p[a.rank]) + base;
  for (size_t g = tid; g < ngroups; g += nthreads) {
    Pack16 p[kMaxRanks];
#pragma unroll
    for (int r = 0; r < kMaxRanks; r++) {
      if (r < a.nranks) p[r] = ld128(mine + r * slotBytes + g * 16);
    }
    typename PT::AccPack acc = PT::widen(p[0]);
#pragma unroll
    for (int r = 1; r < kMaxRanks; r++) {
      if (r < a.nranks) PT::combine(acc, p[r], op);
    }
    if (scale != 1.0f) PT::scale(acc, scale);
    storeLocalGroup(out, extra, g, count, outAligned && extraAligned, PT::narrow(acc));
  }
  retire(a, 1, 1);
}

template <typename T>
__global__ void __launch_bounds__(kThreads)
oneShotAllreduceKernel(CommArgs a, const T* in, T* out, size_t count, DevOp op, float scale, PeerPtrs stage,
                       size_t halfBytes, LocalPtrs extra) {
  using PT = PackTraits<T>;
  const uint32_t e = loadEpoch(a);
  const uint32_t parity = ld_relaxed_sys(&a.self->stageSeq) & 1u;
  const size_t tid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const size_t nthreads = static_cast<size_t>(gridDim.x) * blockDim.x;
  const size_t stageOff = parity * halfBytes;
  char* myStage = static_cast<char*>(stage.p[a.rank]) + stageOff;
  const size_t ngroups = (count + PT::kElems - 1) / PT::kElems;
  const bool inAligned = reinterpret_cast<uintptr_t>(in) % 16 == 0, outAligned = reinterpret_cast<uintptr_t>(out) % 16 == 0;
  bool extraAligned = true;
  for (int k = 0; k < extra.n; k++) extraAligned = extraAligned && reinterpret_cast<uintptr_t>(extra.p[k]) % 16 == 0;

  // Phase 0: publish my contribution in my pool.
  for (size_t g = tid; g < ngroups; g += nthreads) {
    st128(myStage + g * 16, loadLocalGroup(in, extra, g, count, inAligned && extraAligned, op));
  }

  if (!blockBarrier(a, e + 1)) {
    retire(a, 1, 1);
    return;
  }

  // Phase 1: reduce all P staged copies. Summation order is rank order on every
  // rank, so all ranks produce bit-identical results.
  for (size_t g = tid; g < ngroups; g += nthreads) {
    Pack16 p[kMaxRanks];
#pragma unroll
    for (int r = 0; r < kMaxRanks; r++) {
      if (r < a.nranks) p[r] = ld128_stream(static_cast<const char*>(stage.p[r]) + stageOff + g * 16);
    }
    typename PT::AccPack acc = PT::widen(p[0]);
#pragma unroll
    for (int r = 1; r < kMaxRanks; r++) {
      if (r < a.nranks) PT::combine(acc, p[r], op);
    }
    if (scale != 1.0f) PT::scale(acc, scale);
    storeLocalGroup(out, extra, g, count, outAligned && extraAligned, PT::narrow(acc));
  }
  retire(a, 1, 1);
}

// ---- two-shot (fused reduce-scatter + allgather, in place) --------------------------

// Multi-pointer prologue: fold the extra local pointers into `mine`, share by share, with
// the element -> (CTA, thread) mapping of the exchange phase (so the CTA that will read a
// peer's element is the one that is barrier-paired with the CTA that folded it).
template <typename T>
__device__ __forceinline__ void foldLocalShares(char* mine, const LocalPtrs& extra, size_t nvec, size_t count, int P,
                                                DevOp op, size_t tid, size_t nthreads) {
  using PT = PackTraits<T>;
  for (int r = 0; r < P; r++) {
    size_t vb, ve;
    shareOf(nvec, P, r, vb, ve);
    for (size_t v = vb + tid; v < ve; v += nthreads) {
      typename PT::AccPack acc = PT::widen(ld128_stream(mine + v * 16));
      for (int k = 0; k < extra.n; k++) PT::combine(acc, ld128_stream(static_cast<const char*>(extra.p[k]) + v * 16), op);
      st128(mine + v * 16, PT::narrow(acc));
    }
    const size_t tailStart = nvec * PT::kElems;
    size_t tb, te;
    shareOf(count - tailStart, P, r, tb, te);
    for (size_t i = tailStart + tb + tid; i < tailStart + te; i += nthreads) {
      using A = typename AccType<T>::type;
      A acc = toAcc<T>(reinterpret_cast<T*>(mine)[i]);
      for (int k = 0; k < extra.n; k++) acc = applyOp<A>(acc, toAcc<T>(static_cast<const T*>(extra.p[k])[i]), op);
      reinterpret_cast<T*>(mine)[i] = fromAcc<T, A>(acc);
    }
  }
}

// Multi-pointer epilogue: copy the result from `mine` to the extra local pointers (same mapping).
template <typename T>
__device__ __forceinline__ void fanOutLocalShares(const char* mine, const LocalPtrs& extra, size_t nvec, size_t count,
                                                  int P, size_t tid, size_t nthreads) {
  using PT = PackTraits<T>;
  for (int r = 0; r < P; r++) {
    size_t vb, ve;
    shareOf(nvec, P, r, vb, ve);
    for (size_t v = vb + tid; v < ve; v += nthreads) {
      const Pack16 p = ld128(mine + v * 16);
      for (int k = 0; k < extra.n; k++) st128_stream(static_cast<char*>(extra.p[k]) + v * 16, p);
    }
    const size_t tailStart = nvec * PT::kElems;
    size_t tb, te;
    shareOf(count - tailStart, P, r, tb, te);
    for (size_t i = tailStart + tb + tid; i < tailStart + te; i += nthreads) {
      const T x = reinterpret_cast<const T*>(mine)[i];
      for (int k = 0; k < extra.n; k++) static_cast<T*>(extra.p[k])[i] = x;
    }
  }
}

template <typename T, int NR, int UNROLL>
__global__ void __launch_bounds__(kThreads)
twoShotAllreduceKernel(CommArgs a, PeerPtrs bufs, size_t count, DevOp op, float scale, bool vectorOk, LocalPtrs extra) {
  using PT = PackTraits<T>;
  const int P = NR > 0 ? NR : a.nranks;
  const uint32_t e = loadEpoch(a);
  const size_t tid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const size_t nthreads = static_cast<size_t>(gridDim.x) * blockDim.x;
  const size_t nvec = vectorOk ? count / PT::kElems : 0;
  char* mine = static_cast<char*>(bufs.p[a.rank]);

  // Everybody's kernel has started => everybody's input is final. With several local
  // pointers the fold happens first and the barrier also publishes it.
  bool ok;
  if (extra.n > 0) {
    foldLocalShares<T>(mine, extra, nvec, count, P, op, tid, nthreads);
    ok = blockBarrier<true>(a, e + 1);
  } else {
    ok = blockBarrier<false>(a, e + 1);
  }
  if (!ok) {
    retire(a, 2, 0);
    return;
  }

  size_t vb, ve;
  shareOf(nvec, P, a.rank, vb, ve);

  // Peer order is rotated by rank so that at any instant the P readers hit P
  // different sources. Rank r alone computes chunk r, so the (rotated) summation
  // order cannot make ranks disagree.
  constexpr int kSlots = NR > 0 ? NR : kMaxRanks;
  char* peer[kSlots];
#pragma unroll
  for (int i = 0; i < kSlots; i++) peer[i] = i < P ? static_cast<char*>(bufs.p[(a.rank + i) % P]) : nullptr;

  peerAllreducePacks<T, kSlots, UNROLL>(peer, P, vb, ve, op, scale, tid, nthreads);
  // Scalar tail (count not a multiple of the pack width, or unaligned buffers): split across
  // ranks the same way.
  allreduceTailInPlace<T>(bufs, P, a.rank, nvec * PT::kElems, count, op, scale, tid, nthreads);

  // All my stores have landed everywhere and nobody still reads my buffer.
  if (blockBarrier(a, e + 2) && extra.n > 0) fanOutLocalShares<T>(mine, extra, nvec, count, P, tid, nthreads);
  retire(a, 2, 0);
}

// ---- NVLS -----------------------------------------------------------------------------

template <typename T, int UNROLL>
__global__ void __launch_bounds__(kThreads)
nvlsAllreduceKernel(CommArgs a, char* mcBase, PeerPtrs bufs, size_t count, float scale, LocalPtrs extra) {
  using PT = PackTraits<T>;
  const int P = a.nranks;
  const uint32_t e = loadEpoch(a);
  const size_t tid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const size_t nthreads = static_cast<size_t>(gridDim.x) * blockDim.x;
  const size_t nvec = count / PT::kElems;
  char* mine = static_cast<char*>(bufs.p[a.rank]);
  bool ok;
  if (extra.n > 0) {
    foldLocalShares<T>(mine, extra, nvec, count, P, DevOp::SUM, tid, nthreads);
    ok = blockBarrier<true>(a, e + 1);
  } else {
    ok = blockBarrier<false>(a, e + 1);
  }
  if (!ok) {
    retire(a, 2, 0);
    return;
  }
  size_t vb, ve;
  shareOf(nvec, P, a.rank, vb, ve);
  for (size_t v0 = vb + tid; v0 < ve; v0 += nthreads * UNROLL) {
    Pack16 r[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; u++) {
      const size_t v = v0 + static_cast<size_t>(u) * nthreads;
      if (v < ve) r[u] = Multimem<T>::ldReduceAdd(mcBase + v * 16);
    }
#pragma unroll
    for (int u = 0; u < UNROLL; u++) {
      const size_t v = v0 + static_cast<size_t>(u) * nthreads;
      if (v < ve) multimemSt128(mcBase + v * 16, scale != 1.0f ? scalePack<T>(r[u], scale) : r[u]);
    }
  }
  // Sub-pack tail through plain peer pointers, split like the two-shot tail.
  allreduceTailInPlace<T>(bufs, P, a.rank, nvec * PT::kElems, count, DevOp::SUM, scale, tid, nthreads);
  if (blockBarrier(a, e + 2) && extra.n > 0) fanOutLocalShares<T>(mine, extra, nvec, count, P, tid, nthreads);
  retire(a, 2, 0);
}

// ---- NVLS + peer-to-peer hybrid ---------------------------------------------------------------
// Measured on 8 x B200: the in-switch reduction saturates at ~0.75 of the link rate and gets
// SLOWER with more CTAs in flight (tune_P8: 32 CTAs x unroll 2 beats 296 x 8 by 9-30 %), i.e.
// the bound is the switch's reduction path, not NVLink. The links therefore have headroom that
// a plain peer-to-peer two-shot can use at the same time: the vector is cut in two, CTAs
// [0, nvlsBlocks) run the multimem path on the first part, the remaining CTAs run the two-shot
// exchange on the second part, under the same two barriers.
template <typename T, int NR>
__global__ void __launch_bounds__(kThreads)
hybridAllreduceKernel(CommArgs a, char* mcBase, PeerPtrs bufs, size_t count, float scale, int nvlsBlocks,
                      unsigned p2pPermille) {
  using PT = PackTraits<T>;
  constexpr int P = NR;
  constexpr int UP = NR == 2 ? 4 : 2;  // unroll of the peer-to-peer part
  const uint32_t e = loadEpoch(a);
  if (!blockBarrier<false>(a, e + 1)) {
    retire(a, 2, 0);
    return;
  }
  const size_t nvec = count / PT::kElems;
  // split on a multiple of P packs so that both parts share evenly
  size_t p2pVec = nvec / 1000 * p2pPermille / P * P;
  if (gridDim.x <= static_cast<unsigned>(nvlsBlocks)) p2pVec = 0;
  const size_t nvlsVec = nvec - p2pVec;
  if (static_cast<int>(blockIdx.x) < nvlsBlocks) {
    const size_t tid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    const size_t nthreads = static_cast<size_t>(nvlsBlocks) * blockDim.x;
    size_t vb, ve;
    shareOf(nvlsVec, P, a.rank, vb, ve);
    constexpr int U = 2;
    for (size_t v0 = vb + tid; v0 < ve; v0 += nthreads * U) {
      Pack16 r[U];
#pragma unroll
      for (int u = 0; u < U; u++) {
        const size_t v = v0 + static_cast<size_t>(u) * nthreads;
        if (v < ve) r[u] = Multimem<T>::ldReduceAdd(mcBase + v * 16);
      }
#pragma unroll
      for (int u = 0; u < U; u++) {
        const size_t v = v0 + static_cast<size_t>(u) * nthreads;
        if (v < ve) multimemSt128(mcBase + v * 16, scale != 1.0f ? scalePack<T>(r[u], scale) : r[u]);
      }
    }
  } else {
    const size_t tid = static_cast<size_t>(blockIdx.x - nvlsBlocks) * blockDim.x + threadIdx.x;
    const size_t nthreads = static_cast<size_t>(gridDim.x - nvlsBlocks) * blockDim.x;
    size_t vb, ve;
    shareOf(p2pVec, P, a.rank, vb, ve);
    vb += nvlsVec;
    ve += nvlsVec;
    char* peer[P];
#pragma unroll
    for (int i = 0; i < P; i++) peer[i] = static_cast<char*>(bufs.p[(a.rank + i) % P]);
    peerAllreducePacks<T, P, UP>(peer, P, vb, ve, DevOp::SUM, scale, tid, nthreads);
    // sub-pack tail: peer-to-peer group, split like the two-shot tail
    allreduceTailInPlace<T>(bufs, P, a.rank, nvec * PT::kElems, count, DevOp::SUM, scale, tid, nthreads);
  }
  blockBarrier(a, e + 2);
  retire(a, 2, 0);
}

// ---- cast epilogue: out-of-place, output dtype != input dtype --------------------------------
// Rank r reduces items [share r) of every rank's input (peer loads, or multimem.ld_reduce
// when `mcIn` is set), scales, rounds ONCE to TO and stores into every rank's output.
// An item is 8 elements: 32 B of float, 16 B of half / bf16.
template <typename TI, typename TO>
__global__ void __launch_bounds__(kThreads)
castAllreduceKernel(CommArgs a, PeerPtrs ins, char* mcIn, PeerPtrs outs, size_t count, DevOp op, float scale,
                    bool vectorOk) {
  using II = Item8<TI>;
  using OI = Item8<TO>;
  const int P = a.nranks;
  const uint32_t e = loadEpoch(a);
  const size_t tid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const size_t nthreads = static_cast<size_t>(gridDim.x) * blockDim.x;
  if (!blockBarrier<false>(a, e + 1)) {
    retire(a, 2, 0);
    return;
  }
  const size_t nitems = vectorOk ? count / 8 : 0;
  size_t ib, ie;
  shareOf(nitems, P, a.rank, ib, ie);
  for (size_t it = ib + tid; it < ie; it += nthreads) {
    float acc[8];
    if (mcIn != nullptr) {
      if constexpr (std::is_same<TI, float>::value) {
        const Pack16 x = Multimem<float>::ldReduceAdd(mcIn + it * 32), y = Multimem<float>::ldReduceAdd(mcIn + it * 32 + 16);
#pragma unroll
        for (int k = 0; k < 4; k++) {
          acc[k] = __uint_as_float(x.w[k]);
          acc[4 + k] = __uint_as_float(y.w[k]);
        }
      } else {
        const auto w = PackTraits<TI>::widen(Multimem<TI>::ldReduceAdd(mcIn + it * 16));
#pragma unroll
        for (int k = 0; k < 8; k++) acc[k] = w.v[k];
      }
    } else {
      II::load(static_cast<const char*>(ins.p[a.rank]) + it * II::kBytes, acc);
      for (int i = 1; i < P; i++) {
        float x[8];
        II::load(static_cast<const char*>(ins.p[(a.rank + i) % P]) + it * II::kBytes, x);
#pragma unroll
        for (int k = 0; k < 8; k++) acc[k] = applyOp<float>(acc[k], x[k], op);
      }
    }
    if (scale != 1.0f) {
#pragma unroll
      for (int k = 0; k < 8; k++) acc[k] *= scale;
    }
    for (int i = 0; i < P; i++) OI::store(static_cast<char*>(outs.p[(a.rank + i) % P]) + it * OI::kBytes, acc);
  }
  {
    const size_t tailStart = nitems * 8;
    size_t tb, te;
    shareOf(count - tailStart, P, a.rank, tb, te);
    for (size_t i = tailStart + tb + tid; i < tailStart + te; i += nthreads) {
      float acc = toAcc<TI>(static_cast<const TI*>(ins.p[0])[i]);
      for (int r = 1; r < P; r++) acc = applyOp<float>(acc, toAcc<TI>(static_cast<const TI*>(ins.p[r])[i]), op);
      acc *= scale;
      for (int r = 0; r < P; r++) static_cast<TO*>(outs.p[r])[i] = fromAcc<TO>(acc);
    }
  }
  blockBarrier(a, e + 2);
  retire(a, 2, 0);
}

// ---- host-side launchers ----------------------------------------------------------------

namespace {

// The instantiation of the two-shot kernel for (T, P, unroll); unroll 0 = default for P.
template <typename T>
const void* twoShotFn(int P, int unroll) {
  if constexpr (isHotType<T>()) {
    switch (P) {
      case 2:
        if (unroll == 2) return fn(twoShotAllreduceKernel<T, 2, 2>);
        if (unroll == 8) return fn(twoShotAllreduceKernel<T, 2, 8>);
        return fn(twoShotAllreduceKernel<T, 2, 4>);
      case 4:
        if (unroll == 1) return fn(twoShotAllreduceKernel<T, 4, 1>);
        if (unroll == 4) return fn(twoShotAllreduceKernel<T, 4, 4>);
        return fn(twoShotAllreduceKernel<T, 4, 2>);
      case 8:
        if (unroll == 1) return fn(twoShotAllreduceKernel<T, 8, 1>);
        return fn(twoShotAllreduceKernel<T, 8, 2>);
      default: break;
    }
  }
  return fn(twoShotAllreduceKernel<T, 0, 1>);
}

template <typename T>
const void* nvlsFn(int unroll) {
  if constexpr (isHotType<T>()) {
    if (unroll == 2) return fn(nvlsAllreduceKernel<T, 2>);
    if (unroll == 8) return fn(nvlsAllreduceKernel<T, 8>);
    return fn(nvlsAllreduceKernel<T, 4>);
  }
  return nullptr;
}

template <typename T>
const void* hybridFn(int P) {
  if constexpr (isHotType<T>()) {
    switch (P) {
      case 2: return fn(hybridAllreduceKernel<T, 2>);
      case 4: return fn(hybridAllreduceKernel<T, 4>);
      case 8: return fn(hybridAllreduceKernel<T, 8>);
      default: break;
    }
  }
  return nullptr;
}

// LL allreduce: same dtype in and out, or one of the cast epilogue's conversions.
const void* llKernelFor(DataType dt, DataType outDt) {
  if (dt != outDt) {
    return dispatchCast(dt, outDt, [](auto ti, auto to) { return fn(llAllreduceKernel<decltype(ti), decltype(to)>); });
  }
  return dispatchType(dt, [](auto t) { return fn(llAllreduceKernel<decltype(t), decltype(t)>); });
}

const void* oneShotKernelFor(DataType dt, bool push) {
  return dispatchType(dt, [&](auto t) {
    using T = decltype(t);
    return push ? fn(oneShotPushAllreduceKernel<T>) : fn(oneShotAllreduceKernel<T>);
  });
}

const void* llReduceScatterKernelFor(DataType dt) {
  return dispatchType(dt, [](auto t) { return fn(llReduceScatterKernel<decltype(t)>); });
}

}  // namespace

const void* twoShotKernelFor(DataType dt, int nranks, int unroll) {
  return dispatchType(dt, [&](auto t) { return twoShotFn<decltype(t)>(nranks, unroll); });
}

const void* nvlsKernelFor(DataType dt, int unroll) {
  return dispatchType(dt, [&](auto t) { return nvlsFn<decltype(t)>(unroll); });
}

const void* hybridKernelFor(DataType dt, int nranks) {
  return dispatchType(dt, [&](auto t) { return hybridFn<decltype(t)>(nranks); });
}

const void* castKernelFor(DataType in, DataType out) {
  return dispatchCast(in, out, [](auto ti, auto to) { return fn(castAllreduceKernel<decltype(ti), decltype(to)>); });
}

// Force-load every kernel of this file (see touch()).
void preloadAllreduceKernels() {
  touch(fn(barrierKernel));
  for (DataType dt : kAllDataTypes) {
    touch(llReduceScatterKernelFor(dt));
    for (bool push : {false, true}) touch(oneShotKernelFor(dt, push));
    for (int P : {0, 2, 4, 8}) {
      for (int u : {0, 1, 2, 4, 8}) touch(twoShotKernelFor(dt, P, u));
      touch(hybridKernelFor(dt, P));
    }
    for (int u : {2, 4, 8}) touch(nvlsKernelFor(dt, u));
    for (DataType outDt : kAllDataTypes) {
      touch(llKernelFor(dt, outDt));
      touch(castKernelFor(dt, outDt));
    }
  }
  cudaGetLastError();
}

bool& oneShotPushFlag() {
  static bool v = true;
  return v;
}
bool oneShotPushEnabled() { return oneShotPushFlag(); }
void setOneShotPush(bool on) { oneShotPushFlag() = on; }

void launchBarrier(const CommArgs& a, cudaStream_t stream) {
  barrierKernel<<<1, 32, 0, stream>>>(a);
}

bool castSupported(DataType in, DataType out) {
  if (in == out) return true;
  const bool in16 = in == DataType::FLOAT16 || in == DataType::BFLOAT16;
  const bool out16 = out == DataType::FLOAT16 || out == DataType::BFLOAT16;
  return (in == DataType::FLOAT32 && out16) || (in16 && out == DataType::FLOAT32);
}

void launchLLAllreduce(const CommArgs& a, const void* in, void* out, size_t count, DataType dt, DataType outDt,
                       ReduceOp op, float scale, const PeerPtrs& ll, size_t srcStride, size_t parityStride,
                       const LocalPtrs& extra, int blocks, int threads, cudaStream_t stream) {
  const void* k = llKernelFor(dt, outDt);
  if (k == nullptr) return;
  CommArgs ca = a;
  DevOp dop = static_cast<DevOp>(op);
  PeerPtrs pl = ll;
  char* myLL = static_cast<char*>(ll.p[a.rank]);
  LocalPtrs ex = extra;
  void* args[] = {&ca, &in, &out, &count, &dop, &scale, &pl, &myLL, &srcStride, &parityStride, &ex};
  launchKernel(k, blocks, threads, args, stream);
}

void launchLLReduceScatter(const CommArgs& a, const void* in, void* out, size_t perRank, DataType dt, ReduceOp op,
                           float scale, const PeerPtrs& ll, size_t srcStride, size_t parityStride, int blocks, int threads,
                           cudaStream_t stream) {
  CommArgs ca = a;
  DevOp dop = static_cast<DevOp>(op);
  PeerPtrs pl = ll;
  char* myLL = static_cast<char*>(ll.p[a.rank]);
  void* args[] = {&ca, &in, &out, &perRank, &dop, &scale, &pl, &myLL, &srcStride, &parityStride};
  launchKernel(llReduceScatterKernelFor(dt), blocks, threads, args, stream);
}

void launchOneShotAllreduce(const CommArgs& a, const void* in, void* out, size_t count, DataType dt, ReduceOp op,
                            float scale, const PeerPtrs& stage, size_t halfBytes, const LocalPtrs& extra, int blocks,
                            cudaStream_t stream) {
  // Push while every rank's copy fits a slot (half / P), else pull.
  size_t slotBytes = (halfBytes / static_cast<size_t>(a.nranks)) / 16 * 16;
  const size_t padded = (count * elementSize(dt) + 15) / 16 * 16;
  const bool push = padded <= slotBytes && oneShotPushEnabled();
  CommArgs ca = a;
  DevOp dop = static_cast<DevOp>(op);
  PeerPtrs ps = stage;
  LocalPtrs ex = extra;
  void* pushArgs[] = {&ca, &in, &out, &count, &dop, &scale, &ps, &halfBytes, &slotBytes, &ex};
  void* pullArgs[] = {&ca, &in, &out, &count, &dop, &scale, &ps, &halfBytes, &ex};
  launchKernel(oneShotKernelFor(dt, push), blocks, kThreads, push ? pushArgs : pullArgs, stream);
}

void launchTwoShotAllreduce(const CommArgs& a, const PeerPtrs& bufs, size_t count, DataType dt, ReduceOp op,
                            float scale, bool vectorOk, const LocalPtrs& extra, const LaunchCfg& cfg,
                            cudaStream_t stream) {
  DevOp dop = static_cast<DevOp>(op);
  CommArgs ca = a;
  PeerPtrs pb = bufs;
  LocalPtrs ex = extra;
  void* args[] = {&ca, &pb, &count, &dop, &scale, &vectorOk, &ex};
  launchKernel(twoShotKernelFor(dt, a.nranks, cfg.unroll), cfg.blocks, kThreads, args, stream);
}

bool nvlsSupports(DataType dt, ReduceOp op) {
  return op == ReduceOp::SUM && (dt == DataType::FLOAT32 || dt == DataType::FLOAT16 || dt == DataType::BFLOAT16);
}

void launchNvlsAllreduce(const CommArgs& a, void* mcPtr, const PeerPtrs& bufs, size_t count, DataType dt, float scale,
                         const LocalPtrs& extra, const LaunchCfg& cfg, cudaStream_t stream) {
  const void* k = nvlsKernelFor(dt, cfg.unroll);
  if (k == nullptr) return;
  CommArgs ca = a;
  char* mc = static_cast<char*>(mcPtr);
  PeerPtrs pb = bufs;
  LocalPtrs ex = extra;
  void* args[] = {&ca, &mc, &pb, &count, &scale, &ex};
  launchKernel(k, cfg.blocks, kThreads, args, stream);
}

void launchHybridAllreduce(const CommArgs& a, void* mcPtr, const PeerPtrs& bufs, size_t count, DataType dt, float scale,
                           int blocks, int nvlsBlocks, unsigned p2pPermille, cudaStream_t stream) {
  const void* k = hybridKernelFor(dt, a.nranks);
  if (k == nullptr) return;
  CommArgs ca = a;
  char* mc = static_cast<char*>(mcPtr);
  PeerPtrs pb = bufs;
  void* args[] = {&ca, &mc, &pb, &count, &scale, &nvlsBlocks, &p2pPermille};
  launchKernel(k, blocks, kThreads, args, stream);
}

void launchCastAllreduce(const CommArgs& a, const PeerPtrs& ins, void* mcIn, const PeerPtrs& outs, size_t count,
                         DataType dt, DataType outDt, ReduceOp op, float scale, bool vectorOk, int blocks,
                         cudaStream_t stream) {
  const void* k = castKernelFor(dt, outDt);
  if (k == nullptr) return;
  CommArgs ca = a;
  PeerPtrs pi = ins, po = outs;
  char* mc = static_cast<char*>(mcIn);
  DevOp dop = static_cast<DevOp>(op);
  void* args[] = {&ca, &pi, &mc, &po, &count, &dop, &scale, &vectorOk};
  launchKernel(k, blocks, kThreads, args, stream);
}

}  // namespace cuda
}  // namespace glb
