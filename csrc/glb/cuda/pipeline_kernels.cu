// Pipelined allreduce for ARBITRARY device pointers (sm_100a).
//
// The reference API takes plain `T*` (cuda_allreduce_ring_chunked.h:30-36); a pointer that
// is neither registered nor symmetric cannot be read by the peers (and cannot be bound to an
// NVSwitch multicast object), so the data has to pass through the symmetric pool. Instead
// of copy-in / collective / copy-out as three passes, ONE persistent kernel runs a
// three-stage software pipeline over chunks of the vector, one device barrier per step:
//
//     step i:   A(i)    copy chunk i        user input  -> pool slot i % 3      (local HBM)
//               B(i-1)  reduce chunk i-1    in the pool: multimem.ld_reduce + multimem.st
//                                           through the NVSwitch (or peer loads + stores)
//               C(i-2)  copy chunk i-2      pool slot -> user output              (local HBM)
//
// The three stages of a step touch three different slots, so they run concurrently: the
// warps of every CTA are split into an exchange group (B, NVLink-bound) and a copy group
// (A and C, HBM-bound) and the local copies hide under the NVLink time.
//
// Ownership: a chunk is P shares x G tiles x T 16-byte groups; CTA b owns tile b of every
// share in every stage, so the CTA-to-CTA flag barrier is all the synchronisation needed
// (the CTA that reads a peer's tile is barrier-paired with the CTA that wrote it).
#include "glb/cuda/device_common.cuh"
#include "glb/cuda/dispatch.cuh"
#include "glb/cuda/kernels.h"

namespace glb {
namespace cuda {

template <typename T, bool MC, int NR>
__global__ void __launch_bounds__(kThreads)
pipelinedAllreduceKernel(CommArgs a, const T* in, T* out, size_t count, DevOp op, float scale, PeerPtrs stage,
                         char* mcStage, int tileVecs, int exchangeThreads, LocalPtrs extra) {
  using PT = PackTraits<T>;
  const int P = NR > 0 ? NR : a.nranks;
  const int G = gridDim.x;
  const int b = blockIdx.x;
  const size_t T_ = static_cast<size_t>(tileVecs);  // power of two (host enforces)
  const int tileShift = 31 - __clz(tileVecs);
  const size_t chunkVecs = static_cast<size_t>(P) * G * T_;
  const size_t slotBytes = chunkVecs * 16;
  const size_t ngroups = (count + PT::kElems - 1) / PT::kElems;
  const size_t nchunks = (ngroups + chunkVecs - 1) / chunkVecs;
  const uint32_t e = loadEpoch(a);
  char* myStage = static_cast<char*>(stage.p[a.rank]);

  bool aligned = reinterpret_cast<uintptr_t>(in) % 16 == 0 && reinterpret_cast<uintptr_t>(out) % 16 == 0;
  for (int k = 0; k < extra.n; k++) aligned = aligned && reinterpret_cast<uintptr_t>(extra.p[k]) % 16 == 0;

  const bool exchanger = static_cast<int>(threadIdx.x) < exchangeThreads;
  const int xt = threadIdx.x, xn = exchangeThreads;                            // exchange group
  const int ct = threadIdx.x - exchangeThreads, cn = blockDim.x - exchangeThreads;  // copy group

  uint32_t used = 0;
  for (size_t i = 0; i < nchunks + 2; i++) {
    if (exchanger) {
      // ---- B(i-1): reduce my share's tile of chunk i-1 in the pool, deliver to everyone ----
      if (i >= 1 && i - 1 < nchunks) {
        const size_t slot = ((i - 1) % 3) * slotBytes;
        const size_t w0 = (static_cast<size_t>(a.rank) * G + b) * T_;
        if constexpr (MC) {
          char* mc = mcStage + slot + w0 * 16;
          constexpr int U = 4;
          for (size_t o0 = xt; o0 < T_; o0 += static_cast<size_t>(xn) * U) {
            Pack16 r[U];
#pragma unroll
            for (int u = 0; u < U; u++) {
              const size_t o = o0 + static_cast<size_t>(u) * xn;
              if (o < T_) r[u] = Multimem<T>::ldReduceAdd(mc + o * 16);
            }
#pragma unroll
            for (int u = 0; u < U; u++) {
              const size_t o = o0 + static_cast<size_t>(u) * xn;
              if (o < T_) {
                if (scale != 1.0f) r[u] = scalePack<T>(r[u], scale);
                multimemSt128(mc + o * 16, r[u]);
              }
            }
          }
        } else {
          // Peer exchange inside the pool, like the two-shot kernel: kSlots x U independent
          // 128-bit loads in flight per thread (an NVLink round trip is ~2 us).
          constexpr int kSlots = NR > 0 ? NR : kMaxRanks;
          constexpr int U = NR == 2 ? 8 : (NR == 4 ? 4 : (NR == 8 ? 2 : 1));
          char* peer[kSlots];
#pragma unroll
          for (int q = 0; q < kSlots; q++) {
            peer[q] = q < P ? static_cast<char*>(stage.p[(a.rank + q) % P]) + slot + w0 * 16 : nullptr;
          }
          peerAllreducePacks<T, kSlots, U>(peer, P, 0, T_, op, scale, xt, xn);
        }
      }
    } else {
      constexpr int CU = 4;  // independent 128-bit accesses in flight per copy thread
      const size_t PT_ = static_cast<size_t>(P) * T_;
      // ---- C(i-2): pool -> user output ----------------------------------------------------
      if (i >= 2) {
        const size_t c = i - 2;
        const char* slot = myStage + (c % 3) * slotBytes;
        const size_t g0 = c * chunkVecs;
        for (size_t j0 = ct; j0 < PT_; j0 += static_cast<size_t>(cn) * CU) {
          Pack16 p[CU];
          size_t g[CU];
#pragma unroll
          for (int u = 0; u < CU; u++) {
            const size_t j = j0 + static_cast<size_t>(u) * cn;
            const size_t w = (((j >> tileShift) * G + b) << tileShift) + (j & (T_ - 1));
            g[u] = j < PT_ ? g0 + w : ngroups;
            if (g[u] < ngroups) p[u] = ld128(slot + w * 16);
          }
#pragma unroll
          for (int u = 0; u < CU; u++) {
            if (g[u] < ngroups) {
              storeGroup<true>(out, g[u], count, aligned, p[u]);
              for (int k = 0; k < extra.n; k++) storeGroup<true>(static_cast<T*>(extra.p[k]), g[u], count, aligned, p[u]);
            }
          }
        }
      }
      // ---- A(i): user input -> pool -------------------------------------------------------
      if (i < nchunks) {
        char* slot = myStage + (i % 3) * slotBytes;
        const size_t g0 = i * chunkVecs;
        for (size_t j0 = ct; j0 < PT_; j0 += static_cast<size_t>(cn) * CU) {
          Pack16 p[CU];
          size_t w[CU];
#pragma unroll
          for (int u = 0; u < CU; u++) {
            const size_t j = j0 + static_cast<size_t>(u) * cn;
            w[u] = j < PT_ ? (((j >> tileShift) * G + b) << tileShift) + (j & (T_ - 1)) : chunkVecs;
            const size_t g = g0 + w[u];
            if (w[u] < chunkVecs && g < ngroups) {
              p[u] = loadGroup(in, g, count, aligned);
              if (extra.n > 0) {
                typename PT::AccPack acc = PT::widen(p[u]);
                for (int k = 0; k < extra.n; k++) {
                  PT::combine(acc, loadGroup(static_cast<const T*>(extra.p[k]), g, count, aligned), op);
                }
                p[u] = PT::narrow(acc);
              }
            } else {
              p[u].w[0] = p[u].w[1] = p[u].w[2] = p[u].w[3] = 0u;  // keep the reduction of the padding finite
            }
          }
#pragma unroll
          for (int u = 0; u < CU; u++) {
            if (w[u] < chunkVecs) st128(slot + w[u] * 16, p[u]);
          }
        }
      }
    }
    used++;
    if (!blockBarrier(a, e + used)) break;
  }
  retire(a, static_cast<uint32_t>(nchunks + 2), 0);
}

namespace {
template <typename T>
const void* pipeFn(bool mc, int nranks) {
  if constexpr (isHotType<T>()) {
    if (mc) return fn(pipelinedAllreduceKernel<T, true, 0>);
    if (nranks == 2) return fn(pipelinedAllreduceKernel<T, false, 2>);
    if (nranks == 4) return fn(pipelinedAllreduceKernel<T, false, 4>);
    if (nranks == 8) return fn(pipelinedAllreduceKernel<T, false, 8>);
  }
  return fn(pipelinedAllreduceKernel<T, false, 0>);
}
}  // namespace

const void* pipelinedKernelFor(DataType dt, bool mc, int nranks) {
  return dispatchType(dt, [&](auto t) { return pipeFn<decltype(t)>(mc, nranks); });
}

void preloadPipelineKernels() {
  for (DataType dt : kAllDataTypes) {
    for (bool mc : {false, true}) {
      for (int nr : {0, 2, 4, 8}) touch(pipelinedKernelFor(dt, mc, nr));
    }
  }
  cudaGetLastError();
}

void launchPipelinedAllreduce(const CommArgs& a, const void* in, void* out, size_t count, DataType dt, ReduceOp op,
                              float scale, const PeerPtrs& stage, void* mcStage, int tileVecs, int exchangeThreads,
                              const LocalPtrs& extra, int blocks, cudaStream_t stream) {
  const bool mc = mcStage != nullptr && nvlsSupports(dt, op);
  CommArgs ca = a;
  PeerPtrs st = stage;
  LocalPtrs ex = extra;
  char* mcp = mc ? static_cast<char*>(mcStage) : nullptr;
  DevOp dop = static_cast<DevOp>(op);
  void* args[] = {&ca, &in, &out, &count, &dop, &scale, &st, &mcp, &tileVecs, &exchangeThreads, &ex};
  launchKernel(pipelinedKernelFor(dt, mc, a.nranks), blocks, kThreads, args, stream);
}

}  // namespace cuda
}  // namespace glb
