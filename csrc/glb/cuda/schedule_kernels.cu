// Generic step-table executor for the literal allreduce schedules (see schedules.h).
#include "glb/cuda/device_common.cuh"
#include "glb/cuda/dispatch.cuh"
#include "glb/cuda/schedules.h"

namespace glb {
namespace cuda {

template <typename T>
__global__ void __launch_bounds__(kThreads)
scheduleKernel(CommArgs a, PeerPtrs bufs, PeerPtrs stage, const SchedStep* __restrict__ table, int nsteps,
               int nbarriers, DevOp op, float scale, size_t count, bool vectorOk) {
  using PT = PackTraits<T>;
  const uint32_t e = loadEpoch(a);
  const size_t tid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const size_t nthreads = static_cast<size_t>(gridDim.x) * blockDim.x;
  T* local = static_cast<T*>(bufs.p[a.rank]);
  T* myStage = static_cast<T*>(stage.p[a.rank]);

  // Ownership rule: pack (or element) index i of the buffer is always handled by global
  // thread i % nthreads — in every step and on every rank. The inter-rank barrier only
  // synchronises CTAs with the same blockIdx, so a value read in step s must have been
  // written in step s-1 by the SAME (block, thread) slot on the peer; with absolute
  // ownership that holds no matter how the ranges of consecutive steps differ.
  auto firstOwned = [&](size_t begin) { return begin + (tid + nthreads - begin % nthreads) % nthreads; };

  uint32_t used = 0;
  bool alive = true;
  for (int s = 0; s < nsteps; s++) {
    const SchedStep st = table[s];
    // A phase may read what peers produced in the previous phase (and, first, their inputs).
    if (st.sync) {
      used++;
      if (!blockBarrier(a, e + used)) {
        alive = false;
        break;
      }
    }
    const size_t off = st.off, len = st.len;
    if (len == 0) continue;
    // Vector part: whole 16-byte packs inside [off, off+len) (ranges are pack aligned
    // except possibly at their very end); the rest goes element by element.
    const bool v16 = vectorOk && (off * sizeof(T)) % 16 == 0;
    const size_t pvBegin = off * sizeof(T) / 16;
    const size_t pvEnd = v16 ? pvBegin + len / PT::kElems : pvBegin;
    const size_t tailBegin = v16 ? off + (len / PT::kElems) * PT::kElems : off;
    const size_t tailEnd = off + len;
    char* lbase = reinterpret_cast<char*>(local);
    char* sbase = reinterpret_cast<char*>(myStage);
    if (st.mode == SCHED_STAGE) {
      for (size_t pv = firstOwned(pvBegin); pv < pvEnd; pv += nthreads) st128(sbase + pv * 16, ld128_stream(lbase + pv * 16));
      for (size_t i = firstOwned(tailBegin); i < tailEnd; i += nthreads) myStage[i] = local[i];
      continue;
    }
    const PeerPtrs& srcs = st.fromStage ? stage : bufs;
    if (st.mode == SCHED_COPY) {
      const char* src = static_cast<const char*>(srcs.p[st.peers[0]]);
      constexpr int U = 4;
      for (size_t pv0 = firstOwned(pvBegin); pv0 < pvEnd; pv0 += nthreads * U) {
        Pack16 p[U];
#pragma unroll
        for (int u = 0; u < U; u++) {
          const size_t pv = pv0 + u * nthreads;
          if (pv < pvEnd) p[u] = ld128_stream(src + pv * 16);
        }
#pragma unroll
        for (int u = 0; u < U; u++) {
          const size_t pv = pv0 + u * nthreads;
          if (pv < pvEnd) st128(lbase + pv * 16, p[u]);
        }
      }
      for (size_t i = firstOwned(tailBegin); i < tailEnd; i += nthreads) {
        local[i] = static_cast<const T*>(srcs.p[st.peers[0]])[i];
      }
    } else {
      constexpr int U = 4;  // independent packs in flight per thread (each: 1 local + npeers remote loads)
      for (size_t pv0 = firstOwned(pvBegin); pv0 < pvEnd; pv0 += nthreads * U) {
        typename PT::AccPack acc[U];
#pragma unroll
        for (int u = 0; u < U; u++) {
          const size_t pv = pv0 + u * nthreads;
          if (pv < pvEnd) acc[u] = PT::widen(ld128(lbase + pv * 16));
        }
        for (int p = 0; p < st.npeers; p++) {
          const char* src = static_cast<const char*>(srcs.p[st.peers[p]]);
          Pack16 x[U];
#pragma unroll
          for (int u = 0; u < U; u++) {
            const size_t pv = pv0 + u * nthreads;
            if (pv < pvEnd) x[u] = ld128_stream(src + pv * 16);
          }
#pragma unroll
          for (int u = 0; u < U; u++) {
            const size_t pv = pv0 + u * nthreads;
            if (pv < pvEnd) PT::combine(acc[u], x[u], op);
          }
        }
#pragma unroll
        for (int u = 0; u < U; u++) {
          const size_t pv = pv0 + u * nthreads;
          if (pv < pvEnd) st128(lbase + pv * 16, PT::narrow(acc[u]));
        }
      }
      for (size_t i = firstOwned(tailBegin); i < tailEnd; i += nthreads) {
        T acc = local[i];
        for (int p = 0; p < st.npeers; p++) acc = combineOne<T>(acc, static_cast<const T*>(srcs.p[st.peers[p]])[i], op);
        local[i] = acc;
      }
    }
  }
  if (alive) {
    used++;
    if (blockBarrier(a, e + used) && scale != 1.0f) {
      // Fused epilogue: nobody reads my buffer any more; scale my copy in place.
      const size_t nvec = vectorOk ? count / PT::kElems : 0;
      char* lbase = reinterpret_cast<char*>(local);
      for (size_t v = tid; v < nvec; v += nthreads) {
        typename PT::AccPack acc = PT::widen(ld128(lbase + v * 16));
        PT::scale(acc, scale);
        st128(lbase + v * 16, PT::narrow(acc));
      }
      for (size_t i = nvec * PT::kElems + tid; i < count; i += nthreads) local[i] = scaleOne<T>(local[i], scale);
    }
  }
  retire(a, static_cast<uint32_t>(nbarriers), 0);
}

namespace {
const void* scheduleKernelFor(DataType dt) {
  return dispatchType(dt, [](auto t) { return fn(scheduleKernel<decltype(t)>); });
}
}  // namespace

void launchSchedule(const CommArgs& a, const PeerPtrs& bufs, const PeerPtrs& stage, const SchedStep* table,
                    int nsteps, int nbarriers, DataType dt, ReduceOp op, float scale, size_t count, bool vectorOk,
                    int blocks, cudaStream_t stream) {
  CommArgs ca = a;
  PeerPtrs pb = bufs, ps = stage;
  DevOp dop = static_cast<DevOp>(op);
  void* args[] = {&ca, &pb, &ps, &table, &nsteps, &nbarriers, &dop, &scale, &count, &vectorOk};
  launchKernel(scheduleKernelFor(dt), blocks, kThreads, args, stream);
}

void preloadScheduleKernels() {
  for (DataType dt : kAllDataTypes) touch(scheduleKernelFor(dt));
  cudaGetLastError();
}

}  // namespace cuda
}  // namespace glb
